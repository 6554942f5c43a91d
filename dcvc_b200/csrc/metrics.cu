// metrics.cu — the distortion numbers test_video.py writes into its per-job JSON, on the device.
//
// The reference measures every decoded picture on the host (get_distortion, test_video.py:32-66): the unrounded fp16
// reconstruction planes go to numpy and src/utils/metrics.py computes PSNR (calc_psnr, :10-24) and MS-SSIM
// (calc_msssim, :27-93: scipy fftconvolve in float64, about 1.9 s per 1080p 4:2:0 picture on an 8-core Xeon).
// Here the same quantities are three kernel families:
//   * metric planes  — the fp16 arrays get_distortion hands to calc_psnr / calc_msssim, bit-identical (the arithmetic
//                      of frame_to_yuv420 / frame_to_rgb without the final round / truncate);
//   * sse            — sum (src_u8 - rec_f16)^2 per plane in fp64;
//   * msssim         — per level, the mean SSIM and CS maps of an 11x11 Gaussian window (sigma 1.5, 'valid' region)
//                      with all windowed statistics in fp64 (fp32 loses ~1e-7 to the cancellation in
//                      sigma^2 = E[x^2] - mu^2 at magnitudes near 255^2), then the 2x2 reflect-mode mean that feeds
//                      the next level, kept in fp64.  The weighted product of the per-level means is left to the host.
// The planes of one picture share every launch (blockIdx.z = plane).  Every sum is a per-CTA partial followed by a
// fixed-order reduction (no floating-point atomics), so results are bitwise reproducible from run to run.
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/dcvc_b200.h"

namespace dcvc {
namespace met {

constexpr int kMaxPlanes = 3;
constexpr int kMaxLevels = 5;
constexpr int kWin = 11;                  // Gaussian window, calc_ssim: size = 11, sigma = 1.5
constexpr int TH = 16, TW = 32;           // SSIM outputs per CTA (rows x columns); both even so 2x2 downsampling tiles
constexpr int IH = TH + kWin - 1;         // input rows a tile reads
constexpr int NT = 256;
constexpr int kSseBlocks = 256;           // SSE partials per plane
constexpr double C1 = (0.01 * 255) * (0.01 * 255);
constexpr double C2 = (0.03 * 255) * (0.03 * 255);

struct Gauss { double g[kWin]; };

// separable factor of fspecial_gauss(11, 1.5) (metrics.py:27-30): the 2-D window is g (x) g exactly, both normalised
static Gauss gauss1d()
{
    Gauss w;
    double s = 0.0;
    for (int i = 0; i < kWin; ++i) {
        const double x = i - kWin / 2;
        w.g[i] = exp(-(x * x) / (2.0 * 1.5 * 1.5));
        s += w.g[i];
    }
    for (int i = 0; i < kWin; ++i) w.g[i] /= s;
    return w;
}

static inline size_t align256(size_t n) { return (n + 255) & ~static_cast<size_t>(255); }
__host__ __device__ inline int cdiv(int a, int b) { return (a + b - 1) / b; }

// where each plane's downsampled levels and per-CTA partials live inside the caller's workspace
struct Layout {
    int np = 0;
    int L[kMaxPlanes] = {};                      // MS-SSIM levels (0: the plane is too small)
    int h[kMaxPlanes][kMaxLevels] = {}, w[kMaxPlanes][kMaxLevels] = {};
    size_t sse[kMaxPlanes] = {};                 // kSseBlocks doubles
    size_t lx[kMaxPlanes][kMaxLevels] = {}, ly[kMaxPlanes][kMaxLevels] = {};   // levels >= 1, fp64 planes
    size_t part[kMaxPlanes][kMaxLevels] = {};    // 2 doubles per tile
    size_t total = 0;
};

// calc_msssim's level rule (metrics.py:31-38): 5 levels, 4 when a side is below 176, an error below 88
static inline int msssim_levels(int h, int w)
{
    if (h < 88 || w < 88) return 0;
    return (h < 176 || w < 176) ? 4 : 5;
}

static Layout make_layout(int np, const int32_t* hw)
{
    Layout s;
    s.np = np;
    size_t off = 0;
    for (int p = 0; p < np; ++p) {
        s.sse[p] = off;
        off += align256(kSseBlocks * sizeof(double));
    }
    for (int p = 0; p < np; ++p) {
        s.L[p] = msssim_levels(hw[2 * p], hw[2 * p + 1]);
        int h = hw[2 * p], w = hw[2 * p + 1];
        for (int l = 0; l < s.L[p]; ++l) {
            s.h[p][l] = h;
            s.w[p][l] = w;
            if (l > 0) {
                s.lx[p][l] = off;
                off += align256(static_cast<size_t>(h) * w * sizeof(double));
                s.ly[p][l] = off;
                off += align256(static_cast<size_t>(h) * w * sizeof(double));
            }
            s.part[p][l] = off;
            off += align256(static_cast<size_t>(cdiv(h, TH)) * cdiv(w, TW) * 2 * sizeof(double));
            h = (h + 1) / 2;
            w = (w + 1) / 2;
        }
    }
    s.total = off;
    return s;
}

// fixed-order tree sum of one value per thread (NT threads); the result is valid in thread 0
__device__ __forceinline__ void block_sum(double* red, double& a, double& b)
{
    const int t = threadIdx.x;
    red[t] = a;
    red[NT + t] = b;
    __syncthreads();
#pragma unroll
    for (int s = NT / 2; s > 0; s >>= 1) {
        if (t < s) {
            red[t] += red[t + s];
            red[NT + t] += red[NT + t + s];
        }
        __syncthreads();
    }
    a = red[0];
    b = red[NT];
}

// ---- sse: per plane sum (src_u8 - rec_f16)^2 in fp64 (calc_psnr's numerator, metrics.py:14-16) ----
struct SseArgs {
    const uint8_t* src[kMaxPlanes];
    const __half* rec[kMaxPlanes];
    long long n[kMaxPlanes];
    double* part[kMaxPlanes];
};

__global__ void __launch_bounds__(NT) sse_kernel(SseArgs a)
{
    __shared__ double red[2 * NT];
    const int p = blockIdx.z;
    const long long n = a.n[p];
    const uint8_t* s = a.src[p];
    const __half* r = a.rec[p];
    double acc = 0.0, unused = 0.0;
    const long long stride = static_cast<long long>(gridDim.x) * NT;
    for (long long i = static_cast<long long>(blockIdx.x) * NT + threadIdx.x; i < n; i += stride) {
        const double d = static_cast<double>(s[i]) - static_cast<double>(__half2float(r[i]));
        acc += d * d;
    }
    block_sum(red, acc, unused);
    if (threadIdx.x == 0) a.part[p][blockIdx.x] = acc;
}

// ---- msssim: one launch per level for every plane of the picture ----
struct LevelArgs {
    int H[kMaxPlanes], W[kMaxPlanes], active[kMaxPlanes], last[kMaxPlanes];
    const void* x[kMaxPlanes];      // level 0: uint8 source; later levels: fp64
    const void* y[kMaxPlanes];      // level 0: fp16 reconstruction; later levels: fp64
    double* nx[kMaxPlanes];         // next level (unused on a plane's last level)
    double* ny[kMaxPlanes];
    double* part[kMaxPlanes];       // (sum ssim, sum cs) per tile
    Gauss win;
};

template <bool L0>
__device__ __forceinline__ double ld_x(const void* p, long long i)
{
    if (L0) return static_cast<double>(static_cast<const uint8_t*>(p)[i]);
    return static_cast<const double*>(p)[i];
}

template <bool L0>
__device__ __forceinline__ double ld_y(const void* p, long long i)
{
    if (L0) return static_cast<double>(__half2float(static_cast<const __half*>(p)[i]));
    return static_cast<const double*>(p)[i];
}

// One CTA: the TH x TW SSIM outputs whose window starts in its tile (the 'valid' region is (H-10) x (W-10)), and the
// next level's pixels of the same tile (rows/columns 2k, 2k+1 of this level; an odd last row/column is averaged with
// itself, which is what ndimage.convolve(ones(2,2)/4, mode='reflect')[::2, ::2] computes, metrics.py:84-89).
// Horizontal 11-tap pass into shared memory for the five statistics, then the vertical pass per output pixel.
template <bool L0>
__global__ void __launch_bounds__(NT) msssim_level_kernel(LevelArgs a)
{
    __shared__ double hs[5][IH][TW];
    __shared__ double red[2 * NT];
    const int p = blockIdx.z;
    if (!a.active[p]) return;
    const int H = a.H[p], W = a.W[p];
    const int gx = cdiv(W, TW), gy = cdiv(H, TH);
    if (static_cast<int>(blockIdx.x) >= gx || static_cast<int>(blockIdx.y) >= gy) return;
    const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH;
    const int Ho = H - (kWin - 1), Wo = W - (kWin - 1);
    const void* X = a.x[p];
    const void* Y = a.y[p];

    for (int it = threadIdx.x; it < IH * TW; it += NT) {
        const int r = it / TW, c = it % TW;
        double m1 = 0.0, m2 = 0.0, e11 = 0.0, e22 = 0.0, e12 = 0.0;
        if (y0 + r < H && x0 + c < Wo) {
            const long long base = static_cast<long long>(y0 + r) * W + x0 + c;
#pragma unroll
            for (int k = 0; k < kWin; ++k) {
                const double g = a.win.g[k];
                const double u = ld_x<L0>(X, base + k), v = ld_y<L0>(Y, base + k);
                m1 += g * u;
                m2 += g * v;
                e11 += g * (u * u);
                e22 += g * (v * v);
                e12 += g * (u * v);
            }
        }
        hs[0][r][c] = m1;
        hs[1][r][c] = m2;
        hs[2][r][c] = e11;
        hs[3][r][c] = e22;
        hs[4][r][c] = e12;
    }
    __syncthreads();

    double s_ssim = 0.0, s_cs = 0.0;
    for (int it = threadIdx.x; it < TH * TW; it += NT) {
        const int i = it / TW, c = it % TW;
        if (y0 + i >= Ho || x0 + c >= Wo) continue;
        double mu1 = 0.0, mu2 = 0.0, e11 = 0.0, e22 = 0.0, e12 = 0.0;
#pragma unroll
        for (int k = 0; k < kWin; ++k) {
            const double g = a.win.g[k];
            mu1 += g * hs[0][i + k][c];
            mu2 += g * hs[1][i + k][c];
            e11 += g * hs[2][i + k][c];
            e22 += g * hs[3][i + k][c];
            e12 += g * hs[4][i + k][c];
        }
        // calc_ssim (metrics.py:33-57)
        const double mu1_sq = mu1 * mu1, mu2_sq = mu2 * mu2, mu1_mu2 = mu1 * mu2;
        const double s1 = e11 - mu1_sq, s2 = e22 - mu2_sq, s12 = e12 - mu1_mu2;
        const double cs_num = 2.0 * s12 + C2, cs_den = s1 + s2 + C2;
        s_ssim += ((2.0 * mu1_mu2 + C1) * cs_num) / ((mu1_sq + mu2_sq + C1) * cs_den);
        s_cs += cs_num / cs_den;
    }
    block_sum(red, s_ssim, s_cs);
    if (threadIdx.x == 0) {
        double* out = a.part[p] + 2 * (static_cast<long long>(blockIdx.y) * gx + blockIdx.x);
        out[0] = s_ssim;
        out[1] = s_cs;
    }

    if (a.last[p]) return;
    // 2x2 mean for the next level.  Sums of four values are exact here: level-0 inputs are uint8 / fp16 (multiples of
    // 2^-24 below 256) and each level adds two bits, so the summation order cannot matter
    const int nh = (H + 1) / 2, nw = (W + 1) / 2;
    for (int it = threadIdx.x; it < (TH / 2) * (TW / 2); it += NT) {
        const int oy = (y0 >> 1) + it / (TW / 2), ox = (x0 >> 1) + it % (TW / 2);
        if (oy >= nh || ox >= nw) continue;
        const int r0 = 2 * oy, r1 = min(2 * oy + 1, H - 1), c0 = 2 * ox, c1 = min(2 * ox + 1, W - 1);
        const long long i00 = static_cast<long long>(r0) * W + c0, i01 = static_cast<long long>(r0) * W + c1;
        const long long i10 = static_cast<long long>(r1) * W + c0, i11 = static_cast<long long>(r1) * W + c1;
        const long long o = static_cast<long long>(oy) * nw + ox;
        a.nx[p][o] = 0.25 * (ld_x<L0>(X, i00) + ld_x<L0>(X, i01) + ld_x<L0>(X, i10) + ld_x<L0>(X, i11));
        a.ny[p][o] = 0.25 * (ld_y<L0>(Y, i00) + ld_y<L0>(Y, i01) + ld_y<L0>(Y, i10) + ld_y<L0>(Y, i11));
    }
}

// ---- finish: each CTA reduces one partial array in a fixed order and scales it ----
constexpr int kMaxTasks = kMaxPlanes * (2 * kMaxLevels + 1);
struct Task {
    const double* src;
    int n, stride;
    double scale;
    double* dst;
};
struct FinishArgs { Task t[kMaxTasks]; };

__global__ void __launch_bounds__(NT) finish_kernel(FinishArgs a)
{
    __shared__ double red[2 * NT];
    const Task t = a.t[blockIdx.x];
    double s = 0.0, unused = 0.0;
    for (int i = threadIdx.x; i < t.n; i += NT) s += t.src[static_cast<long long>(i) * t.stride];
    block_sum(red, s, unused);
    if (threadIdx.x == 0) *t.dst = s * t.scale;
}

}  // namespace met
}  // namespace dcvc

extern "C" {

int64_t dcvc_metrics_workspace_bytes(int32_t nplanes, const int32_t* hw)
{
    if (nplanes < 1 || nplanes > dcvc::met::kMaxPlanes) return -1;
    return static_cast<int64_t>(dcvc::met::make_layout(nplanes, hw).total);
}

int dcvc_op_metrics_sse(int32_t nplanes, const int32_t* hw, const void* const* src, const void* const* rec,
                        void* workspace, void* out, int32_t out_stride, void* stream)
{
    using namespace dcvc::met;
    if (nplanes < 1 || nplanes > kMaxPlanes) return 3;
    const Layout s = make_layout(nplanes, hw);
    char* ws = static_cast<char*>(workspace);
    SseArgs a = {};
    FinishArgs f = {};
    for (int p = 0; p < nplanes; ++p) {
        if (hw[2 * p] <= 0 || hw[2 * p + 1] <= 0) return 3;
        a.src[p] = static_cast<const uint8_t*>(src[p]);
        a.rec[p] = static_cast<const __half*>(rec[p]);
        a.n[p] = static_cast<long long>(hw[2 * p]) * hw[2 * p + 1];
        a.part[p] = reinterpret_cast<double*>(ws + s.sse[p]);
        f.t[p] = { a.part[p], kSseBlocks, 1, 1.0, static_cast<double*>(out) + static_cast<long long>(p) * out_stride };
    }
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    sse_kernel<<<dim3(kSseBlocks, 1, nplanes), NT, 0, st>>>(a);
    finish_kernel<<<nplanes, NT, 0, st>>>(f);
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

int dcvc_op_msssim(int32_t nplanes, const int32_t* hw, const void* const* src, const void* const* rec, void* workspace,
                   void* out, int32_t out_stride, void* stream)
{
    using namespace dcvc::met;
    if (nplanes < 1 || nplanes > kMaxPlanes) return 3;
    const Layout s = make_layout(nplanes, hw);
    int Lmax = 0;
    for (int p = 0; p < nplanes; ++p) {
        if (s.L[p] == 0) return 2;          // calc_msssim asserts below 88 (metrics.py:37-38)
        Lmax = s.L[p] > Lmax ? s.L[p] : Lmax;
    }
    static const Gauss win = gauss1d();
    char* ws = static_cast<char*>(workspace);
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    FinishArgs f = {};
    int nt = 0;
    for (int l = 0; l < Lmax; ++l) {
        LevelArgs a = {};
        a.win = win;
        int gx = 0, gy = 0;
        for (int p = 0; p < nplanes; ++p) {
            if (l >= s.L[p]) continue;
            const int h = s.h[p][l], w = s.w[p][l];
            a.active[p] = 1;
            a.last[p] = l + 1 == s.L[p];
            a.H[p] = h;
            a.W[p] = w;
            a.x[p] = l == 0 ? src[p] : static_cast<const void*>(ws + s.lx[p][l]);
            a.y[p] = l == 0 ? rec[p] : static_cast<const void*>(ws + s.ly[p][l]);
            if (!a.last[p]) {
                a.nx[p] = reinterpret_cast<double*>(ws + s.lx[p][l + 1]);
                a.ny[p] = reinterpret_cast<double*>(ws + s.ly[p][l + 1]);
            }
            a.part[p] = reinterpret_cast<double*>(ws + s.part[p][l]);
            gx = cdiv(w, TW) > gx ? cdiv(w, TW) : gx;
            gy = cdiv(h, TH) > gy ? cdiv(h, TH) : gy;
            const int tiles = cdiv(w, TW) * cdiv(h, TH);
            const double inv = 1.0 / (static_cast<double>(h - (kWin - 1)) * (w - (kWin - 1)));
            double* o = static_cast<double*>(out) + static_cast<long long>(p) * out_stride + 2 * l;
            f.t[nt++] = { a.part[p], tiles, 2, inv, o };          // mean of the SSIM map
            f.t[nt++] = { a.part[p] + 1, tiles, 2, inv, o + 1 };  // mean of the CS map
        }
        if (l == 0)
            msssim_level_kernel<true><<<dim3(gx, gy, nplanes), NT, 0, st>>>(a);
        else
            msssim_level_kernel<false><<<dim3(gx, gy, nplanes), NT, 0, st>>>(a);
    }
    finish_kernel<<<nt, NT, 0, st>>>(f);
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

}  // extern "C"
