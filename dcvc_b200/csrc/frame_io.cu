// frame_io.cu — the callers' pre/post-processing either side of the codec, on the device (SURVEY.md §8 f2).
//
// The reference does this on the host per frame (numpy / scipy): test_video.py:74-76,115-122 upsamples 4:2:0
// chroma with scipy.ndimage.zoom(order=0), ships fp32 4:4:4 to the GPU and normalises there; test_video.py:355-361
// turns a reconstruction back into 8-bit 4:2:0 (x_hat + 0.5, 2x2 chroma average, * 255, clamp; Y rounded, UV
// truncated) before the device->host copy.  Here both directions are one HBM-bound kernel each, so a 1080p frame
// crosses PCIe as 3.1 MB of 8-bit planes instead of 12.4 MB (fp16 4:4:4) or 24.9 MB (fp32 4:4:4).
// Every fp16 step mirrors the reference's torch half arithmetic (fp32 op-math, one rounding per op), so the
// integer outputs are bit-exact against oracle/ops_ref.py.
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/dcvc_b200.h"

namespace dcvc {

static inline int fio_blocks(long long n, int t) { return static_cast<int>((n + t - 1) / t); }

// x.half() / 255.0 - 0.5 (test_video.py:118-121): fp32 division and subtraction, each rounded to half
__device__ __forceinline__ __half norm_u8(uint8_t v)
{
    const __half h = __float2half_rn(static_cast<float>(v) / 255.0f);
    return __float2half_rn(__half2float(h) - 0.5f);
}

// one thread: 2 rows x 8 columns of luma = 1 row x 4 columns of chroma.  VEC: x is channels_last [H][W][3] with
// 16-byte aligned rows and W % 8 == 0 — 8-byte plane loads and three 16-byte stores per row
template <bool VEC>
__global__ void __launch_bounds__(256)
yuv420_to_frame_kernel(const uint8_t* __restrict__ yp, const uint8_t* __restrict__ up, const uint8_t* __restrict__ vp,
                       int H, int W, __half* __restrict__ x, long long sc, long long sh, long long sw)
{
    const int bw = (W + 7) >> 3;
    const long long tid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (tid >= static_cast<long long>(bw) * (H >> 1)) return;
    const int bx = static_cast<int>(tid % bw);
    const int by = static_cast<int>(tid / bw);
    const int x0 = bx << 3;
    const int Wc = W >> 1;
    if (VEC) {
        // nearest-neighbour chroma (scipy.ndimage.zoom(uv, (1, 2, 2), order=0), transforms.py:69-80)
        const uchar4 u4 = *reinterpret_cast<const uchar4*>(up + static_cast<long long>(by) * Wc + (x0 >> 1));
        const uchar4 v4 = *reinterpret_cast<const uchar4*>(vp + static_cast<long long>(by) * Wc + (x0 >> 1));
        const uint8_t uu[4] = { u4.x, u4.y, u4.z, u4.w }, vv[4] = { v4.x, v4.y, v4.z, v4.w };
        __half hu[4], hv[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) { hu[i] = norm_u8(uu[i]); hv[i] = norm_u8(vv[i]); }
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int yy = 2 * by + r;
            const uint2 y8 = *reinterpret_cast<const uint2*>(yp + static_cast<long long>(yy) * W + x0);
            const uint8_t* yb = reinterpret_cast<const uint8_t*>(&y8);
            __align__(16) __half o[24];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                o[3 * i] = norm_u8(yb[i]);
                o[3 * i + 1] = hu[i >> 1];
                o[3 * i + 2] = hv[i >> 1];
            }
            uint4* dst = reinterpret_cast<uint4*>(x + yy * sh + static_cast<long long>(x0) * 3);
#pragma unroll
            for (int i = 0; i < 3; ++i) dst[i] = reinterpret_cast<const uint4*>(o)[i];
        }
        return;
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int yy = 2 * by + r;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int xx = x0 + i;
            if (xx >= W) break;
            __half* dst = x + yy * sh + xx * sw;
            dst[0] = norm_u8(yp[static_cast<long long>(yy) * W + xx]);
            dst[sc] = norm_u8(up[static_cast<long long>(by) * Wc + (xx >> 1)]);
            dst[2 * sc] = norm_u8(vp[static_cast<long long>(by) * Wc + (xx >> 1)]);
        }
    }
}

// (x_hat + 0.5) * 255 clamped to [0, 255], every op rounded to half (test_video.py:355-361)
__device__ __forceinline__ __half to_255(__half h)
{
    const __half a = __float2half_rn(__half2float(h) * 255.0f);
    const float f = __half2float(a);
    return __float2half_rn(fminf(fmaxf(f, 0.f), 255.f));
}

// one thread: 2 rows x 8 columns -> 2 x 8 Y bytes, 4 U, 4 V.  VEC: x is channels_last [..][Wp][3] with 16-byte
// aligned rows, W % 8 == 0 — three 16-byte loads per row, 8-byte / 4-byte plane stores
template <bool VEC>
__global__ void __launch_bounds__(256)
frame_to_yuv420_kernel(const __half* __restrict__ x, long long sc, long long sh, long long sw, int H, int W,
                       uint8_t* __restrict__ yp, uint8_t* __restrict__ up, uint8_t* __restrict__ vp)
{
    const int bw = (W + 7) >> 3;
    const int Wc = W >> 1;
    const long long tid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (tid >= static_cast<long long>(bw) * (H >> 1)) return;
    const int bx = static_cast<int>(tid % bw);
    const int by = static_cast<int>(tid / bw);
    const int x0 = bx << 3;
    float su[4] = { 0.f, 0.f, 0.f, 0.f }, sv[4] = { 0.f, 0.f, 0.f, 0.f };
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int yy = 2 * by + r;
        __align__(16) __half px[24];
        if (VEC) {
            const uint4* src = reinterpret_cast<const uint4*>(x + yy * sh + static_cast<long long>(x0) * 3);
#pragma unroll
            for (int i = 0; i < 3; ++i) reinterpret_cast<uint4*>(px)[i] = src[i];
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int xx = min(x0 + i, W - 1);
                const __half* src = x + yy * sh + xx * sw;
                px[3 * i] = src[0];
                px[3 * i + 1] = src[sc];
                px[3 * i + 2] = src[2 * sc];
            }
        }
        __align__(8) uint8_t yo[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const __half y05 = __float2half_rn(__half2float(px[3 * i]) + 0.5f);           // x_hat + 0.5
            yo[i] = static_cast<uint8_t>(rintf(__half2float(to_255(y05))));               // .round(): half to even
            su[i >> 1] += __half2float(__float2half_rn(__half2float(px[3 * i + 1]) + 0.5f));  // avg_pool2d: fp32 sum
            sv[i >> 1] += __half2float(__float2half_rn(__half2float(px[3 * i + 2]) + 0.5f));
        }
        if (VEC) {
            *reinterpret_cast<uint2*>(yp + static_cast<long long>(yy) * W + x0) = *reinterpret_cast<const uint2*>(yo);
        } else {
            for (int i = 0; i < 8 && x0 + i < W; ++i) yp[static_cast<long long>(yy) * W + x0 + i] = yo[i];
        }
    }
    __align__(4) uint8_t uo[4], vo[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        uo[i] = static_cast<uint8_t>(__half2float(to_255(__float2half_rn(su[i] / 4.f))));  // .byte(): truncation
        vo[i] = static_cast<uint8_t>(__half2float(to_255(__float2half_rn(sv[i] / 4.f))));
    }
    if (VEC) {
        *reinterpret_cast<uint32_t*>(up + static_cast<long long>(by) * Wc + (x0 >> 1)) = *reinterpret_cast<const uint32_t*>(uo);
        *reinterpret_cast<uint32_t*>(vp + static_cast<long long>(by) * Wc + (x0 >> 1)) = *reinterpret_cast<const uint32_t*>(vo);
    } else {
        for (int i = 0; i < 4 && (x0 >> 1) + i < Wc; ++i) {
            up[static_cast<long long>(by) * Wc + (x0 >> 1) + i] = uo[i];
            vp[static_cast<long long>(by) * Wc + (x0 >> 1) + i] = vo[i];
        }
    }
}

// sum of squared differences of two 8-bit planes (the integer numerator of calc_psnr, metrics.py:10-24)
__global__ void __launch_bounds__(256)
sse_u8_kernel(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b, long long n, unsigned long long* __restrict__ out)
{
    unsigned long long acc = 0;
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int d = static_cast<int>(a[i]) - static_cast<int>(b[i]);
        acc += static_cast<unsigned long long>(d * d);
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, acc);
}

// ---- RGB sources (test_cfg/all_RGB.json: src_type == 'png') ----
// BT.709 constants of src/utils/transforms.py:10-14 as torch applies them to fp32 tensors: a Python scalar becomes an
// fp32 operand, and division by a scalar is a multiplication by its fp32 reciprocal (ATen's div_true CUDA kernel).
// Every op rounds once: __fmul_rn / __fadd_rn keep nvcc from contracting them into FMAs.
struct Bt709 {
    float kr, kg, kb;
    float inv255;        // x.float() / 255.0
    float inv_1mkb;      // / (1 - Kb)
    float inv_1mkr;      // / (1 - Kr)
    float c2mkr, c2mkb;  // (2 - 2 * Kr), (2 - 2 * Kb)
    float inv_kg;        // / Kg
};

static Bt709 bt709()
{
    const double Kr = 0.2126, Kg = 0.7152, Kb = 0.0722;
    Bt709 c;
    c.kr = static_cast<float>(Kr);
    c.kg = static_cast<float>(Kg);
    c.kb = static_cast<float>(Kb);
    c.inv255 = 1.0f / static_cast<float>(255.0);
    c.inv_1mkb = 1.0f / static_cast<float>(1 - Kb);
    c.inv_1mkr = 1.0f / static_cast<float>(1 - Kr);
    c.c2mkr = static_cast<float>(2 - 2 * Kr);
    c.c2mkb = static_cast<float>(2 - 2 * Kb);
    c.inv_kg = 1.0f / static_cast<float>(Kg);
    return c;
}

__device__ __forceinline__ float clamp01(float v) { return fminf(fmaxf(v, 0.f), 1.f); }

// rgb2ycbcr(x.float() / 255.0).half() - 0.5 (test_video.py:93-95, 115-122; transforms.py:17-27), one pixel per thread
__global__ void __launch_bounds__(256)
rgb_to_frame_kernel(const uint8_t* __restrict__ rgb, int H, int W, __half* __restrict__ x, long long sc, long long sh,
                    long long sw, Bt709 k)
{
    const long long n = static_cast<long long>(H) * W;
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int yy = static_cast<int>(i / W), xx = static_cast<int>(i % W);
    const float r = __fmul_rn(static_cast<float>(rgb[i]), k.inv255);
    const float g = __fmul_rn(static_cast<float>(rgb[n + i]), k.inv255);
    const float b = __fmul_rn(static_cast<float>(rgb[2 * n + i]), k.inv255);
    const float y = __fadd_rn(__fadd_rn(__fmul_rn(k.kr, r), __fmul_rn(k.kg, g)), __fmul_rn(k.kb, b));
    const float cb = __fadd_rn(__fmul_rn(__fmul_rn(0.5f, __fsub_rn(b, y)), k.inv_1mkb), 0.5f);
    const float cr = __fadd_rn(__fmul_rn(__fmul_rn(0.5f, __fsub_rn(r, y)), k.inv_1mkr), 0.5f);
    __half* dst = x + yy * sh + xx * sw;
    dst[0] = __float2half_rn(__half2float(__float2half_rn(clamp01(y))) - 0.5f);
    dst[sc] = __float2half_rn(__half2float(__float2half_rn(clamp01(cb))) - 0.5f);
    dst[2 * sc] = __float2half_rn(__half2float(__float2half_rn(clamp01(cr))) - 0.5f);
}

// ycbcr2rgb(x_hat + 0.5) (transforms.py:53-66): half -> fp32 math -> clamp -> half, per channel
__device__ __forceinline__ void ycbcr_to_rgb_half(__half hy, __half hcb, __half hcr, const Bt709& k, __half out[3])
{
    const float y = __half2float(__float2half_rn(__half2float(hy) + 0.5f));
    const float cb = __half2float(__float2half_rn(__half2float(hcb) + 0.5f));
    const float cr = __half2float(__float2half_rn(__half2float(hcr) + 0.5f));
    const float r = __fadd_rn(y, __fmul_rn(k.c2mkr, __fsub_rn(cr, 0.5f)));
    const float b = __fadd_rn(y, __fmul_rn(k.c2mkb, __fsub_rn(cb, 0.5f)));
    const float g = __fmul_rn(__fsub_rn(__fsub_rn(y, __fmul_rn(k.kr, r)), __fmul_rn(k.kb, b)), k.inv_kg);
    out[0] = __float2half_rn(clamp01(r));
    out[1] = __float2half_rn(clamp01(g));
    out[2] = __float2half_rn(clamp01(b));
}

// x_hat[:, :, :H, :W] -> 8-bit planar RGB [3][H][W] as test_video.py:367-369 saves it:
// clamp(ycbcr2rgb(x_hat + 0.5) * 255, 0, 255).round().byte(), every op in half
__global__ void __launch_bounds__(256)
frame_to_rgb_kernel(const __half* __restrict__ x, long long sc, long long sh, long long sw, int H, int W,
                    uint8_t* __restrict__ rgb, Bt709 k)
{
    const long long n = static_cast<long long>(H) * W;
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int yy = static_cast<int>(i / W), xx = static_cast<int>(i % W);
    const __half* src = x + yy * sh + xx * sw;
    __half c[3];
    ycbcr_to_rgb_half(src[0], src[sc], src[2 * sc], k, c);
#pragma unroll
    for (int j = 0; j < 3; ++j) rgb[j * n + i] = static_cast<uint8_t>(rintf(__half2float(to_255(c[j]))));
}

// ---- metric planes: the fp16 arrays get_distortion (test_video.py:32-66) hands to calc_psnr / calc_msssim ----
// yuv420: Y [H][W] = clamp((x_hat + 0.5) * 255), then U, V [H/2][W/2] = the same after the 2x2 average;
// rgb: [3][H][W] = clamp(ycbcr2rgb(x_hat + 0.5) * 255).  No rounding: these are frame_to_yuv420 / frame_to_rgb minus
// their last step.  One thread per output pixel of Y (yuv420) or per pixel (rgb).
template <bool RGB>
__global__ void __launch_bounds__(256)
metric_planes_kernel(const __half* __restrict__ x, long long sc, long long sh, long long sw, int H, int W,
                     __half* __restrict__ rec, Bt709 k)
{
    const long long n = static_cast<long long>(H) * W;
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int yy = static_cast<int>(i / W), xx = static_cast<int>(i % W);
    const __half* src = x + yy * sh + xx * sw;
    if (RGB) {
        __half c[3];
        ycbcr_to_rgb_half(src[0], src[sc], src[2 * sc], k, c);
#pragma unroll
        for (int j = 0; j < 3; ++j) rec[j * n + i] = to_255(c[j]);
        return;
    }
    rec[i] = to_255(__float2half_rn(__half2float(src[0]) + 0.5f));
    if ((yy & 1) || (xx & 1)) return;
    const long long nc = n / 4;
    const long long ci = static_cast<long long>(yy >> 1) * (W >> 1) + (xx >> 1);
#pragma unroll
    for (int ch = 1; ch <= 2; ++ch) {
        float s = 0.f;   // avg_pool2d: fp32 sum in (0,0), (0,1), (1,0), (1,1) order, / 4, to half
#pragma unroll
        for (int r = 0; r < 2; ++r)
#pragma unroll
            for (int c = 0; c < 2; ++c)
                s += __half2float(__float2half_rn(__half2float(src[r * sh + c * sw + ch * sc]) + 0.5f));
        rec[n + (ch - 1) * nc + ci] = to_255(__float2half_rn(s / 4.f));
    }
}

}  // namespace dcvc

extern "C" {

int dcvc_op_yuv420_to_frame(const void* y, const void* u, const void* v, int32_t H, int32_t W, void* x, int64_t sc,
                            int64_t sh, int64_t sw, void* stream)
{
    if ((H & 1) || (W & 1) || H <= 0 || W <= 0) return 1;
    const long long n = static_cast<long long>((W + 7) >> 3) * (H >> 1);
    const bool vec = sc == 1 && sw == 3 && (W % 8) == 0 && (sh % 8) == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 &&
                     (reinterpret_cast<uintptr_t>(y) & 7) == 0 && (reinterpret_cast<uintptr_t>(u) & 3) == 0 &&
                     (reinterpret_cast<uintptr_t>(v) & 3) == 0;
    if (vec)
        dcvc::yuv420_to_frame_kernel<true><<<dcvc::fio_blocks(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
            static_cast<const uint8_t*>(y), static_cast<const uint8_t*>(u), static_cast<const uint8_t*>(v), H, W,
            static_cast<__half*>(x), sc, sh, sw);
    else
        dcvc::yuv420_to_frame_kernel<false><<<dcvc::fio_blocks(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
            static_cast<const uint8_t*>(y), static_cast<const uint8_t*>(u), static_cast<const uint8_t*>(v), H, W,
            static_cast<__half*>(x), sc, sh, sw);
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

int dcvc_op_frame_to_yuv420(const void* x_hat, int64_t sc, int64_t sh, int64_t sw, int32_t H, int32_t W, void* y, void* u,
                            void* v, void* stream)
{
    if ((H & 1) || (W & 1) || H <= 0 || W <= 0) return 1;
    const long long n = static_cast<long long>((W + 7) >> 3) * (H >> 1);
    const bool vec = sc == 1 && sw == 3 && (W % 8) == 0 && (sh % 8) == 0 && (reinterpret_cast<uintptr_t>(x_hat) & 15) == 0 &&
                     (reinterpret_cast<uintptr_t>(y) & 7) == 0 && (reinterpret_cast<uintptr_t>(u) & 3) == 0 &&
                     (reinterpret_cast<uintptr_t>(v) & 3) == 0;
    if (vec)
        dcvc::frame_to_yuv420_kernel<true><<<dcvc::fio_blocks(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
            static_cast<const __half*>(x_hat), sc, sh, sw, H, W, static_cast<uint8_t*>(y), static_cast<uint8_t*>(u),
            static_cast<uint8_t*>(v));
    else
        dcvc::frame_to_yuv420_kernel<false><<<dcvc::fio_blocks(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
            static_cast<const __half*>(x_hat), sc, sh, sw, H, W, static_cast<uint8_t*>(y), static_cast<uint8_t*>(u),
            static_cast<uint8_t*>(v));
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

int dcvc_op_sse_u8(const void* a, const void* b, int64_t n, void* sse_u64, void* stream)
{
    if (n <= 0) return 0;
    long long blocks = (n + 256 * 16 - 1) / (256 * 16);
    if (blocks > 148 * 8) blocks = 148 * 8;
    dcvc::sse_u8_kernel<<<static_cast<int>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const uint8_t*>(a), static_cast<const uint8_t*>(b), n, static_cast<unsigned long long*>(sse_u64));
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

int dcvc_op_rgb_to_frame(const void* rgb, int32_t H, int32_t W, void* x, int64_t sc, int64_t sh, int64_t sw, void* stream)
{
    if (H <= 0 || W <= 0) return 1;
    static const dcvc::Bt709 k = dcvc::bt709();
    const long long n = static_cast<long long>(H) * W;
    dcvc::rgb_to_frame_kernel<<<dcvc::fio_blocks(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const uint8_t*>(rgb), H, W, static_cast<__half*>(x), sc, sh, sw, k);
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

int dcvc_op_frame_to_rgb(const void* x_hat, int64_t sc, int64_t sh, int64_t sw, int32_t H, int32_t W, void* rgb,
                         void* stream)
{
    if (H <= 0 || W <= 0) return 1;
    static const dcvc::Bt709 k = dcvc::bt709();
    const long long n = static_cast<long long>(H) * W;
    dcvc::frame_to_rgb_kernel<<<dcvc::fio_blocks(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __half*>(x_hat), sc, sh, sw, H, W, static_cast<uint8_t*>(rgb), k);
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

int dcvc_op_metric_planes(const void* x_hat, int64_t sc, int64_t sh, int64_t sw, int32_t H, int32_t W, int32_t rgb,
                          void* rec, void* stream)
{
    if (H <= 0 || W <= 0 || (!rgb && ((H & 1) || (W & 1)))) return 1;
    static const dcvc::Bt709 k = dcvc::bt709();
    const long long n = static_cast<long long>(H) * W;
    if (rgb)
        dcvc::metric_planes_kernel<true><<<dcvc::fio_blocks(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
            static_cast<const __half*>(x_hat), sc, sh, sw, H, W, static_cast<__half*>(rec), k);
    else
        dcvc::metric_planes_kernel<false><<<dcvc::fio_blocks(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
            static_cast<const __half*>(x_hat), sc, sh, sw, H, W, static_cast<__half*>(rec), k);
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

}  // extern "C"
