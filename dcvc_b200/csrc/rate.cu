// rate.cu — rate_estimate_kernel: the size the host rANS coder would give a unit at one QP, without running it.
//
// Per symbol the kernel restates enc_symbol (rans_host.cpp): the zig-zag map of the signed value; below the row's escape
// symbol the code length of that symbol; otherwise the escape symbol's code length plus 2 bits for each bypass bin (the
// digit count in unary base 3, then one bin per 2-bit digit).  Code lengths are the Q16 table of rans_cost_table, so
// every sum is an integer: per-thread 64-bit sums, a warp reduction, one integer atomic per block.  The result does not
// depend on the launch order of the blocks, i.e. it is bitwise reproducible.
#include "rate.cuh"

namespace dcvc {

namespace {

constexpr int kThreads = 256;
constexpr int kMaxBlocks = 148 * 4;
constexpr size_t kSmemLimit = 48 * 1024;

__device__ __forceinline__ unsigned long long symbol_cost(int sym, const uint32_t* row, int maxv)
{
    const int value = (sym < 0 ? -sym : sym) * 2 - (sym > 0 ? 1 : 0);
    if (value < maxv) return row[value];
    const uint32_t raw = static_cast<uint32_t>(value - maxv);
    const int n_digits = raw ? (33 - __clz(raw)) / 2 : 0;   // ceil(bit length / 2)
    return row[maxv] + 2ull * 65536ull * static_cast<unsigned long long>(n_digits / 3 + 1 + n_digits);
}

__device__ __forceinline__ unsigned long long warp_sum(unsigned long long v)
{
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__global__ void __launch_bounds__(kThreads) rate_estimate_kernel(const RateArgs a)
{
    extern __shared__ __align__(16) uint8_t smem[];
    uint32_t* ycost = reinterpret_cast<uint32_t*>(smem);
    uint32_t* zcost = ycost + a.y_rows * a.y_width;
    int8_t* ymaxv = reinterpret_cast<int8_t*>(zcost + a.z_ch * a.z_width);
    int8_t* zmaxv = ymaxv + a.y_rows;
    for (int i = threadIdx.x; i < a.y_rows * a.y_width; i += blockDim.x) ycost[i] = a.y_cost[i];
    const uint32_t* zsrc = a.z_cost + static_cast<size_t>(a.z_row0) * a.z_width;
    for (int i = threadIdx.x; i < a.z_ch * a.z_width; i += blockDim.x) zcost[i] = zsrc[i];
    for (int i = threadIdx.x; i < a.y_rows; i += blockDim.x) ymaxv[i] = a.y_maxv[i];
    for (int i = threadIdx.x; i < a.z_ch; i += blockDim.x) zmaxv[i] = a.z_maxv[a.z_row0 + i];
    __syncthreads();

    const long long tid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    unsigned long long ysum = 0, zsum = 0;
    int n_total = 0;
    for (int k = 0; k < a.n_y; ++k) {
        const int n = *a.y_count[k];
        n_total += n;
        const int16_t* y = a.y[k];
        for (long long i = tid; i < n; i += stride) {
            const int16_t packed = y[i];
            const int row = packed & 0xff;
            ysum += symbol_cost(static_cast<int8_t>(packed >> 8), ycost + row * a.y_width, ymaxv[row]);
        }
    }
    for (long long i = tid; i < a.nz; i += stride) {
        const int r = static_cast<int>(i % a.z_ch);
        zsum += symbol_cost(a.z[i], zcost + r * a.z_width, zmaxv[r]);
    }

    __shared__ unsigned long long part[2][kThreads / 32];
    ysum = warp_sum(ysum);
    zsum = warp_sum(zsum);
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    if (lane == 0) { part[0][warp] = ysum; part[1][warp] = zsum; }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long ys = 0, zs = 0;
        for (int w = 0; w < kThreads / 32; ++w) { ys += part[0][w]; zs += part[1][w]; }
        atomicAdd(&a.out->y_q16, ys);
        atomicAdd(&a.out->z_q16, zs);
        if (blockIdx.x == 0) a.out->y_symbols = n_total;
    }
}

}  // namespace

size_t rate_smem_bytes(int y_rows, int y_width, int z_ch, int z_width)
{
    const size_t b = (static_cast<size_t>(y_rows) * y_width + static_cast<size_t>(z_ch) * z_width) * 4 + y_rows + z_ch;
    return b <= kSmemLimit ? b : 0;
}

int launch_rate_estimate(const RateArgs& a, size_t y_capacity, cudaStream_t stream)
{
    const size_t smem = rate_smem_bytes(a.y_rows, a.y_width, a.z_ch, a.z_width);
    if (!smem || a.n_y < 1 || a.n_y > 4 || a.z_ch < 1) return static_cast<int>(cudaErrorInvalidValue);
    cudaError_t e = cudaMemsetAsync(a.out, 0, sizeof(RateSlot), stream);
    if (e != cudaSuccess) return static_cast<int>(e);
    // the counts live on the device: size the grid for the largest possible unit, ~16 symbols per thread
    const size_t work = y_capacity * a.n_y + static_cast<size_t>(a.nz);
    const size_t want = (work + kThreads * 16 - 1) / (kThreads * 16);
    const int blocks = static_cast<int>(want < 1 ? 1 : (want > kMaxBlocks ? kMaxBlocks : want));
    rate_estimate_kernel<<<blocks, kThreads, smem, stream>>>(a);
    return static_cast<int>(cudaGetLastError());
}

}  // namespace dcvc
