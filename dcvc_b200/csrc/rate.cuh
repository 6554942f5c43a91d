// rate.cuh — on-device size estimate of a coded unit (rate.cu).
//
// The host rANS coder spends -log2(f / 2^16) bits per symbol plus 2 bits per bypass bin of an escape
// (rans_host.cpp: enc_symbol).  With one Q16 code-length entry per (CDF row, symbol) the size of a unit is a table
// lookup and an integer sum over the symbols the analysis graph already left on the device.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace dcvc {

// one QP trial: sums in Q16 bits (1.0 bit = 65536) and the y symbol count that fixes ec_parallel
struct RateSlot {
    unsigned long long y_q16;
    unsigned long long z_q16;
    int32_t y_symbols;
    int32_t pad;
};

struct RateArgs {
    const int16_t* y[4];          // compacted y symbols ((symbol << 8) | cdf_row) of each coded step
    const int32_t* y_count[4];    // device counters of those steps
    int n_y;                      // steps in use (4: Intra, HT-L; 1: HT-S, LD)
    const int8_t* z;              // z symbols; row of symbol k = k % z_ch + z_row0 (EncodeJob::Z)
    int nz, z_ch, z_row0;
    const uint32_t* y_cost;       // [y_rows][y_width] Q16 code lengths of the Gaussian CDF set
    const int8_t* y_maxv;         // escape symbol of each row
    int y_rows, y_width;
    const uint32_t* z_cost;       // [z_rows][z_width] of the factorised CDF set
    const int8_t* z_maxv;
    int z_width;
    RateSlot* out;
};

// Zeroes `a.out` and accumulates into it; capturable (no host sync, no allocation).  `y_capacity` bounds the
// symbols a step may hold and only sizes the grid.
int launch_rate_estimate(const RateArgs& a, size_t y_capacity, cudaStream_t stream);
// bytes of dynamic shared memory the kernel needs for these tables (0 when they do not fit)
size_t rate_smem_bytes(int y_rows, int y_width, int z_ch, int z_width);

}  // namespace dcvc
