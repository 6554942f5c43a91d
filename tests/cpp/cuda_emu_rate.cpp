// cuda_emu_rate.cpp — TEST INFRASTRUCTURE ONLY (tests/test_rate_control_cpu.py).
//
// Host restatement of rate_estimate_kernel (dcvc_b200/csrc/rate.cu) for the dry-run shim.  The kernel table of
// cuda_emu_kernels.cpp is extended without editing it: the shim is linked with -Wl,--wrap=emu_lookup,... so that the
// shim's calls land here first; the rate kernel gets an index of its own (kRateIndex), every other name and index is
// passed on to the table (__real_emu_*).
#include <stdint.h>
#include <string.h>

#include "../../dcvc_b200/csrc/rate.cuh"

using namespace dcvc;

namespace {

constexpr int kRateIndex = 1 << 20;   // far beyond the table of cuda_emu_kernels.cpp

// enc_symbol's code length per symbol (rans_host.cpp) from the Q16 tables
uint64_t symbol_cost(int sym, const uint32_t* row, int maxv)
{
    const int value = (sym < 0 ? -sym : sym) * 2 - (sym > 0 ? 1 : 0);
    if (value < maxv) return row[value];
    const uint32_t raw = static_cast<uint32_t>(value - maxv);
    int n_digits = 0;
    while ((raw >> (n_digits * 2)) != 0) ++n_digits;
    return row[maxv] + 2ull * 65536ull * static_cast<uint64_t>(n_digits / 3 + 1 + n_digits);
}

// the launch zeroed `out` (cudaMemsetAsync) before the kernel, as on the device
int rate_estimate(void** g)
{
    const RateArgs& a = *static_cast<const RateArgs*>(g[0]);
    uint64_t ys = 0, zs = 0;
    int n_total = 0;
    for (int k = 0; k < a.n_y; ++k) {
        const int n = *a.y_count[k];
        n_total += n;
        for (int i = 0; i < n; ++i) {
            const int row = a.y[k][i] & 0xff;
            ys += symbol_cost(static_cast<int8_t>(a.y[k][i] >> 8), a.y_cost + static_cast<size_t>(row) * a.y_width,
                              a.y_maxv[row]);
        }
    }
    for (int i = 0; i < a.nz; ++i) {
        const int row = i % a.z_ch + a.z_row0;
        zs += symbol_cost(a.z[i], a.z_cost + static_cast<size_t>(row) * a.z_width, a.z_maxv[row]);
    }
    a.out->y_q16 += ys;
    a.out->z_q16 += zs;
    a.out->y_symbols = n_total;
    return 0;
}

}  // namespace

extern "C" {

int __real_emu_lookup(const char* name);
int __real_emu_num_args(int k);
int __real_emu_arg_size(int k, int i);
int __real_emu_run(int k, void** args);

int __wrap_emu_lookup(const char* name)
{
    return strstr(name, "rate_estimate_kernel") ? kRateIndex : __real_emu_lookup(name);
}
int __wrap_emu_num_args(int k) { return k == kRateIndex ? 1 : __real_emu_num_args(k); }
int __wrap_emu_arg_size(int k, int i)
{
    return k == kRateIndex ? static_cast<int>(sizeof(RateArgs)) : __real_emu_arg_size(k, i);
}
int __wrap_emu_run(int k, void** args) { return k == kRateIndex ? rate_estimate(args) : __real_emu_run(k, args); }

}  // extern "C"
