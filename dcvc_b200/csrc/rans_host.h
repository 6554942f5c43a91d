// Host-side rANS entropy coder — stays on the CPU by contract (BASELINE.json north_star).
//
// Written from scratch; produces / consumes byte streams bit-identical to the reference's
// MLCodec_extensions_cpp (src/cpp/py_rans/rans.cpp:29-181 single-stream arithmetic, 32-bit state,
// 16-bit precision, byte renormalisation, 2-bit bypass escape; src/cpp/py_rans/py_rans.cpp:104-249,
// 412-492 symbol split over <= 8 parallel streams and the pair-merged container).
// Bit-exactness against the reference build is checked in tests/test_rans.py.
#pragma once
#include <stdint.h>

#include <atomic>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>

namespace dcvc {

constexpr int kMaxEcParallel = 8;  // py_rans.h:15

// Fork-join helper: run fn(0..n-1), fn(0) on the caller, the rest on persistent workers.
// The workers busy-wait for the next job for `spin_us` microseconds after finishing one before they block on a
// condition variable (DCVC_B200_RANS_SPIN_US, default 2000; 0 = always block): a picture is decoded in five short
// bursts of entropy decoding with GPU work in between, and a worker that went to sleep costs a futex wake-up per
// burst and runs the burst on a core that has dropped out of its turbo state.
class ForkJoin {
public:
    explicit ForkJoin(int workers);
    ~ForkJoin();
    void run(int n, const std::function<void(int)>& fn);

private:
    void worker_loop(int id);
    std::vector<std::thread> threads_;
    std::mutex mu_;
    std::condition_variable cv_start_, cv_done_;
    const std::function<void(int)>* fn_ = nullptr;
    std::atomic<uint64_t> epoch_{0};   // (job counter << 8) | task count, stored (under mu_) once per run()
    std::atomic<int> pending_{0};      // workers that have not finished the current job
    std::atomic<int> sleepers_{0};     // workers blocked on cv_start_ (modified under mu_)
    std::atomic<bool> stop_{false};
    int spin_us_ = 2000;
};

// One set of quantised CDF rows (index 0: factorised z model, index 1: Gaussian y model).
struct CdfSet {
    int rows = 0;
    int width = 0;                 // entries per row (max_length + 2)
    std::vector<int32_t> cdf;      // [rows][width]
    std::vector<int8_t> max_value; // cdf_length - 2: the escape symbol of each row
};

struct EncodeJob {
    enum Kind { Y, Z } kind = Y;
    const int16_t* y = nullptr;  // Y: (symbol << 8) | cdf_row   (rans.cpp:251-256)
    const int8_t* z = nullptr;   // Z: raw symbols, cdf_row = i % ch + cdf_offset (rans.cpp:289-292)
    int size = 0;
    int cdf_offset = 0;
    int ch = 1;
};

class RansCodec {
public:
    RansCodec();
    void set_cdf(const int32_t* cdf, const int32_t* cdf_sizes, int rows, int width, int index);

    // Encodes the jobs in the order given on every stream (callers pass y steps 3,2,1,0 then z,
    // dmci_proxy.cpp:839-845), flushes and merges the n_parallel streams.
    void encode(const std::vector<EncodeJob>& jobs, int n_parallel, std::vector<uint8_t>& out);

    // Decoder: set_stream once per picture, then decode_z / decode_y calls in bitstream order.
    void set_stream(const uint8_t* data, int size, int n_parallel);
    void decode_z(int8_t* out, int total, int cdf_offset, int ch);
    void decode_y(int8_t* out, const uint8_t* cdf_rows, int total);

    static int ec_parallel_for(int symbol_count);  // dmc_common.cpp:31-35

private:
    CdfSet sets_[2];
    ForkJoin pool_;
    int dec_n_ = 1;
    struct DecStream {
        std::vector<uint8_t> bytes;
        uint32_t state = 0;
        size_t pos = 0;
    };
    DecStream dec_[kMaxEcParallel];
    std::vector<uint8_t> enc_buf_[kMaxEcParallel];
};

// ryg-style pmf -> 16-bit quantised cdf (py_rans.cpp:36-94)
std::vector<uint32_t> pmf_to_quantized_cdf(const float* pmf, int n);

// Code lengths of one CDF set in Q16 bits, [rows][width] like the CDF: entry s of row r (s <= cdf_sizes[r] - 2) is
// round(65536 * (16 - log2(cdf[s + 1] - cdf[s]))), what enc_symbol spends on that symbol; the other entries are 0.
std::vector<uint32_t> rans_cost_table(const int32_t* cdf, const int32_t* cdf_sizes, int rows, int width);

}  // namespace dcvc
