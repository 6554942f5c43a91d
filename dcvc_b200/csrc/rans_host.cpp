// rans_host.cpp — see rans_host.h.  Own implementation of the reference bitstream format.
#include "rans_host.h"

#include <sched.h>
#include <unistd.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <numeric>
#include <stdexcept>

namespace dcvc {

namespace {

constexpr int kScaleBits = 16;                       // probability precision
constexpr int kStateShift = 23;                      // lower bound of the normalised state
constexpr uint32_t kStateLow = 1u << kStateShift;
constexpr int kEncShift = kStateShift - kScaleBits + 8;  // renorm threshold shift (=15)
constexpr uint32_t kProbMask = (1u << kScaleBits) - 1;
constexpr int kBypassBits = 2;
constexpr int kBypassMax = (1 << kBypassBits) - 1;

// Byte sink that grows towards lower addresses (rANS emits the stream back to front).
struct BackWriter {
    std::vector<uint8_t>* buf;
    size_t pos;  // first valid byte; valid bytes are [pos, buf->size())

    void reset(std::vector<uint8_t>* b, size_t capacity)
    {
        buf = b;
        if (buf->size() < capacity) buf->resize(capacity);
        pos = buf->size();
    }
    inline void reserve(size_t need)
    {
        if (pos >= need) return;
        const size_t used = buf->size() - pos;
        const size_t new_size = buf->size() * 2 + need;
        std::vector<uint8_t> nb(new_size);
        memcpy(nb.data() + new_size - used, buf->data() + pos, used);
        buf->swap(nb);
        pos = new_size - used;
    }
    inline void push(uint8_t b) { (*buf)[--pos] = b; }
};

inline void enc_put(uint32_t& x, BackWriter& w, uint32_t start, uint32_t freq)
{
    const uint32_t x_max = freq << kEncShift;
    while (x >= x_max) {
        w.push(static_cast<uint8_t>(x));
        x >>= 8;
    }
    x = ((x / freq) << kScaleBits) + (x % freq) + start;
}

inline void enc_put_bits(uint32_t& x, BackWriter& w, uint32_t val)
{
    constexpr uint32_t freq = 1u << (kScaleBits - kBypassBits);
    constexpr uint32_t x_max = freq << kEncShift;
    while (x >= x_max) {
        w.push(static_cast<uint8_t>(x));
        x >>= 8;
    }
    x = (x << kBypassBits) | val;
}

inline void enc_symbol(uint32_t& x, BackWriter& w, int32_t sym, const int32_t* cdf_row, int maxv)
{
    w.reserve(64);
    int32_t value = (sym < 0 ? -sym : sym) * 2 - (sym > 0 ? 1 : 0);
    if (value >= maxv) {
        // escape: symbol `maxv`, then the remainder in 2-bit digits (count first, unary in base 3)
        const uint32_t raw = static_cast<uint32_t>(value - maxv);
        value = maxv;
        int n_digits = 0;
        while ((raw >> (n_digits * kBypassBits)) != 0) ++n_digits;
        uint8_t bins[48];
        int nb = 0;
        int v = n_digits;
        while (v >= kBypassMax) {
            bins[nb++] = kBypassMax;
            v -= kBypassMax;
        }
        bins[nb++] = static_cast<uint8_t>(v);
        for (int j = 0; j < n_digits; ++j) {
            bins[nb++] = static_cast<uint8_t>((raw >> (j * kBypassBits)) & kBypassMax);
        }
        for (int j = nb - 1; j >= 0; --j) enc_put_bits(x, w, bins[j]);
    }
    const uint32_t start = static_cast<uint16_t>(cdf_row[value]);
    const uint32_t freq = static_cast<uint16_t>(cdf_row[value + 1] - cdf_row[value]);
    enc_put(x, w, start, freq);
}

// Bytes of zero padding behind every decoder stream, and the number of symbols the unchecked decode loop handles
// between two bounds checks: one symbol reads at most kMaxBytesPerSymbol bytes (2 renormalisation bytes + one per
// 2-bit escape digit; an escape has at most 3 * 6 + 16 digits for a 32-bit remainder).
constexpr int kMaxBytesPerSymbol = 48;
constexpr int kDecBlock = 64;
constexpr int kDecPad = kMaxBytesPerSymbol * kDecBlock + 8;

// Reader with a bounds check per byte: reads behind the stream return zero (as the reference's does).  Only used
// for the (at most kDecBlock) symbols decoded after a stream has run past its end, i.e. for corrupt streams.
struct ByteReader {
    const uint8_t* p;
    size_t pos;
    size_t size;
    inline uint8_t next() { return pos < size ? p[pos++] : (++pos, 0); }
};
// Reader without checks: the caller guarantees kMaxBytesPerSymbol readable bytes per symbol.
struct FastReader {
    const uint8_t* p;
    inline uint8_t next() { return *p++; }
};

template <class R>
inline uint32_t dec_bits(uint32_t& x, R& r)
{
    const uint32_t val = x & ((1u << kBypassBits) - 1);
    x >>= kBypassBits;
    if (x < kStateLow) x = (x << 8) | r.next();
    return val;
}

template <class R>
inline int8_t dec_symbol(uint32_t& x, R& r, const int32_t* cdf_row, int maxv)
{
    const int32_t cum = static_cast<int32_t>(x & kProbMask);
    int s = 1;
    while (cdf_row[s] <= cum) ++s;
    --s;
    const uint32_t start = static_cast<uint32_t>(cdf_row[s]);
    const uint32_t freq = static_cast<uint32_t>(cdf_row[s + 1] - cdf_row[s]);
    x = freq * (x >> kScaleBits) + (x & kProbMask) - start;
    while (x < kStateLow) x = (x << 8) | r.next();

    int32_t value = s;
    if (__builtin_expect(value == maxv, 0)) {
        int32_t v = static_cast<int32_t>(dec_bits(x, r));
        int32_t n_digits = v;
        while (v == kBypassMax && n_digits < 30) {
            v = static_cast<int32_t>(dec_bits(x, r));
            n_digits += v;
        }
        uint32_t raw = 0;
        for (int j = 0; j < n_digits; ++j) {
            v = static_cast<int32_t>(dec_bits(x, r));
            if (j < 16) raw |= static_cast<uint32_t>(v) << (j * kBypassBits);
        }
        value = static_cast<int32_t>((raw + static_cast<uint32_t>(maxv)) & 0x3fffffffu);
    }
    return static_cast<int8_t>((value & 1) ? (value + 1) / 2 : -((value + 1) / 2));
}

// Decodes symbols [off, off + len) of one stream.  row_of(k) -> CDF row of symbol k.  Blocks of kDecBlock symbols
// run without per-byte bounds checks while the read position leaves kDecPad - 8 bytes of the (zero-padded) buffer.
template <class RowOf>
inline void decode_run(int8_t* __restrict out, int off, int len, const int32_t* __restrict cdf, int width,
                       const int8_t* __restrict max_value, const uint8_t* __restrict bytes, size_t size_padded,
                       uint32_t& state, size_t& pos, RowOf row_of)
{
    uint32_t x = state;
    int k = off;
    const int end = off + len;
    while (k < end) {
        const int stop = std::min(end, k + kDecBlock);
        if (pos + static_cast<size_t>(kMaxBytesPerSymbol) * kDecBlock <= size_padded) {
            FastReader r{ bytes + pos };
            for (; k < stop; ++k) {
                const int row = row_of(k);
                out[k] = dec_symbol(x, r, cdf + static_cast<size_t>(row) * width, max_value[row]);
            }
            pos = static_cast<size_t>(r.p - bytes);
        } else {
            ByteReader r{ bytes, pos, size_padded };
            for (; k < stop; ++k) {
                const int row = row_of(k);
                out[k] = dec_symbol(x, r, cdf + static_cast<size_t>(row) * width, max_value[row]);
            }
            pos = r.pos;
        }
    }
    state = x;
}

// Trailing bytes two streams may share when the second is stored reversed behind the first
// (py_rans.cpp:14-34).
int shared_tail_bytes(const uint8_t* a, int na, const uint8_t* b, int nb)
{
    int same = 0;
    const int check = std::min({ na, nb, 8 });
    for (int i = 0; i < check; ++i) {
        if (a[na - 1 - i] != 0 || b[nb - 1 - i] != 0) break;
        ++same;
    }
    if (same == 0 && a[na - 1] == b[nb - 1]) same = 1;
    return same;
}

inline void split_range(int total, int n, int i, int& off, int& len)
{
    const int base = total / n;
    off = base * i;
    len = (i == n - 1) ? total - base * (n - 1) : base;
}

}  // namespace

// ------------------------------------------------------------------------------ ForkJoin
namespace {
inline void cpu_relax()
{
#if defined(__x86_64__) || defined(__i386__)
    __builtin_ia32_pause();
#else
    std::this_thread::yield();
#endif
}
inline int64_t now_us()
{
    return std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now().time_since_epoch()).count();
}
}  // namespace

ForkJoin::ForkJoin(int workers)
{
    // busy-waiting only pays when every worker has a hardware thread to itself — counting the sibling processes of a
    // one-process-per-GPU launch (torchrun exports LOCAL_WORLD_SIZE): round 1 measured 0.93 weak-scaling efficiency at 4 and
    // 8 GPUs with unchanged GPU time, i.e. 8 ranks x 8 spinning threads fighting for the cores of two sockets
    // ... unless this process has been given hardware threads of its own (dcvc_b200/shard.py: pin_rank deals whole cores to
    // the local ranks before the first proxy exists): then the workers spin on cores nobody else uses
    int local_world = 1;
    if (const char* e = getenv("LOCAL_WORLD_SIZE")) local_world = std::max(1, atoi(e));
    bool own_cores = false;
#if defined(__linux__)
    cpu_set_t mask;
    if (sched_getaffinity(0, sizeof(mask), &mask) == 0) {
        const int mine = CPU_COUNT(&mask);
        // (configured processors, not hardware_concurrency(): glibc derives that one from the affinity mask itself)
        own_cores = mine < static_cast<int>(sysconf(_SC_NPROCESSORS_CONF)) && mine >= workers + 1;
    }
#endif
    if (!own_cores) {
        spin_us_ /= local_world;
        if (std::thread::hardware_concurrency() < 4u * static_cast<unsigned>(workers + 1) * static_cast<unsigned>(local_world)) spin_us_ = 0;
    }
    if (const char* e = getenv("DCVC_B200_RANS_SPIN_US")) spin_us_ = std::max(0, atoi(e));
    for (int i = 0; i < workers; ++i) threads_.emplace_back(&ForkJoin::worker_loop, this, i + 1);
}

ForkJoin::~ForkJoin()
{
    {
        std::lock_guard<std::mutex> lk(mu_);
        stop_.store(true, std::memory_order_release);
    }
    cv_start_.notify_all();
    for (auto& t : threads_) t.join();
}

void ForkJoin::worker_loop(int id)
{
    uint64_t seen = 0;
    for (;;) {
        // wait for the next epoch: spin first, then block
        const int64_t deadline = now_us() + spin_us_;
        int polls = 0;
        while (epoch_.load(std::memory_order_acquire) == seen && !stop_.load(std::memory_order_acquire)) {
            if ((++polls & 63) == 0) std::this_thread::yield();  // oversubscribed host: let a working thread have the core
            if (spin_us_ == 0 || ((polls & 63) == 0 && now_us() > deadline)) {
                std::unique_lock<std::mutex> lk(mu_);
                sleepers_.fetch_add(1, std::memory_order_relaxed);
                cv_start_.wait(lk, [&] { return stop_.load(std::memory_order_acquire) || epoch_.load(std::memory_order_acquire) != seen; });
                sleepers_.fetch_sub(1, std::memory_order_relaxed);
                break;
            }
            cpu_relax();
        }
        if (stop_.load(std::memory_order_acquire)) return;
        seen = epoch_.load(std::memory_order_acquire);
        // the job's task count travels in the low byte of the epoch word: a worker that is not part of job e may get
        // here after the caller has already started preparing job e + 1
        if (id >= static_cast<int>(seen & 0xff)) continue;
        (*fn_)(id);  // published before the epoch moved; stable until every participant of this job has finished
        if (pending_.fetch_sub(1, std::memory_order_acq_rel) == 1) {
            std::lock_guard<std::mutex> lk(mu_);  // the caller may be between its predicate check and its wait
            cv_done_.notify_one();
        }
    }
}

void ForkJoin::run(int n, const std::function<void(int)>& fn)
{
    if (n <= 1) {
        fn(0);
        return;
    }
    if (n - 1 > static_cast<int>(threads_.size())) throw std::runtime_error("ForkJoin: too many tasks");
    fn_ = &fn;
    pending_.store(n - 1, std::memory_order_relaxed);
    {
        std::lock_guard<std::mutex> lk(mu_);
        const uint64_t e = epoch_.load(std::memory_order_relaxed);
        epoch_.store((((e >> 8) + 1) << 8) | static_cast<uint64_t>(n), std::memory_order_release);
    }
    if (sleepers_.load(std::memory_order_acquire) > 0) cv_start_.notify_all();
    fn(0);
    // the other streams take about as long as ours: spin briefly, then block
    const int64_t deadline = now_us() + 200;
    int polls = 0;
    while (pending_.load(std::memory_order_acquire) != 0) {
        if ((++polls & 63) == 0) std::this_thread::yield();
        if ((polls & 63) == 0 && now_us() > deadline) {
            std::unique_lock<std::mutex> lk(mu_);
            cv_done_.wait(lk, [&] { return pending_.load(std::memory_order_acquire) == 0; });
            break;
        }
        cpu_relax();
    }
}

// ------------------------------------------------------------------------------ RansCodec
RansCodec::RansCodec() : pool_(kMaxEcParallel - 1) {}

int RansCodec::ec_parallel_for(int symbol_count)
{
    const int n = symbol_count / 32768;  // MIN_SYMBOLS_PER_STREAM, def_const.h:18
    return std::max(1, std::min(kMaxEcParallel, n));
}

void RansCodec::set_cdf(const int32_t* cdf, const int32_t* cdf_sizes, int rows, int width, int index)
{
    CdfSet& s = sets_[index];
    s.rows = rows;
    s.width = width;
    s.cdf.assign(cdf, cdf + static_cast<size_t>(rows) * width);
    s.max_value.resize(rows);
    for (int i = 0; i < rows; ++i) s.max_value[i] = static_cast<int8_t>(cdf_sizes[i] - 2);
}

void RansCodec::encode(const std::vector<EncodeJob>& jobs, int n_parallel, std::vector<uint8_t>& out)
{
    const int n = std::max(1, std::min(kMaxEcParallel, n_parallel));
    size_t start_pos[kMaxEcParallel];
    auto body = [&](int i) {
        size_t nsym = 0;
        for (const auto& j : jobs) {
            int off, len;
            split_range(j.size, n, i, off, len);
            nsym += len;
        }
        BackWriter w;
        w.reset(&enc_buf_[i], nsym * 3 + 1024);
        uint32_t x = kStateLow;
        for (const auto& j : jobs) {
            int off, len;
            split_range(j.size, n, i, off, len);
            if (j.kind == EncodeJob::Y) {
                const CdfSet& cs = sets_[1];
                for (int k = off + len - 1; k >= off; --k) {
                    const int16_t packed = j.y[k];
                    const int row = packed & 0xff;
                    const int32_t sym = static_cast<int8_t>(packed >> 8);
                    enc_symbol(x, w, sym, cs.cdf.data() + static_cast<size_t>(row) * cs.width,
                               cs.max_value[row]);
                }
            } else {
                const CdfSet& cs = sets_[0];
                for (int k = off + len - 1; k >= off; --k) {
                    const int row = (k % j.ch) + j.cdf_offset;
                    enc_symbol(x, w, j.z[k], cs.cdf.data() + static_cast<size_t>(row) * cs.width,
                               cs.max_value[row]);
                }
            }
        }
        w.reserve(8);
        w.push(static_cast<uint8_t>(x >> 24));
        w.push(static_cast<uint8_t>(x >> 16));
        w.push(static_cast<uint8_t>(x >> 8));
        w.push(static_cast<uint8_t>(x >> 0));
        start_pos[i] = w.pos;
    };
    pool_.run(n, body);

    const uint8_t* sp[kMaxEcParallel];
    int nb[kMaxEcParallel];
    for (int i = 0; i < n; ++i) {
        sp[i] = enc_buf_[i].data() + start_pos[i];
        nb[i] = static_cast<int>(enc_buf_[i].size() - start_pos[i]);
    }
    if (n == 1) {
        out.assign(sp[0], sp[0] + nb[0]);
        return;
    }
    // streams are stored in pairs: even stream forward, odd stream reversed behind it, sharing
    // trailing zero bytes; a header of int32 cumulative group ends precedes >= 3 streams.
    const int pairs = n / 2;
    const bool tail = (n % 2) != 0;
    int gsize[kMaxEcParallel / 2];
    int share[kMaxEcParallel / 2];
    for (int p = 0; p < pairs; ++p) {
        share[p] = shared_tail_bytes(sp[2 * p], nb[2 * p], sp[2 * p + 1], nb[2 * p + 1]);
        gsize[p] = nb[2 * p] + nb[2 * p + 1] - share[p];
    }
    const int n_off = pairs - 1 + (tail ? 1 : 0);
    size_t total = static_cast<size_t>(n_off) * 4;
    for (int p = 0; p < pairs; ++p) total += gsize[p];
    if (tail) total += nb[n - 1];
    out.resize(total);
    int cumulative = gsize[0];
    for (int k = 0; k < n_off; ++k) {
        const int32_t v = cumulative;
        memcpy(out.data() + k * 4, &v, 4);
        if (k + 1 < pairs) cumulative += gsize[k + 1];
    }
    size_t pos = static_cast<size_t>(n_off) * 4;
    for (int p = 0; p < pairs; ++p) {
        const int i0 = 2 * p, i1 = 2 * p + 1;
        memcpy(out.data() + pos, sp[i0], nb[i0]);
        std::reverse_copy(sp[i1], sp[i1] + nb[i1] - share[p], out.data() + pos + nb[i0]);
        pos += gsize[p];
    }
    if (tail) memcpy(out.data() + pos, sp[n - 1], nb[n - 1]);
}

void RansCodec::set_stream(const uint8_t* data, int size, int n_parallel)
{
    const int n = std::max(1, std::min(kMaxEcParallel, n_parallel));
    dec_n_ = n;
    auto load = [&](int i, const uint8_t* p, int len, bool reversed) {
        DecStream& d = dec_[i];
        d.bytes.resize(static_cast<size_t>(std::max(len, 0)) + kDecPad);
        if (reversed) std::reverse_copy(p, p + len, d.bytes.begin());
        else std::copy(p, p + len, d.bytes.begin());
        std::fill(d.bytes.begin() + len, d.bytes.end(), 0);
        d.state = static_cast<uint32_t>(d.bytes[0]) | (static_cast<uint32_t>(d.bytes[1]) << 8) |
                  (static_cast<uint32_t>(d.bytes[2]) << 16) | (static_cast<uint32_t>(d.bytes[3]) << 24);
        d.pos = 4;
    };
    if (n == 1) {
        load(0, data, size, false);
        return;
    }
    if (n == 2) {
        load(0, data, size, false);
        load(1, data, size, true);
        return;
    }
    const int pairs = n / 2;
    const bool tail = (n % 2) != 0;
    const int n_off = pairs - 1 + (tail ? 1 : 0);
    const int header = n_off * 4;
    if (size < header) throw std::runtime_error("rANS stream shorter than its header");
    std::vector<int> offs(n_off);
    for (int k = 0; k < n_off; ++k) {
        int32_t v;
        memcpy(&v, data + k * 4, 4);
        offs[k] = v;
    }
    const uint8_t* payload = data + header;
    const int payload_size = size - header;
    for (int p = 0; p < pairs; ++p) {
        const int begin = (p == 0) ? 0 : offs[p - 1];
        int end;
        if (p < n_off) end = offs[p];
        else end = tail ? offs[n_off - 1] : payload_size;
        if (begin < 0 || end < begin || end > payload_size) throw std::runtime_error("bad rANS group offsets");
        load(2 * p, payload + begin, end - begin, false);
        load(2 * p + 1, payload + begin, end - begin, true);
    }
    if (tail) {
        const int begin = offs[n_off - 1];
        if (begin < 0 || begin > payload_size) throw std::runtime_error("bad rANS tail offset");
        load(n - 1, payload + begin, payload_size - begin, false);
    }
}

void RansCodec::decode_z(int8_t* out, int total, int cdf_offset, int ch)
{
    const int n = dec_n_;
    const CdfSet& cs = sets_[0];
    auto body = [&](int i) {
        int off, len;
        split_range(total, n, i, off, len);
        DecStream& d = dec_[i];
        decode_run(out, off, len, cs.cdf.data(), cs.width, cs.max_value.data(), d.bytes.data(), d.bytes.size(), d.state,
                   d.pos, [=](int k) { return (k % ch) + cdf_offset; });
    };
    pool_.run(n, body);
}

void RansCodec::decode_y(int8_t* out, const uint8_t* cdf_rows, int total)
{
    const int n = dec_n_;
    const CdfSet& cs = sets_[1];
    auto body = [&](int i) {
        int off, len;
        split_range(total, n, i, off, len);
        DecStream& d = dec_[i];
        decode_run(out, off, len, cs.cdf.data(), cs.width, cs.max_value.data(), d.bytes.data(), d.bytes.size(), d.state,
                   d.pos, [=](int k) { return static_cast<int>(cdf_rows[k]); });
    };
    pool_.run(n, body);
}

// ------------------------------------------------------------------------------ cdf builder
std::vector<uint32_t> pmf_to_quantized_cdf(const float* pmf, int n)
{
    constexpr uint32_t prob_max = 1u << 16;
    std::vector<uint32_t> cdf(static_cast<size_t>(n) + 1);
    cdf[0] = 0;
    for (int i = 0; i < n; ++i) {
        // float * 65536 in float, +0.5 in double, truncate (py_rans.cpp:49-50)
        const float scaled = pmf[i] * static_cast<float>(prob_max);
        cdf[i + 1] = static_cast<uint32_t>(static_cast<double>(scaled) + 0.5);
    }
    int total_i = 0;
    for (uint32_t v : cdf) total_i += static_cast<int>(v);
    const uint32_t total = static_cast<uint32_t>(total_i);
    for (auto& v : cdf) v = static_cast<uint32_t>((static_cast<uint64_t>(prob_max) * v) / total);
    std::partial_sum(cdf.begin(), cdf.end(), cdf.begin());
    cdf.back() = prob_max;
    const int m = static_cast<int>(cdf.size());
    for (int i = 0; i < m - 1; ++i) {
        if (cdf[i] + 1 > cdf[i + 1]) {
            // zero-width symbol: steal one count from the narrowest symbol that can spare it
            uint32_t best_freq = ~0u;
            int best = -1;
            for (int j = 0; j < m - 1; ++j) {
                const uint32_t f = cdf[j + 1] - cdf[j];
                if (f >= 2 && f < best_freq) {
                    best_freq = f;
                    best = j;
                }
            }
            if (best < 0) throw std::runtime_error("pmf_to_quantized_cdf: cannot fix zero frequency");
            if (best < i) {
                for (int j = best + 1; j <= i; ++j) cdf[j] -= 1;
            } else {
                for (int j = i + 1; j <= best; ++j) cdf[j] += 1;
            }
        }
    }
    return cdf;
}

std::vector<uint32_t> rans_cost_table(const int32_t* cdf, const int32_t* cdf_sizes, int rows, int width)
{
    std::vector<uint32_t> out(static_cast<size_t>(rows) * width, 0u);
    for (int r = 0; r < rows; ++r) {
        const int32_t* c = cdf + static_cast<size_t>(r) * width;
        const int maxv = std::min(cdf_sizes[r] - 2, width - 2);
        for (int s = 0; s <= maxv; ++s) {
            const int32_t freq = std::max(c[s + 1] - c[s], 1);   // a valid table has no zero-width symbol
            out[static_cast<size_t>(r) * width + s] =
                static_cast<uint32_t>(std::llround(65536.0 * (kScaleBits - std::log2(static_cast<double>(freq)))));
        }
    }
    return out;
}

}  // namespace dcvc
