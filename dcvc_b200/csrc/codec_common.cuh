// codec_common.cuh — shared runtime of the codec-level C ABI (Intra + HT-S): parameter store, weight
// re-layout, device arenas, the DepthConvBlock op builder, CUDA-graph segments, GPU-only timing and
// per-kernel-family profiling.  See codec.cu (DCVC-UF-Intra) and codec_hts.cu (DCVC-UF HT-S).
//
// Reference counterparts: src/layers/extensions/inference/layers_proxy.{h,cpp} (block proxies, weight
// folding), dmc_common.{h,cpp} (graph capture / run), memory_pool.h (buffer pool).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <functional>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/dcvc_b200.h"
#include "dcb_tail.cuh"
#include "elementwise.cuh"
#include "pw_gemm.cuh"
#include "rans_host.h"
#include "rate.cuh"

namespace dcvc {

constexpr int kQpNum = 64;
constexpr int kMaxRateTrials = 64;   // QPs per dcvc_estimate_bits call
constexpr int kRateZCh = 128;        // z channels of every codec kind: CDF row = k % 128 + qp * 128

#define CK(expr)                                                                           \
    do {                                                                                   \
        cudaError_t e__ = (expr);                                                          \
        if (e__ != cudaSuccess) {                                                          \
            throw std::runtime_error(std::string(#expr) + ": " + cudaGetErrorString(e__)); \
        }                                                                                  \
    } while (0)

inline int round_up(int v, int m) { return (v + m - 1) / m * m; }

struct HostTensor {
    int dtype = DCVC_DTYPE_F16;
    std::vector<int64_t> shape;
    std::vector<uint8_t> bytes;
    int64_t numel() const
    {
        int64_t n = 1;
        for (auto s : shape) n *= s;
        return n;
    }
};

// debugging aid (DCVC_B200_OPSUM): order-sensitive checksum of a device range
static __global__ void view_checksum_kernel(const uint16_t* __restrict__ p, int Cc, int pitch, size_t n_elems,
                                            unsigned long long* out)
{
    unsigned long long acc = 0;
    for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n_elems;
         i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const size_t px = i / Cc;
        acc += static_cast<unsigned long long>(p[px * pitch + (i - px * Cc)]) * (2 * i + 1);
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(out, acc);
}

// bump allocator over one cudaMalloc block
// Device arena of one plan: one cudaMalloc sized from the plan's estimate, carved with 1 KB alignment.  If the estimate
// turns out short (a size / padding combination the formula missed), further blocks are added instead of failing:
// pointers already handed out stay valid, and `overflow_blocks()` tells the tests that the estimate needs fixing.
class Arena {
public:
    ~Arena() { release(); }
    void release()
    {
        if (base_) cudaFree(base_);
        for (void* p : extra_) cudaFree(p);
        extra_.clear();
        base_ = cur_ = nullptr;
        cap_ = used_ = 0;
    }
    void reserve(size_t bytes)
    {
        release();
        CK(cudaMalloc(&base_, bytes));
        cur_ = base_;
        cap_ = bytes;
        used_ = 0;
    }
    void* alloc(size_t bytes)
    {
        size_t off = (used_ + 1023) & ~static_cast<size_t>(1023);
        if (off + bytes > cap_) {
            const size_t block = std::max(bytes + 1024, static_cast<size_t>(32) << 20);
            void* p = nullptr;
            CK(cudaMalloc(&p, block));
            extra_.push_back(p);
            cur_ = p;
            cap_ = block;
            off = 0;
        }
        used_ = off + bytes;
        return static_cast<uint8_t*>(cur_) + off;
    }
    __half* halves(size_t n) { return static_cast<__half*>(alloc(n * 2)); }
    void* base() const { return base_; }
    int overflow_blocks() const { return static_cast<int>(extra_.size()); }

private:
    void* base_ = nullptr;   // first block (the estimate)
    void* cur_ = nullptr;    // block being carved
    std::vector<void*> extra_;
    size_t cap_ = 0, used_ = 0;
};

struct DcbW {
    bool adaptor = false;
    int cin = 0, c = 0, inner = 0;
    const __half *wa = nullptr, *ba = nullptr;
    const __half *w0 = nullptr, *b0 = nullptr;
    const __half* wdw = nullptr;                // [9][inner]
    const __half *w3 = nullptr, *b3 = nullptr;  // b3: dc.3 bias + W3 . dw-bias
    const __half *wf0 = nullptr, *bf0 = nullptr;
    const __half *wf2 = nullptr, *bf2 = nullptr;
};

struct ConvW {
    const __half* w = nullptr;
    const __half* b = nullptr;
    int cout = 0, cin = 0;
};

struct Level {  // one pyramid level: two ping-pong buffers + two scratch buffers
    int H = 0, W = 0;
    __half *A = nullptr, *B = nullptr, *T1 = nullptr, *T2 = nullptr;
};

using OpFn = std::function<int(cudaStream_t)>;

// OP_TAIL: the fused dcb_tail kernel.  OP_GEMM_*: the five instantiations of pw_gemm_kernel as kernels of their own (ncu
// lists them separately too); OP_GEMM stays the family total
enum OpKind { OP_GEMM = 0, OP_DW = 1, OP_ELEM = 2, OP_TAIL = 3, OP_GEMM_64 = 4, OP_GEMM_128 = 5, OP_GEMM_192 = 6, OP_GEMM_256 = 7,
              OP_GEMM_256_FOLD = 8, OP_KINDS = 9 };

struct Segment {
    std::vector<OpFn> ops;
    std::vector<int> kinds;         // OpKind per op (kept in step with `ops`)
    std::vector<double> alg_bytes;  // algorithmic bytes per op (activations in + residuals in + out)
    std::vector<double> flops;
    std::vector<ActView> out_views; // output view per op where known (DCVC_B200_OPSUM debugging)
    std::vector<std::string> notes;
    // capture lane per op.  Lane 0 is the caller's stream; ops of other lanes are captured on side streams that fork
    // from the segment's start and join at its end, i.e. the lanes become parallel branches of the graph (only for
    // op groups that share no buffers: the 8 recon heads of the chunk codecs).  Outside graphs everything runs in list
    // order on one stream.
    std::vector<int> lanes;
    int cur_lane = 0, n_lanes = 1;
    // cross-lane edges: before op `at` is captured, lane `to` waits for everything captured on lane `from` so far
    // (an event record / wait pair inside the capture).  The list order of the ops is always a valid serial order.
    struct LaneSync { size_t at; int from, to; };
    std::vector<LaneSync> syncs;
    cudaGraphExec_t exec = nullptr;
    int launches = 0;
    // the most recent fused DepthConvBlock tail (dcb_tail.cuh), kept so that the NEXT block can hang its dc.0 onto it as
    // phase 4 — valid only while it is still the last op of the segment
    std::shared_ptr<DcbTailOp> tail;
    size_t tail_idx = 0;
    void annotate(int kind, double bytes, double fl)
    {
        while (kinds.size() < ops.size()) {
            kinds.push_back(kind);
            alg_bytes.push_back(bytes);
            flops.push_back(fl);
            lanes.push_back(cur_lane);
        }
    }
    void lane_sync(int from, int to)
    {
        annotate(OP_ELEM, 0, 0);
        syncs.push_back(LaneSync{ ops.size(), from, to });
        const int hi = (from > to ? from : to) + 1;
        if (hi > n_lanes) n_lanes = hi;
    }
    void set_lane(int l)
    {
        annotate(OP_ELEM, 0, 0);  // ops pushed so far keep the lane they were pushed under
        cur_lane = l;
        if (l + 1 > n_lanes) n_lanes = l + 1;
    }
    void elem(OpFn f)
    {
        annotate(OP_ELEM, 0, 0);
        ops.push_back(std::move(f));
        annotate(OP_ELEM, 0, 0);
    }
    void seal()
    {
        annotate(OP_ELEM, 0, 0);
        launches = static_cast<int>(ops.size());
    }
    void reset()
    {
        if (exec) cudaGraphExecDestroy(exec);
        exec = nullptr;
        ops.clear(); kinds.clear(); alg_bytes.clear(); flops.clear(); lanes.clear(); syncs.clear();
        cur_lane = 0; n_lanes = 1;
        launches = 0;
        tail.reset();
    }
};

struct ProfileAcc {
    double ms = 0, bytes = 0, flops = 0;
    long long launches = 0;
};

inline ActView make_view(const void* p, int C, int pitch, int W, int H)
{
    ActView v;
    v.ptr = p; v.C = C; v.pitch = pitch; v.W = W; v.H = H;
    return v;
}

class CodecBase {
public:
    explicit CodecBase(int device) : device_(device) {}
    virtual ~CodecBase()
    {
        if (copy_stream_) cudaStreamDestroy(copy_stream_);
        if (own_stream_) cudaStreamDestroy(own_stream_);
        if (h_rate_slots_) cudaFreeHost(h_rate_slots_);
        if (ev_hop_) cudaEventDestroy(ev_hop_);
        if (ev_y_) cudaEventDestroy(ev_y_);
        if (ev_fork_) cudaEventDestroy(ev_fork_);
        for (auto& st : lane_streams_) cudaStreamDestroy(st);
        for (auto& e : lane_events_) cudaEventDestroy(e);
        for (auto& e : sync_events_) cudaEventDestroy(e);
        for (auto& e : tev_) cudaEventDestroy(e);
        for (auto& e : prof_events_) cudaEventDestroy(e);
    }

    virtual void finalize(float skip_thres) = 0;
    virtual int debug_fetch(const char* name, void* dst, int64_t max_bytes, int64_t* written) = 0;
    // dcvc_estimate_bits: the unit's size at each QP from the analysis graph and the rate kernel alone (no synthesis,
    // no feature-memory update, no rANS).  Leaves every buffer a later compress() reads as it found it.
    virtual void estimate(const void* x, int H, int W, int64_t sc, int64_t sh, int64_t sw, const int32_t* qps, int n_qps,
                          int pad_b, int pad_r, cudaStream_t stream, dcvc_rate_estimate* out) = 0;
    virtual int arena_overflow_blocks() const { return 0; }   // > 0: the plan's arena estimate was short (tests)

    void set_param(const char* name, const void* data, int dtype, int ndim, const int64_t* shape, int on_device)
    {
        HostTensor t;
        t.dtype = dtype;
        t.shape.assign(shape, shape + ndim);
        const size_t esz = (dtype == DCVC_DTYPE_F16) ? 2 : 4;
        t.bytes.resize(static_cast<size_t>(t.numel()) * esz);
        if (on_device) {
            CK(cudaMemcpy(t.bytes.data(), data, t.bytes.size(), cudaMemcpyDeviceToHost));
        } else {
            memcpy(t.bytes.data(), data, t.bytes.size());
        }
        params_[name] = std::move(t);
        finalized_ = false;
    }

    float gpu_ms()
    {
        float total = 0.f;
        for (int i = 0; i + 1 < tev_n_; i += 2) {
            CK(cudaEventSynchronize(tev_[i + 1]));
            float ms = 0.f;
            CK(cudaEventElapsedTime(&ms, tev_[i], tev_[i + 1]));
            total += ms;
        }
        return total;
    }

    bool profile_ = false;
    ProfileAcc prof_[OP_KINDS];
    std::string err;
    int64_t launches = 0;

protected:
    // ------------------------------------------------------------------ parameters
    bool has_param(const std::string& k) const { return params_.count(k) != 0; }
    const HostTensor& param(const std::string& k) const
    {
        auto it = params_.find(k);
        if (it == params_.end()) throw std::runtime_error("missing parameter '" + k + "'");
        return it->second;
    }
    std::vector<__half> param_f16(const std::string& k) const
    {
        const HostTensor& t = param(k);
        std::vector<__half> v(static_cast<size_t>(t.numel()));
        if (t.dtype == DCVC_DTYPE_F16) {
            memcpy(v.data(), t.bytes.data(), t.bytes.size());
        } else if (t.dtype == DCVC_DTYPE_F32) {
            const float* f = reinterpret_cast<const float*>(t.bytes.data());
            for (size_t i = 0; i < v.size(); ++i) v[i] = __float2half_rn(f[i]);
        } else {
            throw std::runtime_error("parameter '" + k + "' is not floating point");
        }
        return v;
    }
    const __half* upload(const std::vector<__half>& v)
    {
        void* d = warena_.alloc(v.size() * sizeof(__half));
        CK(cudaMemcpy(d, v.data(), v.size() * sizeof(__half), cudaMemcpyHostToDevice));
        return static_cast<const __half*>(d);
    }
    const __half* upload_param(const std::string& k) { return upload(param_f16(k)); }

    // DepthConvBlock weights (layers_proxy.cpp:160-206): dw weight -> [9][C'], dw bias folded into dc.3
    DcbW load_dcb(const std::string& p)
    {
        DcbW w;
        if (has_param(p + "adaptor.weight")) {
            w.adaptor = true;
            w.cin = static_cast<int>(param(p + "adaptor.weight").shape[1]);
            w.wa = upload_param(p + "adaptor.weight");
            w.ba = upload_param(p + "adaptor.bias");
        }
        const HostTensor& w0 = param(p + "dc.0.weight");
        w.inner = static_cast<int>(w0.shape[0]);
        w.c = static_cast<int>(w0.shape[1]);
        if (!w.adaptor) w.cin = w.c;
        w.w0 = upload_param(p + "dc.0.weight");
        w.b0 = upload_param(p + "dc.0.bias");
        {
            std::vector<__half> dw = param_f16(p + "dc.2.weight");
            std::vector<__half> t(dw.size());
            for (int c = 0; c < w.inner; ++c)
                for (int k = 0; k < 9; ++k) t[static_cast<size_t>(k) * w.inner + c] = dw[static_cast<size_t>(c) * 9 + k];
            w.wdw = upload(t);
        }
        {
            // fold the depthwise bias into the bias of dc.3 (layers_proxy.cpp:175-178), fp32 then one rounding
            std::vector<__half> w3 = param_f16(p + "dc.3.weight");
            std::vector<__half> bdw = param_f16(p + "dc.2.bias");
            std::vector<__half> b3 = param_f16(p + "dc.3.bias");
            std::vector<__half> folded(b3.size());
            for (int n = 0; n < w.c; ++n) {
                float acc = 0.f;
                for (int c = 0; c < w.inner; ++c)
                    acc += __half2float(w3[static_cast<size_t>(n) * w.inner + c]) * __half2float(bdw[c]);
                folded[n] = __float2half_rn(acc + __half2float(b3[n]));
            }
            w.w3 = upload(w3);
            w.b3 = upload(folded);
        }
        w.wf0 = upload_param(p + "ffn.0.weight");
        w.bf0 = upload_param(p + "ffn.0.bias");
        w.wf2 = upload_param(p + "ffn.2.weight");
        w.bf2 = upload_param(p + "ffn.2.bias");
        return w;
    }

    ConvW load_conv(const std::string& p, int kind)
    {
        ConvW c;
        const HostTensor& wt = param(p + "weight");
        const int cout = static_cast<int>(wt.shape[0]), cin = static_cast<int>(wt.shape[1]);
        const int kh = static_cast<int>(wt.shape[2]), kw = static_cast<int>(wt.shape[3]);
        std::vector<__half> src = param_f16(p + "weight");
        std::vector<__half> dst(src.size());
        if (dcvc_pack_weight(kind, src.data(), cout, cin, kh, kw, dst.data()))
            throw std::runtime_error("pack_weight failed for " + p);
        c.w = upload(dst);
        if (has_param(p + "bias")) {
            std::vector<__half> b = param_f16(p + "bias");
            if (kind == DCVC_GEMM_TCONV2X2 || kind == DCVC_GEMM_CONV3X3_PS2) {
                // GEMM columns of the pixel-shuffle kinds are phase-major: column ph * Cout + co <- channel co * 4 + ph
                std::vector<__half> r(b.size());
                const int co_n = cout / 4;
                for (int co = 0; co < co_n; ++co)
                    for (int ph = 0; ph < 4; ++ph) r[static_cast<size_t>(ph) * co_n + co] = b[static_cast<size_t>(co) * 4 + ph];
                b.swap(r);
            }
            c.b = upload(b);
        }
        c.cout = cout;
        c.cin = cin;
        return c;
    }

    // reserve the weight arena, then (after the model-specific loads) finish with LUT/CDF/streams
    void finalize_begin(float skip_thres)
    {
        CK(cudaSetDevice(device_));
        skip_thres_ = skip_thres;
        size_t total = 0;
        for (auto& kv : params_) total += static_cast<size_t>(kv.second.numel()) * 2 + 2048;
        warena_.reserve(total * 2 + (8u << 20));
    }
    void finalize_end()
    {
        std::vector<uint8_t> h(65536);
        build_scale_lut(h.data());
        lut_ = static_cast<uint8_t*>(warena_.alloc(65536));
        CK(cudaMemcpy(lut_, h.data(), 65536, cudaMemcpyHostToDevice));
        // CDF tables (common_model.py:64-70; dmci_proxy.cpp:639-651)
        const char* names[2] = { "bit_estimator_z.", "gaussian_encoder." };
        for (int i = 0; i < 2; ++i) {
            const HostTensor& c = param(std::string(names[i]) + "quantized_cdf");
            const HostTensor& l = param(std::string(names[i]) + "cdf_length");
            if (c.dtype != DCVC_DTYPE_I32 || l.dtype != DCVC_DTYPE_I32 || c.shape.size() != 2)
                throw std::runtime_error("CDF tables must be int32 [rows][width]");
            const int32_t* cdf = reinterpret_cast<const int32_t*>(c.bytes.data());
            const int32_t* len = reinterpret_cast<const int32_t*>(l.bytes.data());
            const int rows = static_cast<int>(c.shape[0]), width = static_cast<int>(c.shape[1]);
            rans_.set_cdf(cdf, len, rows, width, i);
            // the rate estimate's code-length table and escape symbols of this set (rate.cu)
            const std::vector<uint32_t> cost = rans_cost_table(cdf, len, rows, width);
            std::vector<int8_t> maxv(rows);
            for (int r = 0; r < rows; ++r) maxv[r] = static_cast<int8_t>(len[r] - 2);
            cost_[i] = static_cast<uint32_t*>(warena_.alloc(cost.size() * 4));
            maxv_[i] = static_cast<int8_t*>(warena_.alloc(rows));
            CK(cudaMemcpy(cost_[i], cost.data(), cost.size() * 4, cudaMemcpyHostToDevice));
            CK(cudaMemcpy(maxv_[i], maxv.data(), rows, cudaMemcpyHostToDevice));
            cost_rows_[i] = rows;
            cost_width_[i] = width;
        }
        rate_slots_ = static_cast<RateSlot*>(warena_.alloc(sizeof(RateSlot) * kMaxRateTrials));
        if (!h_rate_slots_) CK(cudaMallocHost(&h_rate_slots_, sizeof(RateSlot) * kMaxRateTrials));
        if (!copy_stream_) {
            int lo, hi;
            CK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
            CK(cudaStreamCreateWithPriority(&copy_stream_, cudaStreamNonBlocking, hi));
            CK(cudaStreamCreateWithFlags(&own_stream_, cudaStreamNonBlocking));
            CK(cudaEventCreateWithFlags(&ev_hop_, cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&ev_y_, cudaEventDisableTiming));
            tev_.resize(48);
            for (auto& e : tev_) CK(cudaEventCreate(&e));
        }
        if (gemm_init() || dcb_tail_init()) throw std::runtime_error(gemm_last_error());
        const char* g = getenv("DCVC_B200_GRAPHS");
        use_graphs_ = !(g && g[0] == '0');
        const char* ft = getenv("DCVC_B200_FUSE_TAIL");
        fuse_tail_ = !(ft && ft[0] == '0');
        if (ft && atoi(ft) > 1) { fuse_min_px_ = atoi(ft); fuse_any_c_ = true; }   // DCVC_B200_FUSE_TAIL=<pixels>: another threshold, any width (measurements, tests)
        finalized_ = true;
    }

    // ------------------------------------------------------------------ op builders
    void add_gemm(Segment& s, int kind, const ActView& in, const ActView& out, const __half* w, const __half* bias,
                  int N, int act, int chunk, const ActView* r1, const ActView* r2, const __half* q)
    {
        auto op = std::make_shared<GemmOp>();
        op->kind = kind;
        op->in = in;
        op->out = out;
        if (r1) op->res1 = *r1;
        if (r2) op->res2 = *r2;
        op->weight = w;
        op->bias = bias;
        op->qscale = q;
        op->N = N;
        op->act = act;
        op->chunk_add = chunk;
        if (gemm_plan(*op)) throw std::runtime_error(std::string("gemm_plan: ") + gemm_last_error());
        s.annotate(OP_ELEM, 0, 0);
        s.ops.push_back([op](cudaStream_t st) { return gemm_launch(*op, st); });
        s.out_views.resize(s.ops.size());
        s.out_views.back() = out;
        {
            char buf[256];
            snprintf(buf, sizeof(buf), "gemm kind=%d in=%dx%dx%d/%d@%p out=%d/%d@%p N=%d act=%d chunk=%d res=%p,%p bn=%d st=%d sb=%d grid=%u",
                     kind, in.H, in.W, in.C, in.pitch, in.ptr, out.C, out.pitch, out.ptr, N, act, chunk,
                     r1 ? r1->ptr : nullptr, r2 ? r2->ptr : nullptr, op->block_n, op->stages, op->p.staging_bufs, op->grid.x);
            s.notes.resize(s.ops.size());
            s.notes.back() = buf;
        }
        const double px_in = static_cast<double>(in.W) * in.H, px_out = static_cast<double>(out.W) * out.H;
        const int taps = (kind == GEMM_CONV3X3_S2 || kind == GEMM_CONV3X3_PS2) ? 9 : (kind == GEMM_CONV2X2_S2 ? 4 : 1);
        double bytes = px_in * in.C * 2 + px_out * out.C * 2;
        if (r1) bytes += px_out * out.C * 2;
        if (r2) bytes += px_out * out.C * 2;
        const double m_px = (kind == GEMM_TCONV2X2 || kind == GEMM_CONV3X3_PS2) ? px_in : px_out;
        const int inst = chunk ? OP_GEMM_256_FOLD : (op->block_n == 64 ? OP_GEMM_64 : op->block_n == 128 ? OP_GEMM_128 : op->block_n == 192 ? OP_GEMM_192 : OP_GEMM_256);
        s.annotate(inst, bytes, 2.0 * m_px * N * taps * in.C);
    }
    void conv1x1(Segment& s, const ActView& in, const ActView& out, const ConvW& c)
    {
        add_gemm(s, GEMM_PW, in, out, c.w, c.b, c.cout, ACT_NONE, 0, nullptr, nullptr, nullptr);
    }

    void gemm_1x1(Segment& s, const ActView& in, const ActView& out, const __half* w, const __half* bias, int N, int act,
                  int chunk, const ActView* r1, const ActView* r2, const __half* q)
    {
        add_gemm(s, GEMM_PW, in, out, w, bias, N, act, chunk, r1, r2, q);
    }

    // DepthConvBlock (layers.py:152-159 == layers_proxy.cpp:71-101): returns the view holding the output.
    // The block input is overwritten in place unless `out` redirects the last GEMM.  `in` may live in one
    // of the level's ping-pong buffers or outside of it (then, without an adaptor, `out` is mandatory
    // and must not be L.A, which holds the dc.3 output).
    ActView dcb(Segment& s, Level& L, const ActView& in, const DcbW& w, bool shortcut, const __half* qscale,
                const ActView* out)
    {
        const int H = in.H, W = in.W;
        __half* bufX;
        ActView x;
        if (w.adaptor) {
            bufX = (in.ptr == L.A) ? L.B : L.A;
            x = make_view(bufX, w.c, w.c, W, H);
            gemm_1x1(s, in, x, w.wa, w.ba, w.c, ACT_NONE, 0, nullptr, nullptr, nullptr);
        } else {
            x = in;
            bufX = static_cast<__half*>(const_cast<void*>(in.ptr));
            const bool internal = (bufX == L.A || bufX == L.B);
            if (!internal && (!out || out->ptr == L.A))
                throw std::runtime_error("dcb: external input without adaptor needs an output outside L.A");
        }
        __half* bufO = (bufX == L.A) ? L.B : L.A;
        const ActView t1 = make_view(L.T1, w.inner, w.inner, W, H);
        const ActView t2 = make_view(L.T2, w.inner, w.inner, W, H);
        const ActView o = make_view(bufO, w.c, w.c, W, H);
        // dc.0: when the previous op of the segment is the fused tail of the block that produced x, this GEMM rides along
        // as that kernel's fourth phase (y is still in its tensor memory); otherwise it is a launch of its own
        bool dc0_fused = false;
        if (!w.adaptor && s.tail && s.tail_idx + 1 == s.ops.size() && !s.tail->t1n.ptr &&
            s.tail->y.ptr == x.ptr && s.tail->y.C == x.C && s.tail->y.pitch == x.pitch && s.tail->y.W == x.W && s.tail->y.H == x.H) {
            DcbTailOp trial = *s.tail;
            trial.t1n = t1;
            trial.w0n = w.w0;
            trial.b0n = w.b0;
            if (dcb_tail_plan(trial) == 0) {
                *s.tail = trial;
                const double px = static_cast<double>(W) * H;
                s.alg_bytes[s.tail_idx] += px * (x.C + w.inner) * 2;
                s.flops[s.tail_idx] += 2.0 * px * w.inner * x.C;
                s.notes[s.tail_idx] += " +dc0";
                dc0_fused = true;
            }
        }
        s.tail.reset();
        if (!dc0_fused) gemm_1x1(s, x, t1, w.w0, w.b0, w.inner, ACT_WSILU, 0, nullptr, nullptr, nullptr);
        {
            const __half* wdw = w.wdw;
            s.annotate(OP_ELEM, 0, 0);
            s.ops.push_back([t1, t2, wdw](cudaStream_t st) { return launch_dw3x3(t1, t2, wdw, st, true); });
            s.out_views.resize(s.ops.size());
            s.out_views.back() = t2;
            s.annotate(OP_DW, 2.0 * 2 * W * H * w.inner, 2.0 * 9 * W * H * w.inner);
        }
        const ActView dst = out ? *out : x;
        // Where the fused kernel is used: measured on B200 (profiles/r2_dcb_tail_timeline.md).  It needs >= 64 pair tiles to fill
        // the chip (fuse_min_px_), and with C = 512 the resident activation tile (128 KB) leaves each issuer's weight ring half
        // a chunk: L2-latency-bound, 153-164 us against 131 us per-op at 135x240 — those blocks keep the per-op kernels.
        if (fuse_tail_ && static_cast<long long>(W) * H >= fuse_min_px_ && (w.c <= 384 || fuse_any_c_)) {
            // dc.3 -> ffn.0 -> ffn.2 as one CTA-pair kernel: o and t1' stay on the SM (dcb_tail.cuh)
            auto op = std::make_shared<DcbTailOp>();
            op->t2 = t2; op->x = x; op->y = dst;
            op->w3 = w.w3; op->b3 = w.b3; op->wf0 = w.wf0; op->bf0 = w.bf0; op->wf2 = w.wf2; op->bf2 = w.bf2;
            op->qscale = qscale;
            op->shortcut = shortcut;
            const int r = dcb_tail_plan(*op);
            if (r == 2) throw std::runtime_error(std::string("dcb_tail_plan: ") + gemm_last_error());
            if (r == 0) {
                s.annotate(OP_ELEM, 0, 0);
                s.ops.push_back([op](cudaStream_t st) { return dcb_tail_launch(*op, st); });
                s.out_views.resize(s.ops.size());
                s.out_views.back() = dst;
                char buf[200];
                snprintf(buf, sizeof(buf), "dcb_tail %dx%d C=%d inner=%d shortcut=%d q=%d tiles=%d pairs=%d stages=%d", H, W, w.c, w.inner,
                         shortcut ? 1 : 0, qscale ? 1 : 0, op->p.tiles, op->p.num_pairs, op->p.stages);
                s.notes.resize(s.ops.size());
                s.notes.back() = buf;
                // algorithmic bytes / flops: the sum over the three ops it replaces (SURVEY.md 8d counts per op)
                const double px = static_cast<double>(W) * H;
                const double bytes = px * 2 * ((w.inner + w.c + w.c) + (w.c + w.inner) + (w.inner + w.c + w.c + (shortcut ? w.c : 0)));
                const double fl = 2.0 * px * (static_cast<double>(w.c) * w.inner + 4.0 * w.inner * w.c + static_cast<double>(w.c) * w.inner);
                s.annotate(OP_TAIL, bytes, fl);
                s.tail = op;
                s.tail_idx = s.ops.size() - 1;
                return dst;
            }
        }
        gemm_1x1(s, t2, o, w.w3, w.b3, w.c, ACT_NONE, 0, &x, nullptr, nullptr);
        gemm_1x1(s, o, t1, w.wf0, w.bf0, 4 * w.inner, ACT_WSILU, 1, nullptr, nullptr, nullptr);
        gemm_1x1(s, t1, dst, w.wf2, w.bf2, w.c, ACT_NONE, 0, &o, shortcut ? &x : nullptr, qscale);
        return dst;
    }

    // ------------------------------------------------------------------ execution
    void run(Segment& s, cudaStream_t stream)
    {
        if (s.ops.empty()) return;
        if (profile_) {
            // per-op CUDA-event timing (graphs off).  All ops of the segment are enqueued back to back with an
            // event before and after each, and read only after the last one: the CPU runs ahead of the GPU, so an
            // interval is the kernel's own duration (plus the inter-kernel gap), not the CPU launch latency.
            const size_t n = s.ops.size();
            while (prof_events_.size() < 2 * n) {
                cudaEvent_t e;
                CK(cudaEventCreate(&e));
                prof_events_.push_back(e);
            }
            for (size_t i = 0; i < n; ++i) {
                CK(cudaEventRecord(prof_events_[2 * i], stream));
                if (s.ops[i](stream)) throw std::runtime_error(std::string("kernel launch failed: ") + gemm_last_error());
                CK(cudaEventRecord(prof_events_[2 * i + 1], stream));
            }
            CK(cudaEventSynchronize(prof_events_[2 * n - 1]));
            const char* path = getenv("DCVC_B200_PROFILE_CSV");
            FILE* f = path ? fopen(path, "a") : nullptr;
            for (size_t i = 0; i < n; ++i) {
                float ms = 0.f;
                CK(cudaEventElapsedTime(&ms, prof_events_[2 * i], prof_events_[2 * i + 1]));
                for (int pass = 0; pass < 2; ++pass) {   // a pw_gemm instantiation also counts towards the family total
                    if (pass == 1 && s.kinds[i] < OP_GEMM_64) break;
                    ProfileAcc& a = prof_[pass == 0 ? s.kinds[i] : OP_GEMM];
                    a.ms += ms; a.bytes += s.alg_bytes[i]; a.flops += s.flops[i]; a.launches += 1;
                }
                if (f) fprintf(f, "%d,%zu,%.3f,%.0f,%.0f\n", s.kinds[i], i, ms * 1e3, s.alg_bytes[i], s.flops[i]);
            }
            if (f) fclose(f);
            launches += s.launches;
            return;
        }
        if (const char* path = getenv("DCVC_B200_OPSUM")) {
            // debugging aid: run op by op and log a checksum of each op's output view (GEMMs, dw3x3), so two
            // runs of the same input can be diffed down to the first op that disagrees
            if (!opsum_dev_) CK(cudaMalloc(&opsum_dev_, 8));
            FILE* f = fopen(path, "a");
            for (size_t i = 0; i < s.ops.size(); ++i) {
                if (s.ops[i](stream)) throw std::runtime_error(std::string("kernel launch failed: ") + gemm_last_error());
                CK(cudaMemsetAsync(opsum_dev_, 0, 8, stream));
                const ActView ov = i < s.out_views.size() ? s.out_views[i] : ActView();
                if (ov.ptr)
                    view_checksum_kernel<<<1184, 256, 0, stream>>>(static_cast<const uint16_t*>(ov.ptr), ov.C, ov.pitch,
                                                                   static_cast<size_t>(ov.W) * ov.H * ov.C, opsum_dev_);
                unsigned long long h = 0;
                CK(cudaMemcpyAsync(&h, opsum_dev_, 8, cudaMemcpyDeviceToHost, stream));
                CK(cudaStreamSynchronize(stream));
                if (f) fprintf(f, "%p %zu kind=%d %s %016llx\n", static_cast<void*>(&s), i, s.kinds[i],
                               i < s.notes.size() ? s.notes[i].c_str() : "-", h);
            }
            if (f) fclose(f);
            launches += s.launches;
            return;
        }
        if (use_graphs_) {
            if (!s.exec) {
                cudaGraph_t graph = nullptr;
                const int n_lanes = s.n_lanes;
                if (n_lanes > 1) {  // side streams / events exist before the capture starts
                    if (!ev_fork_) CK(cudaEventCreateWithFlags(&ev_fork_, cudaEventDisableTiming));
                    while (static_cast<int>(lane_streams_.size()) < n_lanes - 1) {
                        cudaStream_t st = nullptr;
                        cudaEvent_t ev = nullptr;
                        CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
                        lane_streams_.push_back(st);
                        CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
                        lane_events_.push_back(ev);
                    }
                    while (sync_events_.size() < s.syncs.size()) {
                        cudaEvent_t ev = nullptr;
                        CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
                        sync_events_.push_back(ev);
                    }
                }
                CK(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
                int rc = 0;
                std::string lane_err;
                if (n_lanes > 1) {  // fork: every lane starts where the segment starts
                    if (cudaEventRecord(ev_fork_, stream) != cudaSuccess) rc = 1;
                    for (int l = 1; l < n_lanes && !rc; ++l)
                        if (cudaStreamWaitEvent(lane_streams_[l - 1], ev_fork_, 0) != cudaSuccess) rc = 1;
                    if (rc) lane_err = "fork of the capture lanes failed";
                }
                auto lane_stream = [&](int l) { return l == 0 ? stream : lane_streams_[l - 1]; };
                size_t next_sync = 0;
                auto do_syncs = [&](size_t at) {  // cross-lane edges that precede op `at`
                    for (; n_lanes > 1 && next_sync < s.syncs.size() && s.syncs[next_sync].at <= at && !rc; ++next_sync) {
                        const Segment::LaneSync& y = s.syncs[next_sync];
                        if (cudaEventRecord(sync_events_[next_sync], lane_stream(y.from)) != cudaSuccess ||
                            cudaStreamWaitEvent(lane_stream(y.to), sync_events_[next_sync], 0) != cudaSuccess) {
                            lane_err = "cross-lane edge of the capture failed";
                            rc = 1;
                        }
                    }
                };
                for (size_t i = 0; i < s.ops.size() && !rc; ++i) {
                    do_syncs(i);
                    if (rc) break;
                    const int l = (n_lanes > 1 && i < s.lanes.size()) ? s.lanes[i] : 0;
                    rc = s.ops[i](lane_stream(l));
                }
                if (!rc) do_syncs(s.ops.size());
                if (n_lanes > 1) {  // join (also after a failed op: an unjoined capture cannot be ended)
                    for (int l = 1; l < n_lanes; ++l) {
                        if (cudaEventRecord(lane_events_[l - 1], lane_streams_[l - 1]) != cudaSuccess ||
                            cudaStreamWaitEvent(stream, lane_events_[l - 1], 0) != cudaSuccess) {
                            if (!rc) lane_err = "join of the capture lanes failed";
                            rc = 1;
                        }
                    }
                }
                cudaError_t e = cudaStreamEndCapture(stream, &graph);
                if (rc || e != cudaSuccess) {
                    if (graph) cudaGraphDestroy(graph);
                    throw std::runtime_error(std::string("graph capture failed: ") +
                                             (!lane_err.empty() ? lane_err.c_str() : rc ? gemm_last_error() : cudaGetErrorString(e)));
                }
                e = cudaGraphInstantiate(&s.exec, graph, 0);
                cudaGraphDestroy(graph);
                if (e != cudaSuccess) throw std::runtime_error(std::string("cudaGraphInstantiate: ") + cudaGetErrorString(e));
            }
            CK(cudaGraphLaunch(s.exec, stream));
        } else {
            for (auto& op : s.ops) {
                if (op(stream)) throw std::runtime_error(std::string("kernel launch failed: ") + gemm_last_error());
            }
        }
        launches += s.launches;
    }

    // ------------------------------------------------------------------ rate estimate (rate.cu)
    static void check_rate_qps(const int32_t* qps, int n)
    {
        if (n < 1 || n > kMaxRateTrials) throw std::runtime_error("estimate_bits: between 1 and 64 QPs per call");
        for (int i = 0; i < n; ++i)
            if (qps[i] < 0 || qps[i] >= kQpNum) throw std::runtime_error("qp out of range");
    }
    // after enc0 at `qp`: the rate kernel over the y steps and z into result slot `slot`
    void rate_trial(const int16_t* const* y, const int32_t* const* counts, int n_y, size_t y_capacity, const int8_t* z,
                    int nz, int qp, int slot, cudaStream_t stream)
    {
        RateArgs a{};
        for (int k = 0; k < n_y; ++k) { a.y[k] = y[k]; a.y_count[k] = counts[k]; }
        a.n_y = n_y;
        a.z = z; a.nz = nz; a.z_ch = kRateZCh; a.z_row0 = qp * kRateZCh;
        a.y_cost = cost_[1]; a.y_maxv = maxv_[1]; a.y_rows = cost_rows_[1]; a.y_width = cost_width_[1];
        a.z_cost = cost_[0]; a.z_maxv = maxv_[0]; a.z_width = cost_width_[0];
        a.out = rate_slots_ + slot;
        if (a.z_row0 + kRateZCh > cost_rows_[0]) throw std::runtime_error("estimate_bits: the z CDF table has no rows for this qp");
        if (!rate_smem_bytes(a.y_rows, a.y_width, a.z_ch, a.z_width)) throw std::runtime_error("estimate_bits: CDF tables too large");
        if (launch_rate_estimate(a, y_capacity, stream)) throw std::runtime_error("rate_estimate launch failed");
        ++launches;
    }
    // one copy of the slots, one synchronise; bytes = the coded symbols + 4 flush bytes per rANS stream + the offset
    // words of the merged container (RansCodec::encode)
    void rate_finish(int n, cudaStream_t stream, dcvc_rate_estimate* out)
    {
        CK(cudaMemcpyAsync(h_rate_slots_, rate_slots_, sizeof(RateSlot) * n, cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        for (int i = 0; i < n; ++i) {
            const RateSlot& s = h_rate_slots_[i];
            const int ec = RansCodec::ec_parallel_for(s.y_symbols);
            const int n_off = ec / 2 - 1 + ec % 2;
            out[i].y_q16 = static_cast<int64_t>(s.y_q16);
            out[i].z_q16 = static_cast<int64_t>(s.z_q16);
            out[i].y_symbols = s.y_symbols;
            out[i].ec_parallel = ec;
            const uint64_t q16 = s.y_q16 + s.z_q16;
            out[i].bytes = static_cast<int64_t>((q16 + (8ull << 16) - 1) / (8ull << 16)) + 4 * ec + 4 * n_off;
        }
    }

    void tick(cudaStream_t st)
    {
        if (tev_n_ + 2 <= static_cast<int>(tev_.size())) CK(cudaEventRecord(tev_[tev_n_], st));
    }
    void tock(cudaStream_t st)
    {
        if (tev_n_ + 2 <= static_cast<int>(tev_.size())) {
            CK(cudaEventRecord(tev_[tev_n_ + 1], st));
            tev_n_ += 2;
        }
    }

    // CUDA graphs cannot be captured on the legacy default stream: calls made on it hop onto an internal
    // stream and hand the result back with an event (the reference instead requires the caller to set a
    // non-default stream, test_video.py:423-425).
    struct StreamHop {
        CodecBase* c;
        cudaStream_t user, run;
        bool hop;
        StreamHop(CodecBase* codec, cudaStream_t u) : c(codec), user(u), run(u)
        {
            hop = (u == nullptr || u == cudaStreamLegacy || u == cudaStreamPerThread);
            if (hop) {
                if (cudaEventRecord(c->ev_hop_, user) != cudaSuccess ||
                    cudaStreamWaitEvent(c->own_stream_, c->ev_hop_, 0) != cudaSuccess)
                    throw std::runtime_error("stream hop failed");
                run = c->own_stream_;
            }
        }
        ~StreamHop()
        {
            if (hop) {
                cudaEventRecord(c->ev_hop_, run);
                cudaStreamWaitEvent(user, c->ev_hop_, 0);
            }
        }
    };

    int device_;
    bool finalized_ = false;
    bool use_graphs_ = true;
    bool fuse_tail_ = true;                    // DCVC_B200_FUSE_TAIL=0: per-op kernels only (A/B runs, kernel emulation)
    // The fused tail runs 256-pixel tiles on CTA pairs: below ~64 tiles it leaves SMs idle that the per-op kernels (128 x
    // 64..256 tiles on single CTAs) still fill — measured on B200: P16 of 1080p (8160 px, 32 tiles) 66.6 us fused vs 48.1 us
    // per-op for a C = 512 block; P8 of 1080p (32640 px) and everything at 4K are above the threshold.
    long long fuse_min_px_ = 16384;
    bool fuse_any_c_ = false;
    void* dbg_base_ = nullptr;      // activation arena (DCVC_B200_OPSUM)
    size_t dbg_bytes_ = 0;
    unsigned long long* opsum_dev_ = nullptr;
    float skip_thres_ = 0.f;
    std::map<std::string, HostTensor> params_;
    Arena warena_;
    uint8_t* lut_ = nullptr;
    RansCodec rans_;
    cudaStream_t copy_stream_ = nullptr, own_stream_ = nullptr;
    cudaEvent_t ev_hop_ = nullptr, ev_y_ = nullptr, ev_fork_ = nullptr;
    std::vector<cudaStream_t> lane_streams_;   // side streams of multi-lane segments (graph capture only)
    std::vector<cudaEvent_t> lane_events_;
    std::vector<cudaEvent_t> sync_events_;     // one per cross-lane edge of the largest multi-lane segment
    std::vector<cudaEvent_t> tev_;
    std::vector<cudaEvent_t> prof_events_;
    int tev_n_ = 0;
    std::vector<uint8_t> bitstream_;
    // rate estimate: Q16 code lengths and escape symbols of CDF set 0 (z) and 1 (y), one device slot per QP trial
    uint32_t* cost_[2] = { nullptr, nullptr };
    int8_t* maxv_[2] = { nullptr, nullptr };
    int cost_rows_[2] = { 0, 0 }, cost_width_[2] = { 0, 0 };
    RateSlot* rate_slots_ = nullptr;
    RateSlot* h_rate_slots_ = nullptr;
};

}  // namespace dcvc
