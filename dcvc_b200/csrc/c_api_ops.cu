// c_api_ops.cu — op-level and rANS entry points of include/dcvc_b200.h.
#include <string.h>

#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/dcvc_b200.h"
#include "elementwise.cuh"
#include "dcb_tail.cuh"
#include "pw_gemm.cuh"
#include "rans_host.h"

namespace dcvc {
thread_local std::string g_api_err;
void set_api_error(const std::string& s) { g_api_err = s; }
}  // namespace dcvc

using namespace dcvc;

static ActView to_view(const dcvc_view& v)
{
    ActView a;
    a.ptr = v.ptr; a.C = v.C; a.pitch = v.pitch; a.W = v.W; a.H = v.H;
    return a;
}

#define API_TRY try {
#define API_CATCH                                   \
    }                                               \
    catch (const std::exception& e) {               \
        set_api_error(e.what());                    \
        return 1;                                   \
    }                                               \
    catch (...) {                                   \
        set_api_error("unknown C++ exception");     \
        return 1;                                   \
    }

extern "C" {

const char* dcvc_last_error(void) { return g_api_err.c_str(); }
const char* dcvc_build_info(void) { return "dcvc_b200 sm_100a tcgen05/TMA build " __DATE__; }
int dcvc_abi_version(void) { return 1; }

int dcvc_op_gemm(const dcvc_gemm_desc* d, void* stream)
{
    API_TRY
    GemmOp op;
    op.kind = d->kind;
    op.in = to_view(d->in);
    op.out = to_view(d->out);
    op.res1 = to_view(d->res1);
    op.res2 = to_view(d->res2);
    op.weight = static_cast<const __half*>(d->weight);
    op.bias = static_cast<const __half*>(d->bias);
    op.qscale = static_cast<const __half*>(d->qscale);
    op.N = d->N;
    op.act = d->act;
    op.chunk_add = d->chunk_add;
    if (gemm_plan(op)) { set_api_error(gemm_last_error()); return 1; }
    if (gemm_launch(op, static_cast<cudaStream_t>(stream))) { set_api_error(gemm_last_error()); return 1; }
    return 0;
    API_CATCH
}

int dcvc_op_dcb_tail(const dcvc_dcb_tail_desc* d, void* stream)
{
    API_TRY
    DcbTailOp op;
    op.t2 = to_view(d->t2);
    op.x = to_view(d->x);
    op.y = to_view(d->y);
    op.t1n = to_view(d->t1n);
    op.w3 = static_cast<const __half*>(d->w3);   op.b3 = static_cast<const __half*>(d->b3);
    op.wf0 = static_cast<const __half*>(d->wf0); op.bf0 = static_cast<const __half*>(d->bf0);
    op.wf2 = static_cast<const __half*>(d->wf2); op.bf2 = static_cast<const __half*>(d->bf2);
    op.w0n = static_cast<const __half*>(d->w0n); op.b0n = static_cast<const __half*>(d->b0n);
    op.qscale = static_cast<const __half*>(d->qscale);
    op.shortcut = d->shortcut != 0;
    const int r = dcb_tail_plan(op);
    if (r == 1) { set_api_error("dcb_tail: not eligible"); return 2; }
    if (r) { set_api_error(gemm_last_error()); return 1; }
    if (dcb_tail_launch(op, static_cast<cudaStream_t>(stream))) { set_api_error(gemm_last_error()); return 1; }
    return 0;
    API_CATCH
}

int dcvc_pack_weight(int32_t kind, const void* w_host, int32_t cout, int32_t cin, int32_t kh,
                     int32_t kw, void* dst_host)
{
    const uint16_t* w = static_cast<const uint16_t*>(w_host);
    uint16_t* dst = static_cast<uint16_t*>(dst_host);
    switch (kind) {
    case DCVC_GEMM_PW:
        if (kh != 1 || kw != 1) { set_api_error("pack_weight: PW needs 1x1"); return 1; }
        memcpy(dst, w, static_cast<size_t>(cout) * cin * 2);
        return 0;
    case DCVC_GEMM_CONV3X3_S2:
        if (kh != 3 || kw != 3) { set_api_error("pack_weight: conv3x3 needs 3x3"); return 1; }
        for (int n = 0; n < cout; ++n)
            for (int c = 0; c < cin; ++c)
                for (int t = 0; t < 9; ++t)
                    dst[(static_cast<size_t>(n) * 9 + t) * cin + c] = w[(static_cast<size_t>(n) * cin + c) * 9 + t];
        return 0;
    case DCVC_GEMM_CONV2X2_S2: {
        // weight of the 1x1 conv behind pixel_unshuffle(2): input channel = c*4 + py*2 + px
        if (kh != 1 || kw != 1 || cin % 4) { set_api_error("pack_weight: conv2x2 needs [Cout][4C][1][1]"); return 1; }
        const int c1 = cin / 4;
        for (int n = 0; n < cout; ++n)
            for (int c = 0; c < c1; ++c)
                for (int t = 0; t < 4; ++t)
                    dst[(static_cast<size_t>(n) * 4 + t) * c1 + c] = w[static_cast<size_t>(n) * cin + c * 4 + t];
        return 0;
    }
    case DCVC_GEMM_TCONV2X2: {
        // weight of the 1x1 conv in front of pixel_shuffle(2): output channel = co*4 + py*2 + px
        if (kh != 1 || kw != 1 || cout % 4) { set_api_error("pack_weight: tconv needs [4Cout][C][1][1]"); return 1; }
        const int co_n = cout / 4;
        for (int co = 0; co < co_n; ++co)
            for (int ph = 0; ph < 4; ++ph)
                memcpy(dst + (static_cast<size_t>(ph) * co_n + co) * cin,
                       w + (static_cast<size_t>(co) * 4 + ph) * cin, static_cast<size_t>(cin) * 2);
        return 0;
    }
    case DCVC_GEMM_CONV3X3_PS2: {
        // 3x3 conv in front of pixel_shuffle(2): output channel = co*4 + phase -> GEMM row phase*Cout + co, [tap][c]
        if (kh != 3 || kw != 3 || cout % 4) { set_api_error("pack_weight: conv3x3_ps2 needs [4Cout][C][3][3]"); return 1; }
        const int co_n = cout / 4;
        for (int co = 0; co < co_n; ++co)
            for (int ph = 0; ph < 4; ++ph)
                for (int c = 0; c < cin; ++c)
                    for (int t = 0; t < 9; ++t)
                        dst[((static_cast<size_t>(ph) * co_n + co) * 9 + t) * cin + c] =
                            w[((static_cast<size_t>(co) * 4 + ph) * cin + c) * 9 + t];
        return 0;
    }
    }
    set_api_error("pack_weight: bad kind");
    return 1;
}

int dcvc_op_dw3x3(const dcvc_view* in, const dcvc_view* out, const void* w, void* stream)
{
    return launch_dw3x3(to_view(*in), to_view(*out), static_cast<const __half*>(w),
                        static_cast<cudaStream_t>(stream));
}

int dcvc_op_unshuffle8_pad(const void* x, int32_t Cs, int32_t H, int32_t W, int64_t sc, int64_t sh,
                           int64_t sw, const dcvc_view* out, void* stream)
{
    return launch_unshuffle8_pad(static_cast<const __half*>(x), Cs, H, W, sc, sh, sw, to_view(*out),
                                 static_cast<cudaStream_t>(stream));
}

int dcvc_op_shuffle8_clamp(const dcvc_view* in, void* out, int32_t Cs, int32_t clamp, void* stream)
{
    return launch_shuffle8_clamp(to_view(*in), static_cast<__half*>(out), Cs, clamp,
                                 static_cast<cudaStream_t>(stream));
}

int dcvc_op_pad_crop(const dcvc_view* in, const dcvc_view* out, void* stream)
{
    return launch_pad_crop(to_view(*in), to_view(*out), static_cast<cudaStream_t>(stream));
}

int dcvc_op_scale_channels(const dcvc_view* in, const void* q, const dcvc_view* out, void* stream)
{
    return launch_scale_channels(to_view(*in), static_cast<const __half*>(q), to_view(*out),
                                 static_cast<cudaStream_t>(stream));
}

int dcvc_op_round_z(const void* z, void* z_hat, void* z_i8, int64_t n, void* stream)
{
    return launch_round_z(static_cast<const __half*>(z), static_cast<__half*>(z_hat),
                          static_cast<int8_t*>(z_i8), n, static_cast<cudaStream_t>(stream));
}

int dcvc_op_int8_to_half(const void* x, void* out, int64_t n, void* stream)
{
    return launch_int8_to_half(static_cast<const int8_t*>(x), static_cast<__half*>(out), n,
                               static_cast<cudaStream_t>(stream));
}

static uint8_t* device_lut()
{
    static uint8_t* d_lut = nullptr;
    if (!d_lut) {
        std::vector<uint8_t> h(65536);
        build_scale_lut(h.data());
        if (cudaMalloc(&d_lut, 65536) != cudaSuccess) return nullptr;
        cudaMemcpy(d_lut, h.data(), 65536, cudaMemcpyHostToDevice);
    }
    return d_lut;
}

static EntropyStepArgs to_args(const dcvc_entropy_step* a)
{
    EntropyStepArgs e;
    e.H = a->H; e.W = a->W; e.G = a->G; e.step = a->step;
    e.y = static_cast<const __half*>(a->y); e.y_pitch = a->y_pitch;
    e.q_enc = static_cast<const __half*>(a->q_enc);
    e.scales = static_cast<const __half*>(a->scales);
    e.means = static_cast<const __half*>(a->means);
    e.p_pitch = a->p_pitch;
    e.y_hat_acc = static_cast<__half*>(a->y_hat_acc); e.acc_pitch = a->acc_pitch;
    e.skip_thres = a->skip_thres;
    e.scale_lut = device_lut();
    e.sym_raw = static_cast<int16_t*>(a->sym_raw);
    e.idx_raw = static_cast<uint8_t*>(a->idx_raw);
    e.counts = static_cast<int32_t*>(a->counts);
    return e;
}

int dcvc_op_entropy_enc_step(const dcvc_entropy_step* a, void* stream)
{
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    EntropyStepArgs e = to_args(a);
    if (!e.scale_lut) { set_api_error("scale LUT allocation failed"); return 1; }
    if (launch_entropy_enc_step(e, s)) return 1;
    if (launch_scan_counts(e.counts, static_cast<int32_t*>(a->offsets), static_cast<int32_t*>(a->total), a->H * a->W, s)) return 1;
    return launch_compact_i16(e, static_cast<const int32_t*>(a->offsets), static_cast<int16_t*>(a->compact), s);
}

int dcvc_op_entropy_dec_index(const dcvc_entropy_step* a, void* stream)
{
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    EntropyStepArgs e = to_args(a);
    if (!e.scale_lut) { set_api_error("scale LUT allocation failed"); return 1; }
    if (launch_entropy_dec_index(e, s)) return 1;
    if (launch_scan_counts(e.counts, static_cast<int32_t*>(a->offsets), static_cast<int32_t*>(a->total), a->H * a->W, s)) return 1;
    return launch_compact_u8(e, static_cast<const int32_t*>(a->offsets), static_cast<uint8_t*>(a->compact), s);
}

int dcvc_op_entropy_dec_restore(const dcvc_entropy_step* a, void* stream)
{
    EntropyStepArgs e = to_args(a);
    return launch_entropy_dec_restore(e, static_cast<const int32_t*>(a->offsets),
                                      static_cast<const int8_t*>(a->decoded),
                                      static_cast<cudaStream_t>(stream));
}

int dcvc_scale_index_lut(uint8_t* lut65536)
{
    build_scale_lut(lut65536);
    return 0;
}

// ------------------------------------------------------------------------------------ rANS
struct dcvc_rans {
    RansCodec codec;
    std::vector<EncodeJob> jobs;
    std::vector<uint8_t> out;
};

int dcvc_rans_create(dcvc_rans** out)
{
    API_TRY
    *out = new dcvc_rans();
    return 0;
    API_CATCH
}

void dcvc_rans_destroy(dcvc_rans* r) { delete r; }

int dcvc_rans_set_cdf(dcvc_rans* r, const int32_t* cdf, const int32_t* cdf_sizes, int32_t rows,
                      int32_t width, int32_t index)
{
    API_TRY
    if (index < 0 || index > 1) { set_api_error("rans_set_cdf: index must be 0 or 1"); return 1; }
    r->codec.set_cdf(cdf, cdf_sizes, rows, width, index);
    return 0;
    API_CATCH
}

int dcvc_rans_enc_reset(dcvc_rans* r) { r->jobs.clear(); return 0; }

int dcvc_rans_enc_y(dcvc_rans* r, const int16_t* symbols, int32_t n)
{
    EncodeJob j; j.kind = EncodeJob::Y; j.y = symbols; j.size = n;
    r->jobs.push_back(j);
    return 0;
}

int dcvc_rans_enc_z(dcvc_rans* r, const int8_t* symbols, int32_t n, int32_t cdf_offset, int32_t ch)
{
    EncodeJob j; j.kind = EncodeJob::Z; j.z = symbols; j.size = n; j.cdf_offset = cdf_offset; j.ch = ch;
    r->jobs.push_back(j);
    return 0;
}

int dcvc_rans_enc_finish(dcvc_rans* r, int32_t n_parallel, const uint8_t** data, int32_t* size)
{
    API_TRY
    r->codec.encode(r->jobs, n_parallel, r->out);
    *data = r->out.data();
    *size = static_cast<int32_t>(r->out.size());
    return 0;
    API_CATCH
}

int dcvc_rans_dec_set_stream(dcvc_rans* r, const uint8_t* data, int32_t size, int32_t n_parallel)
{
    API_TRY
    r->codec.set_stream(data, size, n_parallel);
    return 0;
    API_CATCH
}

int dcvc_rans_dec_z(dcvc_rans* r, int8_t* out, int32_t n, int32_t cdf_offset, int32_t ch)
{
    API_TRY
    r->codec.decode_z(out, n, cdf_offset, ch);
    return 0;
    API_CATCH
}

int dcvc_rans_dec_y(dcvc_rans* r, int8_t* out, const uint8_t* cdf_rows, int32_t n)
{
    API_TRY
    r->codec.decode_y(out, cdf_rows, n);
    return 0;
    API_CATCH
}

int dcvc_pmf_to_quantized_cdf(const float* pmf, int32_t n, uint32_t* cdf_out)
{
    API_TRY
    std::vector<uint32_t> c = pmf_to_quantized_cdf(pmf, n);
    memcpy(cdf_out, c.data(), c.size() * sizeof(uint32_t));
    return 0;
    API_CATCH
}

int dcvc_rans_cost_table(const int32_t* cdf, const int32_t* cdf_sizes, int32_t rows, int32_t width, uint32_t* out)
{
    API_TRY
    if (rows < 1 || width < 2) throw std::runtime_error("rans_cost_table: bad table shape");
    std::vector<uint32_t> c = rans_cost_table(cdf, cdf_sizes, rows, width);
    memcpy(out, c.data(), c.size() * sizeof(uint32_t));
    return 0;
    API_CATCH
}

}  // extern "C"
