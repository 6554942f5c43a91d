// codec.cu — codec-level runtime behind the C ABI (dcvc_create / set_param / compress / decompress).
//
// B200-native counterpart of the reference's proxy runtime for DCVC-UF-Intra
// (src/layers/extensions/inference/dmci_proxy.{h,cpp}, layers_proxy.{h,cpp}, dmc_common.{h,cpp},
// memory_pool.h), re-designed rather than translated:
//   * weights are re-laid out once on the host (dw bias folded into the next 1x1, stride-2 /
//     transposed-conv weights packed per tap / phase) and live in one device arena;
//   * activations live in a per-resolution arena; every DepthConvBlock ping-pongs between the
//     same four buffers of its pyramid level so the working set stays inside the 126 MB L2;
//   * the QP only selects four per-channel scale vectors: they are staged into fixed device
//     buffers before each call, so ONE CUDA graph per segment serves all 64 QPs (the reference
//     captures 64 graphs per segment, dmc_common.cpp:95-106);
//   * host rANS stays on the CPU (north_star); symbol counts/streams cross PCIe in two small
//     copies per step; the synthesis transform overlaps the CPU encode.
#include <chrono>
#include <cstdio>
#include "codec_common.cuh"

namespace dcvc {

namespace {
constexpr int kChSrc = 192, kChEncDec = 384, kChY = 256, kChZ = 128;
}  // namespace

class IntraCodec : public CodecBase {
public:
    explicit IntraCodec(int device) : CodecBase(device) {}
    ~IntraCodec() override;

    void finalize(float skip_thres) override;
    void compress(const void* x, int H, int W, int64_t sc, int64_t sh, int64_t sw, int qp, int pad_b,
                  int pad_r, cudaStream_t stream, const uint8_t** bs, int32_t* bs_len,
                  int32_t* ec_parallel, void* x_hat_out);
    void decompress(const uint8_t* bs, int len, int qp, int height, int width, int ec_parallel,
                    cudaStream_t stream, void* x_hat_out);
    void estimate(const void* x, int H, int W, int64_t sc, int64_t sh, int64_t sw, const int32_t* qps, int n_qps,
                  int pad_b, int pad_r, cudaStream_t stream, dcvc_rate_estimate* out) override;
    int debug_fetch(const char* name, void* dst, int64_t max_bytes, int64_t* written) override;
    int arena_overflow_blocks() const override { return arena_.overflow_blocks(); }

private:

    // ---- plan
    void plan(int height, int width);
    void clear_plan();
    void build_hyper_tail(Segment& s);  // z_hat -> params, reduced
    void build_spatial_prior(Segment& s, int k);
    void build_synthesis(Segment& s);
    void stage_qp(int qp, cudaStream_t stream);


    // weights on device
    DcbW enc1_, enc2_[6], henc0_, henc1_, henc2_, hdec0_, hdec1_, hdec2_, pf_[3], spa_[3], sp_[3],
        dec1_[13], dec2_;
    ConvW enc_down_, henc1_down_, henc2_down_, hdec0_up_, hdec1_up_, dec_up_, pf3_, sp3_, red_;
    const __half *q_enc_all_ = nullptr, *q_dec_all_ = nullptr, *q_y_enc_all_ = nullptr,
                 *q_y_dec_all_ = nullptr;

    // plan state
    int H8_ = 0, W8_ = 0, H16_ = 0, W16_ = 0, H16p_ = 0, W16p_ = 0, H64_ = 0, W64_ = 0;
    Arena arena_;
    Level l8_, l16_, l32_, l64_;
    __half *in8_ = nullptr, *y_ = nullptr, *ypad_ = nullptr, *hyp_ = nullptr, *params_p_ = nullptr,
           *params_c_ = nullptr, *cat_ = nullptr, *sp_out_ = nullptr, *yhat_ = nullptr,
           *zhat_ = nullptr, *dec_out_ = nullptr;
    int8_t* z_i8_ = nullptr;
    __half *q_enc_ = nullptr, *q_dec_ = nullptr, *q_y_enc_ = nullptr, *q_y_dec_ = nullptr;
    int16_t* sym_raw_ = nullptr;
    uint8_t* idx_raw_ = nullptr;
    int32_t *counts_ = nullptr, *offsets_[4] = { nullptr, nullptr, nullptr, nullptr }, *totals_ = nullptr;
    int16_t* sym_c_[4] = { nullptr, nullptr, nullptr, nullptr };
    uint8_t* idx_c_ = nullptr;
    int8_t* decoded_ = nullptr;
    // pinned host mirrors
    int32_t* h_totals_ = nullptr;
    int16_t* h_sym_[4] = { nullptr, nullptr, nullptr, nullptr };
    uint8_t* h_idx_ = nullptr;
    int8_t* h_decoded_ = nullptr;
    int8_t* h_z_ = nullptr;
    size_t quarter_ = 0;

    Segment enc0_, enc1_seg_, dec0_, dec_step_[4];  // dec_step_[k]: k = 1..3 prior steps, [0] unused
    Segment dec4_;
    const __half* params_cur_ = nullptr;  // params of step 0 (cropped)
};

void IntraCodec::finalize(float skip_thres)
{
    finalize_begin(skip_thres);
    clear_plan();
    enc1_ = load_dcb("enc.enc_1.");
    for (int i = 0; i < 6; ++i) enc2_[i] = load_dcb("enc.enc_2." + std::to_string(i) + ".");
    enc_down_ = load_conv("enc.enc_2.6.", DCVC_GEMM_CONV3X3_S2);
    henc0_ = load_dcb("hyper_enc.conv.0.");
    henc1_down_ = load_conv("hyper_enc.conv.1.down.", DCVC_GEMM_CONV2X2_S2);
    henc1_ = load_dcb("hyper_enc.conv.1.conv.");
    henc2_down_ = load_conv("hyper_enc.conv.2.down.", DCVC_GEMM_CONV2X2_S2);
    henc2_ = load_dcb("hyper_enc.conv.2.conv.");
    hdec0_up_ = load_conv("hyper_dec.conv.0.up.conv.0.", DCVC_GEMM_TCONV2X2);
    hdec0_ = load_dcb("hyper_dec.conv.0.conv.");
    hdec1_up_ = load_conv("hyper_dec.conv.1.up.conv.0.", DCVC_GEMM_TCONV2X2);
    hdec1_ = load_dcb("hyper_dec.conv.1.conv.");
    hdec2_ = load_dcb("hyper_dec.conv.2.");
    for (int i = 0; i < 3; ++i) pf_[i] = load_dcb("y_prior_fusion.conv." + std::to_string(i) + ".");
    pf3_ = load_conv("y_prior_fusion.conv.3.", DCVC_GEMM_PW);
    red_ = load_conv("y_spatial_prior_reduction.", DCVC_GEMM_PW);
    for (int i = 0; i < 3; ++i) spa_[i] = load_dcb("y_spatial_prior_adaptor_" + std::to_string(i + 1) + ".");
    for (int i = 0; i < 3; ++i) sp_[i] = load_dcb("y_spatial_prior.conv." + std::to_string(i) + ".");
    sp3_ = load_conv("y_spatial_prior.conv.3.", DCVC_GEMM_PW);
    dec_up_ = load_conv("dec.dec_1.0.up.conv.0.", DCVC_GEMM_TCONV2X2);
    dec1_[0] = load_dcb("dec.dec_1.0.conv.");
    for (int i = 1; i < 13; ++i) dec1_[i] = load_dcb("dec.dec_1." + std::to_string(i) + ".");
    dec2_ = load_dcb("dec.dec_2.");
    q_enc_all_ = upload(param_f16("q_scale_enc"));
    q_dec_all_ = upload(param_f16("q_scale_dec"));
    q_y_enc_all_ = upload(param_f16("q_scale_y_enc"));
    q_y_dec_all_ = upload(param_f16("q_scale_y_dec"));

    finalize_end();
}

IntraCodec::~IntraCodec() { clear_plan(); }

// =============================================================================== plan
void IntraCodec::clear_plan()
{
    Segment* segs[] = { &enc0_, &enc1_seg_, &dec0_, &dec_step_[0], &dec_step_[1], &dec_step_[2], &dec_step_[3], &dec4_ };
    for (Segment* s : segs) s->reset();
    if (h_totals_) { cudaFreeHost(h_totals_); h_totals_ = nullptr; }
    for (int k = 0; k < 4; ++k) if (h_sym_[k]) { cudaFreeHost(h_sym_[k]); h_sym_[k] = nullptr; }
    if (h_idx_) { cudaFreeHost(h_idx_); h_idx_ = nullptr; }
    if (h_decoded_) { cudaFreeHost(h_decoded_); h_decoded_ = nullptr; }
    if (h_z_) { cudaFreeHost(h_z_); h_z_ = nullptr; }
    arena_.release();
    H8_ = W8_ = 0;
}

void IntraCodec::plan(int height, int width)
{
    const int H = round_up(height, 16), W = round_up(width, 16);
    const int H8 = H / 8, W8 = W / 8;
    if (H8 == H8_ && W8 == W8_) return;
    if (!finalized_) throw std::runtime_error("set_param/finalize_params must be called first");
    clear_plan();
    H8_ = H8; W8_ = W8;
    H16_ = H8 / 2; W16_ = W8 / 2;
    H16p_ = round_up(H16_, 4); W16p_ = round_up(W16_, 4);
    const int H32 = H16p_ / 2, W32 = W16p_ / 2;
    H64_ = H16p_ / 4; W64_ = W16p_ / 4;
    const size_t p8 = static_cast<size_t>(H8) * W8, p16p = static_cast<size_t>(H16p_) * W16p_;
    const size_t p16 = static_cast<size_t>(H16_) * W16_, p32 = static_cast<size_t>(H32) * W32;
    const size_t p64 = static_cast<size_t>(H64_) * W64_;
    quarter_ = p16 * (kChY / 4);

    size_t bytes = 0;
    bytes += 4 * p8 * kChEncDec * 2 + p8 * kChSrc * 2 * 2;          // level 8 + in8 + dec_out
    bytes += 4 * p16p * 512 * 2 + 8 * p16p * 512 * 2;                // level 16 + named P16 buffers
    bytes += 4 * p32 * 128 * 2 + 6 * p64 * 128 * 2;
    bytes += quarter_ * (2 + 1 + 4 * 2 + 1 + 1) + p16 * 4 * 6 + (1u << 20);
    bytes += 64 * 1024;  // alignment slack per allocation
    arena_.reserve(bytes + (4u << 20));
    dbg_base_ = arena_.base();
    dbg_bytes_ = bytes + (4u << 20);
    auto half_buf = [&](size_t n) { return static_cast<__half*>(arena_.alloc(n * 2)); };

    l8_.H = H8; l8_.W = W8;
    l8_.A = half_buf(p8 * kChEncDec); l8_.B = half_buf(p8 * kChEncDec);
    l8_.T1 = half_buf(p8 * kChEncDec); l8_.T2 = half_buf(p8 * kChEncDec);
    in8_ = half_buf(p8 * kChSrc);
    dec_out_ = half_buf(p8 * kChSrc);
    l16_.H = H16p_; l16_.W = W16p_;
    l16_.A = half_buf(p16p * 512); l16_.B = half_buf(p16p * 512);
    l16_.T1 = half_buf(p16p * 512); l16_.T2 = half_buf(p16p * 512);
    l32_.H = H32; l32_.W = W32;
    l32_.A = half_buf(p32 * 128); l32_.B = half_buf(p32 * 128);
    l32_.T1 = half_buf(p32 * 128); l32_.T2 = half_buf(p32 * 128);
    l64_.H = H64_; l64_.W = W64_;
    l64_.A = half_buf(p64 * 128); l64_.B = half_buf(p64 * 128);
    l64_.T1 = half_buf(p64 * 128); l64_.T2 = half_buf(p64 * 128);
    y_ = half_buf(p16 * kChY);
    const bool padded = (H16p_ != H16_) || (W16p_ != W16_);
    ypad_ = padded ? half_buf(p16p * kChY) : y_;
    hyp_ = half_buf(p16p * kChY);
    params_p_ = half_buf(p16p * 512);
    params_c_ = padded ? half_buf(p16 * 512) : params_p_;
    cat_ = half_buf(p16 * 512);
    sp_out_ = half_buf(p16 * 512);
    yhat_ = half_buf(p16 * kChY);
    zhat_ = half_buf(p64 * kChZ);
    z_i8_ = static_cast<int8_t*>(arena_.alloc(p64 * kChZ));
    q_enc_ = half_buf(kChEncDec); q_dec_ = half_buf(kChEncDec);
    q_y_enc_ = half_buf(kChY); q_y_dec_ = half_buf(kChY);
    sym_raw_ = static_cast<int16_t*>(arena_.alloc(quarter_ * 2));
    idx_raw_ = static_cast<uint8_t*>(arena_.alloc(quarter_));
    counts_ = static_cast<int32_t*>(arena_.alloc(p16 * 4));
    totals_ = static_cast<int32_t*>(arena_.alloc(64));
    for (int k = 0; k < 4; ++k) {
        offsets_[k] = static_cast<int32_t*>(arena_.alloc((p16 + 1) * 4));
        sym_c_[k] = static_cast<int16_t*>(arena_.alloc(quarter_ * 2));
    }
    idx_c_ = static_cast<uint8_t*>(arena_.alloc(quarter_));
    decoded_ = static_cast<int8_t*>(arena_.alloc(quarter_));
    CK(cudaMallocHost(&h_totals_, 64));
    for (int k = 0; k < 4; ++k) CK(cudaMallocHost(&h_sym_[k], quarter_ * 2));
    CK(cudaMallocHost(&h_idx_, quarter_));
    CK(cudaMallocHost(&h_decoded_, quarter_));
    CK(cudaMallocHost(&h_z_, p64 * kChZ));

    const ActView v_in8 = make_view(in8_, kChSrc, kChSrc, W8, H8);
    const ActView v_y = make_view(y_, kChY, kChY, W16_, H16_);
    const ActView v_ypad = make_view(ypad_, kChY, kChY, W16p_, H16p_);
    const ActView v_scales0 = make_view(params_c_, kChY, 512, W16_, H16_);

    // ------------------------------------------------------------------ enc_0 (dmci_proxy.cpp:308-394)
    {
        Segment& s = enc0_;
        ActView t = dcb(s, l8_, v_in8, enc1_, false, q_enc_, nullptr);     // enc_1, then * q_enc
        for (int i = 0; i < 6; ++i) t = dcb(s, l8_, t, enc2_[i], false, nullptr, nullptr);
        add_gemm(s, GEMM_CONV3X3_S2, t, v_y, enc_down_.w, enc_down_.b, kChY, ACT_NONE, 0, nullptr, nullptr, nullptr);
        if (padded) s.ops.push_back([v_y, v_ypad](cudaStream_t st) { return launch_pad_crop(v_y, v_ypad, st); });
        // hyper encoder
        ActView h = dcb(s, l16_, v_ypad, henc0_, false, nullptr, nullptr);
        ActView d32 = make_view(l32_.A, kChZ, kChZ, W32, H32);
        add_gemm(s, GEMM_CONV2X2_S2, h, d32, henc1_down_.w, henc1_down_.b, kChZ, ACT_NONE, 0, nullptr, nullptr, nullptr);
        d32 = dcb(s, l32_, d32, henc1_, true, nullptr, nullptr);
        ActView d64 = make_view(l64_.A, kChZ, kChZ, W64_, H64_);
        add_gemm(s, GEMM_CONV2X2_S2, d32, d64, henc2_down_.w, henc2_down_.b, kChZ, ACT_NONE, 0, nullptr, nullptr, nullptr);
        d64 = dcb(s, l64_, d64, henc2_, true, nullptr, nullptr);
        {
            const __half* z = static_cast<const __half*>(d64.ptr);
            __half* zh = zhat_;
            int8_t* zi = z_i8_;
            const long long n = static_cast<long long>(p64) * kChZ;
            s.ops.push_back([z, zh, zi, n](cudaStream_t st) { return launch_round_z(z, zh, zi, n, st); });
        }
        build_hyper_tail(s);
        for (int k = 0; k < 4; ++k) {
            if (k > 0) build_spatial_prior(s, k);
            EntropyStepArgs a;
            a.H = H16_; a.W = W16_; a.G = kChY / 4; a.step = k;
            a.y = y_; a.y_pitch = kChY; a.q_enc = q_y_enc_;
            const __half* pbase = (k == 0) ? params_c_ : sp_out_;
            a.scales = pbase; a.means = pbase + kChY; a.p_pitch = 512;
            a.y_hat_acc = cat_; a.acc_pitch = 512;
            a.skip_thres = skip_thres_; a.scale_lut = lut_;
            a.sym_raw = sym_raw_; a.counts = counts_;
            int32_t* offs = offsets_[k];
            int32_t* tot = totals_ + k;
            int16_t* dst = sym_c_[k];
            const int n = static_cast<int>(p16);
            s.ops.push_back([a](cudaStream_t st) { return launch_entropy_enc_step(a, st); });
            s.ops.push_back([a, offs, tot, n](cudaStream_t st) { return launch_scan_counts(a.counts, offs, tot, n, st); });
            s.ops.push_back([a, offs, dst](cudaStream_t st) { return launch_compact_i16(a, offs, dst, st); });
        }
        const ActView acc = make_view(cat_, kChY, 512, W16_, H16_);
        const ActView yh = make_view(yhat_, kChY, kChY, W16_, H16_);
        const __half* qd = q_y_dec_;
        s.ops.push_back([acc, qd, yh](cudaStream_t st) { return launch_scale_channels(acc, qd, yh, st); });
    }
    (void)v_scales0;
    // ------------------------------------------------------------------ enc_1 = synthesis
    build_synthesis(enc1_seg_);

    // ------------------------------------------------------------------ decoder segments (dmci_proxy.cpp:461-599)
    {
        Segment& s = dec0_;
        const int8_t* zi = z_i8_;
        __half* zh = zhat_;
        const long long n = static_cast<long long>(p64) * kChZ;
        s.ops.push_back([zi, zh, n](cudaStream_t st) { return launch_int8_to_half(zi, zh, n, st); });
        build_hyper_tail(s);
    }
    for (int k = 0; k < 4; ++k) {
        // segment producing the indexes of step k; for k > 0 it first restores step k-1
        Segment& s = (k == 0) ? dec0_ : dec_step_[k];
        if (k > 0) {
            EntropyStepArgs r;
            r.H = H16_; r.W = W16_; r.G = kChY / 4; r.step = k - 1;
            const __half* pb = (k - 1 == 0) ? params_c_ : sp_out_;
            r.scales = pb; r.means = pb + kChY; r.p_pitch = 512;
            r.y_hat_acc = cat_; r.acc_pitch = 512; r.skip_thres = skip_thres_; r.scale_lut = lut_;
            const int32_t* offs = offsets_[k - 1];
            const int8_t* dec = decoded_;
            s.ops.push_back([r, offs, dec](cudaStream_t st) { return launch_entropy_dec_restore(r, offs, dec, st); });
            build_spatial_prior(s, k);
        }
        EntropyStepArgs a;
        a.H = H16_; a.W = W16_; a.G = kChY / 4; a.step = k;
        const __half* pbase = (k == 0) ? params_c_ : sp_out_;
        a.scales = pbase; a.means = pbase + kChY; a.p_pitch = 512;
        a.skip_thres = skip_thres_; a.scale_lut = lut_;
        a.idx_raw = idx_raw_; a.counts = counts_;
        int32_t* offs = offsets_[k];
        int32_t* tot = totals_ + k;
        uint8_t* dst = idx_c_;
        const int n = static_cast<int>(p16);
        s.ops.push_back([a](cudaStream_t st) { return launch_entropy_dec_index(a, st); });
        s.ops.push_back([a, offs, tot, n](cudaStream_t st) { return launch_scan_counts(a.counts, offs, tot, n, st); });
        s.ops.push_back([a, offs, dst](cudaStream_t st) { return launch_compact_u8(a, offs, dst, st); });
    }
    {
        Segment& s = dec4_;
        EntropyStepArgs r;
        r.H = H16_; r.W = W16_; r.G = kChY / 4; r.step = 3;
        r.scales = sp_out_; r.means = sp_out_ + kChY; r.p_pitch = 512;
        r.y_hat_acc = cat_; r.acc_pitch = 512; r.skip_thres = skip_thres_; r.scale_lut = lut_;
        const int32_t* offs = offsets_[3];
        const int8_t* dec = decoded_;
        s.ops.push_back([r, offs, dec](cudaStream_t st) { return launch_entropy_dec_restore(r, offs, dec, st); });
        const ActView acc = make_view(cat_, kChY, 512, W16_, H16_);
        const ActView yh = make_view(yhat_, kChY, kChY, W16_, H16_);
        const __half* qd = q_y_dec_;
        s.ops.push_back([acc, qd, yh](cudaStream_t st) { return launch_scale_channels(acc, qd, yh, st); });
        build_synthesis(s);
    }
    Segment* segs[] = { &enc0_, &enc1_seg_, &dec0_, &dec_step_[1], &dec_step_[2], &dec_step_[3], &dec4_ };
    for (Segment* s : segs) s->seal();
}

// z_hat -> hyper decoder -> prior fusion -> crop -> (scales, means) + reduced params into the cat buffer
void IntraCodec::build_hyper_tail(Segment& s)
{
    const int H32 = l32_.H, W32 = l32_.W;
    const ActView zh = make_view(zhat_, kChZ, kChZ, W64_, H64_);
    ActView u32 = make_view(l32_.A, kChZ, kChZ, W32, H32);
    add_gemm(s, GEMM_TCONV2X2, zh, u32, hdec0_up_.w, nullptr, 4 * kChZ, ACT_NONE, 0, nullptr, nullptr, nullptr);
    u32 = dcb(s, l32_, u32, hdec0_, true, nullptr, nullptr);
    ActView u16 = make_view(l16_.A, kChZ, kChZ, W16p_, H16p_);
    add_gemm(s, GEMM_TCONV2X2, u32, u16, hdec1_up_.w, nullptr, 4 * kChZ, ACT_NONE, 0, nullptr, nullptr, nullptr);
    u16 = dcb(s, l16_, u16, hdec1_, true, nullptr, nullptr);
    const ActView hyp = make_view(hyp_, kChY, kChY, W16p_, H16p_);
    dcb(s, l16_, u16, hdec2_, false, nullptr, &hyp);
    ActView t = dcb(s, l16_, hyp, pf_[0], false, nullptr, nullptr);
    t = dcb(s, l16_, t, pf_[1], false, nullptr, nullptr);
    t = dcb(s, l16_, t, pf_[2], false, nullptr, nullptr);
    const ActView pp = make_view(params_p_, 512, 512, W16p_, H16p_);
    add_gemm(s, GEMM_PW, t, pp, pf3_.w, pf3_.b, 512, ACT_NONE, 0, nullptr, nullptr, nullptr);
    const ActView pc = make_view(params_c_, 512, 512, W16_, H16_);
    if (params_c_ != params_p_) s.ops.push_back([pp, pc](cudaStream_t st) { return launch_pad_crop(pp, pc, st); });
    const ActView red = make_view(cat_ + kChY, kChY, 512, W16_, H16_);
    add_gemm(s, GEMM_PW, pc, red, red_.w, red_.b, kChY, ACT_NONE, 0, nullptr, nullptr, nullptr);
}

// adaptor_k + 3 blocks + 1x1 on cat(y_hat_so_far, reduced) -> sp_out (dmci_proxy.cpp:347-349)
void IntraCodec::build_spatial_prior(Segment& s, int k)
{
    // the spatial prior works on the unpadded latent grid
    Level L = l16_;
    const ActView cat = make_view(cat_, 512, 512, W16_, H16_);
    ActView t = dcb(s, L, cat, spa_[k - 1], false, nullptr, nullptr);
    for (int i = 0; i < 3; ++i) t = dcb(s, L, t, sp_[i], false, nullptr, nullptr);
    const ActView out = make_view(sp_out_, 512, 512, W16_, H16_);
    add_gemm(s, GEMM_PW, t, out, sp3_.w, sp3_.b, 512, ACT_NONE, 0, nullptr, nullptr, nullptr);
}

// y_hat -> x_hat features (dmci_proxy.cpp:14-33); the final shuffle+clamp writes to the caller's buffer
void IntraCodec::build_synthesis(Segment& s)
{
    const ActView yh = make_view(yhat_, kChY, kChY, W16_, H16_);
    ActView t = make_view(l8_.A, kChEncDec, kChEncDec, W8_, H8_);
    add_gemm(s, GEMM_TCONV2X2, yh, t, dec_up_.w, nullptr, 4 * kChEncDec, ACT_NONE, 0, nullptr, nullptr, nullptr);
    t = dcb(s, l8_, t, dec1_[0], true, nullptr, nullptr);
    for (int i = 1; i < 13; ++i) t = dcb(s, l8_, t, dec1_[i], false, (i == 12) ? q_dec_ : nullptr, nullptr);
    const ActView out = make_view(dec_out_, kChSrc, kChSrc, W8_, H8_);
    dcb(s, l8_, t, dec2_, false, nullptr, &out);
}

void IntraCodec::stage_qp(int qp, cudaStream_t stream)
{
    if (qp < 0 || qp >= kQpNum) throw std::runtime_error("qp out of range");
    CK(cudaMemcpyAsync(q_enc_, q_enc_all_ + static_cast<size_t>(qp) * kChEncDec, kChEncDec * 2, cudaMemcpyDeviceToDevice, stream));
    CK(cudaMemcpyAsync(q_dec_, q_dec_all_ + static_cast<size_t>(qp) * kChEncDec, kChEncDec * 2, cudaMemcpyDeviceToDevice, stream));
    CK(cudaMemcpyAsync(q_y_enc_, q_y_enc_all_ + static_cast<size_t>(qp) * kChY, kChY * 2, cudaMemcpyDeviceToDevice, stream));
    CK(cudaMemcpyAsync(q_y_dec_, q_y_dec_all_ + static_cast<size_t>(qp) * kChY, kChY * 2, cudaMemcpyDeviceToDevice, stream));
}

// =============================================================================== compress
void IntraCodec::compress(const void* x, int H, int W, int64_t sc, int64_t sh, int64_t sw, int qp,
                          int pad_b, int pad_r, cudaStream_t stream, const uint8_t** bs,
                          int32_t* bs_len, int32_t* ec_parallel, void* x_hat_out)
{
    CK(cudaSetDevice(device_));
    if ((H + pad_b) % 16 || (W + pad_r) % 16) throw std::runtime_error("padded size must be a multiple of 16");
    plan(H + pad_b, W + pad_r);
    StreamHop hop(this, stream);
    stream = hop.run;
    stage_qp(qp, stream);
    tev_n_ = 0;
    tick(stream);
    // pad + unshuffle (outside the graph: the input pointer changes per call, dmci_proxy.cpp:304-305)
    if (launch_unshuffle8_pad(static_cast<const __half*>(x), 3, H, W, sc, sh, sw,
                              make_view(in8_, kChSrc, kChSrc, W8_, H8_), stream))
        throw std::runtime_error("unshuffle8_pad launch failed");
    ++launches;
    run(enc0_, stream);
    CK(cudaEventRecord(ev_y_, stream));

    // symbols -> host on the copy stream while the synthesis transform runs on `stream`
    CK(cudaStreamWaitEvent(copy_stream_, ev_y_, 0));
    const size_t nz = static_cast<size_t>(H64_) * W64_ * kChZ;
    CK(cudaMemcpyAsync(h_totals_, totals_, 16, cudaMemcpyDeviceToHost, copy_stream_));
    CK(cudaMemcpyAsync(h_z_, z_i8_, nz, cudaMemcpyDeviceToHost, copy_stream_));

    run(enc1_seg_, stream);
    if (launch_shuffle8_clamp(make_view(dec_out_, kChSrc, kChSrc, W8_, H8_),
                              static_cast<__half*>(x_hat_out), 3, 1, stream))
        throw std::runtime_error("shuffle8_clamp launch failed");
    ++launches;
    tock(stream);

    CK(cudaStreamSynchronize(copy_stream_));
    int total = 0;
    for (int k = 0; k < 4; ++k) {
        const int n = h_totals_[k];
        if (n < 0 || static_cast<size_t>(n) > quarter_) throw std::runtime_error("corrupt symbol count");
        total += n;
        if (n) CK(cudaMemcpyAsync(h_sym_[k], sym_c_[k], static_cast<size_t>(n) * 2, cudaMemcpyDeviceToHost, copy_stream_));
    }
    CK(cudaStreamSynchronize(copy_stream_));
    const int n_par = RansCodec::ec_parallel_for(total);
    std::vector<EncodeJob> jobs;
    for (int k = 3; k >= 0; --k) {  // dmci_proxy.cpp:839-841
        EncodeJob j;
        j.kind = EncodeJob::Y; j.y = h_sym_[k]; j.size = h_totals_[k];
        jobs.push_back(j);
    }
    EncodeJob jz;
    jz.kind = EncodeJob::Z; jz.z = h_z_; jz.size = static_cast<int>(nz);
    jz.cdf_offset = qp * kChZ; jz.ch = kChZ;   // dmci_proxy.cpp:843-844
    jobs.push_back(jz);
    rans_.encode(jobs, n_par, bitstream_);
    *bs = bitstream_.data();
    *bs_len = static_cast<int32_t>(bitstream_.size());
    *ec_parallel = n_par;
}

// =============================================================================== estimate
// enc0 writes in8_, y_, the scratch levels, hyper / prior buffers, cat_, yhat_, z_i8_ and the symbol buffers, all of which
// compress() and decompress() rewrite before they read them; x_hat comes from enc1 / dec4, which do not run here.
void IntraCodec::estimate(const void* x, int H, int W, int64_t sc, int64_t sh, int64_t sw, const int32_t* qps, int n_qps,
                          int pad_b, int pad_r, cudaStream_t stream, dcvc_rate_estimate* out)
{
    CK(cudaSetDevice(device_));
    if ((H + pad_b) % 16 || (W + pad_r) % 16) throw std::runtime_error("padded size must be a multiple of 16");
    check_rate_qps(qps, n_qps);
    plan(H + pad_b, W + pad_r);
    StreamHop hop(this, stream);
    stream = hop.run;
    if (launch_unshuffle8_pad(static_cast<const __half*>(x), 3, H, W, sc, sh, sw,
                              make_view(in8_, kChSrc, kChSrc, W8_, H8_), stream))
        throw std::runtime_error("unshuffle8_pad launch failed");
    ++launches;
    const int16_t* ys[4] = { sym_c_[0], sym_c_[1], sym_c_[2], sym_c_[3] };
    const int32_t* counts[4] = { totals_, totals_ + 1, totals_ + 2, totals_ + 3 };
    const int nz = H64_ * W64_ * kChZ;
    for (int i = 0; i < n_qps; ++i) {
        stage_qp(qps[i], stream);
        run(enc0_, stream);
        rate_trial(ys, counts, 4, quarter_, z_i8_, nz, qps[i], i, stream);
    }
    rate_finish(n_qps, stream, out);
}

// =============================================================================== decompress
void IntraCodec::decompress(const uint8_t* bs, int len, int qp, int height, int width,
                            int ec_parallel, cudaStream_t stream, void* x_hat_out)
{
    CK(cudaSetDevice(device_));
    plan(height, width);
    StreamHop hop(this, stream);
    stream = hop.run;
    stage_qp(qp, stream);
    const int zh = (height + 63) / 64, zw = (width + 63) / 64;  // dmci_proxy.cpp:432-433
    if (zh != H64_ || zw != W64_) throw std::runtime_error("z geometry mismatch");
    const int nz = kChZ * zh * zw;
    // DCVC_B200_HOST_TRACE=1: where the host spends a decode (stderr, microseconds) — tools/profile_decode.py
    static const bool host_trace = getenv("DCVC_B200_HOST_TRACE") != nullptr;
    using clk = std::chrono::steady_clock;
    auto us_since = [](clk::time_point t0) { return std::chrono::duration<double, std::micro>(clk::now() - t0).count(); };
    double tr_wait[4] = {}, tr_copy[4] = {}, tr_rans[4] = {};
    int tr_n[4] = {};
    clk::time_point t_all = clk::now(), t0 = t_all;
    rans_.set_stream(bs, len, ec_parallel);
    rans_.decode_z(h_z_, nz, qp * kChZ, kChZ);
    const double tr_z = us_since(t0);
    tev_n_ = 0;
    CK(cudaMemcpyAsync(z_i8_, h_z_, nz, cudaMemcpyHostToDevice, stream));
    for (int k = 0; k < 4; ++k) {
        t0 = clk::now();
        tick(stream);
        run(k == 0 ? dec0_ : dec_step_[k], stream);
        tock(stream);
        // two host waits per step: the count, then exactly that many index bytes.  (Copying the whole index buffer with
        // the count — one wait — was measured on B200: +1.5 % e2e at 1080p for 4 x 0.5 MB of extra D2H traffic; not kept.)
        CK(cudaMemcpyAsync(h_totals_ + k, totals_ + k, 4, cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        tr_wait[k] = us_since(t0);
        const int n = h_totals_[k];
        if (n < 0 || static_cast<size_t>(n) > quarter_) throw std::runtime_error("corrupt index count");
        tr_n[k] = n;
        if (n) {
            t0 = clk::now();
            CK(cudaMemcpyAsync(h_idx_, idx_c_, n, cudaMemcpyDeviceToHost, stream));
            CK(cudaStreamSynchronize(stream));
            tr_copy[k] = us_since(t0);
            t0 = clk::now();
            rans_.decode_y(h_decoded_, h_idx_, n);
            tr_rans[k] = us_since(t0);
            CK(cudaMemcpyAsync(decoded_, h_decoded_, n, cudaMemcpyHostToDevice, stream));
        }
    }
    if (host_trace) {
        fprintf(stderr, "[host trace] intra decode: ec_parallel %d, z %.0f us;", ec_parallel, tr_z);
        for (int k = 0; k < 4; ++k)
            fprintf(stderr, " step %d: launch+gpu+count %.0f, idx d2h %.0f, rANS %.0f (n=%d);", k, tr_wait[k], tr_copy[k], tr_rans[k], tr_n[k]);
        fprintf(stderr, " to last launch %.0f us\n", us_since(t_all));
    }
    tick(stream);
    run(dec4_, stream);
    if (launch_shuffle8_clamp(make_view(dec_out_, kChSrc, kChSrc, W8_, H8_),
                              static_cast<__half*>(x_hat_out), 3, 1, stream))
        throw std::runtime_error("shuffle8_clamp launch failed");
    ++launches;
    tock(stream);
}

int IntraCodec::debug_fetch(const char* name, void* dst, int64_t max_bytes, int64_t* written)
{
    struct Tap { const char* n; const void* p; size_t bytes; };
    const size_t p16 = static_cast<size_t>(H16_) * W16_;
    const Tap taps[] = {
        { "y", y_, p16 * kChY * 2 },
        { "y_hat", yhat_, p16 * kChY * 2 },
        { "params", params_c_, p16 * 512 * 2 },
        { "cat", cat_, p16 * 512 * 2 },
        { "sp_out", sp_out_, p16 * 512 * 2 },
        { "z_i8", z_i8_, static_cast<size_t>(H64_) * W64_ * kChZ },
        { "dec_out", dec_out_, static_cast<size_t>(H8_) * W8_ * kChSrc * 2 },
        { "in8", in8_, static_cast<size_t>(H8_) * W8_ * kChSrc * 2 },
        { "totals", totals_, 16 },
        { "sym0", sym_c_[0], quarter_ * 2 },
        { "sym1", sym_c_[1], quarter_ * 2 },
        { "sym2", sym_c_[2], quarter_ * 2 },
        { "sym3", sym_c_[3], quarter_ * 2 },
    };
    for (const Tap& t : taps) {
        if (strcmp(t.n, name) == 0) {
            if (!t.p) throw std::runtime_error("debug_fetch: buffer not allocated yet");
            const size_t n = std::min<size_t>(t.bytes, static_cast<size_t>(max_bytes));
            CK(cudaDeviceSynchronize());
            CK(cudaMemcpy(dst, t.p, n, cudaMemcpyDeviceToHost));
            *written = static_cast<int64_t>(n);
            return 0;
        }
    }
    throw std::runtime_error(std::string("debug_fetch: unknown buffer '") + name + "'");
}

}  // namespace dcvc

// =================================================================================== C ABI
using dcvc::CodecBase;
using dcvc::IntraCodec;

namespace dcvc {
// codec_hts.cu
CodecBase* make_hts_codec(int device);
CodecBase* make_ld_codec(int device);
int ld_add_ref(CodecBase* c, const void* frame, int H, int W, int64_t sc, int64_t sh, int64_t sw, int apply,
               cudaStream_t stream);
int ld_compress(CodecBase* c, const void* x, int H, int W, int64_t sc, int64_t sh, int64_t sw, int qp, int reset,
                int pad_b, int pad_r, cudaStream_t stream, const uint8_t** bs, int32_t* len, int32_t* ec);
int ld_decompress(CodecBase* c, const uint8_t* bs, int len, int qp, int height, int width, int ec, int reset,
                  cudaStream_t stream, void* const* x_hat_out);
CodecBase* make_htl_codec(int device);
int htl_add_ref(CodecBase* c, const void* frame, int H, int W, int64_t sc, int64_t sh, int64_t sw, int apply,
                cudaStream_t stream);
int htl_compress(CodecBase* c, const void* x, int H, int W, int64_t sc, int64_t sh, int64_t sw, int qp, int reset,
                 int pad_b, int pad_r, cudaStream_t stream, const uint8_t** bs, int32_t* len, int32_t* ec);
int htl_decompress(CodecBase* c, const uint8_t* bs, int len, int qp, int height, int width, int ec, int reset,
                   cudaStream_t stream, void* const* x_hat_out);
int hts_add_ref(CodecBase* c, const void* frame, int H, int W, int64_t sc, int64_t sh, int64_t sw, int apply,
                cudaStream_t stream);
int hts_compress(CodecBase* c, const void* x, int H, int W, int64_t sc, int64_t sh, int64_t sw, int qp, int reset,
                 int pad_b, int pad_r, cudaStream_t stream, const uint8_t** bs, int32_t* len, int32_t* ec);
int hts_decompress(CodecBase* c, const uint8_t* bs, int len, int qp, int height, int width, int ec, int reset,
                   cudaStream_t stream, void* const* x_hat_out);
}  // namespace dcvc

struct dcvc_codec {
    int kind;
    std::unique_ptr<CodecBase> base;
    IntraCodec* intra = nullptr;
    std::string err;
};

namespace dcvc { void set_api_error(const std::string& s); }

#define CODEC_TRY(h) try {
#define CODEC_CATCH(h)                              \
    }                                               \
    catch (const std::exception& e) {               \
        (h)->err = e.what();                        \
        dcvc::set_api_error(e.what());              \
        return 1;                                   \
    }                                               \
    catch (...) {                                   \
        (h)->err = "unknown C++ exception";         \
        dcvc::set_api_error((h)->err);              \
        return 1;                                   \
    }

extern "C" {

int dcvc_create(int32_t kind, int32_t device, dcvc_codec** out)
{
    if (kind != DCVC_KIND_INTRA && kind != DCVC_KIND_HTS && kind != DCVC_KIND_LD && kind != DCVC_KIND_HTL) {
        dcvc::set_api_error("dcvc_create: unknown codec kind");
        return 1;
    }
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) {
        dcvc::set_api_error("dcvc_create: no such CUDA device (this library has no CPU fallback)");
        return 1;
    }
    dcvc_codec* h = new dcvc_codec();
    h->kind = kind;
    if (kind == DCVC_KIND_INTRA) {
        h->intra = new IntraCodec(device);
        h->base.reset(h->intra);
    } else if (kind == DCVC_KIND_LD) {
        h->base.reset(dcvc::make_ld_codec(device));
    } else if (kind == DCVC_KIND_HTL) {
        h->base.reset(dcvc::make_htl_codec(device));
    } else {
        h->base.reset(dcvc::make_hts_codec(device));
    }
    *out = h;
    return 0;
}

int dcvc_destroy(dcvc_codec* h)
{
    delete h;
    return 0;
}

const char* dcvc_codec_error(dcvc_codec* h) { return h ? h->err.c_str() : "null handle"; }

int dcvc_set_param(dcvc_codec* h, const char* name, const void* data, int32_t dtype, int32_t ndim,
                   const int64_t* shape, int32_t on_device)
{
    CODEC_TRY(h)
    h->base->set_param(name, data, dtype, ndim, shape, on_device);
    return 0;
    CODEC_CATCH(h)
}

int dcvc_finalize_params(dcvc_codec* h, float skip_thres)
{
    CODEC_TRY(h)
    h->base->finalize(skip_thres);
    return 0;
    CODEC_CATCH(h)
}

int dcvc_compress(dcvc_codec* h, const void* x, int32_t H, int32_t W, int64_t sc, int64_t sh,
                  int64_t sw, int32_t qp, int32_t pad_b, int32_t pad_r, void* stream,
                  const uint8_t** bit_stream, int32_t* bit_stream_len, int32_t* ec_parallel,
                  void* x_hat_out)
{
    CODEC_TRY(h)
    if (!h->intra) throw std::runtime_error("dcvc_compress is the intra entry point; use dcvc_compress_chunk");
    h->intra->compress(x, H, W, sc, sh, sw, qp, pad_b, pad_r, static_cast<cudaStream_t>(stream),
                       bit_stream, bit_stream_len, ec_parallel, x_hat_out);
    return 0;
    CODEC_CATCH(h)
}

int dcvc_decompress(dcvc_codec* h, const uint8_t* bit_stream, int32_t len, int32_t qp,
                    int32_t height, int32_t width, int32_t ec_parallel, void* stream, void* x_hat_out)
{
    CODEC_TRY(h)
    if (!h->intra) throw std::runtime_error("dcvc_decompress is the intra entry point; use dcvc_decompress_chunk");
    h->intra->decompress(bit_stream, len, qp, height, width, ec_parallel,
                         static_cast<cudaStream_t>(stream), x_hat_out);
    return 0;
    CODEC_CATCH(h)
}

int64_t dcvc_kernel_launches(dcvc_codec* h) { return h->base->launches; }

int dcvc_last_gpu_ms(dcvc_codec* h, float* ms)
{
    CODEC_TRY(h)
    *ms = h->base->gpu_ms();
    return 0;
    CODEC_CATCH(h)
}

int dcvc_profile_enable(dcvc_codec* h, int32_t on)
{
    h->base->profile_ = on != 0;
    if (on) for (auto& a : h->base->prof_) a = dcvc::ProfileAcc();
    return 0;
}

int dcvc_profile_get(dcvc_codec* h, int32_t kind, double* ms, int64_t* launches, double* alg_bytes,
                     double* flops)
{
    if (kind < 0 || kind >= dcvc::OP_KINDS) return 1;
    const dcvc::ProfileAcc& a = h->base->prof_[kind];
    *ms = a.ms; *launches = a.launches; *alg_bytes = a.bytes; *flops = a.flops;
    return 0;
}

int dcvc_add_ref_feature_from_frame(dcvc_codec* h, const void* frame, int32_t H, int32_t W, int64_t sc, int64_t sh,
                                    int64_t sw, int32_t apply_adaptor, void* stream)
{
    CODEC_TRY(h)
    if (h->kind == DCVC_KIND_LD)
        return dcvc::ld_add_ref(h->base.get(), frame, H, W, sc, sh, sw, apply_adaptor, static_cast<cudaStream_t>(stream));
    if (h->kind == DCVC_KIND_HTL)
        return dcvc::htl_add_ref(h->base.get(), frame, H, W, sc, sh, sw, apply_adaptor, static_cast<cudaStream_t>(stream));
    if (h->kind != DCVC_KIND_HTS) throw std::runtime_error("add_ref_feature_from_frame needs a video codec handle");
    return dcvc::hts_add_ref(h->base.get(), frame, H, W, sc, sh, sw, apply_adaptor, static_cast<cudaStream_t>(stream));
    CODEC_CATCH(h)
}

int dcvc_compress_chunk(dcvc_codec* h, const void* x, int32_t H, int32_t W, int64_t sc, int64_t sh, int64_t sw,
                        int32_t qp, int32_t reset_feature_memory, int32_t pad_b, int32_t pad_r, void* stream,
                        const uint8_t** bit_stream, int32_t* bit_stream_len, int32_t* ec_parallel)
{
    CODEC_TRY(h)
    if (h->kind == DCVC_KIND_LD)
        return dcvc::ld_compress(h->base.get(), x, H, W, sc, sh, sw, qp, reset_feature_memory, pad_b, pad_r,
                                 static_cast<cudaStream_t>(stream), bit_stream, bit_stream_len, ec_parallel);
    if (h->kind == DCVC_KIND_HTL)
        return dcvc::htl_compress(h->base.get(), x, H, W, sc, sh, sw, qp, reset_feature_memory, pad_b, pad_r,
                                  static_cast<cudaStream_t>(stream), bit_stream, bit_stream_len, ec_parallel);
    if (h->kind != DCVC_KIND_HTS) throw std::runtime_error("compress_chunk needs a video codec handle");
    return dcvc::hts_compress(h->base.get(), x, H, W, sc, sh, sw, qp, reset_feature_memory, pad_b, pad_r,
                              static_cast<cudaStream_t>(stream), bit_stream, bit_stream_len, ec_parallel);
    CODEC_CATCH(h)
}

int dcvc_decompress_chunk(dcvc_codec* h, const uint8_t* bit_stream, int32_t len, int32_t qp, int32_t height,
                          int32_t width, int32_t ec_parallel, int32_t reset_feature_memory, void* stream,
                          void* const* x_hat_out)
{
    CODEC_TRY(h)
    if (h->kind == DCVC_KIND_LD)
        return dcvc::ld_decompress(h->base.get(), bit_stream, len, qp, height, width, ec_parallel, reset_feature_memory,
                                   static_cast<cudaStream_t>(stream), x_hat_out);
    if (h->kind == DCVC_KIND_HTL)
        return dcvc::htl_decompress(h->base.get(), bit_stream, len, qp, height, width, ec_parallel, reset_feature_memory,
                                    static_cast<cudaStream_t>(stream), x_hat_out);
    if (h->kind != DCVC_KIND_HTS) throw std::runtime_error("decompress_chunk needs a video codec handle");
    return dcvc::hts_decompress(h->base.get(), bit_stream, len, qp, height, width, ec_parallel, reset_feature_memory,
                                static_cast<cudaStream_t>(stream), x_hat_out);
    CODEC_CATCH(h)
}

int dcvc_estimate_bits(dcvc_codec* h, const void* x, int32_t H, int32_t W, int64_t sc, int64_t sh, int64_t sw,
                       const int32_t* qps, int32_t n_qps, int32_t reset_feature_memory, int32_t pad_b, int32_t pad_r,
                       void* stream, dcvc_rate_estimate* out)
{
    CODEC_TRY(h)
    (void)reset_feature_memory;   // selects the memory update after the unit, which the estimate does not run
    h->base->estimate(x, H, W, sc, sh, sw, qps, n_qps, pad_b, pad_r, static_cast<cudaStream_t>(stream), out);
    return 0;
    CODEC_CATCH(h)
}

int dcvc_debug_fetch(dcvc_codec* h, const char* name, void* host_dst, int64_t max_bytes,
                     int64_t* bytes_written)
{
    CODEC_TRY(h)
    if (strcmp(name, "arena_overflow_blocks") == 0) {
        // how many times the activation arena had to grow beyond the plan's estimate (0 when the estimate is right)
        if (max_bytes < 4) throw std::runtime_error("debug_fetch: buffer too small");
        const int32_t n = h->base->arena_overflow_blocks();
        memcpy(host_dst, &n, 4);
        *bytes_written = 4;
        return 0;
    }
    return h->base->debug_fetch(name, host_dst, max_bytes, bytes_written);
    CODEC_CATCH(h)
}

}  // extern "C"
