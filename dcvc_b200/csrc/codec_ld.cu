// codec_ld.cu — DCVC-UF low-delay codec (one frame per call) behind the C ABI.
//
// B200-native counterpart of src/layers/extensions/inference/dmc_ld_proxy.{h,cpp}: same state machine (reference
// feature -> feature memory -> context + temporal prior; the encoder updates them at the end of compress(), the
// decoder lazily at the start of the next decompress(), dmc_ld_proxy.cpp:468-472, 512-516, 639-658), one symbol
// stream per frame (:444-453, 541-544), means-only refinement over the two checkerboard masks of
// common_model.py:157-172 (:444-449 encoder, :579-581 decoder).  Networks: src/models/video_model_ld.py:24-211.
// Same building blocks as the HT-S codec (codec_hts.cu): every GEMM runs through pw_gemm, QP-dependent scale vectors
// are staged so one CUDA graph per segment serves all 64 QPs.
#include "codec_common.cuh"

namespace dcvc {

namespace {
constexpr int kSrc = 192, kY = 128, kZ = 128, kD = 256, kM = 256;  // video_model_ld.py:16-21
constexpr int kP = 3 * kY;                                          // prior-fusion width: (q_dec | scales | means)
constexpr int kCatSp = kY + kP;                                     // spatial-prior input: y_hat_0 | common params
}  // namespace

class LdCodec : public CodecBase {
public:
    explicit LdCodec(int device) : CodecBase(device) {}
    ~LdCodec() override { clear_plan(); }

    void finalize(float skip_thres) override;
    int debug_fetch(const char* name, void* dst, int64_t max_bytes, int64_t* written) override;
    int arena_overflow_blocks() const override { return arena_.overflow_blocks(); }

    void add_ref(const void* frame, int H, int W, int64_t sc, int64_t sh, int64_t sw, int apply, cudaStream_t stream);
    void compress(const void* x, int H, int W, int64_t sc, int64_t sh, int64_t sw, int qp, int reset, int pad_b,
                  int pad_r, cudaStream_t stream, const uint8_t** bs, int32_t* len, int32_t* ec);
    void decompress(const uint8_t* bs, int len, int qp, int height, int width, int ec, int reset,
                    cudaStream_t stream, void* const* x_hat_out);
    void estimate(const void* x, int H, int W, int64_t sc, int64_t sh, int64_t sw, const int32_t* qps, int n_qps,
                  int pad_b, int pad_r, cudaStream_t stream, dcvc_rate_estimate* out) override;

private:
    void plan(int height, int width);
    void clear_plan();
    void stage_qp(int qp, cudaStream_t stream);
    ActView chain(Segment& s, Level& L, ActView in, const DcbW* blocks, int n, const __half* q_last, const ActView* out);

    // weights
    DcbW fa_i_[4], fa_m_[4], fe_[5], enc_[3], henc0_, henc1_, henc2_, hdec0_, hdec1_, hdec2_, tpe_, pf_[3], sp_[2],
        dec_[3], rh_[3];
    ConvW enc_down_, henc1_down_, henc2_down_, hdec0_up_, hdec1_up_, tpe_down_, pf3_, sp2_, dec_up_, dec_out_, rh_out_;
    const __half *q_encoder_all_ = nullptr, *q_decoder_all_ = nullptr, *q_feature_all_ = nullptr;

    // plan
    int H8_ = 0, W8_ = 0, H16_ = 0, W16_ = 0, H16p_ = 0, W16p_ = 0, H64_ = 0, W64_ = 0;
    Arena arena_;
    Level l8_, l16_, l32_, l64_;
    __half *cat8_ = nullptr, *cat_fam_ = nullptr, *feature_i_ = nullptr;
    __half *y_ = nullptr, *ypad_ = nullptr, *hyp_p_ = nullptr, *cat_pf_ = nullptr, *cat_sp_ = nullptr, *temporal_raw_ = nullptr,
           *means_ = nullptr, *yhat_ = nullptr, *zhat_ = nullptr;
    int8_t *z_i8_ = nullptr, *yq_ = nullptr, *decoded_ = nullptr;
    __half *q_enc_ = nullptr, *q_dec_ = nullptr, *q_feat_ = nullptr;
    int16_t *sym_raw_ = nullptr, *sym_c_ = nullptr;
    uint8_t *idx_raw_ = nullptr, *idx_c_ = nullptr;
    int32_t *counts_ = nullptr, *offsets_ = nullptr, *total_ = nullptr;
    int32_t* h_total_ = nullptr;
    int16_t* h_sym_ = nullptr;
    uint8_t* h_idx_ = nullptr;
    int8_t *h_decoded_ = nullptr, *h_z_ = nullptr;
    size_t n_lat_ = 0;
    bool memory_has_value_ = false;

    Segment s_enc0_, s_decoder_, s_reset_head_, s_fa_i_, s_fa_m_, s_fe_, s_temporal_, s_dec1_, s_dec3_, s_recon_;
};

// =============================================================================== parameters
void LdCodec::finalize(float skip_thres)
{
    finalize_begin(skip_thres);
    clear_plan();
    auto dcbs = [&](DcbW* dst, const std::string& prefix, int n) {
        for (int i = 0; i < n; ++i) dst[i] = load_dcb(prefix + std::to_string(i) + ".");
    };
    dcbs(fa_i_, "feature_adaptor_i.conv.", 4);
    dcbs(fa_m_, "feature_adaptor_m.conv.", 4);
    dcbs(fe_, "feature_extractor.conv.", 5);
    dcbs(enc_, "encoder.conv1.", 2);
    enc_[2] = load_dcb("encoder.conv2.");
    enc_down_ = load_conv("encoder.down.", DCVC_GEMM_CONV3X3_S2);
    henc0_ = load_dcb("hyper_encoder.conv.0.");
    henc1_down_ = load_conv("hyper_encoder.conv.1.down.", DCVC_GEMM_CONV2X2_S2);
    henc1_ = load_dcb("hyper_encoder.conv.1.conv.");
    henc2_down_ = load_conv("hyper_encoder.conv.2.down.", DCVC_GEMM_CONV2X2_S2);
    henc2_ = load_dcb("hyper_encoder.conv.2.conv.");
    hdec0_up_ = load_conv("hyper_decoder.conv.0.up.conv.0.", DCVC_GEMM_TCONV2X2);
    hdec0_ = load_dcb("hyper_decoder.conv.0.conv.");
    hdec1_up_ = load_conv("hyper_decoder.conv.1.up.conv.0.", DCVC_GEMM_TCONV2X2);
    hdec1_ = load_dcb("hyper_decoder.conv.1.conv.");
    hdec2_ = load_dcb("hyper_decoder.conv.2.");
    tpe_down_ = load_conv("temporal_prior_encoder.conv.down.", DCVC_GEMM_CONV2X2_S2);
    tpe_ = load_dcb("temporal_prior_encoder.conv.conv.");
    dcbs(pf_, "y_prior_fusion.conv.", 3);
    pf3_ = load_conv("y_prior_fusion.conv.3.", DCVC_GEMM_PW);
    dcbs(sp_, "y_spatial_prior.conv.", 2);
    sp2_ = load_conv("y_spatial_prior.conv.2.", DCVC_GEMM_PW);
    dec_up_ = load_conv("decoder.up.conv.0.", DCVC_GEMM_TCONV2X2);
    dcbs(dec_, "decoder.conv1.", 3);
    dec_out_ = load_conv("decoder.conv2.", DCVC_GEMM_PW);
    dcbs(rh_, "recon_head.conv.", 3);
    rh_out_ = load_conv("recon_head.head.", DCVC_GEMM_PW);
    q_encoder_all_ = upload_param("q_encoder");
    q_decoder_all_ = upload_param("q_decoder");
    q_feature_all_ = upload_param("q_feature");
    finalize_end();
}

// =============================================================================== plan
void LdCodec::clear_plan()
{
    Segment* segs[] = { &s_enc0_, &s_decoder_, &s_reset_head_, &s_fa_i_, &s_fa_m_, &s_fe_, &s_temporal_, &s_dec1_, &s_dec3_, &s_recon_ };
    for (Segment* s : segs) s->reset();
    if (h_total_) { cudaFreeHost(h_total_); h_total_ = nullptr; }
    if (h_sym_) { cudaFreeHost(h_sym_); h_sym_ = nullptr; }
    if (h_idx_) { cudaFreeHost(h_idx_); h_idx_ = nullptr; }
    if (h_decoded_) { cudaFreeHost(h_decoded_); h_decoded_ = nullptr; }
    if (h_z_) { cudaFreeHost(h_z_); h_z_ = nullptr; }
    arena_.release();
    H8_ = W8_ = 0;
    memory_has_value_ = false;
}

ActView LdCodec::chain(Segment& s, Level& L, ActView in, const DcbW* blocks, int n, const __half* q_last, const ActView* out)
{
    // n DepthConvBlocks in sequence; the first may take an external input (then it lands in L.B unless it has an
    // adaptor), the last is redirected to `out` when given and carries the fused per-channel quant scale.
    ActView t = in;
    for (int i = 0; i < n; ++i) {
        const bool last = (i == n - 1);
        const bool external = (t.ptr != L.A && t.ptr != L.B);
        ActView first_out = make_view(L.B, blocks[i].c, blocks[i].c, t.W, t.H);
        const ActView* o = last ? out : nullptr;
        if (!o && external && !blocks[i].adaptor) o = &first_out;
        t = dcb(s, L, t, blocks[i], false, last ? q_last : nullptr, o);
    }
    return t;
}

void LdCodec::plan(int height, int width)
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
    const size_t p8 = static_cast<size_t>(H8) * W8, p16 = static_cast<size_t>(H16_) * W16_;
    const size_t p16p = static_cast<size_t>(H16p_) * W16p_, p32 = static_cast<size_t>(H32) * W32;
    const size_t p64 = static_cast<size_t>(H64_) * W64_;
    n_lat_ = p16 * kY;
    const bool padded = (H16p_ != H16_) || (W16p_ != W16_);

    size_t bytes = p8 * 2 * (512 + 512 + kSrc + 4 * kD);
    bytes += p16p * 2 * (4 * kP + 2 * kY + kP + kCatSp + 2 * kY + 3 * kY);
    bytes += p32 * 2 * 4 * kY + p64 * 2 * 4 * kY + p64 * kZ * 3;
    bytes += n_lat_ * (1 + 2 + 2 + 1 + 1 + 1) + p16 * 8 + (2u << 20) + 64 * 4096;
    arena_.reserve(bytes);
    dbg_base_ = arena_.base();
    dbg_bytes_ = bytes;

    cat8_ = arena_.halves(p8 * 512);
    cat_fam_ = arena_.halves(p8 * 512);
    feature_i_ = arena_.halves(p8 * kSrc);
    l8_.H = H8; l8_.W = W8;
    l8_.A = arena_.halves(p8 * kD); l8_.B = arena_.halves(p8 * kD);
    l8_.T1 = arena_.halves(p8 * kD); l8_.T2 = arena_.halves(p8 * kD);
    l16_.H = H16p_; l16_.W = W16p_;
    l16_.A = arena_.halves(p16p * kP); l16_.B = arena_.halves(p16p * kP);
    l16_.T1 = arena_.halves(p16p * kP); l16_.T2 = arena_.halves(p16p * kP);
    l32_.H = H32; l32_.W = W32;
    l32_.A = arena_.halves(p32 * kY); l32_.B = arena_.halves(p32 * kY);
    l32_.T1 = arena_.halves(p32 * kY); l32_.T2 = arena_.halves(p32 * kY);
    l64_.H = H64_; l64_.W = W64_;
    l64_.A = arena_.halves(p64 * kY); l64_.B = arena_.halves(p64 * kY);
    l64_.T1 = arena_.halves(p64 * kY); l64_.T2 = arena_.halves(p64 * kY);
    y_ = arena_.halves(p16 * kY);
    ypad_ = padded ? arena_.halves(p16p * kY) : y_;
    cat_pf_ = arena_.halves(p16 * kP);
    hyp_p_ = padded ? arena_.halves(p16p * kY) : nullptr;
    cat_sp_ = arena_.halves(p16 * kCatSp);
    temporal_raw_ = arena_.halves(p16 * 2 * kY);
    means_ = arena_.halves(p16 * kY);
    yhat_ = arena_.halves(p16 * kY);
    zhat_ = arena_.halves(p64 * kZ);
    z_i8_ = static_cast<int8_t*>(arena_.alloc(p64 * kZ));
    yq_ = static_cast<int8_t*>(arena_.alloc(n_lat_));
    decoded_ = static_cast<int8_t*>(arena_.alloc(n_lat_));
    sym_raw_ = static_cast<int16_t*>(arena_.alloc(n_lat_ * 2));
    sym_c_ = static_cast<int16_t*>(arena_.alloc(n_lat_ * 2));
    idx_raw_ = static_cast<uint8_t*>(arena_.alloc(n_lat_));
    idx_c_ = static_cast<uint8_t*>(arena_.alloc(n_lat_));
    counts_ = static_cast<int32_t*>(arena_.alloc(p16 * 4));
    offsets_ = static_cast<int32_t*>(arena_.alloc((p16 + 1) * 4));
    total_ = static_cast<int32_t*>(arena_.alloc(64));
    q_enc_ = arena_.halves(kD); q_dec_ = arena_.halves(kD); q_feat_ = arena_.halves(2 * kY);
    CK(cudaMallocHost(&h_total_, 64));
    CK(cudaMallocHost(&h_sym_, n_lat_ * 2));
    CK(cudaMallocHost(&h_idx_, n_lat_));
    CK(cudaMallocHost(&h_decoded_, n_lat_));
    CK(cudaMallocHost(&h_z_, p64 * kZ));

    // "cat" buffers.  cat8_ = [up(y_hat) 256 | ctx 256] is the decoder's input; the encoder's input [x 192 | ctx 256]
    // is the view that starts 64 channels in (x overlaps the part of `up` the decoder writes later).
    const ActView v_cat_dec = make_view(cat8_, 512, 512, W8, H8);
    const ActView v_up_out = make_view(cat8_, kD, 512, W8, H8);
    const ActView v_ctx = make_view(cat8_ + kD, kM, 512, W8, H8);
    const ActView v_cat_enc = make_view(cat8_ + 64, kSrc + kM, 512, W8, H8);
    const ActView v_cat_fam = make_view(cat_fam_, 512, 512, W8, H8);
    const ActView v_memory = make_view(cat_fam_, kM, 512, W8, H8);
    const ActView v_feature_p = make_view(cat_fam_ + kM, kD, 512, W8, H8);
    const ActView v_feature_i = make_view(feature_i_, kSrc, kSrc, W8, H8);
    const ActView v_y = make_view(y_, kY, kY, W16_, H16_);
    const ActView v_ypad = make_view(ypad_, kY, kY, W16p_, H16p_);
    const ActView v_hyper = make_view(cat_pf_, kY, kP, W16_, H16_);
    const ActView v_temporal = make_view(cat_pf_ + kY, 2 * kY, kP, W16_, H16_);
    const ActView v_temporal_raw = make_view(temporal_raw_, 2 * kY, 2 * kY, W16_, H16_);
    const ActView v_cat_pf = make_view(cat_pf_, kP, kP, W16_, H16_);
    const ActView v_cat_sp = make_view(cat_sp_, kCatSp, kCatSp, W16_, H16_);
    const ActView v_acc = make_view(cat_sp_, kY, kCatSp, W16_, H16_);
    const ActView v_common = make_view(cat_sp_ + kY, kP, kCatSp, W16_, H16_);
    const ActView v_qdec = make_view(cat_sp_ + kY, kY, kCatSp, W16_, H16_);
    const ActView v_means1 = make_view(means_, kY, kY, W16_, H16_);
    const ActView v_yhat = make_view(yhat_, kY, kY, W16_, H16_);
    const int npix16 = static_cast<int>(p16);

    auto step_args = [&](int k) {
        EntropyStepArgs a;
        a.H = H16_; a.W = W16_; a.G = kY / 2; a.ng = 2; a.step = k;
        a.scales = cat_sp_ + 2 * kY; a.p_pitch = kCatSp;
        if (k == 0) { a.means = cat_sp_ + 3 * kY; a.m_pitch = kCatSp; } else { a.means = means_; a.m_pitch = kY; }
        a.y_hat_acc = cat_sp_; a.acc_pitch = kCatSp;
        a.skip_thres = skip_thres_; a.scale_lut = lut_;
        a.yq_dense = yq_;
        return a;
    };
    auto full_args = [&]() {
        EntropyStepArgs a;
        a.H = H16_; a.W = W16_; a.G = kY; a.step = 0; a.full = 1;
        a.scales = cat_sp_ + 2 * kY; a.p_pitch = kCatSp;
        a.skip_thres = skip_thres_; a.scale_lut = lut_;
        a.yq_dense = yq_; a.sym_raw = sym_raw_; a.idx_raw = idx_raw_; a.counts = counts_;
        return a;
    };
    // z_hat -> hyper params (cropped) into cat_pf[0:128]; temporal params * q_feature into cat_pf[128:384];
    // prior fusion -> (q_dec | scales | means) inside the spatial prior's cat buffer  (dmc_ld_proxy.cpp:436-442, 529-538)
    auto build_params = [&](Segment& s) {
        ActView u32 = make_view(l32_.A, kY, kY, W32, H32);
        add_gemm(s, GEMM_TCONV2X2, make_view(zhat_, kZ, kZ, W64_, H64_), u32, hdec0_up_.w, nullptr, 4 * kY, ACT_NONE, 0, nullptr, nullptr, nullptr);
        u32 = dcb(s, l32_, u32, hdec0_, false, nullptr, nullptr);
        ActView u16 = make_view(l16_.A, kY, kY, W16p_, H16p_);
        add_gemm(s, GEMM_TCONV2X2, u32, u16, hdec1_up_.w, nullptr, 4 * kY, ACT_NONE, 0, nullptr, nullptr, nullptr);
        u16 = dcb(s, l16_, u16, hdec1_, false, nullptr, nullptr);
        if (padded) {
            const ActView hp = make_view(hyp_p_, kY, kY, W16p_, H16p_);
            dcb(s, l16_, u16, hdec2_, false, nullptr, &hp);
            s.elem([hp, v_hyper](cudaStream_t st) { return launch_pad_crop(hp, v_hyper, st); });
        } else {
            dcb(s, l16_, u16, hdec2_, false, nullptr, &v_hyper);
        }
        const __half* qf = q_feat_;
        s.elem([v_temporal_raw, qf, v_temporal](cudaStream_t st) { return launch_scale_channels(v_temporal_raw, qf, v_temporal, st); });
        Level L = l16_;
        ActView t = chain(s, L, v_cat_pf, pf_, 3, nullptr, nullptr);
        conv1x1(s, t, v_common, pf3_);
    };
    auto build_spatial_prior = [&](Segment& s) {
        // SpatialPrior(cat(y_hat_0, common)) -> means of the second step  (dmc_ld_proxy.cpp:447, 580)
        Level L = l16_;
        ActView t = chain(s, L, v_cat_sp, sp_, 2, nullptr, nullptr);
        conv1x1(s, t, v_means1, sp2_);
    };

    // ------------------------------------------------------------------ feature memory / context / temporal prior
    chain(s_fa_i_, l8_, v_feature_i, fa_i_, 4, nullptr, &v_memory);
    chain(s_fa_m_, l8_, v_cat_fam, fa_m_, 4, nullptr, &v_memory);
    chain(s_fe_, l8_, v_memory, fe_, 5, nullptr, &v_ctx);
    {
        // TemporalPriorEncoder(memory): 2x2/s2 + block -> temporal_raw (q_feature is applied where it is consumed)
        Segment& s = s_temporal_;
        Level L = l16_;
        ActView d = make_view(L.A, 2 * kY, 2 * kY, W16_, H16_);
        add_gemm(s, GEMM_CONV2X2_S2, v_memory, d, tpe_down_.w, tpe_down_.b, 2 * kY, ACT_NONE, 0, nullptr, nullptr, nullptr);
        dcb(s, L, d, tpe_, false, nullptr, &v_temporal_raw);
    }

    // ------------------------------------------------------------------ enc_0 (dmc_ld_proxy.cpp:431-454)
    {
        Segment& s = s_enc0_;
        ActView t = chain(s, l8_, v_cat_enc, enc_, 3, q_enc_, nullptr);
        add_gemm(s, GEMM_CONV3X3_S2, t, v_y, enc_down_.w, enc_down_.b, kY, ACT_NONE, 0, nullptr, nullptr, nullptr);
        if (padded) s.elem([v_y, v_ypad](cudaStream_t st) { return launch_pad_crop(v_y, v_ypad, st); });
        Level L16 = l16_;
        ActView h = chain(s, L16, v_ypad, &henc0_, 1, nullptr, nullptr);
        ActView d32 = make_view(l32_.A, kY, kY, W32, H32);
        add_gemm(s, GEMM_CONV2X2_S2, h, d32, henc1_down_.w, henc1_down_.b, kY, ACT_NONE, 0, nullptr, nullptr, nullptr);
        d32 = dcb(s, l32_, d32, henc1_, false, nullptr, nullptr);
        ActView d64 = make_view(l64_.A, kZ, kZ, W64_, H64_);
        add_gemm(s, GEMM_CONV2X2_S2, d32, d64, henc2_down_.w, henc2_down_.b, kZ, ACT_NONE, 0, nullptr, nullptr, nullptr);
        d64 = dcb(s, l64_, d64, henc2_, false, nullptr, nullptr);
        {
            const __half* z = static_cast<const __half*>(d64.ptr);
            __half* zh = zhat_;
            int8_t* zi = z_i8_;
            const long long n = static_cast<long long>(p64) * kZ;
            s.elem([z, zh, zi, n](cudaStream_t st) { return launch_round_z(z, zh, zi, n, st); });
        }
        build_params(s);
        for (int k = 0; k < 2; ++k) {
            if (k > 0) build_spatial_prior(s);
            EntropyStepArgs a = step_args(k);
            a.y = y_; a.y_pitch = kY;
            a.q_div = cat_sp_ + kY; a.q_pitch = kCatSp;
            s.elem([a](cudaStream_t st) { return launch_entropy_enc_step(a, st); });
        }
        s.elem([v_acc, v_qdec, v_yhat](cudaStream_t st) { return launch_mul_clamp_min(v_acc, v_qdec, v_yhat, st); });
        const EntropyStepArgs f = full_args();
        int32_t* offs = offsets_;
        int32_t* tot = total_;
        int16_t* dst = sym_c_;
        s.elem([f](cudaStream_t st) { return launch_entropy_build_symbols_full(f, st); });
        s.elem([f, offs, tot, npix16](cudaStream_t st) { return launch_scan_counts(f.counts, offs, tot, npix16, st); });
        s.elem([f, offs, dst](cudaStream_t st) { return launch_compact_i16(f, offs, dst, st); });
    }
    // ------------------------------------------------------------------ synthesis: y_hat -> feature_p (Decoder, :35-40)
    {
        Segment& s = s_decoder_;
        add_gemm(s, GEMM_TCONV2X2, v_yhat, v_up_out, dec_up_.w, nullptr, 4 * kD, ACT_NONE, 0, nullptr, nullptr, nullptr);
        ActView t = chain(s, l8_, v_cat_dec, dec_, 3, nullptr, nullptr);
        add_gemm(s, GEMM_PW, t, v_feature_p, dec_out_.w, dec_out_.b, kD, ACT_NONE, 0, nullptr, nullptr, q_dec_);
    }
    // recon head without the shuffle -> feature_i: the reset reference (encoder) and every decoded frame's head output
    auto build_head = [&](Segment& s) {
        ActView t = chain(s, l8_, v_feature_p, rh_, 3, nullptr, nullptr);
        conv1x1(s, t, v_feature_i, rh_out_);
    };
    build_head(s_reset_head_);
    build_head(s_recon_);
    // ------------------------------------------------------------------ decoder segments
    {
        Segment& s = s_dec1_;  // dmc_ld_proxy.cpp:527-545
        const int8_t* zi = z_i8_;
        __half* zh = zhat_;
        const long long n = static_cast<long long>(p64) * kZ;
        s.elem([zi, zh, n](cudaStream_t st) { return launch_int8_to_half(zi, zh, n, st); });
        build_params(s);
        const EntropyStepArgs f = full_args();
        int32_t* offs = offsets_;
        int32_t* tot = total_;
        uint8_t* dst = idx_c_;
        s.elem([f](cudaStream_t st) { return launch_entropy_dec_index(f, st); });
        s.elem([f, offs, tot, npix16](cudaStream_t st) { return launch_scan_counts(f.counts, offs, tot, npix16, st); });
        s.elem([f, offs, dst](cudaStream_t st) { return launch_compact_u8(f, offs, dst, st); });
    }
    {
        Segment& s = s_dec3_;  // dmc_ld_proxy.cpp:575-582 up to y_hat
        const EntropyStepArgs f = full_args();
        const int32_t* offs = offsets_;
        const int8_t* dec = decoded_;
        s.elem([f, offs, dec](cudaStream_t st) { return launch_entropy_recover_dense(f, offs, dec, st); });
        for (int k = 0; k < 2; ++k) {
            if (k > 0) build_spatial_prior(s);
            const EntropyStepArgs a = step_args(k);
            s.elem([a](cudaStream_t st) { return launch_entropy_restore_dense(a, st); });
        }
        s.elem([v_acc, v_qdec, v_yhat](cudaStream_t st) { return launch_mul_clamp_min(v_acc, v_qdec, v_yhat, st); });
    }
    Segment* segs[] = { &s_enc0_, &s_decoder_, &s_reset_head_, &s_fa_i_, &s_fa_m_, &s_fe_, &s_temporal_, &s_dec1_, &s_dec3_, &s_recon_ };
    for (Segment* s : segs) s->seal();
}

void LdCodec::stage_qp(int qp, cudaStream_t stream)
{
    if (qp < 0 || qp >= kQpNum) throw std::runtime_error("qp out of range");
    CK(cudaMemcpyAsync(q_enc_, q_encoder_all_ + static_cast<size_t>(qp) * kD, kD * 2, cudaMemcpyDeviceToDevice, stream));
    CK(cudaMemcpyAsync(q_dec_, q_decoder_all_ + static_cast<size_t>(qp) * kD, kD * 2, cudaMemcpyDeviceToDevice, stream));
    CK(cudaMemcpyAsync(q_feat_, q_feature_all_ + static_cast<size_t>(qp) * 2 * kY, 2 * kY * 2, cudaMemcpyDeviceToDevice, stream));
}

// =============================================================================== reference feature
void LdCodec::add_ref(const void* frame, int H, int W, int64_t sc, int64_t sh, int64_t sw, int apply, cudaStream_t stream)
{
    CK(cudaSetDevice(device_));
    plan(H, W);
    StreamHop hop(this, stream);
    stream = hop.run;
    // feature_i = pixel_unshuffle(frame, 8)   (dmc_ld_proxy.cpp:409-411; the frame is the padded reconstruction)
    if (launch_unshuffle8_pad(static_cast<const __half*>(frame), 3, H, W, sc, sh, sw, make_view(feature_i_, kSrc, kSrc, W8_, H8_), stream))
        throw std::runtime_error("unshuffle8 launch failed");
    ++launches;
    if (apply) {
        run(s_fa_i_, stream);
        run(s_fe_, stream);
        run(s_temporal_, stream);
    }
    memory_has_value_ = apply != 0;
}

// =============================================================================== compress
void LdCodec::compress(const void* x, int H, int W, int64_t sc, int64_t sh, int64_t sw, int qp, int reset, int pad_b,
                       int pad_r, cudaStream_t stream, const uint8_t** bs, int32_t* len, int32_t* ec)
{
    CK(cudaSetDevice(device_));
    if ((H + pad_b) % 16 || (W + pad_r) % 16) throw std::runtime_error("padded size must be a multiple of 16");
    plan(H + pad_b, W + pad_r);
    StreamHop hop(this, stream);
    stream = hop.run;
    stage_qp(qp, stream);
    tev_n_ = 0;
    tick(stream);
    if (launch_unshuffle8_pad(static_cast<const __half*>(x), 3, H, W, sc, sh, sw, make_view(cat8_ + 64, kSrc, 512, W8_, H8_), stream))
        throw std::runtime_error("unshuffle8_pad launch failed");
    ++launches;
    run(s_enc0_, stream);
    CK(cudaEventRecord(ev_y_, stream));
    CK(cudaStreamWaitEvent(copy_stream_, ev_y_, 0));
    const size_t nz = static_cast<size_t>(H64_) * W64_ * kZ;
    CK(cudaMemcpyAsync(h_total_, total_, 4, cudaMemcpyDeviceToHost, copy_stream_));
    CK(cudaMemcpyAsync(h_z_, z_i8_, nz, cudaMemcpyDeviceToHost, copy_stream_));

    // enc_1: synthesis + memory / context / temporal prior of the NEXT frame (dmc_ld_proxy.cpp:468-472, 639-649)
    run(s_decoder_, stream);
    if (reset) {
        run(s_reset_head_, stream);
        run(s_fa_i_, stream);
    } else {
        run(s_fa_m_, stream);
    }
    run(s_fe_, stream);
    run(s_temporal_, stream);
    tock(stream);

    CK(cudaStreamSynchronize(copy_stream_));
    const int n = h_total_[0];
    if (n < 0 || static_cast<size_t>(n) > n_lat_) throw std::runtime_error("corrupt symbol count");
    if (n) CK(cudaMemcpyAsync(h_sym_, sym_c_, static_cast<size_t>(n) * 2, cudaMemcpyDeviceToHost, copy_stream_));
    CK(cudaStreamSynchronize(copy_stream_));
    const int n_par = RansCodec::ec_parallel_for(n);
    std::vector<EncodeJob> jobs(2);
    jobs[0].kind = EncodeJob::Y; jobs[0].y = h_sym_; jobs[0].size = n;
    jobs[1].kind = EncodeJob::Z; jobs[1].z = h_z_; jobs[1].size = static_cast<int>(nz);
    jobs[1].cdf_offset = qp * kZ; jobs[1].ch = kZ;
    rans_.encode(jobs, n_par, bitstream_);
    *bs = bitstream_.data();
    *len = static_cast<int32_t>(bitstream_.size());
    *ec = n_par;
}

// =============================================================================== estimate
// The unshuffle writes channels 64..256 of cat8_ (the part of `up` the decoder rewrites; the context is 256..512), and
// enc0 reads the temporal prior without writing it; everything else enc0 writes, compress() and decompress() rewrite
// before they read.  So the state the next frame is coded from is untouched.
void LdCodec::estimate(const void* x, int H, int W, int64_t sc, int64_t sh, int64_t sw, const int32_t* qps, int n_qps,
                       int pad_b, int pad_r, cudaStream_t stream, dcvc_rate_estimate* out)
{
    CK(cudaSetDevice(device_));
    if ((H + pad_b) % 16 || (W + pad_r) % 16) throw std::runtime_error("padded size must be a multiple of 16");
    check_rate_qps(qps, n_qps);
    plan(H + pad_b, W + pad_r);
    StreamHop hop(this, stream);
    stream = hop.run;
    if (launch_unshuffle8_pad(static_cast<const __half*>(x), 3, H, W, sc, sh, sw, make_view(cat8_ + 64, kSrc, 512, W8_, H8_), stream))
        throw std::runtime_error("unshuffle8_pad launch failed");
    ++launches;
    const int16_t* ys[1] = { sym_c_ };
    const int32_t* counts[1] = { total_ };
    const int nz = H64_ * W64_ * kZ;
    for (int i = 0; i < n_qps; ++i) {
        stage_qp(qps[i], stream);
        run(s_enc0_, stream);
        rate_trial(ys, counts, 1, n_lat_, z_i8_, nz, qps[i], i, stream);
    }
    rate_finish(n_qps, stream, out);
}

// =============================================================================== decompress
void LdCodec::decompress(const uint8_t* bs, int len, int qp, int height, int width, int ec, int reset,
                         cudaStream_t stream, void* const* x_hat_out)
{
    CK(cudaSetDevice(device_));
    plan(height, width);
    StreamHop hop(this, stream);
    stream = hop.run;
    stage_qp(qp, stream);
    const int zh = (height + 63) / 64, zw = (width + 63) / 64;
    if (zh != H64_ || zw != W64_) throw std::runtime_error("z geometry mismatch");
    const int nz = kZ * zh * zw;
    tev_n_ = 0;
    // dec_0 runs on the GPU while the CPU decodes z (dmc_ld_proxy.cpp:510-516)
    tick(stream);
    run(memory_has_value_ ? s_fa_m_ : s_fa_i_, stream);
    run(s_temporal_, stream);
    tock(stream);
    rans_.set_stream(bs, len, ec);
    rans_.decode_z(h_z_, nz, qp * kZ, kZ);
    CK(cudaMemcpyAsync(z_i8_, h_z_, nz, cudaMemcpyHostToDevice, stream));
    tick(stream);
    run(s_dec1_, stream);
    tock(stream);
    CK(cudaMemcpyAsync(h_total_, total_, 4, cudaMemcpyDeviceToHost, stream));
    CK(cudaEventRecord(ev_y_, stream));
    // dec_2 (context) overlaps the CPU entropy decode of y (:557-560)
    tick(stream);
    run(s_fe_, stream);
    tock(stream);
    CK(cudaEventSynchronize(ev_y_));
    const int n = h_total_[0];
    if (n < 0 || static_cast<size_t>(n) > n_lat_) throw std::runtime_error("corrupt index count");
    if (n) {
        CK(cudaStreamWaitEvent(copy_stream_, ev_y_, 0));
        CK(cudaMemcpyAsync(h_idx_, idx_c_, n, cudaMemcpyDeviceToHost, copy_stream_));
        CK(cudaStreamSynchronize(copy_stream_));
        rans_.decode_y(h_decoded_, h_idx_, n);
        CK(cudaMemcpyAsync(decoded_, h_decoded_, n, cudaMemcpyHostToDevice, stream));
    }
    tick(stream);
    run(s_dec3_, stream);
    run(s_decoder_, stream);
    run(s_recon_, stream);  // head output lands in feature_i (doubles as the reset reference, :585-586)
    if (launch_shuffle8_clamp(make_view(feature_i_, kSrc, kSrc, W8_, H8_), static_cast<__half*>(x_hat_out[0]), 3, 1, stream))
        throw std::runtime_error("shuffle8_clamp launch failed");
    ++launches;
    tock(stream);
    memory_has_value_ = !reset;  // host-side state (dmc_ld_proxy.cpp:590)
}

int LdCodec::debug_fetch(const char* name, void* dst, int64_t max_bytes, int64_t* written)
{
    struct Tap { const char* n; const void* p; size_t bytes; };
    const size_t p8 = static_cast<size_t>(H8_) * W8_, p16 = static_cast<size_t>(H16_) * W16_;
    const Tap taps[] = {
        { "y", y_, p16 * kY * 2 }, { "y_hat", yhat_, p16 * kY * 2 }, { "cat_sp", cat_sp_, p16 * kCatSp * 2 },
        { "cat_fam", cat_fam_, p8 * 512 * 2 }, { "cat8", cat8_, p8 * 512 * 2 },
        { "feature_i", feature_i_, p8 * kSrc * 2 }, { "z_i8", z_i8_, static_cast<size_t>(H64_) * W64_ * kZ },
        { "total", total_, 4 }, { "sym", sym_c_, n_lat_ * 2 }, { "yq", yq_, n_lat_ },
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

// ------------------------------------------------------------------------------- glue for codec.cu
CodecBase* make_ld_codec(int device) { return new LdCodec(device); }

int ld_add_ref(CodecBase* c, const void* frame, int H, int W, int64_t sc, int64_t sh, int64_t sw, int apply, cudaStream_t stream)
{
    static_cast<LdCodec*>(c)->add_ref(frame, H, W, sc, sh, sw, apply, stream);
    return 0;
}

int ld_compress(CodecBase* c, const void* x, int H, int W, int64_t sc, int64_t sh, int64_t sw, int qp, int reset,
                int pad_b, int pad_r, cudaStream_t stream, const uint8_t** bs, int32_t* len, int32_t* ec)
{
    static_cast<LdCodec*>(c)->compress(x, H, W, sc, sh, sw, qp, reset, pad_b, pad_r, stream, bs, len, ec);
    return 0;
}

int ld_decompress(CodecBase* c, const uint8_t* bs, int len, int qp, int height, int width, int ec, int reset,
                  cudaStream_t stream, void* const* x_hat_out)
{
    static_cast<LdCodec*>(c)->decompress(bs, len, qp, height, width, ec, reset, stream, x_hat_out);
    return 0;
}

}  // namespace dcvc
