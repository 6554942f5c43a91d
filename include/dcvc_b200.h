/*
 * dcvc_b200.h — C ABI of libdcvc_b200.so: the B200-native drop-in for the DCVC-UF per-frame
 * inference hot path.  Plain pointers and sizes only; no torch / ATen types cross this boundary.
 *
 * Every entry point names the reference interface it replaces (paths relative to the
 * microsoft/DCVC tree; the pybind11 module `inference_extensions_cuda` is defined in
 * src/layers/extensions/inference/bind.cpp:11-38).
 *
 * Conventions: all functions return 0 on success, non-zero on failure; the message is available
 * through dcvc_last_error() (thread-local for op-level calls, per-handle for codec calls).
 * Activations are fp16, NHWC ("channels_last"), batch 1, with an explicit channel pitch so that
 * channel slices of concatenated buffers can be passed without copies.  `stream` is a
 * cudaStream_t passed as void*.
 */
#ifndef DCVC_B200_H
#define DCVC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

const char* dcvc_last_error(void);
/* compiled-for architecture string ("sm_100a") and ABI version */
const char* dcvc_build_info(void);
int dcvc_abi_version(void);

/* ---------------------------------------------------------------------------------------------
 * Op-level ABI — one entry per kernel family of SURVEY.md §2.2.
 * ------------------------------------------------------------------------------------------- */

/* NHWC view: element (y,x,c) = ptr[(y*W + x)*pitch + c] */
typedef struct dcvc_view {
    const void* ptr;
    int32_t C, pitch, W, H;
} dcvc_view;

/* DCVC_GEMM_CONV3X3_PS2 (3x3 / stride 1 / pad 1 + pixel_shuffle(2), the HT-L SubpelConv2x) is experimental: it is not
 * validated on hardware yet (SURVEY.md §8 f3). */
enum { DCVC_GEMM_PW = 0, DCVC_GEMM_CONV3X3_S2 = 1, DCVC_GEMM_CONV2X2_S2 = 2, DCVC_GEMM_TCONV2X2 = 3, DCVC_GEMM_CONV3X3_PS2 = 4 };
/* GDN / IGDN: out = res1 * rsqrt(acc + bias) / res1 * sqrt(acc + bias) (DCVC-family/DCVC/src/layers/gdn.py:52-67) */
enum { DCVC_ACT_NONE = 0, DCVC_ACT_WSILU = 1, DCVC_ACT_GDN = 2, DCVC_ACT_IGDN = 3 };

/*
 * Dense contraction with fused epilogue: out = [chunk_add4]( act( in (*) W + bias ) ) [+ res1] [+ res2] [* qscale]
 * Replaces conv1x1_bias / _wsilu / _shortcut / _shortcut2 / _with_quant / _shortcut_with_quant /
 * _wsilu_chunk_add (cutlass/conv1x1_*.cu), conv_bias (cutlass/conv_bias.cu:131-150, 3x3/s2 and
 * 2x2/s2) and transposed_conv (cutlass/transposed_conv.cu:101-119).
 * `weight` is the packed [N][taps*Cin] K-major matrix produced by dcvc_pack_weight().
 */
typedef struct dcvc_gemm_desc {
    int32_t kind;          /* DCVC_GEMM_* */
    dcvc_view in, out, res1, res2; /* res*.ptr == NULL: absent */
    const void* weight;    /* fp16 packed */
    const void* bias;      /* fp16 [N] or NULL */
    const void* qscale;    /* fp16 [out.C] or NULL */
    int32_t N;             /* GEMM columns */
    int32_t act;           /* DCVC_ACT_* */
    int32_t chunk_add;     /* 1: N -> N/4 by summing groups of 4 consecutive columns after act */
} dcvc_gemm_desc;

int dcvc_op_gemm(const dcvc_gemm_desc* d, void* stream);

/*
 * The pixel-local run of a DepthConvBlock (reference: DepthConvBlockProxy::forward, layers_proxy.cpp:71-101 — the four
 * conv1x1_* calls behind the depthwise 3x3; layers.py:152-159) as ONE kernel:
 *     o   = t2 . w3 + b3 + x                       (dc.3 + shortcut)
 *     t1' = chunk_add4(wsilu(o . wf0 + bf0))       (ffn.0)
 *     y   = (t1' . wf2 + bf2 + o [+ x]) [* qscale] (ffn.2 + shortcut [+ block shortcut] [* q])
 *     t1n = wsilu(y . w0n + b0n)                   (the NEXT block's dc.0; t1n.ptr == NULL: absent)
 * o and t1' never leave the SM.  Returns 2 (dcvc_last_error(): "not eligible") for shapes the fused kernel does not
 * take (C % 128, inner % 64, > 512 channels); the codecs fall back to four dcvc_op_gemm-equivalent launches then.
 */
typedef struct dcvc_dcb_tail_desc {
    dcvc_view t2, x, y, t1n;
    const void *w3, *b3, *wf0, *bf0, *wf2, *bf2, *w0n, *b0n; /* fp16; weights [N][K] K-major */
    const void* qscale;    /* fp16 [C] or NULL */
    int32_t shortcut;      /* 1: y also adds x */
} dcvc_dcb_tail_desc;

int dcvc_op_dcb_tail(const dcvc_dcb_tail_desc* d, void* stream);

/* Host helper: re-lay a PyTorch conv weight (fp16, contiguous [Cout][Cin][kh][kw] on the HOST)
 * into the packed layout of `kind` (layers_proxy.cpp:260-266, 314-323).  dst holds N*Ktot halves. */
int dcvc_pack_weight(int32_t kind, const void* w_host, int32_t cout, int32_t cin, int32_t kh,
                     int32_t kw, void* dst_host);

/* depthwise 3x3, pad 1, no bias; w = [9][C] fp16 tap-major (cutlass/d3x3.cu:443-446) */
int dcvc_op_dw3x3(const dcvc_view* in, const dcvc_view* out, const void* w, void* stream);

/* pad_and_unshuffle_8_cuda (elementwise/cat_and_pad.cu:7-51): x is [1,Cs,H,W] with element
 * strides (sc,sh,sw); replicate-pads to the size of `out` * 8 */
int dcvc_op_unshuffle8_pad(const void* x, int32_t Cs, int32_t H, int32_t W, int64_t sc, int64_t sh,
                           int64_t sw, const dcvc_view* out, void* stream);
/* pixel_shuffle_8_cuda(clamp) (elementwise/shuffle.cu:123-137): out is NHWC [in.H*8][in.W*8][Cs] */
int dcvc_op_shuffle8_clamp(const dcvc_view* in, void* out, int32_t Cs, int32_t clamp, void* stream);
/* replicate_pad_cuda / slice_cuda (elementwise/cat_and_pad.cu:53-110) */
int dcvc_op_pad_crop(const dcvc_view* in, const dcvc_view* out, void* stream);
/* multiply_with_broadcast_cuda (elementwise/stream.cu:484-546) */
int dcvc_op_scale_channels(const dcvc_view* in, const void* q, const dcvc_view* out, void* stream);
/* round_z_cuda / int8_to_dtype_cuda (elementwise/stream.cu:862-894, 454-482) */
int dcvc_op_round_z(const void* z, void* z_hat, void* z_i8, int64_t n, void* stream);
int dcvc_op_int8_to_half(const void* x, void* out, int64_t n, void* stream);

/* ---- frame IO on the device: the callers' pre/post-processing either side of the codec (SURVEY.md §8 f2) ----
 * 8-bit YUV 4:2:0 planes (y [H][W], u, v [H/2][W/2], device) -> fp16 model input channels 0..2 of x
 * ([1,3,H,W] with element strides sc,sh,sw): nearest-neighbour chroma upsampling (ycbcr420_to_444_np,
 * src/utils/transforms.py:69-80) and x.half() / 255 - 0.5 (test_video.py:115-122).  H, W even. */
int dcvc_op_yuv420_to_frame(const void* y, const void* u, const void* v, int32_t H, int32_t W, void* x,
                            int64_t sc, int64_t sh, int64_t sw, void* stream);
/* fp16 reconstruction x_hat[:, :, :H, :W] -> 8-bit YUV 4:2:0 planes exactly as the reference saves frames
 * (test_video.py:355-361: x_hat + 0.5, yuv_444_to_420 = 2x2 chroma average (transforms.py:83-90), * 255, clamp,
 * Y rounded half-to-even, UV truncated). */
int dcvc_op_frame_to_yuv420(const void* x_hat, int64_t sc, int64_t sh, int64_t sw, int32_t H, int32_t W,
                            void* y, void* u, void* v, void* stream);
/* *sse_u64 += sum (a[i] - b[i])^2 over two 8-bit device arrays: the integer numerator of calc_psnr
 * (src/utils/metrics.py:10-24), so PSNR needs no frame on the host */
int dcvc_op_sse_u8(const void* a, const void* b, int64_t n, void* sse_u64, void* stream);
/* 8-bit planar RGB [3][H][W] (PNGReader.read_one_frame, device) -> fp16 model input channels 0..2 of x (element
 * strides sc,sh,sw): rgb2ycbcr(x.float() / 255.0).half() - 0.5 (test_video.py:93-95, 115-122; BT.709,
 * src/utils/transforms.py:17-27), bit-exact: fp32 ops rounded one at a time, division by a scalar as a multiplication
 * by its fp32 reciprocal.  Any H, W. */
int dcvc_op_rgb_to_frame(const void* rgb, int32_t H, int32_t W, void* x, int64_t sc, int64_t sh, int64_t sw,
                         void* stream);
/* fp16 reconstruction x_hat[:, :, :H, :W] -> 8-bit planar RGB [3][H][W] as the reference saves PNG frames
 * (test_video.py:367-369: ycbcr2rgb(x_hat + 0.5) in fp32 with clamp (transforms.py:53-66), back to half, * 255,
 * clamp, round half-to-even, byte()). */
int dcvc_op_frame_to_rgb(const void* x_hat, int64_t sc, int64_t sh, int64_t sw, int32_t H, int32_t W, void* rgb,
                         void* stream);

/* ---- distortion metrics of test_video.py's per-job JSON (get_distortion, test_video.py:32-66) ----
 * Metric planes: the unrounded fp16 arrays get_distortion measures, written to rec (fp16, contiguous):
 * rgb == 0: Y [H][W] = clamp((x_hat + 0.5) * 255, 0, 255), then U, V [H/2][W/2] after the 2x2 chroma average
 *           (yuv_444_to_420, transforms.py:83-90); H, W even;
 * rgb != 0: [3][H][W] = clamp(ycbcr2rgb(x_hat + 0.5) * 255, 0, 255). */
int dcvc_op_metric_planes(const void* x_hat, int64_t sc, int64_t sh, int64_t sw, int32_t H, int32_t W, int32_t rgb,
                          void* rec, void* stream);
/* Scratch for dcvc_op_metrics_sse / dcvc_op_msssim over nplanes (1..3) planes of sizes hw[2p] x hw[2p+1], in bytes
 * (-1 on bad arguments).  One workspace serves both ops and every picture of that geometry. */
int64_t dcvc_metrics_workspace_bytes(int32_t nplanes, const int32_t* hw);
/* out[p * out_stride] = sum (src[p] - rec[p])^2 in fp64: calc_psnr's numerator (src/utils/metrics.py:10-24) for
 * uint8 source planes and fp16 metric planes (contiguous rows).  Per-CTA partials + a fixed-order reduction:
 * bitwise reproducible. */
int dcvc_op_metrics_sse(int32_t nplanes, const int32_t* hw, const void* const* src, const void* const* rec,
                        void* workspace, void* out, int32_t out_stride, void* stream);
/* MS-SSIM levels of calc_msssim (src/utils/metrics.py:27-93) per plane pair: out[p * out_stride + 2l] and [.. + 2l + 1]
 * = mean of the SSIM map and of the CS map at level l (11x11 Gaussian, sigma 1.5, 'valid' region, C1 = (0.01*255)^2,
 * C2 = (0.03*255)^2; statistics and downsampled levels in fp64).  5 levels, 4 when a side is below 176; returns 2
 * when a side is below 88 (the reference asserts).  The weighted product
 * prod(mcs[:L-1] ** w[:L-1]) * mssim[L-1] ** w[L-1] is the caller's.  One launch per level + one; reproducible. */
int dcvc_op_msssim(int32_t nplanes, const int32_t* hw, const void* const* src, const void* const* rec, void* workspace,
                   void* out, int32_t out_stride, void* stream);

/* ---- ops of the older DCVC-family codecs that north_star names (SURVEY.md §8 f4) ----
 * out = in * in, elementwise: the A operand of the GDN GEMM (gdn.py:58: F.conv2d(x ** 2, gamma, beta)) */
int dcvc_op_square(const dcvc_view* in, const dcvc_view* out, void* stream);
/* bilinear backward warp with border clamp (DCVC-family/DCVC-FM/src/models/extensions/block_mc_kernel.cu:25-73,
 * == grid_sample(bilinear, border, align_corners=True), block_mc.py:47-58): out(y, x, :) = sum of the 4 neighbours
 * of im at (x + flow_x(y, x), y + flow_y(y, x)); im / out NHWC fp16, flow fp16 [2][H][W] with element strides
 * (fc, fh, fw); half arithmetic as the reference's __half kernel (fp32 positions, half weights, hfma chain). */
int dcvc_op_warp_bilinear(const dcvc_view* im, const void* flow, int64_t fc, int64_t fh, int64_t fw,
                          const dcvc_view* out, void* stream);

/* Entropy-parameter path, one 4x-mask step (elementwise/stream.cu:77-173, 175-420, 548-630,
 * 756-818, 896-949).  Buffers: see dcvc_entropy_step. */
typedef struct dcvc_entropy_step {
    int32_t H, W, G, step;
    const void* y; int32_t y_pitch;
    const void* q_enc;
    const void* scales; const void* means; int32_t p_pitch;
    void* y_hat_acc; int32_t acc_pitch;
    float skip_thres;
    void* sym_raw;   /* int16 [H*W][G]  (encoder) */
    void* idx_raw;   /* uint8 [H*W][G]  (decoder) */
    void* counts;    /* int32 [H*W] */
    void* offsets;   /* int32 [H*W+1] */
    void* total;     /* int32 [1] */
    void* compact;   /* int16 (enc) or uint8 (dec) [H*W*G] */
    const void* decoded; /* int8 compacted decoded symbols (decoder restore) */
} dcvc_entropy_step;

/* process_with_mask + fold + build_index_enc + compaction */
int dcvc_op_entropy_enc_step(const dcvc_entropy_step* a, void* stream);
/* fold + build_index_dec + compaction */
int dcvc_op_entropy_dec_index(const dcvc_entropy_step* a, void* stream);
/* conditional_recover + restore_y_4x */
int dcvc_op_entropy_dec_restore(const dcvc_entropy_step* a, void* stream);
/* 65536-entry fp16-bits -> scale-table index LUT (host) */
int dcvc_scale_index_lut(uint8_t* lut65536);

/* ---------------------------------------------------------------------------------------------
 * Host rANS coder (stays on the CPU).  Replaces MLCodec_extensions_cpp RansEncoder/RansDecoder/
 * pmf_to_quantized_cdf (src/cpp/py_rans/bind.cpp:14-40) with bit-identical streams.
 * ------------------------------------------------------------------------------------------- */
typedef struct dcvc_rans dcvc_rans;
int dcvc_rans_create(dcvc_rans** out);
void dcvc_rans_destroy(dcvc_rans* r);
/* index 0: z (factorised) tables, 1: y (Gaussian) tables; cdf is [rows][width] int32 */
int dcvc_rans_set_cdf(dcvc_rans* r, const int32_t* cdf, const int32_t* cdf_sizes, int32_t rows,
                      int32_t width, int32_t index);
/* encoder: queue jobs in coding order, then finish() -> merged stream */
int dcvc_rans_enc_reset(dcvc_rans* r);
int dcvc_rans_enc_y(dcvc_rans* r, const int16_t* symbols, int32_t n);
int dcvc_rans_enc_z(dcvc_rans* r, const int8_t* symbols, int32_t n, int32_t cdf_offset, int32_t ch);
int dcvc_rans_enc_finish(dcvc_rans* r, int32_t n_parallel, const uint8_t** data, int32_t* size);
/* decoder */
int dcvc_rans_dec_set_stream(dcvc_rans* r, const uint8_t* data, int32_t size, int32_t n_parallel);
int dcvc_rans_dec_z(dcvc_rans* r, int8_t* out, int32_t n, int32_t cdf_offset, int32_t ch);
int dcvc_rans_dec_y(dcvc_rans* r, int8_t* out, const uint8_t* cdf_rows, int32_t n);
int dcvc_pmf_to_quantized_cdf(const float* pmf, int32_t n, uint32_t* cdf_out /* n+1 */);
/* code lengths of a CDF set in Q16 bits, out = uint32 [rows][width]: entry s of row r (s <= cdf_sizes[r] - 2) is
 * round(65536 * (16 - log2(cdf[r][s+1] - cdf[r][s]))), the rest 0.  The table dcvc_estimate_bits sums on the device. */
int dcvc_rans_cost_table(const int32_t* cdf, const int32_t* cdf_sizes, int32_t rows, int32_t width, uint32_t* out);

/* ---------------------------------------------------------------------------------------------
 * Codec-level ABI — what the pybind classes DMCIProxy / DMCHTSProxy bind (bind.cpp:13-31).
 * ------------------------------------------------------------------------------------------- */
typedef struct dcvc_codec dcvc_codec;
enum { DCVC_KIND_INTRA = 0, DCVC_KIND_HTS = 1, DCVC_KIND_HTL = 2, DCVC_KIND_LD = 3 };
enum { DCVC_DTYPE_F16 = 0, DCVC_DTYPE_I32 = 1, DCVC_DTYPE_F32 = 2 };

/* DMCIProxy() / DMCHTSProxy() constructors (dmci_proxy.cpp:269-276) */
int dcvc_create(int32_t kind, int32_t device, dcvc_codec** out);
int dcvc_destroy(dcvc_codec* h);
const char* dcvc_codec_error(dcvc_codec* h);

/* set_param(state_dict, skip_thres) (dmci_proxy.cpp:604-652), one tensor at a time: `data` is a
 * device pointer for fp16 params, a host pointer for the int32 CDF tables; contiguous in `shape`. */
int dcvc_set_param(dcvc_codec* h, const char* name, const void* data, int32_t dtype, int32_t ndim,
                   const int64_t* shape, int32_t on_device);
int dcvc_finalize_params(dcvc_codec* h, float skip_thres);

/* DMCIProxy::compress (dmci_proxy.cpp:296-421): x = fp16 [1,3,H,W] device tensor with element
 * strides (sc,sh,sw); x_hat_out = caller-owned fp16 NHWC [H16*16][W16*16][3] device buffer.
 * The bitstream stays valid until the next call on this handle. */
int dcvc_compress(dcvc_codec* h, const void* x, int32_t H, int32_t W, int64_t sc, int64_t sh,
                  int64_t sw, int32_t qp, int32_t pad_b, int32_t pad_r, void* stream,
                  const uint8_t** bit_stream, int32_t* bit_stream_len, int32_t* ec_parallel,
                  void* x_hat_out);
/* DMCIProxy::decompress (dmci_proxy.cpp:423-602) */
int dcvc_decompress(dcvc_codec* h, const uint8_t* bit_stream, int32_t len, int32_t qp,
                    int32_t height, int32_t width, int32_t ec_parallel, void* stream,
                    void* x_hat_out);

/* Video codecs.  DCVC_KIND_LD (DMCLDProxy, dmc_ld_proxy.cpp:407-593; bind.cpp:32-38): the same three entry points with
 * x = fp16 [1,3,H,W] (one frame) and x_hat_out = ONE caller-owned fp16 NHWC [Hp][Wp][3] buffer.
 * Chunk codecs (DCVC_KIND_HTS): DMCHTSProxy::add_ref_feature_from_frame / compress / decompress
 * (dmc_hts_proxy.cpp:492-502, 504-585, 587-710; bind.cpp:24-31).
 * frame: fp16 [1,3,Hp,Wp] reconstruction (already padded to x16) with element strides;
 * x: fp16 [1,24,H,W] = 8 stacked YUV444 frames; x_hat_out: 8 caller-owned fp16 NHWC [Hp][Wp][3] buffers. */
int dcvc_add_ref_feature_from_frame(dcvc_codec* h, const void* frame, int32_t H, int32_t W, int64_t sc,
                                    int64_t sh, int64_t sw, int32_t apply_adaptor, void* stream);
int dcvc_compress_chunk(dcvc_codec* h, const void* x, int32_t H, int32_t W, int64_t sc, int64_t sh,
                        int64_t sw, int32_t qp, int32_t reset_feature_memory, int32_t pad_b,
                        int32_t pad_r, void* stream, const uint8_t** bit_stream,
                        int32_t* bit_stream_len, int32_t* ec_parallel);
int dcvc_decompress_chunk(dcvc_codec* h, const uint8_t* bit_stream, int32_t len, int32_t qp,
                          int32_t height, int32_t width, int32_t ec_parallel,
                          int32_t reset_feature_memory, void* stream, void* const* x_hat_out);

/* Rate estimate of one coded unit at each of n_qps QPs (1..64), for rate control.  x, H, W, strides and padding as for
 * dcvc_compress (Intra, LD) / dcvc_compress_chunk (HT-S, HT-L); reset_feature_memory does not change the estimate (it
 * only selects the memory update after the unit) and is ignored for Intra.  Runs the analysis graph and an integer
 * reduction of the symbols' code lengths on the device per QP, one copy and one synchronise at the end; no synthesis,
 * no feature-memory update, no rANS, and the next compress gives the same bytes as without the call.
 * y_q16 / z_q16: bits of the y / z symbols in Q16; ec_parallel: the stream count compress would use;
 * bytes = ceil((y_q16 + z_q16) / 2^19) + 4 * ec_parallel + 4 * (offset words of the merged container). */
typedef struct dcvc_rate_estimate {
    int64_t y_q16, z_q16;
    int32_t y_symbols, ec_parallel;
    int64_t bytes;
} dcvc_rate_estimate;
int dcvc_estimate_bits(dcvc_codec* h, const void* x, int32_t H, int32_t W, int64_t sc, int64_t sh, int64_t sw,
                       const int32_t* qps, int32_t n_qps, int32_t reset_feature_memory, int32_t pad_b, int32_t pad_r,
                       void* stream, dcvc_rate_estimate* out);

/* instrumentation for bench.py: kernels launched by this handle since creation, and the GPU-only
 * duration (ms) of the segments of the last compress/decompress (CUDA events on `stream`). */
int64_t dcvc_kernel_launches(dcvc_codec* h);
int dcvc_last_gpu_ms(dcvc_codec* h, float* ms);
/* per-kernel-family profiling (bench.py roofline): when enabled, segments run un-graphed with a
 * CUDA-event pair around every launch; kind 0 = pw_gemm, 1 = dw3x3, 2 = elementwise/entropy, 3 = dcb_tail (fused),
 * 4..8 = the pw_gemm instantiations <64>, <128>, <192>, <256>, <256, fold> on their own (0 is their total).
 * alg_bytes = algorithmic bytes (activation operands in + residuals in + out, fp16). */
int dcvc_profile_enable(dcvc_codec* h, int32_t on);
int dcvc_profile_get(dcvc_codec* h, int32_t kind, double* ms, int64_t* launches, double* alg_bytes,
                     double* flops);
/* debug taps for parity tests: copy a named internal buffer (fp16) to host. */
int dcvc_debug_fetch(dcvc_codec* h, const char* name, void* host_dst, int64_t max_bytes,
                     int64_t* bytes_written);

#ifdef __cplusplus
}
#endif
#endif /* DCVC_B200_H */
