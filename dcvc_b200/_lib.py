"""ctypes binding of libdcvc_b200.so (include/dcvc_b200.h).

There is deliberately no fallback: if the shared library is missing or does not load, importing the
product path raises — the CUDA extension *is* the product (no CPU / PyTorch route for the transform
path).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libdcvc_b200.so")


class View(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("C", C.c_int32), ("pitch", C.c_int32), ("W", C.c_int32),
                ("H", C.c_int32)]


class GemmDesc(C.Structure):
    _fields_ = [("kind", C.c_int32), ("inp", View), ("out", View), ("res1", View), ("res2", View),
                ("weight", C.c_void_p), ("bias", C.c_void_p), ("qscale", C.c_void_p),
                ("N", C.c_int32), ("act", C.c_int32), ("chunk_add", C.c_int32)]


class DcbTailDesc(C.Structure):
    _fields_ = [("t2", View), ("x", View), ("y", View), ("t1n", View),
                ("w3", C.c_void_p), ("b3", C.c_void_p), ("wf0", C.c_void_p), ("bf0", C.c_void_p),
                ("wf2", C.c_void_p), ("bf2", C.c_void_p), ("w0n", C.c_void_p), ("b0n", C.c_void_p),
                ("qscale", C.c_void_p), ("shortcut", C.c_int32)]


class RateEstimate(C.Structure):
    _fields_ = [("y_q16", C.c_int64), ("z_q16", C.c_int64), ("y_symbols", C.c_int32), ("ec_parallel", C.c_int32),
                ("bytes", C.c_int64)]


class EntropyStep(C.Structure):
    _fields_ = [("H", C.c_int32), ("W", C.c_int32), ("G", C.c_int32), ("step", C.c_int32),
                ("y", C.c_void_p), ("y_pitch", C.c_int32),
                ("q_enc", C.c_void_p),
                ("scales", C.c_void_p), ("means", C.c_void_p), ("p_pitch", C.c_int32),
                ("y_hat_acc", C.c_void_p), ("acc_pitch", C.c_int32),
                ("skip_thres", C.c_float),
                ("sym_raw", C.c_void_p), ("idx_raw", C.c_void_p), ("counts", C.c_void_p),
                ("offsets", C.c_void_p), ("total", C.c_void_p), ("compact", C.c_void_p),
                ("decoded", C.c_void_p)]


GEMM_PW, GEMM_CONV3X3_S2, GEMM_CONV2X2_S2, GEMM_TCONV2X2, GEMM_CONV3X3_PS2 = 0, 1, 2, 3, 4
ACT_NONE, ACT_WSILU, ACT_GDN, ACT_IGDN = 0, 1, 2, 3
KIND_INTRA, KIND_HTS, KIND_HTL, KIND_LD = 0, 1, 2, 3
DTYPE_F16, DTYPE_I32, DTYPE_F32 = 0, 1, 2

# name -> (restype, argtypes); also the list of symbols the header declares (tests check exports)
_P = C.c_void_p
_I = C.c_int32
_L = C.c_int64
SIGNATURES = {
    "dcvc_last_error": (C.c_char_p, []),
    "dcvc_build_info": (C.c_char_p, []),
    "dcvc_abi_version": (C.c_int, []),
    "dcvc_op_gemm": (C.c_int, [C.POINTER(GemmDesc), _P]),
    "dcvc_op_dcb_tail": (C.c_int, [C.POINTER(DcbTailDesc), _P]),
    "dcvc_pack_weight": (C.c_int, [_I, _P, _I, _I, _I, _I, _P]),
    "dcvc_op_dw3x3": (C.c_int, [C.POINTER(View), C.POINTER(View), _P, _P]),
    "dcvc_op_unshuffle8_pad": (C.c_int, [_P, _I, _I, _I, _L, _L, _L, C.POINTER(View), _P]),
    "dcvc_op_shuffle8_clamp": (C.c_int, [C.POINTER(View), _P, _I, _I, _P]),
    "dcvc_op_pad_crop": (C.c_int, [C.POINTER(View), C.POINTER(View), _P]),
    "dcvc_op_scale_channels": (C.c_int, [C.POINTER(View), _P, C.POINTER(View), _P]),
    "dcvc_op_round_z": (C.c_int, [_P, _P, _P, _L, _P]),
    "dcvc_op_yuv420_to_frame": (C.c_int, [_P, _P, _P, _I, _I, _P, _L, _L, _L, _P]),
    "dcvc_op_frame_to_yuv420": (C.c_int, [_P, _L, _L, _L, _I, _I, _P, _P, _P, _P]),
    "dcvc_op_sse_u8": (C.c_int, [_P, _P, _L, _P, _P]),
    "dcvc_op_rgb_to_frame": (C.c_int, [_P, _I, _I, _P, _L, _L, _L, _P]),
    "dcvc_op_frame_to_rgb": (C.c_int, [_P, _L, _L, _L, _I, _I, _P, _P]),
    "dcvc_op_metric_planes": (C.c_int, [_P, _L, _L, _L, _I, _I, _I, _P, _P]),
    "dcvc_metrics_workspace_bytes": (C.c_int64, [_I, C.POINTER(_I)]),
    "dcvc_op_metrics_sse": (C.c_int, [_I, C.POINTER(_I), C.POINTER(_P), C.POINTER(_P), _P, _P, _I, _P]),
    "dcvc_op_msssim": (C.c_int, [_I, C.POINTER(_I), C.POINTER(_P), C.POINTER(_P), _P, _P, _I, _P]),
    "dcvc_op_square": (C.c_int, [C.POINTER(View), C.POINTER(View), _P]),
    "dcvc_op_warp_bilinear": (C.c_int, [C.POINTER(View), _P, _L, _L, _L, C.POINTER(View), _P]),
    "dcvc_op_int8_to_half": (C.c_int, [_P, _P, _L, _P]),
    "dcvc_op_entropy_enc_step": (C.c_int, [C.POINTER(EntropyStep), _P]),
    "dcvc_op_entropy_dec_index": (C.c_int, [C.POINTER(EntropyStep), _P]),
    "dcvc_op_entropy_dec_restore": (C.c_int, [C.POINTER(EntropyStep), _P]),
    "dcvc_scale_index_lut": (C.c_int, [_P]),
    "dcvc_rans_create": (C.c_int, [C.POINTER(_P)]),
    "dcvc_rans_destroy": (None, [_P]),
    "dcvc_rans_set_cdf": (C.c_int, [_P, _P, _P, _I, _I, _I]),
    "dcvc_rans_enc_reset": (C.c_int, [_P]),
    "dcvc_rans_enc_y": (C.c_int, [_P, _P, _I]),
    "dcvc_rans_enc_z": (C.c_int, [_P, _P, _I, _I, _I]),
    "dcvc_rans_enc_finish": (C.c_int, [_P, _I, C.POINTER(_P), C.POINTER(_I)]),
    "dcvc_rans_dec_set_stream": (C.c_int, [_P, _P, _I, _I]),
    "dcvc_rans_dec_z": (C.c_int, [_P, _P, _I, _I, _I]),
    "dcvc_rans_dec_y": (C.c_int, [_P, _P, _P, _I]),
    "dcvc_pmf_to_quantized_cdf": (C.c_int, [_P, _I, _P]),
    "dcvc_rans_cost_table": (C.c_int, [_P, _P, _I, _I, _P]),
    "dcvc_create": (C.c_int, [_I, _I, C.POINTER(_P)]),
    "dcvc_destroy": (C.c_int, [_P]),
    "dcvc_codec_error": (C.c_char_p, [_P]),
    "dcvc_set_param": (C.c_int, [_P, C.c_char_p, _P, _I, _I, C.POINTER(_L), _I]),
    "dcvc_finalize_params": (C.c_int, [_P, C.c_float]),
    "dcvc_compress": (C.c_int, [_P, _P, _I, _I, _L, _L, _L, _I, _I, _I, _P, C.POINTER(_P),
                                C.POINTER(_I), C.POINTER(_I), _P]),
    "dcvc_decompress": (C.c_int, [_P, _P, _I, _I, _I, _I, _I, _P, _P]),
    "dcvc_add_ref_feature_from_frame": (C.c_int, [_P, _P, _I, _I, _L, _L, _L, _I, _P]),
    "dcvc_compress_chunk": (C.c_int, [_P, _P, _I, _I, _L, _L, _L, _I, _I, _I, _I, _P, C.POINTER(_P),
                                      C.POINTER(_I), C.POINTER(_I)]),
    "dcvc_decompress_chunk": (C.c_int, [_P, _P, _I, _I, _I, _I, _I, _I, _P, C.POINTER(_P)]),
    "dcvc_estimate_bits": (C.c_int, [_P, _P, _I, _I, _L, _L, _L, _P, _I, _I, _I, _I, _P, C.POINTER(RateEstimate)]),
    "dcvc_kernel_launches": (C.c_int64, [_P]),
    "dcvc_last_gpu_ms": (C.c_int, [_P, C.POINTER(C.c_float)]),
    "dcvc_profile_enable": (C.c_int, [_P, _I]),
    "dcvc_profile_get": (C.c_int, [_P, _I, C.POINTER(C.c_double), C.POINTER(_L), C.POINTER(C.c_double),
                                   C.POINTER(C.c_double)]),
    "dcvc_debug_fetch": (C.c_int, [_P, C.c_char_p, _P, _L, C.POINTER(_L)]),
}

_lib = None


def load() -> C.CDLL:
    """Load libdcvc_b200.so (building nothing): raises if it is not there."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m dcvc_b200.build` "
            "(or __graft_entry__.build()). There is no CPU fallback for the transform path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export it
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().dcvc_last_error().decode(errors="replace")
        raise RuntimeError(f"libdcvc_b200: {what} failed: {msg}")
