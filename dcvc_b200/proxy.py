"""Python face of the codec-level C ABI: drop-in for the reference's pybind11 classes
(src/layers/extensions/inference/bind.cpp:11-38).  Same class names, method names, argument order
and return values; torch is used only for device memory and the current stream.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib


class _CodecHandle:
    def __init__(self, kind: int):
        if not torch.cuda.is_available():
            raise RuntimeError("inference_extensions_cuda (dcvc_b200) needs a CUDA device: there is no CPU path")
        self.lib = _lib.load()
        self.h = C.c_void_p()
        self.device = torch.cuda.current_device()
        rc = self.lib.dcvc_create(kind, self.device, C.byref(self.h))
        if rc:
            raise RuntimeError("dcvc_create failed: " + self.lib.dcvc_last_error().decode())

    def same_device(self, t):
        if t.device.index is not None and t.device.index != self.device:
            raise RuntimeError(f"tensor on cuda:{t.device.index}, but this proxy was created on cuda:{self.device}")

    def check(self, rc, what):
        if rc:
            raise RuntimeError(f"{what}: " + self.lib.dcvc_codec_error(self.h).decode(errors="replace"))

    def __del__(self):
        try:
            if self.h:
                self.lib.dcvc_destroy(self.h)
        except Exception:
            pass


def _push_state_dict(hd: _CodecHandle, state_dict, skip_threshold: float):
    """Hands every tensor of the state_dict to the C side (`dcvc_set_param` copies it with a blocking cudaMemcpy on the
    legacy stream).  The layout / dtype conversions below run as kernels on torch's CURRENT stream, which is usually a
    non-blocking stream the legacy stream does not order against (test_video.py runs the models under its own stream and
    finalises them to channels_last, so every k > 1 conv weight needs such a kernel; the P model's set_param runs right
    behind the I model's queued synthesis).  So: materialise every tensor first, synchronise that stream ONCE, then copy."""
    staged = []
    for name, t in state_dict.items():
        if not isinstance(t, torch.Tensor):
            continue
        if t.dtype in (torch.int32, torch.int64):
            tt = t.detach().to("cpu", torch.int32).contiguous()
            dtype, on_dev = _lib.DTYPE_I32, 0
        elif t.is_floating_point():
            # logical (row-major) order, whatever the memory_format of the module was
            tt = t.detach().contiguous(memory_format=torch.contiguous_format)
            if tt.dtype == torch.float16:
                dtype = _lib.DTYPE_F16
            else:
                tt = tt.float()
                dtype = _lib.DTYPE_F32
            on_dev = 1 if tt.is_cuda else 0
            if tt.is_cuda and tt.device.index is not None and tt.device.index != hd.device:
                raise RuntimeError(f"set_param({name}): tensor lives on cuda:{tt.device.index}, the proxy on cuda:{hd.device}")
        else:
            continue
        staged.append((name, tt, dtype, on_dev))
    if any(on_dev for _, _, _, on_dev in staged):
        torch.cuda.current_stream(hd.device).synchronize()
    for name, tt, dtype, on_dev in staged:
        shape = (C.c_int64 * max(1, tt.dim()))(*tt.shape)
        hd.check(hd.lib.dcvc_set_param(hd.h, name.encode(), C.c_void_p(tt.data_ptr()), dtype, tt.dim(), shape, on_dev),
                 f"set_param({name})")
    hd.check(hd.lib.dcvc_finalize_params(hd.h, C.c_float(float(skip_threshold))), "finalize_params")


def _estimate_bits(hd: _CodecHandle, x, qps, reset_feature_memory, padding_b, padding_r):
    """dcvc_estimate_bits: one record per QP, in the order given"""
    qps = [int(q) for q in qps]
    hd.same_device(x)
    _, _, H, W = x.shape
    q = (C.c_int32 * len(qps))(*qps)
    res = (_lib.RateEstimate * len(qps))()
    stream = C.c_void_p(torch.cuda.current_stream(hd.device).cuda_stream)
    hd.check(hd.lib.dcvc_estimate_bits(hd.h, C.c_void_p(x.data_ptr()), H, W, x.stride(1), x.stride(2), x.stride(3), q,
                                       len(qps), 1 if reset_feature_memory else 0, int(padding_b), int(padding_r), stream,
                                       res), "estimate_bits")
    return [{"qp": qp, "bits_y": r.y_q16 / 65536.0, "bits_z": r.z_q16 / 65536.0, "y_symbols": r.y_symbols,
             "ec_parallel": r.ec_parallel, "bytes": r.bytes} for qp, r in zip(qps, res)]


class DMCIProxy:
    """DCVC-UF-Intra proxy (reference: DMCIProxy, dmci_proxy.h:142-144)."""

    def __init__(self):
        self._hd = _CodecHandle(_lib.KIND_INTRA)
        self._x_hat = {}

    def set_param(self, state_dict, skip_threshold: float):
        _push_state_dict(self._hd, state_dict, skip_threshold)

    def _out(self, side, hp, wp, device):
        # Reconstructions are written into proxy-owned buffers (no allocation per frame), one for the encoder side and one
        # for the decoder side: the x_hat of a compress() stays valid through the following decompress() (the usual
        # encode-then-decode comparison), and is overwritten by the NEXT compress(); clone() what must outlive that.
        t = self._x_hat.get(side)
        if t is None or t.shape[2] != hp or t.shape[3] != wp:
            t = torch.empty((1, 3, hp, wp), dtype=torch.float16, device=device, memory_format=torch.channels_last)
            self._x_hat[side] = t
        return t

    def compress(self, x: torch.Tensor, qp: int, padding_b: int, padding_r: int):
        """-> (bit_stream: np.ndarray[uint8], x_hat: fp16 channels_last [1,3,H16p,W16p], ec_parallel).
        x_hat is a proxy-owned buffer, reused by the next compress() call (see _out)."""
        hd = self._hd
        assert x.is_cuda and x.dtype == torch.float16 and x.dim() == 4 and x.shape[0] == 1 and x.shape[1] == 3
        hd.same_device(x)
        _, _, H, W = x.shape
        out = self._out("enc", H + padding_b, W + padding_r, x.device)
        bs, n, ec = C.c_void_p(), C.c_int32(), C.c_int32()
        stream = C.c_void_p(torch.cuda.current_stream(hd.device).cuda_stream)
        hd.check(hd.lib.dcvc_compress(hd.h, C.c_void_p(x.data_ptr()), H, W, x.stride(1), x.stride(2), x.stride(3),
                                      int(qp), int(padding_b), int(padding_r), stream, C.byref(bs), C.byref(n),
                                      C.byref(ec), C.c_void_p(out.data_ptr())), "compress")
        stream_np = np.ctypeslib.as_array(C.cast(bs, C.POINTER(C.c_uint8)), (n.value,)).copy()
        return stream_np, out, ec.value

    def estimate_bits(self, x: torch.Tensor, qps, padding_b: int, padding_r: int):
        """Size of compress(x, qp, ...) for each qp in `qps` without coding it: a list of dicts with bits_y / bits_z
        (the y and z symbols' code lengths, exact in Q16), y_symbols, ec_parallel and bytes (the stream length to within
        a few bytes per rANS stream).  Runs the analysis graph per QP and changes no state of the proxy."""
        assert x.is_cuda and x.dtype == torch.float16 and x.dim() == 4 and x.shape[0] == 1 and x.shape[1] == 3
        return _estimate_bits(self._hd, x, qps, False, padding_b, padding_r)

    def decompress(self, bit_stream: np.ndarray, qp: int, height: int, width: int, ec_parallel: int):
        """-> x_hat: fp16 channels_last [1,3,H16p,W16p], a proxy-owned buffer reused by the next decompress() call"""
        hd = self._hd
        bs = np.ascontiguousarray(bit_stream, dtype=np.uint8)
        hp, wp = (height + 15) // 16 * 16, (width + 15) // 16 * 16
        out = self._out("dec", hp, wp, torch.device("cuda", hd.device))
        stream = C.c_void_p(torch.cuda.current_stream(hd.device).cuda_stream)
        hd.check(hd.lib.dcvc_decompress(hd.h, C.c_void_p(bs.ctypes.data), bs.size, int(qp), int(height), int(width),
                                        int(ec_parallel), stream, C.c_void_p(out.data_ptr())), "decompress")
        return out

    # ---- instrumentation (not part of the reference surface)
    def kernel_launches(self) -> int:
        return int(self._hd.lib.dcvc_kernel_launches(self._hd.h))

    def last_gpu_ms(self) -> float:
        ms = C.c_float()
        self._hd.check(self._hd.lib.dcvc_last_gpu_ms(self._hd.h, C.byref(ms)), "last_gpu_ms")
        return ms.value

    def profile_enable(self, on: bool):
        self._hd.lib.dcvc_profile_enable(self._hd.h, 1 if on else 0)

    def profile_get(self):
        """{family: dict(ms, launches, alg_bytes, flops)} accumulated since profile_enable(True)"""
        out = {}
        for kind, name in enumerate(("pw_gemm", "dw3x3", "elementwise", "dcb_tail", "pw_gemm<64>", "pw_gemm<128>", "pw_gemm<192>",
                                     "pw_gemm<256>", "pw_gemm<256,fold>")):
            ms, n, b, f = C.c_double(), C.c_int64(), C.c_double(), C.c_double()
            self._hd.lib.dcvc_profile_get(self._hd.h, kind, C.byref(ms), C.byref(n), C.byref(b), C.byref(f))
            out[name] = {"ms": ms.value, "launches": n.value, "alg_bytes": b.value, "flops": f.value}
        return out

    def debug_fetch(self, name: str, dtype=np.float16) -> np.ndarray:
        buf = np.zeros(64 << 20, dtype=np.uint8)
        n = C.c_int64()
        self._hd.check(self._hd.lib.dcvc_debug_fetch(self._hd.h, name.encode(), C.c_void_p(buf.ctypes.data), buf.size,
                                                     C.byref(n)), "debug_fetch")
        return buf[: n.value].view(dtype).copy()


class DMCHTSProxy:
    """DCVC-UF HT-S chunk codec proxy (reference: DMCHTSProxy, dmc_hts_proxy.h:229-233; bind.cpp:24-31)."""

    FRAMES = 8

    def __init__(self):
        self._hd = _CodecHandle(_lib.KIND_HTS)
        self._x_hat = None

    def set_param(self, state_dict, skip_threshold: float):
        _push_state_dict(self._hd, state_dict, skip_threshold)

    def add_ref_feature_from_frame(self, frame: torch.Tensor, apply_adaptor: bool):
        hd = self._hd
        assert frame.is_cuda and frame.dtype == torch.float16 and frame.dim() == 4 and frame.shape[1] == 3
        hd.same_device(frame)
        _, _, H, W = frame.shape
        stream = C.c_void_p(torch.cuda.current_stream(hd.device).cuda_stream)
        hd.check(hd.lib.dcvc_add_ref_feature_from_frame(hd.h, C.c_void_p(frame.data_ptr()), H, W, frame.stride(1),
                                                        frame.stride(2), frame.stride(3), 1 if apply_adaptor else 0,
                                                        stream), "add_ref_feature_from_frame")

    def compress(self, x: torch.Tensor, qp: int, reset_feature_memory: bool, padding_b: int, padding_r: int):
        """x: fp16 [1, 24, H, W] -> (bit_stream np.ndarray[uint8], ec_parallel)"""
        hd = self._hd
        assert x.is_cuda and x.dtype == torch.float16 and x.dim() == 4 and x.shape[1] == 3 * self.FRAMES
        hd.same_device(x)
        _, _, H, W = x.shape
        bs, n, ec = C.c_void_p(), C.c_int32(), C.c_int32()
        stream = C.c_void_p(torch.cuda.current_stream(hd.device).cuda_stream)
        hd.check(hd.lib.dcvc_compress_chunk(hd.h, C.c_void_p(x.data_ptr()), H, W, x.stride(1), x.stride(2), x.stride(3),
                                            int(qp), 1 if reset_feature_memory else 0, int(padding_b), int(padding_r),
                                            stream, C.byref(bs), C.byref(n), C.byref(ec)), "compress")
        return np.ctypeslib.as_array(C.cast(bs, C.POINTER(C.c_uint8)), (n.value,)).copy(), ec.value

    def estimate_bits(self, x: torch.Tensor, qps, reset_feature_memory: bool, padding_b: int, padding_r: int):
        """Size of compress(x, qp, reset_feature_memory, ...) for each qp in `qps` without coding it (see
        DMCIProxy.estimate_bits).  The feature memory, context and every other state the next compress() reads stay
        as they were."""
        assert x.is_cuda and x.dtype == torch.float16 and x.dim() == 4 and x.shape[1] == 3 * self.FRAMES
        return _estimate_bits(self._hd, x, qps, reset_feature_memory, padding_b, padding_r)

    def decompress(self, bit_stream: np.ndarray, qp: int, height: int, width: int, ec_parallel: int,
                   reset_feature_memory: bool):
        """-> list of 8 fp16 channels_last tensors [1,3,H16p,W16p] (proxy-owned, reused by the next call)"""
        hd = self._hd
        bs = np.ascontiguousarray(bit_stream, dtype=np.uint8)
        hp, wp = (height + 15) // 16 * 16, (width + 15) // 16 * 16
        if self._x_hat is None or self._x_hat[0].shape[2] != hp or self._x_hat[0].shape[3] != wp:
            dev = torch.device("cuda", hd.device)
            self._x_hat = [torch.empty((1, 3, hp, wp), dtype=torch.float16, device=dev,
                                       memory_format=torch.channels_last) for _ in range(self.FRAMES)]
        ptrs = (C.c_void_p * self.FRAMES)(*[t.data_ptr() for t in self._x_hat])
        stream = C.c_void_p(torch.cuda.current_stream(hd.device).cuda_stream)
        hd.check(hd.lib.dcvc_decompress_chunk(hd.h, C.c_void_p(bs.ctypes.data), bs.size, int(qp), int(height), int(width),
                                              int(ec_parallel), 1 if reset_feature_memory else 0, stream, ptrs),
                 "decompress")
        return self._x_hat

    kernel_launches = DMCIProxy.kernel_launches
    last_gpu_ms = DMCIProxy.last_gpu_ms
    profile_enable = DMCIProxy.profile_enable
    profile_get = DMCIProxy.profile_get
    debug_fetch = DMCIProxy.debug_fetch


class DMCLDProxy(DMCHTSProxy):
    """DCVC-UF low-delay codec proxy (reference: DMCLDProxy, dmc_ld_proxy.h; bind.cpp:32-38): one frame per call,
    `decompress` returns ONE tensor."""

    FRAMES = 1

    def __init__(self):
        self._hd = _CodecHandle(_lib.KIND_LD)
        self._x_hat = None

    def decompress(self, bit_stream: np.ndarray, qp: int, height: int, width: int, ec_parallel: int,
                   reset_feature_memory: bool):
        """-> fp16 channels_last tensor [1,3,H16p,W16p] (proxy-owned, reused by the next call)"""
        return super().decompress(bit_stream, qp, height, width, ec_parallel, reset_feature_memory)[0]


class DMCHTLProxy(DMCHTSProxy):
    """DCVC-UF HT-L chunk codec proxy (reference: DMCHTLProxy, dmc_htl_proxy.h; bind.cpp:18-23)."""

    def __init__(self):
        self._hd = _CodecHandle(_lib.KIND_HTL)
        self._x_hat = None
