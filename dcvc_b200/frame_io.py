"""Frame IO on the device: the callers' pre/post-processing either side of the codec (SURVEY.md §8 f2).

Host-side mirror of what the reference's driver does around `compress` / `decompress`
(test_video.py:74-76,115-122: 4:2:0 -> 4:4:4, `/255 - 0.5`; test_video.py:355-361: reconstruction -> 8-bit
4:2:0; test_video.py:88-101,366-369: the same for RGB sources; src/utils/metrics.py:10-24: PSNR), as HBM-bound
kernels of libdcvc_b200.so: a 1080p frame crosses PCIe as 3.1 MB of 8-bit planes instead of 12-25 MB of floating-point 4:4:4.  Integer outputs are bit-exact
against the reference arithmetic (oracle/ops_ref.py: yuv420_to_frame / frame_to_yuv420).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib


def _stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def yuv420_to_frame(y: torch.Tensor, u: torch.Tensor, v: torch.Tensor, out: torch.Tensor | None = None,
                    channel: int = 0) -> torch.Tensor:
    """uint8 device planes y [H,W], u, v [H/2,W/2] -> fp16 [1,3,H,W] channels_last model input
    (`get_src_frame`, test_video.py:66-122).  `out` / `channel`: write into channels channel..channel+2 of an
    existing [1,C,H,W] tensor (the 8-frame chunk input of the HT codecs stacks frames on the channel axis)."""
    assert y.is_cuda and y.dtype == torch.uint8 and y.is_contiguous() and u.is_contiguous() and v.is_contiguous()
    H, W = y.shape
    assert u.shape == (H // 2, W // 2) and v.shape == u.shape and H % 2 == 0 and W % 2 == 0
    if out is None:
        out = torch.empty((1, 3, H, W), dtype=torch.float16, device=y.device).contiguous(memory_format=torch.channels_last)
    assert out.dtype == torch.float16 and out.shape[2] == H and out.shape[3] == W and out.shape[1] >= channel + 3
    lib = _lib.load()
    ptr = out.data_ptr() + channel * out.stride(1) * 2
    _lib.check(lib.dcvc_op_yuv420_to_frame(y.data_ptr(), u.data_ptr(), v.data_ptr(), H, W, ptr, out.stride(1),
                                           out.stride(2), out.stride(3), _stream()), "op_yuv420_to_frame")
    return out


def frame_to_yuv420(x_hat: torch.Tensor, height: int, width: int, out=None):
    """fp16 reconstruction [1,3,Hp,Wp] (any strides) -> uint8 planes (y [H,W], u, v [H/2,W/2]) of the top-left
    height x width window, exactly as the reference writes decoded frames (test_video.py:352-361)."""
    assert x_hat.is_cuda and x_hat.dtype == torch.float16 and x_hat.dim() == 4 and x_hat.shape[1] == 3
    assert height % 2 == 0 and width % 2 == 0 and height <= x_hat.shape[2] and width <= x_hat.shape[3]
    if out is None:
        y = torch.empty((height, width), dtype=torch.uint8, device=x_hat.device)
        u = torch.empty((height // 2, width // 2), dtype=torch.uint8, device=x_hat.device)
        v = torch.empty_like(u)
    else:
        y, u, v = out
    lib = _lib.load()
    _lib.check(lib.dcvc_op_frame_to_yuv420(x_hat.data_ptr(), x_hat.stride(1), x_hat.stride(2), x_hat.stride(3),
                                           height, width, y.data_ptr(), u.data_ptr(), v.data_ptr(), _stream()),
               "op_frame_to_yuv420")
    return y, u, v


def rgb_to_frame(rgb: torch.Tensor, out: torch.Tensor | None = None, channel: int = 0) -> torch.Tensor:
    """uint8 planar RGB device tensor [3,H,W] (what PNGReader.read_one_frame returns) -> fp16 [1,3,H,W] channels_last
    model input, bit-exact with rgb2ycbcr(x.float() / 255.0).half() - 0.5 (test_video.py:93-95, 115-122).
    `out` / `channel` as in yuv420_to_frame."""
    assert rgb.is_cuda and rgb.dtype == torch.uint8 and rgb.dim() == 3 and rgb.shape[0] == 3 and rgb.is_contiguous()
    _, H, W = rgb.shape
    if out is None:
        out = torch.empty((1, 3, H, W), dtype=torch.float16, device=rgb.device).contiguous(memory_format=torch.channels_last)
    assert out.dtype == torch.float16 and out.shape[2] == H and out.shape[3] == W and out.shape[1] >= channel + 3
    lib = _lib.load()
    ptr = out.data_ptr() + channel * out.stride(1) * 2
    _lib.check(lib.dcvc_op_rgb_to_frame(rgb.data_ptr(), H, W, ptr, out.stride(1), out.stride(2), out.stride(3),
                                        _stream()), "op_rgb_to_frame")
    return out


def frame_to_rgb(x_hat: torch.Tensor, height: int, width: int, out: torch.Tensor | None = None) -> torch.Tensor:
    """fp16 reconstruction [1,3,Hp,Wp] (any strides) -> uint8 planar RGB [3,height,width] of the top-left window,
    exactly as the reference writes decoded PNG frames (test_video.py:366-369)."""
    assert x_hat.is_cuda and x_hat.dtype == torch.float16 and x_hat.dim() == 4 and x_hat.shape[1] == 3
    assert 0 < height <= x_hat.shape[2] and 0 < width <= x_hat.shape[3]
    if out is None:
        out = torch.empty((3, height, width), dtype=torch.uint8, device=x_hat.device)
    assert out.dtype == torch.uint8 and out.shape == (3, height, width) and out.is_contiguous()
    lib = _lib.load()
    _lib.check(lib.dcvc_op_frame_to_rgb(x_hat.data_ptr(), x_hat.stride(1), x_hat.stride(2), x_hat.stride(3), height,
                                        width, out.data_ptr(), _stream()), "op_frame_to_rgb")
    return out


def sse_u8(a: torch.Tensor, b: torch.Tensor, acc: torch.Tensor | None = None) -> torch.Tensor:
    """acc (uint64-as-int64 device scalar) += sum((a - b)^2) over two uint8 device tensors."""
    assert a.is_cuda and b.is_cuda and a.dtype == torch.uint8 and b.dtype == torch.uint8 and a.numel() == b.numel()
    assert a.is_contiguous() and b.is_contiguous()
    if acc is None:
        acc = torch.zeros(1, dtype=torch.int64, device=a.device)
    lib = _lib.load()
    _lib.check(lib.dcvc_op_sse_u8(a.data_ptr(), b.data_ptr(), a.numel(), acc.data_ptr(), _stream()), "op_sse_u8")
    return acc


def psnr_from_sse(sse: int, n: int, data_range: int = 255) -> float:
    """calc_psnr (src/utils/metrics.py:10-24) from the integer sum of squared errors"""
    mse = sse / float(n)
    if mse > 1e-10:
        return min(10.0 * np.log10(data_range * data_range / mse), 99.9)
    return 99.9
