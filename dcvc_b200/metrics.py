"""Distortion of decoded pictures on the device: the PSNR / MS-SSIM numbers of test_video.py's per-job JSON.

The reference measures every decoded picture on the host (get_distortion, test_video.py:32-66, with calc_psnr /
calc_msssim / calc_msssim_rgb of src/utils/metrics.py).  `Distortion` computes the same values from the fp16
reconstruction and the 8-bit source planes already on the device (csrc/metrics.cu): the metric planes, the per-plane
sum of squared errors and the per-level MS-SSIM means are enqueued on the current stream with no allocation and no
host synchronisation (so `.add` can be captured into a CUDA graph); `.results()` copies everything down once and
finishes the few scalar operations the reference does in numpy.

    d = Distortion("yuv420", H, W, calc_ssim=True, capacity=frame_num)
    for x_hat, (y, u, v) in ...: d.add(x_hat, (y, u, v))
    psnrs, ssims = d.results()          # per picture, shaped like get_distortion's (curr_psnr, curr_ssim)
    log = log_json(frame_num, H * W, test_time, frame_types, bits, psnrs, ssims, verbose=True)
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib

MSSSIM_WEIGHTS_5 = np.array([0.0448, 0.2856, 0.3001, 0.2363, 0.1333])
MSSSIM_WEIGHTS_4 = np.array([0.0517, 0.3295, 0.3462, 0.2726])
_SLOT = 11          # per plane: sum of squared errors, then (mean SSIM, mean CS) for up to 5 levels


def msssim_levels(h: int, w: int) -> int:
    """calc_msssim's level count (src/utils/metrics.py:31-38): 5, 4 when a side is below 176; ValueError below 88"""
    if h < 88 or w < 88:
        raise ValueError(f"MS-SSIM needs both sides of every plane >= 88, got {h}x{w}")
    return 4 if (h < 176 or w < 176) else 5


def psnr_from_mse(mse: float, data_range: int = 255) -> float:
    """calc_psnr's mapping of a mean squared error to dB (src/utils/metrics.py:10-24)"""
    if np.isnan(mse) or np.isinf(mse):
        return -999.9
    psnr = 10 * np.log10(data_range * data_range / mse) if mse > 1e-10 else 999.9
    return float(min(psnr, 99.9))


def msssim_from_levels(mssim: Sequence[float], mcs: Sequence[float]) -> float:
    """calc_msssim's weighted product of the per-level means (src/utils/metrics.py:91)"""
    level = len(mssim)
    weight = MSSSIM_WEIGHTS_5 if level == 5 else MSSSIM_WEIGHTS_4
    mssim, mcs = np.asarray(mssim, dtype=np.float64), np.asarray(mcs, dtype=np.float64)
    return float(np.prod(mcs[0:level - 1] ** weight[0:level - 1]) * (mssim[level - 1] ** weight[level - 1]))


def _ptrs(ts) -> C.Array:
    return (C.c_void_p * len(ts))(*[t.data_ptr() for t in ts])


class Distortion:
    """Per-picture distortion of one sequence, accumulated on the device.

    src_type "yuv420": `add(x_hat, (y, u, v))` with uint8 planes y [H,W], u, v [H/2,W/2];
    src_type "png":    `add(x_hat, rgb)` with a uint8 [3,H,W] tensor.
    x_hat is the fp16 reconstruction [1,3,Hp,Wp] (any strides, Hp >= H, Wp >= W); its top-left H x W window is
    measured, as test_video.py:340 crops it.  `capacity` bounds the number of pictures (the results array is allocated
    once)."""

    def __init__(self, src_type: str, height: int, width: int, calc_ssim: bool, capacity: int, device=None):
        if src_type not in ("yuv420", "png"):
            raise ValueError(f"src_type must be 'yuv420' or 'png', got {src_type!r}")
        if src_type == "yuv420" and (height % 2 or width % 2):
            raise ValueError("yuv420 sources need even picture sizes")
        self.src_type, self.H, self.W = src_type, height, width
        self.calc_ssim, self.capacity = bool(calc_ssim), int(capacity)
        device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if src_type == "yuv420":
            self.hw = [(height, width), (height // 2, width // 2), (height // 2, width // 2)]
        else:
            self.hw = [(height, width)] * 3
        self.levels = [msssim_levels(h, w) for h, w in self.hw] if self.calc_ssim else [0, 0, 0]
        sizes = [h * w for h, w in self.hw]
        rec = torch.empty(sum(sizes), dtype=torch.float16, device=device)
        self.rec_planes = list(torch.split(rec, sizes))
        self._rec = rec
        self._hw = (C.c_int32 * 6)(*[v for hw in self.hw for v in hw])
        self._rec_ptrs = _ptrs(self.rec_planes)
        lib = _lib.load()
        nbytes = lib.dcvc_metrics_workspace_bytes(3, self._hw)
        if nbytes < 0:
            raise RuntimeError("dcvc_metrics_workspace_bytes rejected the plane sizes")
        self.workspace = torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device=device)
        self.out = torch.zeros((self.capacity, 3, _SLOT), dtype=torch.float64, device=device)
        self.count = 0

    def reset(self) -> None:
        self.count = 0

    def _src_planes(self, src) -> List[torch.Tensor]:
        if self.src_type == "yuv420":
            y, u, v = src
            planes = [y, u, v]
        else:
            assert src.dim() == 3 and src.shape[0] == 3
            planes = [src[0], src[1], src[2]]
        for t, (h, w) in zip(planes, self.hw):
            assert t.is_cuda and t.dtype == torch.uint8 and tuple(t.shape) == (h, w) and t.is_contiguous()
        return planes

    def add(self, x_hat: torch.Tensor, src) -> None:
        """enqueue the metrics of one picture on the current stream (no allocation, no synchronisation)"""
        if self.count >= self.capacity:
            raise IndexError(f"Distortion holds at most {self.capacity} pictures")
        assert x_hat.is_cuda and x_hat.dtype == torch.float16 and x_hat.dim() == 4 and x_hat.shape[1] == 3
        assert x_hat.shape[2] >= self.H and x_hat.shape[3] >= self.W
        planes = self._src_planes(src)
        lib = _lib.load()
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        _lib.check(lib.dcvc_op_metric_planes(x_hat.data_ptr(), x_hat.stride(1), x_hat.stride(2), x_hat.stride(3),
                                             self.H, self.W, int(self.src_type == "png"), self._rec.data_ptr(), stream),
                   "op_metric_planes")
        src_ptrs = _ptrs(planes)
        slot = self.out.data_ptr() + self.count * 3 * _SLOT * 8
        _lib.check(lib.dcvc_op_metrics_sse(3, self._hw, src_ptrs, self._rec_ptrs, self.workspace.data_ptr(), slot,
                                           _SLOT, stream), "op_metrics_sse")
        if self.calc_ssim:
            rc = lib.dcvc_op_msssim(3, self._hw, src_ptrs, self._rec_ptrs, self.workspace.data_ptr(), slot + 8, _SLOT,
                                    stream)
            if rc == 2:
                raise ValueError("MS-SSIM needs both sides of every plane >= 88")
            _lib.check(rc, "op_msssim")
        self.count += 1

    def raw(self) -> np.ndarray:
        """[count, 3, 11] float64: per plane the sum of squared errors, then (mean SSIM, mean CS) per level"""
        return self.out[:self.count].cpu().numpy()

    def results(self) -> Tuple[List[list], List[list]]:
        """(psnrs, ssims) per picture, as get_distortion returns them (test_video.py:32-66):
        yuv420 [psnr, psnr_y, psnr_u, psnr_v] / [ssim, ssim_y, ssim_u, ssim_v] with psnr = (6 y + u + v) / 8;
        png [psnr] over all three channels / [mean of the three channels' MS-SSIM].  MS-SSIM is 0 when calc_ssim is
        off.  One device-to-host copy."""
        raw = self.raw()
        psnrs, ssims = [], []
        for pic in raw:
            if self.calc_ssim:
                ms = [msssim_from_levels(pic[p, 1:1 + 2 * L:2], pic[p, 2:2 + 2 * L:2])
                      for p, L in enumerate(self.levels)]
            else:
                ms = [0., 0., 0.]
            if self.src_type == "yuv420":
                py, pu, pv = (psnr_from_mse(pic[p, 0] / float(h * w)) for p, (h, w) in enumerate(self.hw))
                psnrs.append([(6 * py + pu + pv) / 8, py, pu, pv])
                ssims.append([(6 * ms[0] + ms[1] + ms[2]) / 8, ms[0], ms[1], ms[2]])
            else:
                n = 3 * self.H * self.W
                psnrs.append([psnr_from_mse((pic[0, 0] + pic[1, 0] + pic[2, 0]) / float(n))])
                ssims.append([(ms[0] + ms[1] + ms[2]) / 3 if self.calc_ssim else 0.])
        return psnrs, ssims


def log_json(frame_num: int, frame_pixel_num: int, test_time: float, frame_types: Sequence[int],
             bits: Sequence[int], psnrs: Sequence[Sequence[float]], ssims: Sequence[Sequence[float]],
             verbose: bool = False, avg_encoding_time: Optional[float] = None,
             avg_decoding_time: Optional[float] = None) -> dict:
    """The per-job record test_video.py writes (schema of generate_log_json, src/utils/common.py:46-116): I / P /
    all averages of bpp, PSNR and MS-SSIM (plus the Y, U, V components for yuv420 sources), per-picture lists when
    `verbose`, the test time and, when both are given, the average unit encoding / decoding times."""
    yuv = len(psnrs[0]) > 1
    if yuv and (len(psnrs[0]) != 4 or len(ssims[0]) != 4):
        raise ValueError("yuv420 records carry [all, y, u, v] per picture")
    comps = [("psnr", 0, psnrs), ("ssim", 0, ssims)]
    if yuv:
        comps += [(f"psnr_{c}", i, psnrs) for i, c in enumerate("yuv", 1)]
        comps += [(f"ssim_{c}", i, ssims) for i, c in enumerate("yuv", 1)]
    # running sums per picture class, accumulated in display order from an integer 0 (as the reference does)
    acc = {t: {"bits": 0, **{key: 0 for key, _, _ in comps}} for t in ("i", "p")}
    count = {"i": 0, "p": 0}
    for f in range(frame_num):
        t = "i" if frame_types[f] == 0 else "p"
        acc[t]["bits"] += bits[f]
        for key, idx, src in comps:
            acc[t][key] += src[f][idx]
        count[t] += 1

    def avg(t, key, scale=1):
        return acc[t][key] / count[t] / scale if count[t] > 0 else 0

    log = {"frame_pixel_num": frame_pixel_num, "i_frame_num": count["i"], "p_frame_num": count["p"]}
    for t in ("i", "p"):
        log[f"ave_{t}_frame_bpp"] = avg(t, "bits", frame_pixel_num)
        log[f"ave_{t}_frame_psnr"] = avg(t, "psnr")
        log[f"ave_{t}_frame_msssim"] = avg(t, "ssim")
        if yuv:
            for c in "yuv":
                log[f"ave_{t}_frame_psnr_{c}"] = avg(t, f"psnr_{c}")
                log[f"ave_{t}_frame_msssim_{c}"] = avg(t, f"ssim_{c}")
    if verbose:
        log["frame_bpp"] = list(np.array(bits) / frame_pixel_num)
        log["frame_psnr"] = [p[0] for p in psnrs]
        log["frame_msssim"] = [s[0] for s in ssims]
        log["frame_type"] = frame_types
        if yuv:
            for i, c in enumerate("yuv", 1):
                log[f"frame_psnr_{c}"] = [p[i] for p in psnrs]
                log[f"frame_msssim_{c}"] = [s[i] for s in ssims]
    log["test_time"] = test_time
    log["ave_all_frame_bpp"] = (acc["i"]["bits"] + acc["p"]["bits"]) / (frame_num * frame_pixel_num)
    log["ave_all_frame_psnr"] = (acc["i"]["psnr"] + acc["p"]["psnr"]) / frame_num
    log["ave_all_frame_msssim"] = (acc["i"]["ssim"] + acc["p"]["ssim"]) / frame_num
    if avg_encoding_time is not None and avg_decoding_time is not None:
        log["avg_frame_encoding_time"] = avg_encoding_time
        log["avg_frame_decoding_time"] = avg_decoding_time
    if yuv:
        for c in "yuv":
            log[f"ave_all_frame_psnr_{c}"] = (acc["i"][f"psnr_{c}"] + acc["p"][f"psnr_{c}"]) / frame_num
            log[f"ave_all_frame_msssim_{c}"] = (acc["i"][f"ssim_{c}"] + acc["p"][f"ssim_{c}"]) / frame_num
    return log
