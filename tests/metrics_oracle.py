"""Host restatement of the reference's distortion metrics (test infrastructure; never imported by dcvc_b200).

calc_psnr / calc_msssim / calc_msssim_rgb (src/utils/metrics.py:10-100) and the arrays get_distortion measures
(test_video.py:32-66), written the way csrc/metrics.cu computes them rather than the way the reference does:
the 11x11 Gaussian window as two 11-tap passes over the 'valid' region in float64 (the reference uses scipy
fftconvolve), and the next level as an explicit 2x2 mean of rows / columns (2k, 2k+1) with an odd last row / column
averaged with itself (the reference: ndimage.convolve(ones(2,2)/4, mode='reflect')[::2, ::2]).  Pinned to the
reference's own functions by tests/golden/metrics_reference.json."""
from __future__ import annotations

import numpy as np
import torch

WEIGHTS_5 = np.array([0.0448, 0.2856, 0.3001, 0.2363, 0.1333])
WEIGHTS_4 = np.array([0.0517, 0.3295, 0.3462, 0.2726])
C1 = (0.01 * 255) ** 2
C2 = (0.03 * 255) ** 2


def gauss1d(size: int = 11, sigma: float = 1.5) -> np.ndarray:
    x = np.arange(size, dtype=np.float64) - size // 2
    g = np.exp(-(x * x) / (2.0 * sigma * sigma))
    return g / g.sum()


def _window_valid(a: np.ndarray, g: np.ndarray) -> np.ndarray:
    k = len(g)
    h = sum(g[i] * a[:, i:a.shape[1] - k + 1 + i] for i in range(k))
    return sum(g[i] * h[i:h.shape[0] - k + 1 + i, :] for i in range(k))


def ssim_cs_means(x: np.ndarray, y: np.ndarray):
    """(mean SSIM map, mean CS map) of one level"""
    g = gauss1d()
    mu1, mu2 = _window_valid(x, g), _window_valid(y, g)
    e11, e22, e12 = _window_valid(x * x, g), _window_valid(y * y, g), _window_valid(x * y, g)
    s1, s2, s12 = e11 - mu1 * mu1, e22 - mu2 * mu2, e12 - mu1 * mu2
    cs = (2 * s12 + C2) / (s1 + s2 + C2)
    ssim = (2 * mu1 * mu2 + C1) / (mu1 * mu1 + mu2 * mu2 + C1) * cs
    return float(ssim.mean()), float(cs.mean())


def downsample2(a: np.ndarray) -> np.ndarray:
    p = np.pad(a, ((0, a.shape[0] % 2), (0, a.shape[1] % 2)), mode="edge")
    return 0.25 * (p[0::2, 0::2] + p[0::2, 1::2] + p[1::2, 0::2] + p[1::2, 1::2])


def msssim_levels(img1: np.ndarray, img2: np.ndarray):
    """per-level (mssim, mcs) lists; ValueError where the reference asserts (a side below 88)"""
    h, w = img1.shape
    if h < 88 or w < 88:
        raise ValueError(f"MS-SSIM needs both sides >= 88, got {h}x{w}")
    level = 4 if (h < 176 or w < 176) else 5
    x, y = img1.astype(np.float64), img2.astype(np.float64)
    mssim, mcs = [], []
    for _ in range(level):
        s, c = ssim_cs_means(x, y)
        mssim.append(s)
        mcs.append(c)
        x, y = downsample2(x), downsample2(y)
    return mssim, mcs


def msssim(img1: np.ndarray, img2: np.ndarray) -> float:
    mssim, mcs = msssim_levels(img1, img2)
    L = len(mssim)
    w = WEIGHTS_5 if L == 5 else WEIGHTS_4
    return float(np.prod(np.array(mcs[:L - 1]) ** w[:L - 1]) * np.array(mssim[L - 1]) ** w[L - 1])


def msssim_rgb(img1: np.ndarray, img2: np.ndarray) -> float:
    return sum(msssim(img1[i], img2[i]) for i in range(3)) / 3


def psnr(img1: np.ndarray, img2: np.ndarray, data_range: int = 255) -> float:
    mse = float(np.mean(np.square(img1.astype(np.float64) - img2.astype(np.float64))))
    if np.isnan(mse) or np.isinf(mse):
        return -999.9
    return float(min(10 * np.log10(data_range * data_range / mse) if mse > 1e-10 else 999.9, 99.9))


# ---- colour transforms and metric planes as test_video.py composes them (torch, host) ----
KR, KG, KB = 0.2126, 0.7152, 0.0722


def rgb2ycbcr(rgb: torch.Tensor) -> torch.Tensor:
    r, g, b = rgb.chunk(3, -3)
    y = KR * r + KG * g + KB * b
    cb = 0.5 * (b - y) / (1 - KB) + 0.5
    cr = 0.5 * (r - y) / (1 - KR) + 0.5
    return torch.clamp(torch.cat((y, cb, cr), dim=-3), 0., 1.)


def ycbcr2rgb(ycbcr: torch.Tensor) -> torch.Tensor:
    dtype = ycbcr.dtype
    y, cb, cr = ycbcr.float().chunk(3, -3)
    r = y + (2 - 2 * KR) * (cr - 0.5)
    b = y + (2 - 2 * KB) * (cb - 0.5)
    g = (y - KR * r - KB * b) / KG
    return torch.clamp(torch.cat((r, g, b), dim=-3), 0., 1.).to(dtype)


def metric_planes(x_hat: torch.Tensor, src_type: str, height: int, width: int):
    """the fp16 arrays get_distortion measures, as numpy: [y, u, v] (yuv420) or [r, g, b] (png)"""
    x = x_hat[:, :, :height, :width] + 0.5
    if src_type == "yuv420":
        uv = torch.nn.functional.avg_pool2d(x[:, 1:].float(), 2, 2).to(x.dtype)
        y = torch.clamp(x[:, :1] * 255, 0, 255)
        uv = torch.clamp(uv * 255, 0, 255)
        return [y[0, 0].numpy(), uv[0, 0].numpy(), uv[0, 1].numpy()]
    rgb = torch.clamp(ycbcr2rgb(x) * 255, 0, 255)
    return [rgb[0, i].numpy() for i in range(3)]


def distortion(src_type: str, x_hat: torch.Tensor, src, calc_ssim: bool, height: int, width: int):
    """(curr_psnr, curr_ssim) of get_distortion for one picture"""
    rec = metric_planes(x_hat, src_type, height, width)
    if src_type == "yuv420":
        ps = [psnr(s, r) for s, r in zip(src, rec)]
        ms = [msssim(s, r) for s, r in zip(src, rec)] if calc_ssim else [0., 0., 0.]
        return [(6 * ps[0] + ps[1] + ps[2]) / 8] + ps, [(6 * ms[0] + ms[1] + ms[2]) / 8] + ms
    rgb = np.asarray(src)
    return [psnr(rgb, np.stack(rec))], [msssim_rgb(rgb, np.stack(rec)) if calc_ssim else 0.]


class HostDistortion:
    """Distortion's interface (dcvc_b200.metrics) on the host, for driving run_job without a device"""

    def __init__(self, src_type, height, width, calc_ssim, capacity):
        self.args = (src_type, height, width)
        self.calc_ssim, self.capacity = calc_ssim, capacity
        self.psnrs, self.ssims = [], []

    def add(self, x_hat, src):
        assert len(self.psnrs) < self.capacity
        src_type, h, w = self.args
        p, s = distortion(src_type, x_hat, src, self.calc_ssim, h, w)
        self.psnrs.append(p)
        self.ssims.append(s)

    def results(self):
        return self.psnrs, self.ssims


def pair(h: int, w: int, seed: int):
    """seeded (uint8 source, fp16 reconstruction) plane pair: smooth content plus noise, both saturating somewhere"""
    rng = np.random.default_rng(seed)
    a = rng.random((h + 6, w + 6))
    k = np.ones(7) / 7
    a = np.apply_along_axis(lambda r: np.convolve(r, k, mode="valid"), 1, a)
    a = np.apply_along_axis(lambda c: np.convolve(c, k, mode="valid"), 0, a)
    a = (a - a.mean()) / a.std() * 60 + 128
    src = np.clip(np.round(a), 0, 255).astype(np.uint8)
    rec = np.clip(src.astype(np.float64) + rng.normal(0, 4, (h, w)), 0, 255).astype(np.float16)
    return src, rec
