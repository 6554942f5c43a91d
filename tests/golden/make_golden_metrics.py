"""Generates tests/golden/metrics_reference.json from the REFERENCE's own functions: calc_psnr, calc_ssim,
calc_msssim and calc_msssim_rgb (src/utils/metrics.py) on seeded plane pairs, and generate_log_json
(src/utils/common.py:46-116) on seeded per-picture records.  Run with a checkout of the reference:

    python tests/golden/make_golden_metrics.py path/to/reference

Inputs are regenerated from their seeds by tests/metrics_oracle.pair (their SHA-256 is stored to catch drift).
Per-level values come from the reference's calc_ssim applied level by level with the reference's own downsampling
call (ndimage.convolve(ones(2,2)/4, mode='reflect')[::2, ::2], metrics.py:84-89).
"""
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "tests"))
if len(sys.argv) != 2 or not os.path.isdir(os.path.join(sys.argv[1], "src", "utils")):
    sys.exit("usage: python tests/golden/make_golden_metrics.py path/to/reference")
sys.path.insert(0, os.path.abspath(sys.argv[1]))
from scipy import ndimage  # noqa: E402

from src.utils.common import generate_log_json  # noqa: E402  (reference)
from src.utils.metrics import calc_msssim, calc_msssim_rgb, calc_psnr, calc_ssim  # noqa: E402  (reference)

from metrics_oracle import pair  # noqa: E402

SIZES = [(88, 88), (88, 120), (175, 177), (176, 176), (270, 481), (540, 960)]
RGB_SIZES = [(88, 120), (270, 481)]


def levels(src, rec):
    level = 4 if min(src.shape) < 176 else 5
    im1, im2 = src.astype(np.float64), rec.astype(np.float64)
    mssim, mcs = [], []
    f = np.ones((2, 2)) / 4.0
    for _ in range(level):
        s, c = calc_ssim(im1, im2)
        mssim.append(float(s.mean()))
        mcs.append(float(c.mean()))
        im1 = ndimage.convolve(im1, f, mode="reflect")[::2, ::2]
        im2 = ndimage.convolve(im2, f, mode="reflect")[::2, ::2]
    return mssim, mcs


def digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def main():
    out = {"planes": [], "rgb": [], "log_json": []}
    for i, (h, w) in enumerate(SIZES):
        src, rec = pair(h, w, 100 + i)
        mssim, mcs = levels(src, rec)
        out["planes"].append({"h": h, "w": w, "seed": 100 + i, "sha256": digest(src, rec),
                              "psnr": float(calc_psnr(src, rec)), "msssim": float(calc_msssim(src, rec)),
                              "mssim": mssim, "mcs": mcs})
    for i, (h, w) in enumerate(RGB_SIZES):
        ps = [pair(h, w, 200 + 3 * i + c) for c in range(3)]
        src, rec = np.stack([p[0] for p in ps]), np.stack([p[1] for p in ps])
        out["rgb"].append({"h": h, "w": w, "seeds": [200 + 3 * i + c for c in range(3)], "sha256": digest(src, rec),
                           "psnr": float(calc_psnr(src, rec)), "msssim": float(calc_msssim_rgb(src, rec))})
    rng = np.random.default_rng(7)
    for src_type in ("yuv420", "png"):
        for verbose in (False, True):
            for timed in (False, True):
                n = 19
                frame_types = [0] + [1] * 8 + [1] * 8 + [0] + [1]
                bits = [int(b) for b in rng.integers(1000, 90000, n)]
                k = 4 if src_type == "yuv420" else 1
                psnrs = [[float(v) for v in rng.uniform(25, 45, k)] for _ in range(n)]
                ssims = [[float(v) for v in rng.uniform(0.8, 1.0, k)] for _ in range(n)]
                args = dict(frame_num=n, frame_pixel_num=180 * 264, test_time=12.5, frame_types=frame_types,
                            bits=bits, psnrs=psnrs, ssims=ssims, verbose=verbose,
                            avg_encoding_time=0.0125 if timed else None, avg_decoding_time=0.0111 if timed else None)
                log = generate_log_json(**args)
                out["log_json"].append({"args": args, "log": json.loads(json.dumps(log))})
    with open(os.path.join(HERE, "metrics_reference.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
