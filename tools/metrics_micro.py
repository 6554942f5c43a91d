"""Timing of the device distortion metrics (dcvc_b200.metrics.Distortion) against the reference's host get_distortion,
and the wall time of a 97-frame 1080p HT-S job through dcvc_b200.sequence.run_job with MS-SSIM on and off.

    python tools/metrics_micro.py [--iters 200] [--host-iters 3] [--out results.json]

Device times are CUDA events around each Distortion.add; between timed calls a 512 MB buffer is overwritten so every
call reads its inputs from HBM, not from the 126 MB L2.  The reference's get_distortion is timed on this host's CPU
(it needs the reference byte-code in oracle/_ref/py)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from dcvc_b200 import model  # noqa: E402
from dcvc_b200.metrics import Distortion  # noqa: E402
from dcvc_b200.sequence import run_job  # noqa: E402
from util_frames import synth_frame  # noqa: E402

H, W, HP = 1080, 1920, 1088


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def picture(src_type, seed):
    base = synth_frame(HP, W, seed)
    g = torch.Generator().manual_seed(seed)
    x_hat = (base + (torch.rand(base.shape, generator=g) - 0.5) * 0.06).half()
    u8 = ((base[0, :, :H] + 0.5) * 255).round().clamp(0, 255).byte()
    if src_type == "png":
        return x_hat, None, None, None, u8.numpy().copy()
    return (x_hat, u8[0].numpy().copy(), np.ascontiguousarray(u8[1, ::2, ::2].numpy()),
            np.ascontiguousarray(u8[2, ::2, ::2].numpy()), None)


def time_device(src_type, calc_ssim, iters, flush):
    x_hat, y, u, v, rgb = picture(src_type, 3)
    x_hat = x_hat.cuda().contiguous(memory_format=torch.channels_last)
    src = torch.from_numpy(rgb).cuda() if src_type == "png" else tuple(torch.from_numpy(p).cuda() for p in (y, u, v))
    d = Distortion(src_type, H, W, calc_ssim, capacity=1)
    for _ in range(20):
        d.reset()
        d.add(x_hat, src)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for e0, e1 in ev:
        flush.fill_(1)
        d.reset()
        e0.record()
        d.add(x_hat, src)
        e1.record()
    torch.cuda.synchronize()
    ms = np.array([e0.elapsed_time(e1) for e0, e1 in ev])
    return {"median_ms": float(np.median(ms)), "p10_ms": float(np.percentile(ms, 10)),
            "p90_ms": float(np.percentile(ms, 90)), "iters": iters}


def time_host(src_type, iters):
    from oracle.build_ref import py_surface_root
    root = py_surface_root()
    if root is None:
        return None
    for p in (root, os.path.join(ROOT, "oracle", "_ref")):
        sys.path.insert(0, p)
    import test_video
    x_hat, y, u, v, rgb = picture(src_type, 3)
    x_hat = x_hat.cuda()[:, :, :H, :W]
    out = []
    for _ in range(iters):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        test_video.get_distortion({"src_type": src_type, "calc_ssim": True}, x_hat, y, u, v, rgb)
        out.append(time.perf_counter() - t0)
    return {"median_s": float(np.median(out)), "iters": iters}


def time_job(calc_ssim, frames=97, qp=32):
    pics = [((synth_frame(H, W, 500 + i)[0] + 0.5) * 255).round().clamp(0, 255).byte() for i in range(frames)]
    src = [(p[0].contiguous().cuda(), p[1, ::2, ::2].contiguous().cuda(), p[2, ::2, ::2].contiguous().cuda()) for p in pics]
    i_net = model.DMCI.synthetic(0)
    i_net.update(0.15)
    i_net = i_net.half().to("cuda")
    p_net = model.DMC.synthetic()
    p_net.update(0.15)
    p_net = p_net.half().to("cuda")
    run_job(i_net, p_net, src[:17], H, W, qp, qp, 8, calc_ssim=calc_ssim)        # warm-up: plans, arenas, kernels
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    _, log = run_job(i_net, p_net, src, H, W, qp, qp, 8, calc_ssim=calc_ssim, verbose=1)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    return {"frames": frames, "wall_s": wall, "test_time_s": log["test_time"],
            "avg_unit_encoding_s": log.get("avg_frame_encoding_time"),
            "avg_unit_decoding_s": log.get("avg_frame_decoding_time"),
            "ave_all_frame_psnr": log["ave_all_frame_psnr"], "ave_all_frame_msssim": log["ave_all_frame_msssim"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--host-iters", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("metrics_micro.py needs a CUDA device")
    res = {"card": card(), "picture": f"{H}x{W} (x_hat {HP}x{W})",
           "l2": "512 MB buffer overwritten before every timed call (inputs read from HBM)"}
    print("[card]", res["card"])
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    for src_type in ("yuv420", "png"):
        for ssim in (False, True):
            r = time_device(src_type, ssim, a.iters, flush)
            res[f"device_{src_type}_ssim{int(ssim)}"] = r
            print(f"[device] {src_type} calc_ssim={int(ssim)}: median {r['median_ms']:.3f} ms "
                  f"(p10 {r['p10_ms']:.3f}, p90 {r['p90_ms']:.3f}) over {r['iters']}")
    del flush
    for src_type in ("yuv420", "png"):
        r = time_host(src_type, a.host_iters)
        res[f"host_get_distortion_{src_type}"] = r
        print(f"[host] reference get_distortion {src_type} calc_ssim=1: {r}")
    for ssim in (False, True):
        r = time_job(ssim)
        res[f"job_hts_97f_ssim{int(ssim)}"] = r
        print(f"[job] HT-S 97 frames 1080p calc_ssim={int(ssim)}: {r}")
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
