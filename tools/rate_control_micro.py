"""Cost of rate control at 1080p for every codec kind (synthetic checkpoints and pictures):

* one compress() against one estimate_bits() pass (one QP), host clock around calls that end in a device synchronise;
* the rate kernel alone (torch.profiler, CUDA activities, the rate_estimate_kernel launches of a 16-QP estimate);
* encode FPS of a sequence at fixed QP against the same sequence rate-controlled to the fixed run's bitrate at q 40,
  with the mean number of trials per unit and the achieved against the target bitrate.

    python tools/rate_control_micro.py [--frames 17] [--iters 10] [--out results.json]

Prints its results; writes JSON only with --out."""
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
from dcvc_b200.model import DMC, DMCHTL, DMCI, DMCLD  # noqa: E402
from dcvc_b200.rate_control import RateController  # noqa: E402
from dcvc_b200.sequence import SequenceEncoder  # noqa: E402
from util_frames import synth_frame  # noqa: E402

H, W, SKIP, FPS = 1080, 1920, 0.15, 30.0


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def planes(n):
    out = []
    for t in range(n):
        f = synth_frame(H, W, 100 + t)[0]
        u8 = ((f + 0.5) * 255).round().clamp(0, 255).byte()
        out.append((u8[0].cuda().contiguous(), u8[1, ::2, ::2].cuda().contiguous(), u8[2, ::2, ::2].cuda().contiguous()))
    return out


def wall(fn, iters):
    fn()
    torch.cuda.synchronize()
    t = []
    for _ in range(iters):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        t.append(time.perf_counter() - t0)
    return 1e3 * float(np.median(t))


def kernel_us(fn):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    ts = [e.device_time for e in prof.events() if "rate_estimate_kernel" in e.name]
    return float(np.mean(ts)) if ts else float("nan"), len(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=17)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    i_net = DMCI.synthetic(0)
    i_net.update(SKIP)
    i_net = i_net.half().to("cuda")
    pad_r, pad_b = i_net.get_padding_size(H, W, 16)
    res = {"card": card(), "size": f"{H}x{W}", "frames": args.frames, "kinds": {}}
    print(f"[rate] {res['card']}, {H}x{W}")
    frames = planes(args.frames)
    for kind, cls, seed, delay in (("intra", None, 0, 1), ("hts", DMC, 1, 8), ("ld", DMCLD, 2, 1), ("htl", DMCHTL, 3, 8)):
        if cls is None:
            net, n_in = i_net, 1
        else:
            net = cls.synthetic(seed)
            net.update(SKIP)
            net = net.half().to("cuda")
            n_in = 8 if delay == 8 else 1
        x = torch.cat([synth_frame(H, W, 7 + i) for i in range(n_in)], dim=1).half().cuda()
        x = x.contiguous(memory_format=torch.channels_last)
        if kind == "intra":
            comp = lambda: net.compress(x, 40, pad_b, pad_r)                         # noqa: E731
            est = lambda qps=(40,): net.estimate_bits(x, list(qps), pad_b, pad_r)   # noqa: E731
        else:
            e = i_net.compress(synth_frame(H, W, 5).half().cuda().contiguous(memory_format=torch.channels_last), 40, pad_b, pad_r)
            net.clear_dpb()
            net.add_ref_feature_from_frame(e["x_hat"])
            comp = lambda: net.compress(x, 40, 0, pad_b, pad_r)                      # noqa: E731
            est = lambda qps=(40,): net.estimate_bits(x, list(qps), 0, pad_b, pad_r)  # noqa: E731
        ms_comp, ms_est = wall(comp, args.iters), wall(est, args.iters)
        k_us, k_n = kernel_us(lambda: est(range(0, 64, 4)))

        def encode(rc, qp=40):
            enc = SequenceEncoder(i_net, net if kind != "intra" else i_net, H, W, qp, qp, frame_delay=delay,
                                  force_intra=kind == "intra", rate_control=rc)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            data = enc.encode(frames)
            torch.cuda.synchronize()
            return data, time.perf_counter() - t0
        encode(None)
        fixed, t_fixed = encode(None)
        target = len(fixed) * 8 / (args.frames / FPS) / 1000
        rc = RateController(target, fps=FPS)
        data, t_rc = encode(rc)
        trials = float(np.mean([len(u["tried"]) for u in rc.history]))
        r = {"compress_ms": ms_comp, "estimate_ms": ms_est, "rate_kernel_us": k_us, "rate_kernel_launches": k_n,
             "fixed_fps": args.frames / t_fixed, "rc_fps": args.frames / t_rc, "trials_per_unit": trials,
             "target_kbps": target, "achieved_kbps": len(data) * 8 / (args.frames / FPS) / 1000,
             "qps": [u["qp"] for u in rc.history]}
        res["kinds"][kind] = r
        print(f"[rate] {kind}: compress {ms_comp:.2f} ms, estimate {ms_est:.2f} ms, rate kernel {k_us:.1f} us "
              f"({k_n} launches); encode {r['fixed_fps']:.1f} FPS fixed q40, {r['rc_fps']:.1f} FPS rate-controlled "
              f"({trials:.2f} trials/unit); {r['achieved_kbps']:.0f} of {target:.0f} kbps, qps {r['qps']}")
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
