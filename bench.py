#!/usr/bin/env python
"""bench.py — DCVC-UF-Intra 1080p decode/encode throughput on N x B200 (BASELINE.json configs[1]).

A "step" is one pass of the hot path over one synthetic 1080p 4:4:4 frame: `DMCI.decompress` of a
bitstream produced beforehand by `DMCI.compress` (neural synthesis + entropy-parameter path on the
GPU, rANS on the host CPU, exactly the reference's FPS protocol: test_video.py:295-325).  `value`
keeps the reconstruction in HBM; `e2e` additionally copies the reconstruction to pinned host memory
inside the timed region.  Encode FPS, GPU-only segment time, the per-kernel-family roofline and the
CPU baseline (oracle port on the host cores) ride along in the same JSON line.

  python bench.py --gpus 1 --steps 20 --warmup 5
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference        # the reference's CPU path (oracle port + reference rANS)
  python bench.py --dump-outputs DIR      # also writes what the last timed Intra decode / e2e / encode step returned
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

H, W = 1080, 1920
# Test hook of the CPU tier only (tests/dry_bench_runner.py runs this file's control flow on the emulated runtime at a
# tiny size to check the JSON contract): the driver never sets it, and a line produced with it says so.
_SIZE_OVERRIDE = os.environ.get("DCVC_B200_BENCH_TEST_SIZE")
if _SIZE_OVERRIDE:
    H, W = (int(v) for v in _SIZE_OVERRIDE.split("x"))
QP = 32
SKIP = 0.15  # test_compress_time.py:41
METRIC = "1080p_yuv_decode_fps"
# SURVEY.md §8(d): algorithmic bytes of the Intra decode side at the reference's fusion granularity
ALG_BYTES_DECODE = 5.89e9
ALG_GMAC_DECODE = 701.2


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1590.0, "fallback"


class ClockSampler(threading.Thread):
    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples = []
        self.stop_flag = False

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([s.strip() for s in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        mx = [int(s[1]) for s in self.samples if s[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples if len(s) > 2 + i)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons}


# at most this many bytes of .npy per --dump-outputs directory
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """Writes each array as path/<name>.npy in float32 (float64 stays float64): what a caller of the timed path received
    in the last timed step, so that two builds run with the same arguments (hence the same seeded inputs) can be compared
    output for output."""
    out = {}
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
        out[name] = a if a.dtype == np.float64 else a.astype(np.float32)
    total = sum(a.nbytes for a in out.values())
    assert total <= DUMP_LIMIT_BYTES, f"--dump-outputs: {total} bytes exceed {DUMP_LIMIT_BYTES}"
    os.makedirs(path, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a)


def make_model(device, world, rank):
    """rank 0 generates the synthetic checkpoint; it is broadcast once over NCCL (SURVEY.md §8e)."""
    import torch.distributed as dist
    from dcvc_b200.model import DMCI
    from dcvc_b200.spec import dmci_spec, synth_state_dict
    from dcvc_b200.shard import broadcast_state_dict
    spec = dmci_spec()
    if world == 1:
        sd = synth_state_dict(spec, 0)
    else:
        sd = broadcast_state_dict(synth_state_dict(spec, 0) if rank == 0 else None, spec, 0, device)
    m = DMCI()
    m.load_state_dict(sd)
    m.update(SKIP)
    return m.half().to(device)


def run_ours(args):
    import torch.distributed as dist
    from util_frames import psnr, synth_frame
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (the product has no CPU path)"
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    # DCVC_B200_PIN=1: host threads of this rank (the rANS pool is created with the first proxy) on the GPU's socket and
    # on their own cores (opt-in: within the run-to-run spread when measured, dcvc_b200/shard.py)
    from dcvc_b200.shard import pin_rank
    numa = pin_rank(local, int(os.environ.get("LOCAL_WORLD_SIZE", str(world))))
    model = make_model(device, world, rank)
    stream = torch.cuda.Stream(device)
    torch.cuda.set_stream(stream)  # a non-default stream, like test_video.py:423-425

    x = synth_frame(H, W, 1234 + rank).half().to(device).contiguous(memory_format=torch.channels_last)
    pad_r, pad_b = model.get_padding_size(H, W, 16)
    sps = {"height": H, "width": W}
    enc = model.compress(x, QP, pad_b, pad_r)
    x_hat_enc = enc["x_hat"].clone()
    bs = enc["bit_stream"]
    dec = model.decompress(bs, sps, QP, enc["ec_parallel"])
    torch.cuda.synchronize()
    assert torch.equal(x_hat_enc, dec["x_hat"]), "decode does not match encode"
    # now, not at the end: the reconstruction lives in a proxy-owned buffer that the later legs (which share this Intra
    # model for their I frames, also at another resolution) write again
    psnr_ours = psnr(x_hat_enc.float().cpu()[:, :, :H, :W], x.float().cpu())
    totals = model.proxy.debug_fetch("totals", np.int32)
    n_sym = int(totals.sum())
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
    # e2e result = the decoded picture as the reference's driver writes it: 8-bit YUV 4:2:0 planes
    # (test_video.py:352-361), converted on the device (dcvc_b200/frame_io.py) and copied to pinned host memory
    from dcvc_b200 import frame_io
    dev_planes = (torch.empty((H, W), dtype=torch.uint8, device=device),
                  torch.empty((H // 2, W // 2), dtype=torch.uint8, device=device),
                  torch.empty((H // 2, W // 2), dtype=torch.uint8, device=device))
    host_planes = tuple(torch.empty(t.shape, dtype=torch.uint8).pin_memory() for t in dev_planes)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier()
        for e0, e1 in evs:
            flush.zero_()            # evict L2 between timed iterations (outside the timed interval)
            e0.record()
            fn()
            e1.record()
        barrier()
        return [e0.elapsed_time(e1) for e0, e1 in evs]

    last = {}   # what the latest step returned (read for --dump-outputs after its timed loop)

    def step_dec():
        last["dec"] = model.decompress(bs, sps, QP, enc["ec_parallel"])

    def step_dec_e2e():
        out = model.decompress(bs, sps, QP, enc["ec_parallel"])["x_hat"]
        frame_io.frame_to_yuv420(out, H, W, out=dev_planes)
        for hp, dp in zip(host_planes, dev_planes):
            hp.copy_(dp, non_blocking=True)
        torch.cuda.current_stream().synchronize()   # the caller owns the host planes when the step ends

    def step_enc():
        last["enc"] = model.compress(x, QP, pad_b, pad_r)

    for _ in range(args.warmup):
        step_dec(); step_dec_e2e(); step_enc()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = model.proxy.kernel_launches()
    t_dec = timed(step_dec, args.steps)
    l1 = model.proxy.kernel_launches()
    gpu_only_ms = model.proxy.last_gpu_ms()
    dumps = {}
    if args.dump_outputs:
        # x_hat is a proxy-owned buffer that the next decode writes again: copied before the e2e loop
        dumps["decode_x_hat"] = last["dec"]["x_hat"].float().cpu()
    t_e2e = timed(step_dec_e2e, args.steps)
    t_enc = timed(step_enc, args.steps)
    if args.dump_outputs:
        for name, t in zip(("e2e_y", "e2e_u", "e2e_v"), host_planes):
            dumps[name] = t.clone()
        dumps["encode_bit_stream"] = np.frombuffer(last["enc"]["bit_stream"], dtype=np.uint8)
    sampler.stop_flag = True
    sampler.join(timeout=2)

    def reduce_max(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    tot_dec = reduce_max(sum(t_dec))
    tot_e2e = reduce_max(sum(t_e2e))
    tot_enc = reduce_max(sum(t_enc))

    # ---- per-kernel-family roofline (CUDA events around every launch, graphs off)
    hbm_peak, tf_peak, peak_src = _peaks()
    model.proxy.profile_enable(True)
    for _ in range(3):
        step_dec()
    torch.cuda.synchronize()
    prof = model.proxy.profile_get()
    model.proxy.profile_enable(False)
    # the dominant KERNEL of the step = the __global__ function with the largest share of the GPU time: the fused
    # DepthConvBlock tail (dcb_tail_kernel) or one of the five instantiations of the per-op GEMM (pw_gemm_kernel<BN, fold>; ncu
    # lists them as separate kernels too).  "pw_gemm" is the sum over the instantiations (reported alongside).
    families = ("pw_gemm", "dw3x3", "elementwise", "dcb_tail")
    kernels = ("dcb_tail",) + tuple(k for k in prof if k.startswith("pw_gemm<"))
    fam = max(kernels, key=lambda k: prof.get(k, {"ms": 0.0})["ms"])
    g = prof[fam]
    roofline = None
    if g["launches"]:
        n_prof = 3
        total_ms = max(1e-9, sum(prof[k]["ms"] for k in families if k in prof))
        share = g["ms"] / total_ms
        # Duration of the dominant kernel inside the timed step: its share of the GPU time (CUDA events around every
        # launch, graphs off: those intervals include launch gaps and lose the PDL overlap, so they are reported
        # separately as *_isolated) x the GPU-only time of the timed, graph-launched decode (CUDA events around the
        # graph segments).  ncu's launch list gives the same share (profiles/README.md).
        ms_in_step = share * gpu_only_ms
        alg_per_step = g["alg_bytes"] / n_prof
        flops_per_step = g["flops"] / n_prof
        gbs = alg_per_step / (ms_in_step * 1e-3) / 1e9
        tfs = flops_per_step / (ms_in_step * 1e-3) / 1e12
        gbs_iso = g["alg_bytes"] / (g["ms"] * 1e-3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", f"traffic_{'dcb_tail' if fam == 'dcb_tail' else 'pw_gemm'}.json")
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get("dram_bytes_per_launch")
        launches_per_step = g["launches"] // n_prof
        roofline = {"bound": "hbm", "kernel": ("dcb_tail_kernel" if fam == "dcb_tail" else fam.replace("pw_gemm<", "pw_gemm_kernel<")), "achieved": round(gbs, 1), "peak": hbm_peak, "unit": "GB/s",
                    "frac": round(gbs / hbm_peak, 4), "traffic": traffic, "peak_source": peak_src,
                    "method": "algorithmic bytes of the kernel's launches in one step / (share_of_gpu_time x GPU-only ms of the timed step)",
                    "launches_per_step": launches_per_step,
                    "avg_launch_us": round(ms_in_step * 1e3 / launches_per_step, 2),
                    "alg_bytes_per_launch": round(g["alg_bytes"] / g["launches"]),
                    "tensor_tflops": round(tfs, 1), "tensor_frac": round(tfs / tf_peak, 4),
                    "share_of_gpu_time": round(share, 3),
                    "achieved_isolated": round(gbs_iso, 1), "frac_isolated": round(gbs_iso / hbm_peak, 4),
                    "avg_launch_us_isolated": round(g["ms"] * 1e3 / g["launches"], 2),
                    "families_ms_per_step_isolated": {k: round(v["ms"] / n_prof, 3) for k, v in prof.items()},
                    "families_launches_per_step": {k: int(v["launches"] // n_prof) for k, v in prof.items()},
                    "families_alg_gbs_in_step": {k: round(v["alg_bytes"] / n_prof / max(1e-9, v["ms"] / total_ms * gpu_only_ms * 1e-3) / 1e9, 1)
                                                 for k, v in prof.items() if v["alg_bytes"] > 0},
                    "whole_decode_alg_gbs": round(ALG_BYTES_DECODE / (gpu_only_ms * 1e-3) / 1e9, 1),
                    "whole_decode_frac": round(ALG_BYTES_DECODE / (gpu_only_ms * 1e-3) / 1e9 / hbm_peak, 4)}

    # ---- HT-S chunk codec (configs[2]: the reference's published B200 headline, BASELINE.md) rides along
    hts = None
    if not args.no_hts:
        hts = bench_hts(model, device, world, rank, args, timed, reduce_max)

    # ---- LD codec rides along too; it must never take the headline numbers down with it
    ld = None
    if not args.no_hts and world == 1:   # single-GPU runs only: no collective may depend on this optional leg
        try:
            ld = bench_ld(model, device, world, rank, args, timed, reduce_max)
        except Exception as e:  # noqa: BLE001 — reported in the JSON line instead of failing the bench
            ld = {"error": f"{type(e).__name__}: {e}"}

    # ---- HT-L: same leg with the large model, failure-isolated like LD
    htl = None
    if not args.no_hts and world == 1:
        try:
            htl = bench_hts(model, device, world, rank, args, timed, reduce_max, large=True)
        except Exception as e:  # noqa: BLE001
            htl = {"error": f"{type(e).__name__}: {e}"}

    # ---- configs[4]: the HT-S leg again at 4K (single-GPU runs; --hts-size HxW picks another size, "none" skips it)
    hts_extra = None
    if args.hts_size.lower() != "none" and not args.no_hts and world == 1 and not (_SIZE_OVERRIDE and args.hts_size == "2160x3840"):
        try:
            eh, ew = (int(v) for v in args.hts_size.lower().split("x"))
            hts_extra = bench_hts(model, device, world, rank, args, timed, reduce_max, hw=(eh, ew))
        except Exception as e:  # noqa: BLE001
            hts_extra = {"error": f"{type(e).__name__}: {e}"}

    # ---- configs[3]: the runtime job list (8 sequences x 4 rate points) sharded over the ranks
    seq8 = None
    if not args.no_hts and not args.no_seq8:
        try:
            seq8 = bench_seq8(model, device, world, rank, args, **({"n_seq": 2, "n_frames": 17} if _SIZE_OVERRIDE else {}))
        except Exception as e:  # noqa: BLE001 (set-up failures only: the job loop reports through the gather)
            seq8 = {"error": f"{type(e).__name__}: {e}"}
            if world > 1:
                raise

    # ---- two independent decodes in flight per GPU (two proxies, two streams, two host threads): serving-style throughput
    # beside the headline (--no-pipelined skips it; not run under the CPU test tier's size override)
    pipelined = None
    if not args.no_pipelined and world == 1 and not os.environ.get("DCVC_B200_BENCH_TEST_SIZE"):
        try:
            pipelined = bench_pipelined(model, device, bs, sps, enc["ec_parallel"], args)
        except Exception as e:  # noqa: BLE001
            pipelined = {"error": f"{type(e).__name__}: {e}"}

    # ---- the reference's own CUDA extension (CUTLASS, compiled for sm_100a by baseline/build_ref_cuda.py) under the
    # reference's own models, same box, same checkpoints / frames / protocol, in its own process (rank 0, N=1 only)
    reference_cuda = None
    if rank == 0 and world == 1 and not args.no_reference_cuda and not _SIZE_OVERRIDE:
        reference_cuda = run_reference_cuda(args)

    # ---- CPU baseline: the oracle port on the host cores (rank 0, N=1 only), bounded sample
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline = cpu_reference_sample(steps=1, sample_hw=(H, W))
        try:  # what the reference's own driver pins (src/utils/common.py:264-272: torch.set_num_threads(1))
            one = cpu_reference_sample(steps=1, sample_hw=(H, W), threads=1)
            cpu_baseline["single_thread"] = {k: one[k] for k in ("value", "unit", "cores", "sample", "seconds_per_sample")}
        except Exception as e:  # noqa: BLE001
            cpu_baseline["single_thread"] = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        fps = world * args.steps / (tot_dec * 1e-3)
        out = {
            "metric": METRIC, "value": round(fps, 2), "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(tot_dec / args.steps, 4), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {"workload": "DCVC-UF-Intra 1080p single-frame decode (configs[1]), q_index 32, skip_thres 0.15, "
                                   "one independent frame per GPU", "resolution": [H, W], "qp": QP,
                       "l2": "flushed between timed steps (256 MiB memset outside the timed interval)",
                       "weights": "seeded synthetic checkpoint (no checkpoints offline)"},
            "e2e": {"value": round(world * args.steps / (tot_e2e * 1e-3), 2), "unit": "frames/s",
                    "h2d_bytes_per_step": int(65280 + n_sym), "d2h_bytes_per_step": int(n_sym + 16 + sum(t.numel() for t in host_planes)),
                    "result": "8-bit YUV 4:2:0 planes in pinned host memory (frame_to_yuv420 on the device)",
                    "bitstream_bytes": len(bs)},
            "encode_fps": round(world * args.steps / (tot_enc * 1e-3), 2),
            "gpu_only_ms_per_decode": round(gpu_only_ms, 4),
            "gpu_launches": int(l1 - l0),
            "bpp": round(len(bs) * 8 / (H * W), 4),
            "psnr_db": round(psnr_ours, 3),
            "clocks": sampler.summary(),
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
            "hts": hts,
            "ld": ld,
            "htl": htl,
            "pipelined": pipelined,
            "seq8": seq8,
            "hts_extra": hts_extra,
            "reference_cuda": reference_cuda,
            "host": {"cpus": os.cpu_count(), "numa_pinned_cpus": (len(numa) if numa else None)},
            # every DCVC_B200_* switch of the environment (none in the driver's runs): an A/B line describes itself
            "switches": {k: v for k, v in sorted(os.environ.items()) if k.startswith("DCVC_B200_")},
        }
        if reference_cuda and "intra" in reference_cuda:
            # same frame, same checkpoint, same q_index: the product next to the reference's CUDA path
            ri = reference_cuda["intra"]
            out["parity"] = {"against": "reference CUDA extension, same box", "frame": "1080p synth seed 1234, q_index 32",
                             "bytes": [len(bs), ri["bytes"]], "d_bpp": round(abs(len(bs) - ri["bytes"]) * 8 / (H * W), 6),
                             "psnr_db": [round(psnr_ours, 4), ri["psnr_db"]], "d_psnr_db": round(abs(psnr_ours - ri["psnr_db"]), 5)}
            sp = {"intra_decode": round(out["value"] / ri["decode_fps"], 3), "intra_encode": round(out["encode_fps"] / ri["encode_fps"], 3)}
            for leg, name in ((hts, "hts"), (ld, "ld"), (htl, "htl")):
                if leg and name in reference_cuda and "decode_fps" in leg:
                    sp[name + "_decode"] = round(leg["decode_fps"] / reference_cuda[name]["decode_fps"], 3)
                    sp[name + "_encode"] = round(leg["encode_fps"] / reference_cuda[name]["encode_fps"], 3)
            out["speedup_vs_reference_cuda"] = sp
        if _SIZE_OVERRIDE:
            out["INVALID_test_size_override"] = _SIZE_OVERRIDE
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dumps)
            out["dumped_outputs"] = sorted(dumps)
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def bench_seq8(i_net, device, world, rank, args, n_seq=8, n_frames=97, rate_num=4):
    """BASELINE.json configs[3]: the reference's runtime job — test_cfg/runtime_avg.json has 1080p sequences of 97 frames,
    intra period -1, four rate points each (test_video.py:527-564 submits sequence-major, rate-minor) — here 8 synthetic
    sequences, dealt in rotated blocks to the ranks (one process per GPU, no cross-GPU dependency), each job coded and decoded
    through the sequence driver (dcvc_b200/sequence.py = the loop of test_video.py:204-372) with the reference's timing
    protocol per coded unit (first four units dropped, test_video.py:375-381).  Results are gathered on rank 0."""
    import torch.distributed as dist
    from dcvc_b200.model import DMC
    from dcvc_b200.sequence import SequenceDecoder, SequenceEncoder, UnitTimer
    from dcvc_b200.shard import broadcast_state_dict, shard_jobs
    from dcvc_b200.spec import hts_spec, synth_state_dict
    spec = hts_spec()
    sd = synth_state_dict(spec, 1) if world == 1 else broadcast_state_dict(synth_state_dict(spec, 1) if rank == 0 else None, spec, 0, device)
    p_net = DMC()
    p_net.load_state_dict(sd)
    p_net.update(SKIP)
    p_net = p_net.half().to(device)
    qps = [int(i + 0.5) for i in np.linspace(0, 63, num=rate_num)]          # test_video.py:507-510
    jobs = [(seq, r) for seq in range(n_seq) for r in range(rate_num)]       # test_video.py:527-564 order
    mine = shard_jobs(jobs, rank, world)

    def sequence_planes(seq):
        """a drifting band-limited texture: 97 pictures of 8-bit 4:2:0 planes, made on the device"""
        g = torch.Generator(device="cpu").manual_seed(7000 + seq)
        base = torch.rand((1, 1, H + 104, W + 104), generator=g)
        base = torch.nn.functional.avg_pool2d(base, 5, 1).to(device)
        base = ((base - base.mean()) / base.std() * 0.18 + 0.5).clamp(0, 1)[0, 0]
        out = []
        for t in range(n_frames):
            img = base[t:t + H, (t // 2):(t // 2) + W]
            y = (img * 255).round().to(torch.uint8).contiguous()
            u = ((img[::2, ::2] * 0.5 + 0.25) * 255).round().to(torch.uint8).contiguous()
            v = ((img[1::2, 1::2] * 0.4 + 0.3) * 255).round().to(torch.uint8).contiguous()
            out.append((y, u, v))
        return out

    results = []
    frames_cache = {}
    t_enc_sum = t_dec_sum = 0.0
    err = None
    for seq, r in mine:
        try:
            if seq not in frames_cache:
                frames_cache.clear()
                frames_cache[seq] = sequence_planes(seq)
            frames = frames_cache[seq]
            enc = SequenceEncoder(i_net, p_net, H, W, qp_i=qps[r], qp_p=qps[r], frame_delay=8, intra_period=-1, reset_interval=32)
            enc.timer = UnitTimer(device)
            data = enc.encode(frames)
            dec = SequenceDecoder(i_net, p_net, frame_delay=8)
            dec.timer = UnitTimer(device)
            sse = 0.0
            for k, (y, u, v) in enumerate(dec.decode(data, n_frames)):
                if k % 16 == 0:   # PSNR-Y of a few pictures: a sanity value for the line, not a quality claim (random weights)
                    sse += float(((y.float() - frames[k][0].float()) ** 2).mean())
            torch.cuda.synchronize()
            e_ms, d_ms = enc.unit_ms[4:], dec.unit_ms[4:]
            t_enc_sum += sum(enc.unit_ms)
            t_dec_sum += sum(dec.unit_ms)
            results.append({"seq": seq, "rate_idx": r, "qp": qps[r], "bytes": len(data), "bpp": len(data) * 8 / (n_frames * H * W),
                            "avg_unit_enc_ms": sum(e_ms) / len(e_ms), "avg_unit_dec_ms": sum(d_ms) / len(d_ms),
                            "psnr_y_db": 10 * np.log10(255.0 ** 2 / max(sse / ((n_frames + 15) // 16), 1e-9))})
        except Exception as e:  # noqa: BLE001 — a failing job must not keep this rank out of the gather below
            err = f"{type(e).__name__}: {e}"
            break
    local = {"rank": rank, "jobs": results, "enc_ms": t_enc_sum, "dec_ms": t_dec_sum, "error": err}
    if world > 1:
        gathered = [None] * world if rank == 0 else None
        dist.gather_object(local, gathered, dst=0)
    else:
        gathered = [local]
    del p_net
    if rank != 0:
        return None
    errors = [f"rank {part['rank']}: {part['error']}" for part in gathered if part.get("error")]
    if errors or sum(len(part["jobs"]) for part in gathered) != len(jobs):
        return {"error": "; ".join(errors) or "jobs missing"}
    alljobs = sorted((j for part in gathered for j in part["jobs"]), key=lambda j: (j["seq"], j["rate_idx"]))
    enc_fps = 8e3 / (sum(j["avg_unit_enc_ms"] for j in alljobs) / len(alljobs))
    dec_fps = 8e3 / (sum(j["avg_unit_dec_ms"] for j in alljobs) / len(alljobs))
    total_frames = n_frames * len(alljobs)
    return {"workload": f"{n_seq} synthetic {W}x{H} sequences x {n_frames} frames x {rate_num} rate points (q_index {qps}), HT-S, intra period -1, "
                        f"reset interval 32; {len(alljobs)} jobs dealt in rotated blocks to {world} rank(s) (configs[3]; test_cfg/runtime_avg.json, test_video.py:527-564)",
            "jobs": len(alljobs), "jobs_per_rank": [len(part["jobs"]) for part in gathered],
            "protocol_decode_fps": round(dec_fps, 1), "protocol_encode_fps": round(enc_fps, 1),
            "protocol": "reference per-unit timing: 8 / mean unit time, first 4 units of every job dropped (test_video.py:375-381, test_compress_time.py:48-69)",
            "aggregate_decode_fps": round(total_frames / (max(part["dec_ms"] for part in gathered) * 1e-3), 1),
            "aggregate_encode_fps": round(total_frames / (max(part["enc_ms"] for part in gathered) * 1e-3), 1),
            "aggregate": "all jobs' frames / the busiest rank's summed unit times (strong scaling: the job list is fixed)",
            "published_b200_reference_fps": {"encode": 1415.1, "decode": 945.8, "source": "BASELINE.md (HT-S, 1 GPU)"},
            "bpp_by_rate": [round(float(np.mean([j["bpp"] for j in alljobs if j["rate_idx"] == r])), 4) for r in range(rate_num)],
            "psnr_y_by_rate": [round(float(np.mean([j["psnr_y_db"] for j in alljobs if j["rate_idx"] == r])), 2) for r in range(rate_num)]}


def bench_pipelined(model, device, bs, sps, ec, args, ways=2):
    """Serving-style throughput, NOT the reference's FPS protocol (which times one call at a time): `ways` independent
    Intra decoders (own proxy, own CUDA stream, own host thread; ctypes releases the GIL inside the C ABI) decode the
    same bitstream concurrently, so one decoder's host rANS round trips overlap the other's GPU segments and one
    persistent GEMM's tail overlaps the other stream's kernels.  Timed on the device: first start event to last end
    event over all streams.  Reported beside the headline, never instead of it."""
    from dcvc_b200.model import DMCI
    from dcvc_b200.spec import dmci_spec, synth_state_dict
    nets = [model]
    for _ in range(ways - 1):
        m = DMCI()
        m.load_state_dict(synth_state_dict(dmci_spec(), 0))
        m.update(SKIP)
        nets.append(m.half().to(device))
    streams = [torch.cuda.Stream(device) for _ in nets]
    ref = model.decompress(bs, sps, QP, ec)["x_hat"].clone()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in nets]
    origin = torch.cuda.Event(enable_timing=True)
    ok = [False] * len(nets)
    gate = threading.Barrier(len(nets) + 1)

    errs = []

    def worker(i):
        try:
            torch.cuda.set_device(device)
            with torch.cuda.stream(streams[i]):
                for _ in range(args.warmup):
                    nets[i].decompress(bs, sps, QP, ec)
                streams[i].synchronize()
                gate.wait(timeout=120)
                gate.wait(timeout=120)           # the main thread has recorded `origin`
                ev[i][0].record()
                out = None
                for _ in range(args.steps):
                    out = nets[i].decompress(bs, sps, QP, ec)["x_hat"]
                ev[i][1].record()
                streams[i].synchronize()
                ok[i] = bool(torch.equal(out, ref))
        except Exception as e:  # noqa: BLE001 — a dead worker must not leave the others waiting at the gate
            errs.append(e)
            gate.abort()

    threads = [threading.Thread(target=worker, args=(i,), daemon=True) for i in range(len(nets))]
    for t in threads:
        t.start()
    try:
        gate.wait(timeout=120)
        torch.cuda.synchronize()
        origin.record(torch.cuda.default_stream(device))
        torch.cuda.synchronize()
        gate.wait(timeout=120)
    except threading.BrokenBarrierError:
        pass
    for t in threads:
        t.join(timeout=300)
    if errs or any(t.is_alive() for t in threads):
        raise RuntimeError(f"pipelined leg failed: {errs[0] if errs else 'worker did not finish'}")
    torch.cuda.synchronize()
    t_first = min(origin.elapsed_time(e0) for e0, _ in ev)
    t_last = max(origin.elapsed_time(e1) for _, e1 in ev)
    ms = t_last - t_first
    return {"ways": ways, "decode_fps": round(len(nets) * args.steps / (ms * 1e-3), 2), "ms_total": round(ms, 3),
            "bit_identical_to_single": all(ok),
            "protocol": "throughput of concurrent independent decodes on one GPU (not the reference's per-call FPS protocol)"}


def bench_hts(i_net, device, world, rank, args, timed, reduce_max, large=False, hw=None):
    """DCVC-UF HT-S 1080p chunk (8 frames) encode / decode after one intra frame (configs[2]); published B200
    numbers of the reference's CUTLASS build: 1415.1 / 945.8 FPS (BASELINE.md).  large=True: the HT-L model
    (published reference CUTLASS build on B200: 811.7 / 551.6 FPS)."""
    import torch.distributed as dist
    from util_frames import psnr, synth_frame
    from dcvc_b200.model import DMC, DMCHTL
    from dcvc_b200.shard import broadcast_state_dict
    from dcvc_b200.spec import htl_spec, hts_spec, synth_state_dict
    h, w = hw or (H, W)
    spec = htl_spec() if large else hts_spec()
    seed = 3 if large else 1
    published = {"encode": 811.7, "decode": 551.6} if large else {"encode": 1415.1, "decode": 945.8}
    if (h, w) == (2160, 3840):                           # BASELINE.md, assets/complexity.png table (d)
        published = {"encode": 237.9, "decode": 177.2} if large else {"encode": 424.0, "decode": 289.5}
    elif (h, w) != (1080, 1920):
        published = None
    # SURVEY.md §8d, per chunk at 1088x1920; scaled by the padded area for other sizes
    area = ((h + 15) // 16 * 16) * ((w + 15) // 16 * 16) / float(1088 * 1920)
    alg_bytes_decode = (17.33e9 if large else 14.09e9) * area
    if world == 1:
        sd = synth_state_dict(spec, seed)
    else:
        sd = broadcast_state_dict(synth_state_dict(spec, seed) if rank == 0 else None, spec, 0, device)
    p_net = DMCHTL() if large else DMC()
    p_net.load_state_dict(sd)
    p_net.update(SKIP)
    p_net = p_net.half().to(device)
    pad_r, pad_b = i_net.get_padding_size(h, w, 16)
    sps = {"height": h, "width": w}
    x0 = synth_frame(h, w, 4000 + rank).half().to(device).contiguous(memory_format=torch.channels_last)
    n_chunks = args.steps + args.warmup
    chunks = [synth_frame(h, w, 4100 + 10 * rank + (c % 3), channels=24).half().to(device)
              .contiguous(memory_format=torch.channels_last) for c in range(min(n_chunks, 3))]
    enc = i_net.compress(x0, QP, pad_b, pad_r)
    p_net.add_ref_feature_from_frame(enc["x_hat"])
    state = {"c": 0, "streams": []}

    def step_enc():
        c = state["c"]
        e = p_net.compress(chunks[c % len(chunks)], QP, 0, pad_b, pad_r)
        state["streams"].append((e["bit_stream"], e["ec_parallel"]))
        state["c"] += 1

    for _ in range(args.warmup):
        step_enc()
    t_enc = timed(step_enc, args.steps)
    streams = state["streams"]
    d = i_net.decompress(enc["bit_stream"], sps, QP, enc["ec_parallel"])
    p_net.add_ref_feature_from_frame(d["x_hat"], False)
    state["c"] = 0

    def step_dec():
        bs, ec = streams[state["c"]]
        state["x_hat"] = p_net.decompress(bs, sps, QP, ec, 0)["x_hat"]
        state["c"] += 1

    for _ in range(args.warmup):
        step_dec()
    l0 = p_net.proxy.kernel_launches()
    t_dec = timed(step_dec, args.steps)
    l1 = p_net.proxy.kernel_launches()
    gpu_ms = p_net.proxy.last_gpu_ms()
    tot_enc, tot_dec = reduce_max(sum(t_enc)), reduce_max(sum(t_dec))
    last = (args.warmup + args.steps - 1) % len(chunks)
    src = chunks[last][:, 0:3].float().cpu()
    out = {
        "workload": f"DCVC-UF {'HT-L' if large else 'HT-S'} {w}x{h}, 8-frame chunks after one intra frame, q_index 32, skip_thres 0.15 (configs[2])",
        "decode_fps": round(world * 8 * args.steps / (tot_dec * 1e-3), 1),
        "encode_fps": round(world * 8 * args.steps / (tot_enc * 1e-3), 1),
        "ms_per_chunk_decode": round(tot_dec / args.steps, 3), "ms_per_chunk_encode": round(tot_enc / args.steps, 3),
        "gpu_only_ms_per_chunk_decode": round(gpu_ms, 3),
        "gpu_launches_per_chunk_decode": int((l1 - l0) // args.steps),
        "bytes_per_chunk": int(np.mean([len(s[0]) for s in streams])),
        "psnr_db_frame0": round(psnr(state["x_hat"][0].float().cpu()[:, :, :h, :w], src), 3),
        "published_b200_reference_fps": dict(published, source="BASELINE.md (assets/complexity.png)") if published else None,
        "decode_vs_published": round(world * 8 * args.steps / (tot_dec * 1e-3) / published["decode"], 3) if published else None,
        "alg_gbs_decode": round(alg_bytes_decode / (gpu_ms * 1e-3) / 1e9, 1),
        "hbm_frac_decode": round(alg_bytes_decode / (gpu_ms * 1e-3) / 1e9 / _peaks()[0], 4),
    }
    del p_net
    return out


def bench_ld(i_net, device, world, rank, args, timed, reduce_max):
    """DCVC-UF LD 1080p, one frame per call after one intra frame; published B200 numbers of the reference's CUTLASS
    build: 625.6 / 621.9 FPS (BASELINE.md).  Same protocol as the HT-S leg."""
    from util_frames import psnr, synth_frame
    from dcvc_b200.model import DMCLD
    from dcvc_b200.shard import broadcast_state_dict
    from dcvc_b200.spec import ld_spec, synth_state_dict
    spec = ld_spec()
    if world == 1:
        sd = synth_state_dict(spec, 2)
    else:
        sd = broadcast_state_dict(synth_state_dict(spec, 2) if rank == 0 else None, spec, 0, device)
    p_net = DMCLD()
    p_net.load_state_dict(sd)
    p_net.update(SKIP)
    p_net = p_net.half().to(device)
    pad_r, pad_b = i_net.get_padding_size(H, W, 16)
    sps = {"height": H, "width": W}
    x0 = synth_frame(H, W, 5000 + rank).half().to(device).contiguous(memory_format=torch.channels_last)
    frames = [synth_frame(H, W, 5100 + 10 * rank + c).half().to(device).contiguous(memory_format=torch.channels_last)
              for c in range(3)]
    enc = i_net.compress(x0, QP, pad_b, pad_r)
    p_net.add_ref_feature_from_frame(enc["x_hat"])
    state = {"c": 0, "streams": []}

    def step_enc():
        c = state["c"]
        e = p_net.compress(frames[c % len(frames)], QP, 0, pad_b, pad_r)
        state["streams"].append((e["bit_stream"], e["ec_parallel"]))
        state["c"] += 1

    for _ in range(args.warmup):
        step_enc()
    t_enc = timed(step_enc, args.steps)
    streams = state["streams"]
    d = i_net.decompress(enc["bit_stream"], sps, QP, enc["ec_parallel"])
    p_net.add_ref_feature_from_frame(d["x_hat"], False)
    state["c"] = 0

    def step_dec():
        bs, ec = streams[state["c"]]
        state["x_hat"] = p_net.decompress(bs, sps, QP, ec, 0)["x_hat"]
        state["c"] += 1

    for _ in range(args.warmup):
        step_dec()
    l0 = p_net.proxy.kernel_launches()
    t_dec = timed(step_dec, args.steps)
    l1 = p_net.proxy.kernel_launches()
    gpu_ms = p_net.proxy.last_gpu_ms()
    tot_enc, tot_dec = reduce_max(sum(t_enc)), reduce_max(sum(t_dec))
    last = (args.warmup + args.steps - 1) % len(frames)
    out = {
        "workload": "DCVC-UF LD 1080p, one frame per call after one intra frame, q_index 32, skip_thres 0.15",
        "decode_fps": round(world * args.steps / (tot_dec * 1e-3), 1),
        "encode_fps": round(world * args.steps / (tot_enc * 1e-3), 1),
        "ms_per_frame_decode": round(tot_dec / args.steps, 3), "ms_per_frame_encode": round(tot_enc / args.steps, 3),
        "gpu_only_ms_per_frame_decode": round(gpu_ms, 3),
        "gpu_launches_per_frame_decode": int((l1 - l0) // args.steps),
        "bytes_per_frame": int(np.mean([len(s[0]) for s in streams])),
        "psnr_db": round(psnr(state["x_hat"].float().cpu()[:, :, :H, :W], frames[last].float().cpu()), 3),
        "published_b200_reference_fps": {"encode": 625.6, "decode": 621.9, "source": "BASELINE.md (assets/complexity.png)"},
        "decode_vs_published": round(world * args.steps / (tot_dec * 1e-3) / 621.9, 3),
    }
    del p_net
    return out


def run_reference_cuda(args):
    """baseline/run_ref_cuda.py in a subprocess (the module name inference_extensions_cuda can only mean one thing per
    process).  A missing build or a failing run is reported in the line, never raised."""
    script = os.path.join(ROOT, "baseline", "run_ref_cuda.py")
    try:
        r = subprocess.run([sys.executable, script, "--steps", str(args.steps), "--warmup", str(args.warmup)],
                           capture_output=True, text=True, timeout=900)
        if r.returncode != 0:
            return {"error": (r.stderr or r.stdout)[-600:]}
        return json.loads(r.stdout.strip().splitlines()[-1])
    except Exception as e:  # noqa: BLE001
        return {"error": f"{type(e).__name__}: {e}"}


def cpu_reference_sample(steps, sample_hw, threads=None):
    """The reference's CPU path = oracle port (PyTorch fp32-accumulate restatement of the proxy control
    flow + the reference's own rANS coder from oracle/_ref), timed on the host cores on a bounded
    sample of whole frames at the bench's own picture size (no area scaling)."""
    from util_frames import synth_frame
    from dcvc_b200.spec import dmci_spec, synth_state_dict
    from oracle.dmci_oracle import DmciOracle
    # more than ~32 threads slows the small CPU convolutions of this model down (measured on the 128-core box)
    cores = threads or min(os.cpu_count() or 1, 32)
    torch.set_num_threads(cores)
    h, w = sample_hw
    o = DmciOracle(synth_state_dict(dmci_spec(), 0), skip_thres=SKIP, emulate_fp16=True, threads=cores)
    x = synth_frame(h, w, 1234)
    pad_b, pad_r = (16 - h % 16) % 16, (16 - w % 16) % 16
    enc = _CPU_STREAM_CACHE.get((h, w))
    if enc is None:
        enc = _CPU_STREAM_CACHE[(h, w)] = o.compress(x, QP, pad_b, pad_r)
    t0 = time.perf_counter()
    for _ in range(steps):
        o.decompress(enc["bit_stream"], QP, h, w, enc["ec_parallel"])
    dt = (time.perf_counter() - t0) / steps
    return {"value": round(1.0 / dt, 4), "unit": "frames/s", "cores": cores, "kind": "port",
            "cpu_model": _cpu_model(), "host_cpus": os.cpu_count(),
            "sample": f"{steps} whole decode(s) of the bench's own {h}x{w} frame (q_index {QP}) with the oracle port + the reference's own "
                      f"rANS coder on {cores} thread(s), {dt:.2f} s each", "seconds_per_sample": round(dt, 3)}


_CPU_STREAM_CACHE = {}


def _cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = args.steps + args.warmup
    t0 = time.time()
    # each step = one whole decode of the product arm's own 1080p frame on the host cores (the same config: no sampling)
    from util_frames import synth_frame
    from dcvc_b200.spec import dmci_spec, synth_state_dict
    from oracle.dmci_oracle import DmciOracle
    cores = min(os.cpu_count() or 1, 32)
    torch.set_num_threads(cores)
    h, w = H, W
    o = DmciOracle(synth_state_dict(dmci_spec(), 0), skip_thres=SKIP, emulate_fp16=True, threads=cores)
    x = synth_frame(h, w, 1234)
    enc = o.compress(x, QP, (16 - h % 16) % 16, (16 - w % 16) % 16)
    # a step costs seconds here
    for _ in range(args.warmup):
        o.decompress(enc["bit_stream"], QP, h, w, enc["ec_parallel"])
    t1 = time.perf_counter()
    dec = None
    for _ in range(args.steps):
        dec = o.decompress(enc["bit_stream"], QP, h, w, enc["ec_parallel"])
    dt = time.perf_counter() - t1
    done = args.steps
    fps = done / dt
    out = {"impl": "reference", "metric": METRIC, "value": round(fps, 4), "unit": "frames/s",
           "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": done, "warmup": args.warmup,
           "ms_per_step": round(dt / done * 1e3, 2), "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": "DCVC-UF-Intra 1080p single-frame decode (configs[1]), q_index 32, skip_thres 0.15, "
                                  "one independent frame per GPU", "resolution": [H, W], "qp": QP,
                      "l2": "n/a (CPU)", "weights": "seeded synthetic checkpoint (no checkpoints offline)"},
           "cpu_baseline": {"value": round(fps, 4), "unit": "frames/s", "cores": cores, "kind": "port",
                            "cpu_model": _cpu_model(), "host_cpus": os.cpu_count(),
                            "sample": f"each step = one whole decode of the {h}x{w} frame with the oracle port + the reference's own "
                                      f"rANS coder on {cores} threads; {done} steps"},
           "e2e": {"value": round(fps, 4), "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "wall_s": round(time.time() - t0, 1)}
    if args.dump_outputs and dec is not None:
        dump_outputs(args.dump_outputs, {"decode_x_hat": dec["x_hat"]})
        out["dumped_outputs"] = ["decode_x_hat"]
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-hts", action="store_true")
    ap.add_argument("--hts-size", default="2160x3840", help="second HT-S leg at HxW (configs[4]: 4K; single GPU; 'none' skips it)")
    ap.add_argument("--no-seq8", action="store_true", help="skip the configs[3] leg (8 sequences x 4 rate points over the ranks)")
    ap.add_argument("--no-reference-cuda", action="store_true", help="skip the same-box run of the reference's own CUDA extension")
    ap.add_argument("--no-pipelined", action="store_true", help="skip the two-concurrent-decodes-per-GPU leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step returned as DIR/<name>.npy (float32, at most 64 MB)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
