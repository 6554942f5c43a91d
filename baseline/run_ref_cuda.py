#!/usr/bin/env python
"""Times the REFERENCE's own CUDA path on this box: the reference's unmodified Python models (src/models, the
byte-code in oracle/_ref/py) on top of the reference's own CUTLASS extension compiled for sm_100a
(baseline/build_ref_cuda.py -> baseline/_ref/inference_extensions_cuda_ref*.so) — none of this repository's kernels on the
path.  Same synthetic checkpoints, frames, q_index, skip_thres and timing protocol as bench.py's product arm (CUDA events
per call, L2 flushed between calls; test_video.py:204-325 times one call at a time the same way).

Runs in its own process because the module name `inference_extensions_cuda` can only mean one thing per process.
Prints one JSON line.  With --dump DIR also writes the streams and reconstructions (parity anchor for
tests/test_reference_cuda_gpu.py).

  python baseline/run_ref_cuda.py --steps 10 --warmup 3 [--models intra,hts,ld,htl] [--size 1080x1920]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)

QP = 32
SKIP = 0.15


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--models", default="intra,hts,ld,htl")
    ap.add_argument("--size", default="1080x1920")
    ap.add_argument("--qp", type=int, default=QP)
    ap.add_argument("--dump", default=None)
    args = ap.parse_args()
    import torch
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    import build_ref_cuda
    ext = build_ref_cuda.load(as_plugin=True)
    if ext is None:
        print(json.dumps({"unavailable": "baseline/_ref/inference_extensions_cuda_ref*.so not built"}))
        return
    from oracle.build_ref import py_surface_root
    ref_root = py_surface_root()
    if ref_root is None:
        print(json.dumps({"unavailable": "oracle/_ref/py (the reference's models as byte-code) not built"}))
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))   # MLCodec_extensions_cpp (the reference's rANS module)
    sys.path.insert(0, ref_root)
    from src.models.image_model import DMCI
    from src.models import video_model_ht, video_model_ld
    from src.utils.common import ModelStructure
    import inference_extensions_cuda as plugin
    assert plugin is ext, "the reference's models must resolve the REFERENCE extension in this process"
    from dcvc_b200.spec import dmci_spec, hts_spec, htl_spec, ld_spec, synth_state_dict   # parameter shapes + seeds only
    from util_frames import psnr, synth_frame

    h, w = (int(v) for v in args.size.lower().split("x"))
    qp = args.qp
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)          # test_video.py:423-425: graphs cannot be captured on stream 0
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def fin(net):
        return net.half().to(dev).to(memory_format=torch.channels_last)     # test_video.py:28-30

    def timed(fn, steps):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        torch.cuda.synchronize()
        for e0, e1 in evs:
            flush.zero_()
            e0.record()
            fn()
            e1.record()
        torch.cuda.synchronize()
        return sum(e0.elapsed_time(e1) for e0, e1 in evs) / steps

    i_net = DMCI().eval()
    i_net.load_state_dict(synth_state_dict(dmci_spec(), 0))
    i_net.update(SKIP)
    i_net = fin(i_net)
    pad_r, pad_b = DMCI.get_padding_size(h, w, 16)
    sps = {"height": h, "width": w}
    x0 = synth_frame(h, w, 1234).half().to(dev).contiguous(memory_format=torch.channels_last)
    out = {"impl": "reference_cuda", "size": [h, w], "qp": qp, "steps": args.steps, "warmup": args.warmup,
           "cutlass": "4.5.0 (flashinfer/data/cutlass; the reference pins 4.4.1)", "gpu": torch.cuda.get_device_name(0)}
    dump = {}
    models = args.models.split(",")

    enc = i_net.compress(x0, qp, pad_b, pad_r)
    x_hat_i = enc["x_hat"].clone()
    dec = i_net.decompress(enc["bit_stream"], sps, qp, enc["ec_parallel"])
    torch.cuda.synchronize()
    if "intra" in models:
        for _ in range(args.warmup):
            i_net.decompress(enc["bit_stream"], sps, qp, enc["ec_parallel"])
            i_net.compress(x0, qp, pad_b, pad_r)
        ms_d = timed(lambda: i_net.decompress(enc["bit_stream"], sps, qp, enc["ec_parallel"]), args.steps)
        ms_e = timed(lambda: i_net.compress(x0, qp, pad_b, pad_r), args.steps)
        out["intra"] = {"decode_fps": round(1e3 / ms_d, 2), "encode_fps": round(1e3 / ms_e, 2), "ms_per_decode": round(ms_d, 4),
                        "ms_per_encode": round(ms_e, 4), "bytes": len(enc["bit_stream"]),
                        "bpp": round(len(enc["bit_stream"]) * 8 / (h * w), 5),
                        "psnr_db": round(psnr(dec["x_hat"].float().cpu()[:, :, :h, :w], x0.float().cpu()), 4),
                        "decode_equals_encode": bool(torch.equal(x_hat_i, dec["x_hat"]))}
        dump["intra_stream"] = np.frombuffer(enc["bit_stream"], dtype=np.uint8)
        dump["intra_x_hat"] = dec["x_hat"].float().cpu().numpy()[:, :, :h, :w].astype(np.float16)

    for name in ("hts", "ld", "htl"):
        if name not in models:
            continue
        nf = 1 if name == "ld" else 8
        if name == "ld":
            p_net, spec, seed = video_model_ld.DMC(), ld_spec(), 2
        elif name == "hts":
            p_net, spec, seed = video_model_ht.DMC(model_structure=ModelStructure.HTS), hts_spec(), 1
        else:
            p_net, spec, seed = video_model_ht.DMC(model_structure=ModelStructure.HTL), htl_spec(), 3
        p_net = p_net.eval()
        p_net.load_state_dict(synth_state_dict(spec, seed))
        p_net.update(SKIP)
        p_net = fin(p_net)
        # bench.py's bench_hts / bench_ld protocol, frame seeds included: encode warmup + steps units one after the other,
        # then decode exactly that sequence (encoder and decoder state stay consistent)
        base = {"hts": 4000, "htl": 4000, "ld": 5000}[name]
        xi = synth_frame(h, w, base).half().to(dev).contiguous(memory_format=torch.channels_last)
        units = [synth_frame(h, w, base + 100 + c, channels=3 * nf).half().to(dev).contiguous(memory_format=torch.channels_last)
                 for c in range(3)]
        enc_i = i_net.compress(xi, qp, pad_b, pad_r)
        p_net.clear_dpb()
        p_net.add_ref_feature_from_frame(enc_i["x_hat"])
        encs = []
        k = [0]

        def step_enc():
            encs.append(p_net.compress(units[k[0] % 3], qp, 0, pad_b, pad_r))
            k[0] += 1

        for _ in range(args.warmup):
            step_enc()
        ms_e = timed(step_enc, args.steps)
        dec_i = i_net.decompress(enc_i["bit_stream"], sps, qp, enc_i["ec_parallel"])
        p_net.clear_dpb()
        p_net.add_ref_feature_from_frame(dec_i["x_hat"], apply_feature_adaptor=False)
        k[0] = 0
        recon = []

        def step_dec():
            e = encs[k[0]]
            d = p_net.decompress(e["bit_stream"], sps, qp, e["ec_parallel"], 0)["x_hat"]
            if k[0] == 0:
                recon.append([t.clone() for t in (d if isinstance(d, list) else [d])])
            k[0] += 1

        for _ in range(args.warmup):
            step_dec()
        ms_d = timed(step_dec, args.steps)
        nbytes = [len(e["bit_stream"]) for e in encs]
        out[name] = {"decode_fps": round(nf * 1e3 / ms_d, 2), "encode_fps": round(nf * 1e3 / ms_e, 2),
                     "ms_per_unit_decode": round(ms_d, 4), "ms_per_unit_encode": round(ms_e, 4), "frames_per_unit": nf,
                     "bytes_per_unit": nbytes,
                     "psnr_db_frame0": round(psnr(recon[0][0].float().cpu()[:, :, :h, :w], units[0][:, :3].float().cpu()), 4)}
        dump[name + "_streams"] = np.concatenate([np.frombuffer(e["bit_stream"], dtype=np.uint8) for e in encs])
        dump[name + "_stream_sizes"] = np.array(nbytes, dtype=np.int64)
        dump[name + "_x_hat0"] = recon[0][0].float().cpu().numpy()[:, :, :h, :w].astype(np.float16)
        del p_net
        torch.cuda.empty_cache()

    if args.dump:
        os.makedirs(args.dump, exist_ok=True)
        np.savez(os.path.join(args.dump, f"ref_cuda_{h}x{w}_q{qp}.npz"), **dump)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
