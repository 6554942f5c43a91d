"""The drop-in claim, exercised: the REFERENCE's own Python surface drives this repository's plugin, unmodified.

`north_star`: "keeping the src/models and src/layers Python operator API surface so test_video.py and
test_compress_time.py run unmodified".  Here the reference's model classes (src/models/image_model.py:194-217,
video_model_ht.py:413-450, video_model_ld.py:273-306) and its driver scripts (test_video.py:166-399,
test_compress_time.py:23-69) are imported / executed as they are — from the sourceless byte-code `oracle/build_ref.py`
emits into oracle/_ref/py — with `inference_extensions_cuda` resolving to THIS repository's package and
`MLCodec_extensions_cpp` to the reference coder built into oracle/_ref.  Nothing of the reference is patched.

Checks: the reference classes produce the same bytes and reconstructions as the repo's host-side mirrors
(dcvc_b200/model.py) for the same synthetic checkpoint; test_video.py completes a 17-frame 4-rate job per model
structure and its JSON holds finite PSNR / bpp for every frame; test_compress_time.py prints its two FPS lines.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from util_frames import synth_frame

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SKIP = 0.15


def _ref_py_root():
    from oracle.build_ref import py_surface_root
    p = py_surface_root()
    return (p, ".pyc") if p else (None, None)


REF_ROOT, REF_EXT = _ref_py_root()
needs_ref = pytest.mark.skipif(REF_ROOT is None, reason="reference Python surface not built (python oracle/build_ref.py)")


@pytest.fixture(scope="module")
def ref_modules():
    """the reference's model modules, imported with our plugin and the reference coder on the path"""
    added = [REF_ROOT, os.path.join(ROOT, "oracle", "_ref"), ROOT]
    for p in added:
        if p not in sys.path:
            sys.path.insert(0, p)
    import inference_extensions_cuda
    assert os.path.dirname(os.path.dirname(inference_extensions_cuda.__file__)) == ROOT, "plugin must be this repository's"
    from src.models.image_model import DMCI
    from src.models import video_model_ht, video_model_ld
    from src.utils.common import ModelStructure
    return {"DMCI": DMCI, "ht": video_model_ht, "ld": video_model_ld, "MS": ModelStructure}


def _finalize(net):
    # test_video.py:28-30
    net = net.half().to("cuda")
    return net.to(memory_format=torch.channels_last)


def _ref_intra(mods, seed=0):
    from dcvc_b200.spec import dmci_spec, synth_state_dict
    net = mods["DMCI"]().eval()
    net.load_state_dict(synth_state_dict(dmci_spec(), seed))
    net.update(SKIP)
    return _finalize(net)


def _mirror_intra(seed=0):
    from dcvc_b200.model import DMCI
    m = DMCI.synthetic(seed)
    m.update(SKIP)
    return m.half().to("cuda")


@needs_ref
@pytest.mark.parametrize("h,w,qp", [(128, 192, 32), (200, 328, 5), (1080, 1920, 48)])
def test_reference_dmci_through_plugin(ref_modules, h, w, qp):
    """image_model.py:194-217 unmodified, under a side stream with work queued ahead (what test_video.py does): the
    channels_last fp16 state_dict is pushed correctly and the bytes / reconstruction equal the mirror's."""
    x = synth_frame(h, w, 11).half().cuda().contiguous(memory_format=torch.channels_last)
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        ref = _ref_intra(ref_modules)
        junk = torch.randn(4096, 4096, device="cuda")
        for _ in range(20):
            junk = junk @ junk * 1e-3          # ~ms of queued work ahead of set_param's conversions
        pad_r, pad_b = ref.get_padding_size(h, w, 16)
        e1 = ref.compress(x, qp, pad_b, pad_r)
        xe1 = e1["x_hat"].clone()
        d1 = ref.decompress(e1["bit_stream"], {"height": h, "width": w}, qp, e1["ec_parallel"])
        xd1 = d1["x_hat"].clone()
        mir = _mirror_intra()
        e2 = mir.compress(x, qp, pad_b, pad_r)
        xe2 = e2["x_hat"].clone()
    torch.cuda.synchronize()
    assert isinstance(e1["bit_stream"], bytes) and e1["bit_stream"] == e2["bit_stream"]
    assert e1["ec_parallel"] == e2["ec_parallel"]
    assert torch.equal(xe1, xe2) and torch.equal(xe1, xd1)
    assert xd1.shape == (1, 3, h + pad_b, w + pad_r) and xd1.dtype == torch.float16


def _ref_video(mods, structure):
    from dcvc_b200.spec import hts_spec, htl_spec, ld_spec, synth_state_dict
    if structure == "ld":
        net, spec, seed = mods["ld"].DMC(), ld_spec(), 2
    elif structure == "hts":
        net, spec, seed = mods["ht"].DMC(model_structure=mods["MS"].HTS), hts_spec(), 1
    else:
        net, spec, seed = mods["ht"].DMC(model_structure=mods["MS"].HTL), htl_spec(), 3
    net = net.eval()
    net.load_state_dict(synth_state_dict(spec, seed))
    net.update(SKIP)
    return _finalize(net)


def _mirror_video(structure):
    from dcvc_b200 import model
    m = {"ld": model.DMCLD, "hts": model.DMC, "htl": model.DMCHTL}[structure].synthetic()
    m.update(SKIP)
    return m.half().to("cuda")


@needs_ref
@pytest.mark.parametrize("structure", ["hts", "ld", "htl"])
def test_reference_video_models_through_plugin(ref_modules, structure):
    """video_model_ht.py:413-450 / video_model_ld.py:273-306 unmodified: I frame + two units with a memory reset, encoder
    and decoder; bytes and reconstructions equal the mirror's."""
    h, w, qp = 128, 192, 30
    nf = 1 if structure == "ld" else 8
    pad_r, pad_b = ref_modules["DMCI"].get_padding_size(h, w, 16)
    sps = {"height": h, "width": w}
    x0 = synth_frame(h, w, 21).half().cuda().contiguous(memory_format=torch.channels_last)
    units = [synth_frame(h, w, 22 + i, channels=3 * nf).half().cuda().contiguous(memory_format=torch.channels_last) for i in range(2)]
    out = {}
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        for who in ("ref", "mirror"):
            i_net = _ref_intra(ref_modules) if who == "ref" else _mirror_intra()
            p_net = _ref_video(ref_modules, structure) if who == "ref" else _mirror_video(structure)
            enc = i_net.compress(x0, qp, pad_b, pad_r)
            p_net.clear_dpb()
            p_net.add_ref_feature_from_frame(enc["x_hat"])
            streams = [(enc["bit_stream"], enc["ec_parallel"], 0)]
            for i, x in enumerate(units):
                e = p_net.compress(x, qp, i, pad_b, pad_r)
                streams.append((e["bit_stream"], e["ec_parallel"], i))
            dec = i_net.decompress(streams[0][0], sps, qp, streams[0][1])
            p_net.clear_dpb()
            p_net.add_ref_feature_from_frame(dec["x_hat"], apply_feature_adaptor=False)
            recon = [dec["x_hat"].clone()]
            for bs, ec, reset in streams[1:]:
                d = p_net.decompress(bs, sps, qp, ec, reset)
                xs = d["x_hat"] if isinstance(d["x_hat"], list) else [d["x_hat"]]
                assert len(xs) == nf
                recon += [t.clone() for t in xs]
            out[who] = (streams, recon)
    torch.cuda.synchronize()
    for (b1, e1, _), (b2, e2, _) in zip(out["ref"][0], out["mirror"][0]):
        assert b1 == b2 and e1 == e2
    for a, b in zip(out["ref"][1], out["mirror"][1]):
        assert torch.equal(a, b)
        assert torch.isfinite(a.float()).all()


# ------------------------------------------------------------------------------------------------ the driver scripts

def _write_job(tmp, structure, frames, h, w, n_seq=1):
    """synthetic checkpoints (.pth.tar, the container get_state_dict reads: src/utils/common.py:174-181), a YUV 4:2:0
    sequence and the JSON job description of test_cfg/*.json"""
    from dcvc_b200.spec import dmci_spec, hts_spec, htl_spec, ld_spec, synth_state_dict
    spec, seed = {"hts": (hts_spec, 1), "htl": (htl_spec, 3), "ld": (ld_spec, 2)}[structure]
    ck = os.path.join(tmp, "checkpoints")
    os.makedirs(ck, exist_ok=True)
    torch.save({"state_dict": dict(synth_state_dict(dmci_spec(), 0))}, os.path.join(ck, "cvpr2026_image.pth.tar"))
    torch.save({"state_dict": dict(synth_state_dict(spec(), seed))}, os.path.join(ck, f"cvpr2026_video_{structure}.pth.tar"))
    ds = os.path.join(tmp, "data", "HEVC_B")
    os.makedirs(ds, exist_ok=True)
    seqs = {}
    for s in range(n_seq):
        name = f"Synth{s}_{w}x{h}_30.yuv"
        with open(os.path.join(ds, name), "wb") as f:
            for i in range(frames):
                fr = ((synth_frame(h, w, 900 + 31 * s + i)[0] + 0.5) * 255).round().clamp(0, 255).byte().numpy()
                f.write(fr[0].tobytes())
                f.write(np.ascontiguousarray(fr[1, ::2, ::2]).tobytes())
                f.write(np.ascontiguousarray(fr[2, ::2, ::2]).tobytes())
        seqs[name] = {"width": w, "height": h, "frames": frames, "intra_period": -1}
    cfg = {"root_path": os.path.join(tmp, "data"),
           "test_classes": {"HEVC_B": {"test": 1, "base_path": "HEVC_B", "src_type": "yuv420", "sequences": seqs}}}
    os.makedirs(os.path.join(tmp, "test_cfg"), exist_ok=True)
    with open(os.path.join(tmp, "test_cfg", "runtime_avg.json"), "w") as f:
        json.dump(cfg, f)
    return cfg


def _env():
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([ROOT, os.path.join(ROOT, "oracle", "_ref"), REF_ROOT, env.get("PYTHONPATH", "")])
    env.pop("DCVC_B200_PROFILE_CSV", None)
    return env


@needs_ref
@pytest.mark.parametrize("structure,force_intra", [("hts", 0), ("ld", 0), ("htl", 0), ("hts", 1)])
def test_reference_test_video_unmodified(tmp_path, structure, force_intra):
    """python test_video.py … exactly as the reference's README / test_compress_time.py invoke it (4 rate points, one
    worker, --skip_thres 0.15, verbose 2): spawned worker, custom stream, finalize_model, bitstream container, decoder
    loop, metrics — all the reference's code, our plugin underneath."""
    tmp = str(tmp_path)
    frames, h, w = (17, 144, 208) if structure != "ld" else (9, 144, 208)
    _write_job(tmp, structure, frames, h, w)
    out_json = os.path.join(tmp, "out.json")
    cmd = [sys.executable, os.path.join(REF_ROOT, "test_video" + REF_EXT), "--verbose", "2", "--rate_num", "4",
           "--force_intra", str(force_intra), "--test_config", os.path.join(tmp, "test_cfg", "runtime_avg.json"),
           "--force_frame_num", "-1", "--cuda_idx", "0", "-w", "1", "--skip_thres", "0.15", "--output_path", out_json,
           "--model_path_i", os.path.join(tmp, "checkpoints", "cvpr2026_image.pth.tar"),
           "--model_path_p", os.path.join(tmp, "checkpoints", f"cvpr2026_video_{structure}.pth.tar"),
           "--model_structure", structure, "--stream_path", os.path.join(tmp, "out_bin")]
    r = subprocess.run(cmd, cwd=tmp, env=_env(), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "Test finished" in r.stdout
    res = json.load(open(out_json))["HEVC_B"]
    assert len(res) == 1
    for seq, rates in res.items():
        assert sorted(rates) == ["000", "001", "002", "003"]
        bpps = []
        for k in sorted(rates):
            p = rates[k]
            assert p["i_frame_num"] + p["p_frame_num"] == frames
            assert p["i_frame_num"] == (frames if force_intra else 1)
            assert np.isfinite(p["ave_all_frame_psnr"]) and 5.0 < p["ave_all_frame_psnr"] < 60.0
            assert np.isfinite(p["ave_all_frame_bpp"]) and p["ave_all_frame_bpp"] > 0
            bpps.append(p["ave_all_frame_bpp"])
        assert len(set(bpps)) > 1, "the four rate points must differ"


@needs_ref
def test_reference_test_compress_time_unmodified(tmp_path):
    """python test_compress_time.py --model_structure hts: the reference's timing driver (it shells out to `python
    test_video.py` with relative checkpoint / config paths, so the job is laid out the way the reference tree has it)."""
    tmp = str(tmp_path)
    _write_job(tmp, "hts", 41, 144, 208)   # > 4 timed units: the script drops the first 4 as warm-up
    for name in ("test_video", "test_compress_time"):
        os.symlink(os.path.join(REF_ROOT, name + REF_EXT), os.path.join(tmp, name + ".py"))
    r = subprocess.run([sys.executable, "test_compress_time.py", "--model_structure", "hts", "--output_path", "t.json"],
                       cwd=tmp, env=_env(), capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("Average ")]
    assert len(lines) == 2 and all(" fps" in l for l in lines), r.stdout[-2000:]
