"""RGB frame IO and device distortion metrics against the reference's own functions, on the device.

The reference functions are the byte-code oracle/build_ref.py emits into oracle/_ref/py: get_src_frame and
get_distortion of test_video.py, ycbcr2rgb of src/utils/transforms.py, calc_msssim of src/utils/metrics.py, and finally
test_video.py itself run unmodified next to dcvc_b200.sequence.run_job."""
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


def _ref_py_root():
    from oracle.build_ref import py_surface_root
    return py_surface_root()


REF_ROOT = _ref_py_root()
needs_ref = pytest.mark.skipif(REF_ROOT is None, reason="reference Python surface not built (python oracle/build_ref.py)")

# measured on a B200: |dPSNR| <= 1.8e-15 dB, |dMS-SSIM| <= 8.3e-15 (fp64 statistics; only the summation order differs
# from scipy's FFT convolution)
PSNR_TOL = 1e-12       # dB
MSSSIM_TOL = 1e-13


@pytest.fixture(scope="module")
def ref():
    for p in (REF_ROOT, os.path.join(ROOT, "oracle", "_ref"), ROOT):
        if p not in sys.path:
            sys.path.insert(0, p)
    import test_video
    from src.utils import metrics, transforms
    return {"tv": test_video, "metrics": metrics, "transforms": transforms}


def _rgb(h, w, seed):
    """uint8 [3,h,w] with smooth content plus full-range corners (0 and 255 saturate every clamp)"""
    x = ((synth_frame(h, w, seed)[0] + 0.5) * 255).round().clamp(0, 255).byte().numpy()
    rng = np.random.default_rng(seed)
    x[:, :4, :4] = rng.integers(0, 256, (3, 4, 4), dtype=np.uint8)
    x[:, -2:, -2:] = np.array([0, 255], dtype=np.uint8)[rng.integers(0, 2, (3, 2, 2))]
    return np.ascontiguousarray(x)


class _Reader:
    def __init__(self, frames):
        self.frames = list(frames)

    def read_one_frame(self):
        return self.frames.pop(0)


# ------------------------------------------------------------------------------------------------ RGB frame IO

@needs_ref
@pytest.mark.parametrize("h,w", [(64, 64), (37, 91), (176, 208), (1080, 1920)])
def test_rgb_to_frame_bit_exact(ref, h, w):
    from dcvc_b200.frame_io import rgb_to_frame
    src = _rgb(h, w, h + w)
    if h == 64:      # every 8-bit value in every channel, in random combinations
        rng = np.random.default_rng(1)
        src = np.stack([rng.permutation(np.tile(np.arange(256, dtype=np.uint8), 16)).reshape(64, 64) for _ in range(3)])
    x_ref, *_ = ref["tv"].get_src_frame({"src_type": "png"}, _Reader([src]), "cuda", 1, True)
    mine = rgb_to_frame(torch.from_numpy(src).cuda())
    torch.cuda.synchronize()
    assert mine.shape == x_ref.shape and mine.dtype == x_ref.dtype
    assert torch.equal(mine, x_ref)


@needs_ref
def test_rgb_to_frame_channel_stacking_and_plain_layout(ref):
    """8 pictures stacked on the channel axis (the HT chunk input, test_video.py:108-122), into a channels_last and a
    plain NCHW `out`"""
    from dcvc_b200.frame_io import rgb_to_frame
    h, w = 96, 160
    srcs = [_rgb(h, w, 50 + i) for i in range(8)]
    ref["tv"].g_frame_delay = 8
    x_ref, *_ = ref["tv"].get_src_frame({"src_type": "png"}, _Reader(srcs), "cuda", 8, False)
    for fmt in (torch.channels_last, torch.contiguous_format):
        out = torch.empty((1, 24, h, w), dtype=torch.float16, device="cuda").contiguous(memory_format=fmt)
        for i, s in enumerate(srcs):
            rgb_to_frame(torch.from_numpy(s).cuda(), out=out, channel=3 * i)
        torch.cuda.synchronize()
        assert torch.equal(out, x_ref)


@needs_ref
@pytest.mark.parametrize("hp,wp,h,w", [(64, 64, 64, 64), (1088, 1920, 1080, 1920), (192, 272, 180, 264)])
def test_frame_to_rgb_bit_exact(ref, hp, wp, h, w):
    """test_video.py:367-369 on the device with the reference's ycbcr2rgb; inputs reach beyond [-0.5, 0.5]"""
    from dcvc_b200.frame_io import frame_to_rgb
    g = torch.Generator().manual_seed(hp + wp)
    x_hat = ((torch.rand((1, 3, hp, wp), generator=g) - 0.5) * 1.3).half().cuda().contiguous(memory_format=torch.channels_last)
    crop = x_hat[:, :, :h, :w]
    rgb_ref = ref["transforms"].ycbcr2rgb(crop + 0.5)
    rgb_ref = torch.clamp(rgb_ref * 255, 0, 255).round().byte().squeeze(0)
    mine = frame_to_rgb(x_hat, h, w)
    torch.cuda.synchronize()
    assert torch.equal(mine, rgb_ref)


# ------------------------------------------------------------------------------------------------ Distortion

def _case(src_type, h, w, hp, seed):
    g = torch.Generator().manual_seed(seed)
    base = synth_frame(hp, w, seed)
    x_hat = (base + (torch.rand(base.shape, generator=g) - 0.5) * 0.06).half()
    x_hat[:, :, :3, :3] = 0.7           # saturating values
    x_hat = x_hat.cuda().contiguous(memory_format=torch.channels_last)
    src = ((base[0, :, :h] + 0.5) * 255).round().clamp(0, 255).byte()
    if src_type == "png":
        rgb = ((synth_frame(h, w, seed + 1)[0] + 0.5) * 255).round().clamp(0, 255).byte().numpy()
        return x_hat, None, None, None, np.ascontiguousarray(rgb)
    y = src[0].numpy().copy()
    u = np.ascontiguousarray(src[1, ::2, ::2].numpy())
    v = np.ascontiguousarray(src[2, ::2, ::2].numpy())
    return x_hat, y, u, v, None


def _mine(src_type, h, w, calc_ssim, x_hat, y, u, v, rgb):
    from dcvc_b200.metrics import Distortion
    d = Distortion(src_type, h, w, calc_ssim, capacity=2)
    src = (torch.from_numpy(rgb).cuda() if src_type == "png" else
           tuple(torch.from_numpy(p).cuda() for p in (y, u, v)))
    d.add(x_hat, src)
    d.add(x_hat, src)
    return d


@needs_ref
@pytest.mark.parametrize("src_type,h,w,hp", [("yuv420", 176, 176, 176), ("yuv420", 1080, 1920, 1088),
                                             ("yuv420", 2160, 3840, 2160), ("png", 1080, 1920, 1088)])
def test_distortion_matches_get_distortion(ref, src_type, h, w, hp):
    x_hat, y, u, v, rgb = _case(src_type, h, w, hp, h + w)
    psnr_ref, ssim_ref = ref["tv"].get_distortion({"src_type": src_type, "calc_ssim": True}, x_hat[:, :, :h, :w],
                                                  y, u, v, rgb)
    d = _mine(src_type, h, w, True, x_hat, y, u, v, rgb)
    psnrs, ssims = d.results()
    assert len(psnrs) == 2 and psnrs[0] == psnrs[1] and ssims[0] == ssims[1]
    dp = max(abs(a - b) for a, b in zip(psnrs[0], psnr_ref))
    ds = max(abs(a - b) for a, b in zip(ssims[0], ssim_ref))
    print(f"[metrics] {src_type} {h}x{w}: max |dPSNR| {dp:.3e} dB, max |dMS-SSIM| {ds:.3e}; "
          f"PSNR {psnrs[0][0]:.4f}, MS-SSIM {ssims[0][0]:.6f}")
    assert len(psnrs[0]) == len(psnr_ref) and len(ssims[0]) == len(ssim_ref)
    assert dp <= PSNR_TOL and ds <= MSSSIM_TOL


@needs_ref
def test_metric_planes_are_get_distortions_arrays(ref):
    """the fp16 planes the kernels measure are bit-identical to the arrays get_distortion hands to calc_psnr"""
    for src_type in ("yuv420", "png"):
        h, w = 180, 264
        x_hat, y, u, v, rgb = _case(src_type, h, w, 192, 7)
        d = _mine(src_type, h, w, False, x_hat, y, u, v, rgb)
        torch.cuda.synchronize()
        xc = x_hat[:, :, :h, :w] + 0.5
        if src_type == "yuv420":
            y_rec, uv_rec = ref["transforms"].yuv_444_to_420(xc)
            want = [torch.clamp(y_rec * 255, 0, 255)[0, 0], torch.clamp(uv_rec * 255, 0, 255)[0, 0],
                    torch.clamp(uv_rec * 255, 0, 255)[0, 1]]
        else:
            want = list(torch.clamp(ref["transforms"].ycbcr2rgb(xc) * 255, 0, 255)[0])
        for got, exp in zip(d.rec_planes, want):
            assert torch.equal(got.view(exp.shape), exp)


def test_distortion_rejects_small_chroma_for_msssim():
    """144x208 4:2:0: chroma is 72x104, below calc_msssim's 88 (the reference asserts); PSNR alone works"""
    from dcvc_b200.metrics import Distortion
    with pytest.raises(ValueError):
        Distortion("yuv420", 144, 208, True, capacity=1)
    x_hat, y, u, v, _ = _case("yuv420", 144, 208, 144, 3)
    psnrs, ssims = _mine("yuv420", 144, 208, False, x_hat, y, u, v, None).results()
    assert np.isfinite(psnrs[0][0]) and ssims[0] == [0.0, 0.0, 0.0, 0.0]


def test_distortion_reproducible_and_graph_capturable():
    """two runs are bitwise identical; .add captured into a CUDA graph and replayed gives the same numbers (so it
    neither allocates nor synchronises)"""
    from dcvc_b200.metrics import Distortion
    h, w = 1080, 1920
    x_hat, y, u, v, _ = _case("yuv420", h, w, 1088, 5)
    src = tuple(torch.from_numpy(p).cuda() for p in (y, u, v))
    runs = []
    for _ in range(2):
        d = Distortion("yuv420", h, w, True, capacity=1)
        d.add(x_hat, src)
        runs.append(d.raw())
    assert np.array_equal(runs[0], runs[1])
    d = Distortion("yuv420", h, w, True, capacity=1)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            d.add(x_hat, src)
    graph.replay()
    graph.replay()
    torch.cuda.synchronize()
    assert np.array_equal(d.raw(), runs[0])


# ------------------------------------------------------------------------------------------------ end to end

def _write_job(tmp, structure, src_type, frames, h, w):
    """checkpoints + one sequence (YUV file or a directory of im00001.png ...) + the test_cfg JSON"""
    from PIL import Image
    from dcvc_b200.spec import dmci_spec, hts_spec, ld_spec, synth_state_dict
    spec, seed = {"hts": (hts_spec, 1), "ld": (ld_spec, 2)}[structure]
    ck = os.path.join(tmp, "checkpoints")
    os.makedirs(ck, exist_ok=True)
    torch.save({"state_dict": dict(synth_state_dict(dmci_spec(), 0))}, os.path.join(ck, "image.pth.tar"))
    torch.save({"state_dict": dict(synth_state_dict(spec(), seed))}, os.path.join(ck, f"video_{structure}.pth.tar"))
    ds = os.path.join(tmp, "data", "DS")
    os.makedirs(ds, exist_ok=True)
    pics = [((synth_frame(h, w, 900 + i)[0] + 0.5) * 255).round().clamp(0, 255).byte().numpy() for i in range(frames)]
    if src_type == "yuv420":
        name = f"Synth_{w}x{h}_30.yuv"
        planes = [(p[0].copy(), np.ascontiguousarray(p[1, ::2, ::2]), np.ascontiguousarray(p[2, ::2, ::2])) for p in pics]
        with open(os.path.join(ds, name), "wb") as f:
            for yuv in planes:
                for q in yuv:
                    f.write(q.tobytes())
        src = [tuple(torch.from_numpy(q).cuda() for q in yuv) for yuv in planes]
    else:
        name = f"Synth_{w}x{h}"
        os.makedirs(os.path.join(ds, name))
        for i, p in enumerate(pics):
            Image.fromarray(np.ascontiguousarray(p.transpose(1, 2, 0))).save(os.path.join(ds, name, f"im{i + 1:05d}.png"))
        src = [torch.from_numpy(np.ascontiguousarray(p)).cuda() for p in pics]
    cfg = {"root_path": os.path.join(tmp, "data"),
           "test_classes": {"DS": {"test": 1, "base_path": "DS", "src_type": src_type,
                                   "sequences": {name: {"width": w, "height": h, "frames": frames, "intra_period": -1}}}}}
    with open(os.path.join(tmp, "cfg.json"), "w") as f:
        json.dump(cfg, f)
    return name, src


@needs_ref
@pytest.mark.parametrize("structure,src_type", [("hts", "yuv420"), ("hts", "png"), ("ld", "yuv420"), ("ld", "png")])
def test_run_job_matches_test_video(tmp_path, structure, src_type):
    """the unmodified test_video.py (--calc_ssim 1 --verbose_json 1) and run_job on the same job: identical bitstream,
    frame_bpp and frame_type; every per-picture PSNR and MS-SSIM within the tolerances above"""
    from dcvc_b200 import model
    from dcvc_b200.sequence import run_job
    tmp = str(tmp_path)
    h, w, qp = 180, 264, 30
    frames = 10 if structure == "hts" else 4
    name, src = _write_job(tmp, structure, src_type, frames, h, w)
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([ROOT, os.path.join(ROOT, "oracle", "_ref"), REF_ROOT, env.get("PYTHONPATH", "")])
    cmd = [sys.executable, os.path.join(REF_ROOT, "test_video.pyc"), "--rate_num", "1", "--qp_i", str(qp),
           "--qp_p", str(qp), "--test_config", os.path.join(tmp, "cfg.json"), "--cuda_idx", "0", "-w", "1",
           "--skip_thres", "0.15", "--output_path", os.path.join(tmp, "out.json"), "--calc_ssim", "1",
           "--verbose_json", "1", "--model_path_i", os.path.join(tmp, "checkpoints", "image.pth.tar"),
           "--model_path_p", os.path.join(tmp, "checkpoints", f"video_{structure}.pth.tar"),
           "--model_structure", structure, "--stream_path", os.path.join(tmp, "out_bin")]
    r = subprocess.run(cmd, cwd=tmp, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    ref_bin = open(os.path.join(tmp, "out_bin", "DS", f"{name}_q{qp}.bin"), "rb").read()
    ref_log = json.load(open(os.path.join(tmp, "out_bin", "DS", f"{name}_q{qp}.json")))

    i_net = model.DMCI.synthetic(0)
    i_net.update(0.15)
    i_net = i_net.half().to("cuda")
    p_net = (model.DMC if structure == "hts" else model.DMCLD).synthetic()
    p_net.update(0.15)
    p_net = p_net.half().to("cuda")
    stream = torch.cuda.Stream()        # test_video.py codes on a side stream too
    with torch.cuda.stream(stream):
        data, log = run_job(i_net, p_net, src, h, w, qp, qp, frame_delay=8 if structure == "hts" else 1,
                            src_type=src_type, calc_ssim=True, verbose_json=True)
    assert data == ref_bin
    assert log["frame_type"] == ref_log["frame_type"] and log["frame_bpp"] == ref_log["frame_bpp"]
    assert set(log) == set(ref_log)
    dp = ds = 0.0
    for k in ref_log:
        if k.startswith("frame_psnr"):
            dp = max(dp, max(abs(a - b) for a, b in zip(log[k], ref_log[k])))
        elif k.startswith("frame_msssim"):
            ds = max(ds, max(abs(a - b) for a, b in zip(log[k], ref_log[k])))
    print(f"[run_job] {structure} {src_type} {h}x{w}: max |dPSNR| {dp:.3e} dB, max |dMS-SSIM| {ds:.3e}")
    assert dp <= PSNR_TOL and ds <= MSSSIM_TOL
