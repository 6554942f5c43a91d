"""Distortion metrics and the job driver without a device (CPU tier).

* the host restatement tests/metrics_oracle.py (the algorithm csrc/metrics.cu implements: separable fp64 window,
  explicit 2x2 downsampling) against values minted from the reference's calc_psnr / calc_msssim / calc_msssim_rgb;
* dcvc_b200.metrics.log_json against the reference's generate_log_json output;
* the sequence driver with src_type="png" and run_job, driven through stand-in models and the host metrics."""
import hashlib
import io
import json
import os
import pickle

import numpy as np
import pytest
import torch

import metrics_oracle as mo
from dcvc_b200 import stream
from dcvc_b200.metrics import log_json, msssim_from_levels, psnr_from_mse
from dcvc_b200.sequence import SequenceDecoder, SequenceEncoder, frame_schedule, run_job

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = json.load(open(os.path.join(HERE, "golden", "metrics_reference.json")))


def _digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


@pytest.mark.parametrize("case", GOLD["planes"], ids=lambda c: f"{c['h']}x{c['w']}")
def test_oracle_msssim_and_psnr_match_the_reference(case):
    src, rec = mo.pair(case["h"], case["w"], case["seed"])
    assert _digest(src, rec) == case["sha256"], "seeded inputs drifted"
    mssim, mcs = mo.msssim_levels(src, rec)
    assert len(mssim) == len(case["mssim"]) == (4 if min(case["h"], case["w"]) < 176 else 5)
    assert np.max(np.abs(np.array(mssim) - case["mssim"])) < 1e-13
    assert np.max(np.abs(np.array(mcs) - case["mcs"])) < 1e-13
    assert abs(mo.msssim(src, rec) - case["msssim"]) < 1e-13
    # the product of the per-level means the device returns is finished on the host by dcvc_b200.metrics
    assert abs(msssim_from_levels(case["mssim"], case["mcs"]) - case["msssim"]) < 1e-15
    assert abs(mo.psnr(src, rec) - case["psnr"]) < 1e-12
    sse = float(np.sum(np.square(src.astype(np.float64) - rec.astype(np.float64))))
    assert abs(psnr_from_mse(sse / src.size) - case["psnr"]) < 1e-12


@pytest.mark.parametrize("case", GOLD["rgb"], ids=lambda c: f"{c['h']}x{c['w']}")
def test_oracle_rgb_metrics_match_the_reference(case):
    ps = [mo.pair(case["h"], case["w"], s) for s in case["seeds"]]
    src, rec = np.stack([p[0] for p in ps]), np.stack([p[1] for p in ps])
    assert _digest(src, rec) == case["sha256"]
    assert abs(mo.msssim_rgb(src, rec) - case["msssim"]) < 1e-13
    assert abs(mo.psnr(src, rec) - case["psnr"]) < 1e-12


def test_msssim_below_88_is_an_error():
    src, rec = mo.pair(87, 200, 1)
    with pytest.raises(ValueError):
        mo.msssim_levels(src, rec)
    from dcvc_b200.metrics import msssim_levels
    with pytest.raises(ValueError):
        msssim_levels(200, 87)
    assert msssim_levels(88, 88) == 4 and msssim_levels(175, 400) == 4 and msssim_levels(176, 176) == 5


@pytest.mark.parametrize("i", range(len(GOLD["log_json"])))
def test_log_json_equals_generate_log_json(i):
    case = GOLD["log_json"][i]
    mine = json.loads(json.dumps(log_json(**case["args"])))
    assert mine == case["log"]
    assert list(mine) == list(case["log"]), "same key order as the reference's JSON"


# ------------------------------------------------------------------------------------------------ driver, png sources
class _Pic:
    def __init__(self, frame):
        self.frame = frame


class _FakeIntra:
    def __init__(self, log):
        self.log = log

    @staticmethod
    def get_padding_size(height, width, p=64):
        return (-width) % p, (-height) % p

    def compress(self, x, qp, padding_b, padding_r):
        self.log.append(("i.compress", qp))
        return {"bit_stream": pickle.dumps(x), "ec_parallel": 1, "x_hat": x}

    def decompress(self, bit_stream, sps, qp, ec_part):
        self.log.append(("i.decompress", qp))
        return {"x_hat": pickle.loads(bit_stream)}


class _FakeVideo:
    def __init__(self, log, n):
        self.log, self.n = log, n

    def clear_dpb(self):
        self.log.append(("p.clear_dpb",))

    def add_ref_feature_from_frame(self, frame, apply_feature_adaptor=True):
        self.log.append(("p.add_ref", apply_feature_adaptor))

    def compress(self, x, qp, reset_feature_memory, padding_b, padding_r):
        assert len(x) == self.n
        self.log.append(("p.compress", qp, reset_feature_memory))
        return {"bit_stream": pickle.dumps(x), "ec_parallel": 3}

    def decompress(self, bit_stream, sps, qp, ec_part, reset_feature_memory):
        self.log.append(("p.decompress", qp, reset_feature_memory))
        x = pickle.loads(bit_stream)
        return {"x_hat": x if self.n > 1 else x[0]}


def _rgb_frames(n, h, w, seed):
    rng = np.random.default_rng(seed)
    return [rng.integers(0, 256, (3, h, w), dtype=np.uint8) for _ in range(n)]


@pytest.mark.parametrize("n_frames,delay", [(19, 8), (6, 1)])
def test_sequence_driver_png_roundtrip(n_frames, delay):
    H, W = 36, 52
    frames = _rgb_frames(n_frames, H, W, n_frames)
    log_e, log_d = [], []
    to_model = lambda group, d: [_Pic(g) for g in group]    # noqa: E731
    enc = SequenceEncoder(_FakeIntra(log_e), _FakeVideo(log_e, delay), H, W, 21, 33, frame_delay=delay,
                          to_model=to_model, src_type="png")
    data = enc.encode(frames)
    from_model = lambda x, h, w: (x[0] if isinstance(x, list) else x).frame     # noqa: E731
    out = list(SequenceDecoder(_FakeIntra(log_d), _FakeVideo(log_d, delay), frame_delay=delay, from_model=from_model,
                               src_type="png").decode(data, n_frames))
    assert len(out) == n_frames and all(np.array_equal(a, b) for a, b in zip(out, frames))
    units = frame_schedule(n_frames, delay)
    assert [e for e in log_e if e[0].endswith("compress")] == \
        [("i.compress", 21) if u.is_intra else ("p.compress", 33, u.reset_feature_memory) for u in units]
    assert len(enc.bits) == n_frames and sum(enc.bits) == 8 * len(data)
    with pytest.raises(ValueError):
        SequenceEncoder(_FakeIntra([]), _FakeVideo([], delay), H, W, 21, 33, src_type="rgb24")


class _Timer:
    def start(self):
        pass

    def stop(self):
        return 2.0


@pytest.mark.parametrize("src_type,delay,n_frames", [("yuv420", 8, 19), ("png", 8, 12), ("png", 1, 6)])
def test_run_job_bookkeeping(src_type, delay, n_frames):
    """bits (SPS bytes on the first unit, chunk bits on its first picture), frame_types (the padded tail of the last
    chunk not counted), unit times by the drop-first-4 rule, and the record = log_json of the host metrics"""
    H, W = (96, 100) if src_type == "png" else (176, 176)     # 4:2:0 chroma at the 88 MS-SSIM minimum
    rng = np.random.default_rng(3)
    if src_type == "png":
        frames = _rgb_frames(n_frames, H, W, 5)
        models = [torch.from_numpy(f).float().div(255).unsqueeze(0) for f in frames]
        models = [(mo.rgb2ycbcr(m).half() - 0.5) for m in models]
    else:
        frames = [(rng.integers(0, 256, (H, W), dtype=np.uint8), rng.integers(0, 256, (H // 2, W // 2), dtype=np.uint8),
                   rng.integers(0, 256, (H // 2, W // 2), dtype=np.uint8)) for _ in range(n_frames)]
        models = [torch.from_numpy(np.stack([y, np.repeat(np.repeat(u, 2, 0), 2, 1), np.repeat(np.repeat(v, 2, 0), 2, 1)]))
                  .unsqueeze(0).half().div(255) - 0.5 for y, u, v in frames]
    index = {id(f): i for i, f in enumerate(frames)}
    to_model = lambda group, d: [models[index[id(g)]] for g in group]    # noqa: E731
    log = []
    data, rec = run_job(_FakeIntra(log), _FakeVideo(log, delay), frames, H, W, 21, 33, frame_delay=delay,
                        src_type=src_type, calc_ssim=True, verbose_json=True, verbose=1, to_model=to_model,
                        metrics=mo.HostDistortion, timer=_Timer)
    units = frame_schedule(n_frames, delay)
    frame_types = []
    for u in units:
        frame_types += [0] if u.is_intra else [1] * u.count
    assert rec["frame_type"] == frame_types and len(frame_types) == n_frames
    # bits: parse the stream back; the SPS unit's bytes count towards the first coded unit
    f, bits = io.BytesIO(data), []
    pos = 0
    for u in units:
        while True:
            hdr = stream.read_header(f)
            if hdr["nal_type"] != stream.NalType.NAL_SPS:
                break
            stream.read_sps_remaining(f, hdr["sps_id"])
        stream.read_ip_remaining(f)
        bits += [8 * (f.tell() - pos)] + [0] * (u.count - 1)
        pos = f.tell()
    assert f.read() == b""
    assert rec["frame_bpp"] == list(np.array(bits) / (H * W))
    psnrs, ssims = [], []
    for i, fr in enumerate(frames):
        p, s = mo.distortion(src_type, models[i], fr, True, H, W)
        psnrs.append(p)
        ssims.append(s)
    timed = len(units) > 4
    want = log_json(n_frames, H * W, rec["test_time"], frame_types, bits, psnrs, ssims, verbose=True,
                    avg_encoding_time=0.002 if timed else None, avg_decoding_time=0.002 if timed else None)
    assert rec == want
    assert ("avg_frame_encoding_time" in rec) == timed
