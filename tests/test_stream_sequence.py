"""Callers either side of the codec (SURVEY.md §8 f2, CPU tier): the bitstream container (dcvc_b200/stream.py vs the
reference's src/utils/stream_helper.py, pinned by a fixture minted from the reference's own functions) and the sequence
driver (dcvc_b200/sequence.py vs the loops of test_video.py:204-372), the latter with stand-in models so that no device
is needed: what is checked is the schedule, the call protocol and the framing, not the codec."""
import hashlib
import io
import json
import os
import pickle

import numpy as np
import pytest

from dcvc_b200 import stream
from dcvc_b200.sequence import SequenceDecoder, SequenceEncoder, Unit, frame_schedule

HERE = os.path.dirname(os.path.abspath(__file__))


def _payload(n, seed):
    return np.random.default_rng(seed).integers(0, 256, n, dtype=np.uint8).tobytes()


def _replay(mod, ops):
    f = io.BytesIO()
    for op in ops:
        if op[0] == "sps":
            mod.write_sps(f, {"sps_id": op[1], "height": op[2], "width": op[3]})
        else:
            mod.write_ip(f, op[1], op[2], op[3], op[4], op[5], _payload(op[6], op[7]))
    return f.getvalue()


def test_container_bytes_match_the_reference_fixture():
    g = json.load(open(os.path.join(HERE, "golden", "stream_container.json")))
    data = _replay(stream, g["ops"])
    assert len(data) == g["length"] and data[:512].hex() == g["head_hex"]
    assert hashlib.sha256(data).hexdigest() == g["sha256"]
    # and it parses back to what was written
    f = io.BytesIO(data)
    for op in g["ops"]:
        h = stream.read_header(f)
        if op[0] == "sps":
            assert h["nal_type"] == stream.NalType.NAL_SPS and h["sps_id"] == op[1]
            assert stream.read_sps_remaining(f, h["sps_id"]) == {"sps_id": op[1], "height": op[2], "width": op[3]}
        else:
            assert h["nal_type"] == (stream.NalType.NAL_I if op[1] else stream.NalType.NAL_P) and h["sps_id"] == op[2]
            qp, ec, reset, bs = stream.read_ip_remaining(f)
            assert (qp, ec, reset) == (op[3], op[4], op[5]) and bs == _payload(op[6], op[7])
    assert f.read() == b""


def test_container_random_writes_match_the_reference_fixture():
    """random ids / sizes / payload lengths across the varint widths: the bytes the reference's own helpers wrote for
    them (fixture minted by tests/golden/make_golden.py), read back by our parser; write_uint_adaptive on its boundaries"""
    g = json.load(open(os.path.join(HERE, "golden", "stream_container_random.json")))
    ops = g["ops"]
    mine = _replay(stream, ops)
    assert len(mine) == g["length"] and hashlib.sha256(mine).hexdigest() == g["sha256"]
    f = io.BytesIO(mine)
    for op in ops:
        h = stream.read_header(f)
        if op[0] == "sps":
            assert stream.read_sps_remaining(f, h["sps_id"]) == {"sps_id": op[1], "height": op[2], "width": op[3]}
        else:
            assert stream.read_ip_remaining(f)[:3] == (op[3], op[4], op[5])
    assert f.read() == b""
    for v, want in g["uint_adaptive"].items():
        a = io.BytesIO()
        assert stream.write_uint_adaptive(a, int(v)) == want["returned"] and a.getvalue().hex() == want["hex"]
        a.seek(0)
        assert stream.read_uint_adaptive(a) == int(v)


def test_container_rejects_damage_loudly():
    f = io.BytesIO()
    stream.write_ip(f, True, 0, 10, 3, 0, b"abcdef")
    data = f.getvalue()
    with pytest.raises(EOFError):
        g = io.BytesIO(data[:-2])
        stream.read_header(g)
        stream.read_ip_remaining(g)
    with pytest.raises(ValueError):
        stream.write_uint_adaptive(io.BytesIO(), 1 << 30)
    with pytest.raises(ValueError):
        stream.write_ip(io.BytesIO(), False, 16, 0, 0, 0, b"")
    h = stream.SPSHelper()
    for i in range(16):
        assert h.get_sps_id({"sps_id": -1, "height": 16 * (i + 1), "width": 16}) == (i, True)
    assert h.get_sps_id({"sps_id": -1, "height": 32, "width": 16}) == (1, False)
    with pytest.raises(ValueError):
        h.get_sps_id({"sps_id": -1, "height": 8, "width": 8})


# ------------------------------------------------------------------------------------------------ schedule
def _reference_loop(frame_num, g, intra_period, reset_interval):
    """the reference's while-loop (test_video.py:204-236, 264) restated literally, as the expectation"""
    out, frame_idx = [], 0
    while frame_idx < frame_num:
        is_intra = False
        if frame_idx == 0 or intra_period == 1:
            is_intra = True
        if intra_period > 1 and frame_idx != 1:
            if frame_idx % intra_period == 1:
                is_intra = True
        maximum_read = min(g, frame_num - frame_idx)
        if is_intra:
            maximum_read = 1
        reset = 0
        if not is_intra and reset_interval > 0 and (frame_idx + g) % reset_interval == 1:
            reset = 1
        out.append(Unit(frame_idx, maximum_read, is_intra, reset))
        frame_idx += maximum_read
    return out


@pytest.mark.parametrize("frame_num,g,ip,ri", [(97, 8, -1, 32), (96, 8, -1, 32), (33, 8, 32, 32), (100, 8, 16, 24), (10, 1, -1, 32),
                                               (70, 1, 8, 4), (5, 8, -1, 32), (1, 8, -1, 32), (0, 8, -1, 32), (40, 8, 1, 32),
                                               (97, 8, -1, 0)])
def test_frame_schedule_equals_the_reference_loop(frame_num, g, ip, ri):
    got = frame_schedule(frame_num, g, ip, ri)
    assert got == _reference_loop(frame_num, g, ip, ri)
    assert sum(u.count for u in got) == frame_num
    if frame_num:
        assert got[0].is_intra and got[0].count == 1


def test_frame_schedule_of_the_headline_config():
    """configs[2]: 97 frames, IP -1, 8-frame chunks, reset every 32: 1 intra + 12 chunks, resets at pictures 25, 57, 89"""
    u = frame_schedule(97, 8, -1, 32)
    assert len(u) == 13 and [x.first for x in u if x.reset_feature_memory] == [25, 57, 89]
    with pytest.raises(ValueError):
        frame_schedule(97, 8, 12, 32)


# ------------------------------------------------------------------------------------------------ driver with stand-in models
class _Pic:
    """stand-in for a model tensor holding one picture"""

    def __init__(self, planes):
        self.planes = planes


class _FakeIntra:
    """lossless stand-in: the "bit stream" is the pickled model input; records the protocol"""

    def __init__(self, log):
        self.log = log

    @staticmethod
    def get_padding_size(height, width, p=64):
        return (-width) % p, (-height) % p

    def compress(self, x, qp, padding_b, padding_r):
        self.log.append(("i.compress", qp, padding_b, padding_r))
        return {"bit_stream": pickle.dumps(x), "ec_parallel": 1, "x_hat": x}

    def decompress(self, bit_stream, sps, qp, ec_part):
        self.log.append(("i.decompress", qp, sps["height"], sps["width"], ec_part))
        return {"x_hat": pickle.loads(bit_stream)}


class _FakeVideo:
    def __init__(self, log, frames_per_call):
        self.log, self.n = log, frames_per_call

    def clear_dpb(self):
        self.log.append(("p.clear_dpb",))

    def add_ref_feature_from_frame(self, frame, apply_feature_adaptor=True):
        self.log.append(("p.add_ref", apply_feature_adaptor))

    def compress(self, x, qp, reset_feature_memory, padding_b, padding_r):
        assert len(x) == self.n, "the driver must pad the tail chunk to the frame delay"
        self.log.append(("p.compress", qp, reset_feature_memory))
        return {"bit_stream": pickle.dumps(x), "ec_parallel": 3}

    def decompress(self, bit_stream, sps, qp, ec_part, reset_feature_memory):
        self.log.append(("p.decompress", qp, ec_part, reset_feature_memory))
        x = pickle.loads(bit_stream)
        return {"x_hat": x if self.n > 1 else x[0]}


@pytest.mark.parametrize("n_frames,delay,intra_period", [(19, 8, -1), (17, 8, 8), (6, 1, -1), (9, 1, 4), (1, 8, -1)])
def test_sequence_driver_protocol_and_roundtrip(n_frames, delay, intra_period):
    rng = np.random.default_rng(n_frames)
    H, W = 36, 52            # not a multiple of 16: padding is passed through to the models
    frames = [(rng.integers(0, 256, (H, W), dtype=np.uint8), rng.integers(0, 256, (H // 2, W // 2), dtype=np.uint8),
               rng.integers(0, 256, (H // 2, W // 2), dtype=np.uint8)) for _ in range(n_frames)]
    log_e, log_d = [], []
    to_model = lambda group, delay_: [_Pic(g) for g in group]    # noqa: E731  stand-in "tensor": a list of pictures
    i_e, p_e = _FakeIntra(log_e), _FakeVideo(log_e, delay)
    enc = SequenceEncoder(i_e, p_e, H, W, qp_i=21, qp_p=33, frame_delay=delay, intra_period=intra_period, reset_interval=8,
                          to_model=to_model)
    data = enc.encode(frames)
    # intra pictures come out of the fake as a 1-element list
    i_d, p_d = _FakeIntra(log_d), _FakeVideo(log_d, delay)
    from_model = lambda x, h, w: (x[0] if isinstance(x, list) else x).planes      # noqa: E731
    out = list(SequenceDecoder(i_d, p_d, frame_delay=delay, from_model=from_model).decode(data, n_frames))
    assert len(out) == n_frames
    for a, b in zip(out, frames):
        assert all(np.array_equal(p, q) for p, q in zip(a, b))
    units = frame_schedule(n_frames, delay, intra_period, 8)
    # encoder protocol: intra -> clear_dpb + add_ref(apply adaptor); P -> compress with the scheduled reset flag
    want_e, want_d = [], []
    for u in units:
        if u.is_intra:
            want_e += [("i.compress", 21, 12, 12), ("p.clear_dpb",), ("p.add_ref", True)]
            want_d += [("i.decompress", 21, H, W, 1), ("p.clear_dpb",), ("p.add_ref", False)]
        else:
            want_e.append(("p.compress", 33, u.reset_feature_memory))
            want_d.append(("p.decompress", 33, 3, u.reset_feature_memory))
    assert log_e == want_e and log_d == want_d
    assert len(enc.bits) == n_frames and sum(enc.bits) == 8 * len(data)
    # exactly one SPS unit, first in the stream
    f = io.BytesIO(data)
    assert stream.read_header(f)["nal_type"] == stream.NalType.NAL_SPS
