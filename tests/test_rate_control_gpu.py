"""Rate estimate and rate control on the device (dcvc_estimate_bits, dcvc_b200.rate_control).

* the rate kernel's Q16 sums equal a numpy restatement of enc_symbol on the same symbols, bit for bit;
* `bytes` is within twice the largest error tests/test_rate_control_cpu.py measures against the real coder;
* estimates interleaved with compress change no byte of the stream (the handle's state is untouched);
* a per-unit QP schedule decodes with the mirrors and with the reference's own models;
* the controller hits a reachable target within 5 % and is deterministic; run_job carries it.

The `small` cases also run under emulation on the CPU tier (tests/test_rate_control_cpu.py)."""
import numpy as np
import pytest
import torch

from test_reference_surface_gpu import REF_ROOT, _ref_intra, _ref_video, ref_modules  # noqa: F401  (fixture)
from test_sequence_gpu import _planes

pytestmark = pytest.mark.gpu
SKIP = 0.15
# twice the error model of the CPU comparison with the real coder (tests/test_rate_control_cpu.py:
# MEASURED_MAX_RELATIVE_ERROR of the stream + 1 byte per rANS stream)
MEASURED_MAX_RELATIVE_ERROR = 2.1e-4


def _size_tolerance(n_bytes, ec_parallel):
    return 2 * (MEASURED_MAX_RELATIVE_ERROR * n_bytes + ec_parallel)


def _nets():
    from dcvc_b200.model import DMC, DMCHTL, DMCI, DMCLD
    nets = {}
    for name, cls, seed in (("intra", DMCI, 0), ("hts", DMC, 1), ("ld", DMCLD, 2), ("htl", DMCHTL, 3)):
        m = cls.synthetic(seed)
        m.update(SKIP)
        nets[name] = m.half().to("cuda")
    return nets


@pytest.fixture(scope="module")
def nets():
    return _nets()


def _cost_tables(lib, cdf, lengths):
    import ctypes as C
    cdf = np.ascontiguousarray(cdf, dtype=np.int32)
    lengths = np.ascontiguousarray(lengths, dtype=np.int32)
    out = np.zeros(cdf.shape, dtype=np.uint32)
    assert lib.dcvc_rans_cost_table(cdf.ctypes.data, lengths.ctypes.data, cdf.shape[0], cdf.shape[1],
                                    out.ctypes.data_as(C.c_void_p)) == 0
    return out.astype(np.int64), (lengths - 2).astype(np.int64)


def _np_cost(sym, rows, cost, maxv):
    """enc_symbol's code length in Q16 per symbol (rans_host.cpp), summed"""
    sym = sym.astype(np.int64)
    value = np.abs(sym) * 2 - (sym > 0)
    mv = maxv[rows]
    esc = value >= mv
    raw = np.where(esc, value - mv, 0)
    n_digits = np.zeros_like(raw)
    r = raw.copy()
    while np.any(r):
        n_digits += r > 0
        r >>= 2
    idx = np.where(esc, mv, value)
    c = cost[rows, idx] + np.where(esc, 2 * 65536 * (n_digits // 3 + 1 + n_digits), 0)
    return int(c.sum())


def _restated(net, kind, qp):
    """(y_q16, z_q16, y_symbols) of the symbols the estimate left on the device"""
    from dcvc_b200 import _lib
    lib = _lib.load()
    zc, zl, yc, yl = net._cdf
    ycost, ymaxv = _cost_tables(lib, yc, yl)
    zcost, zmaxv = _cost_tables(lib, zc, zl)
    p = net.proxy
    if kind in ("intra", "htl"):
        counts = p.debug_fetch("totals", np.int32)[:4]
        packed = [p.debug_fetch(f"sym{k}", np.int16)[:counts[k]] for k in range(4)]
    else:
        counts = p.debug_fetch("total", np.int32)[:1]
        packed = [p.debug_fetch("sym", np.int16)[:counts[0]]]
    y = np.concatenate(packed) if packed else np.zeros(0, np.int16)
    rows = (y.astype(np.int64) & 0xff)
    syms = (y.astype(np.int64) >> 8).astype(np.int8)
    z = p.debug_fetch("z_i8", np.int8)
    zrows = np.arange(z.size) % 128 + qp * 128
    return _np_cost(syms, rows, ycost, ymaxv), _np_cost(z, zrows, zcost, zmaxv), int(counts.sum())


def _input(kind, h, w, seed=3):
    from util_frames import synth_frame
    n = {"intra": 1, "ld": 1, "hts": 8, "htl": 8}[kind]
    x = torch.cat([synth_frame(h, w, seed + i) for i in range(n)], dim=1)
    return x.half().cuda().contiguous(memory_format=torch.channels_last)


def _prime(nets, kind, h, w):
    """a reference for the P codecs, as after an intra picture"""
    if kind == "intra":
        return
    i_net, p_net = nets["intra"], nets[kind]
    pad_r, pad_b = i_net.get_padding_size(h, w, 16)
    e = i_net.compress(_input("intra", h, w, 11), 30, pad_b, pad_r)
    p_net.clear_dpb()
    p_net.add_ref_feature_from_frame(e["x_hat"])


def _estimate(net, kind, x, qps, pad_b, pad_r):
    if kind == "intra":
        return net.estimate_bits(x, qps, pad_b, pad_r)
    return net.estimate_bits(x, qps, 0, pad_b, pad_r)


def _compress(net, kind, x, qp, pad_b, pad_r):
    if kind == "intra":
        return net.compress(x, qp, pad_b, pad_r)
    return net.compress(x, qp, 0, pad_b, pad_r)


SIZES = [pytest.param(64, 96, id="small"), pytest.param(256, 384, id="256x384"), pytest.param(1080, 1920, id="1080p")]


@pytest.mark.parametrize("h,w", SIZES)
@pytest.mark.parametrize("kind", ["intra", "hts", "ld", "htl"])
def test_estimate_is_the_exact_table_sum_and_close_to_the_stream(nets, kind, h, w):
    net = nets[kind]
    _prime(nets, kind, h, w)
    pad_r, pad_b = net.get_padding_size(h, w, 16)
    x = _input(kind, h, w)
    for qp in (0, 21, 42, 63):
        r = _estimate(net, kind, x, [qp], pad_b, pad_r)[0]
        torch.cuda.synchronize()
        y_q16, z_q16, n_sym = _restated(net, kind, qp)
        assert r["bits_y"] * 65536 == y_q16 and r["bits_z"] * 65536 == z_q16, (kind, qp, r, y_q16, z_q16)
        assert r["y_symbols"] == n_sym
        e = _compress(net, kind, x, qp, pad_b, pad_r)
        assert e["ec_parallel"] == r["ec_parallel"]
        n = len(e["bit_stream"])
        assert abs(r["bytes"] - n) <= _size_tolerance(n, r["ec_parallel"]), (kind, qp, r["bytes"], n)


class _Probing:
    """a model whose compress() is preceded by estimates at random QPs"""

    def __init__(self, net, intra, rng):
        self.net, self.intra, self.rng = net, intra, rng

    def __getattr__(self, name):
        return getattr(self.net, name)

    def compress(self, x, qp, *args):
        qps = [int(q) for q in self.rng.integers(0, 64, 3)]
        self.net.estimate_bits(x, qps, *args)
        out = self.net.compress(x, qp, *args)
        if self.intra:
            self.x_hats.append(out["x_hat"].clone())
        return out


SEQ = {"intra": (1, 3, 32), "ld": (1, 6, 4), "hts": (8, 25, 16), "htl": (8, 25, 16)}


def _encode(nets, kind, frames, h, w, probe, rate_control=None, qp_i=30, qp_p=25):
    from dcvc_b200.sequence import SequenceEncoder
    delay, _, reset = SEQ[kind]
    i_net, p_net = nets["intra"], nets["ld" if kind == "intra" else kind]
    if probe:
        rng = np.random.default_rng(7)
        i_net, p_net = _Probing(i_net, True, rng), _Probing(p_net, False, rng)
        i_net.x_hats = []
    enc = SequenceEncoder(i_net, p_net, h, w, qp_i, qp_p, frame_delay=delay, reset_interval=reset,
                          force_intra=kind == "intra", rate_control=rate_control)
    return enc.encode(frames), (i_net.x_hats if probe else None)


@pytest.mark.parametrize("kind", ["intra", "hts", "ld", "htl"])
def test_estimates_between_units_change_nothing(nets, kind):
    from dcvc_b200.sequence import SequenceDecoder
    h, w = 72, 104
    delay, n, _ = SEQ[kind]
    frames = _planes(n, 5)
    plain, _ = _encode(nets, kind, frames, h, w, False)
    probed, x_hats = _encode(nets, kind, frames, h, w, True)
    assert probed == plain
    p_net = nets["ld" if kind == "intra" else kind]
    dec = SequenceDecoder(nets["intra"], p_net, frame_delay=delay, force_intra=kind == "intra",
                          from_model=lambda x, hh, ww: x.clone())
    hats = list(dec.decode(probed, n))
    torch.cuda.synchronize()
    if kind == "intra":
        assert all(torch.equal(a, b) for a, b in zip(hats, x_hats))


class _Cycle:
    """a fixed per-unit QP schedule with the controller's interface"""

    def __init__(self, qps):
        self.qps, self.i, self.history = qps, 0, []

    def choose(self, first, count, is_intra, estimate):
        qp = self.qps[self.i % len(self.qps)]
        self.i += 1
        return qp

    def update(self, n):
        self.history.append(n)


@pytest.mark.parametrize("kind", ["hts", "ld"])
@pytest.mark.skipif(REF_ROOT is None, reason="reference Python surface not built (python oracle/build_ref.py)")
def test_variable_qp_stream_decodes_with_the_mirrors_and_the_reference(nets, ref_modules, kind):
    import io

    from dcvc_b200 import stream
    from dcvc_b200.sequence import SequenceDecoder
    h, w = 72, 104
    delay, n, _ = SEQ[kind]
    frames = _planes(n, 9)
    data, x_hats = _encode(nets, kind, frames, h, w, True, rate_control=_Cycle([5, 40, 63, 17, 29]))
    f, qps = io.BytesIO(data), []
    while f.tell() < len(data):
        hd = stream.read_header(f)
        if hd["nal_type"] == stream.NalType.NAL_SPS:
            stream.read_sps_remaining(f, hd["sps_id"])
            continue
        qps.append(stream.read_ip_remaining(f)[0])
    assert len(set(qps)) > 2
    mine = [x.clone() for x in SequenceDecoder(nets["intra"], nets[kind], frame_delay=delay,
                                               from_model=lambda x, hh, ww: x).decode(data, n)]
    ref_i = _ref_intra(ref_modules)
    pad_r, pad_b = ref_i.get_padding_size(h, w, 16)
    ref_i.compress(_input("intra", h, w), 0, pad_b, pad_r)     # the reference's DMCI builds its proxy in compress()
    ref = [x.clone() for x in SequenceDecoder(ref_i, _ref_video(ref_modules, kind), frame_delay=delay,
                                              from_model=lambda x, hh, ww: x).decode(data, n)]
    torch.cuda.synchronize()
    assert torch.equal(mine[0], x_hats[0])
    assert all(torch.equal(a, b) for a, b in zip(mine, ref))


@pytest.mark.parametrize("kind", ["ld", "hts"])
def test_controller_hits_a_fixed_qp_rate(nets, kind):
    from dcvc_b200.rate_control import RateController
    h, w, n, fps = 256, 384, 65, 30.0
    frames = _planes_at(n, h, w)
    fixed, _ = _encode_at(nets, kind, frames, h, w, 40, 40)
    target_kbps = len(fixed) * 8 / (n / fps) / 1000
    runs = []
    for _ in range(2):
        rc = RateController(target_kbps, fps=fps)
        data, _ = _encode_at(nets, kind, frames, h, w, 0, 0, rc)
        runs.append((data, rc))
    (d0, rc0), (d1, _) = runs
    assert d0 == d1
    assert all(0 <= u["qp"] <= 63 for u in rc0.history)
    assert sum(u["bytes"] for u in rc0.history) == len(d0)
    spread = len(d0) / len(fixed) - 1
    print(f"[rate] {kind}: target {len(fixed)} B, achieved {len(d0)} B ({100 * spread:+.2f} %), "
          f"qps {[u['qp'] for u in rc0.history]}, trials/unit {np.mean([len(u['tried']) for u in rc0.history]):.2f}")
    assert abs(spread) <= 0.05


def _planes_at(n, h, w):
    rng = np.random.default_rng(21)
    base = rng.random((h + 80, w + 80)).astype(np.float32)
    out = []
    for t in range(n):
        img = np.roll(base, (t, t // 2), axis=(0, 1))[40:40 + h, 40:40 + w]
        y = torch.from_numpy(np.clip(img * 200 + 20, 0, 255).astype(np.uint8)).cuda().contiguous()
        u = torch.from_numpy(np.clip(img[::2, ::2] * 90 + 80, 0, 255).astype(np.uint8)).cuda().contiguous()
        v = torch.from_numpy(np.clip(img[1::2, 1::2] * 70 + 100, 0, 255).astype(np.uint8)).cuda().contiguous()
        out.append((y, u, v))
    return out


def _encode_at(nets, kind, frames, h, w, qp_i, qp_p, rc=None):
    from dcvc_b200.sequence import SequenceEncoder
    delay = 1 if kind == "ld" else 8
    enc = SequenceEncoder(nets["intra"], nets[kind], h, w, qp_i, qp_p, frame_delay=delay, rate_control=rc)
    return enc.encode(frames), enc


def test_run_job_with_rate_control(nets):
    from dcvc_b200.rate_control import RateController
    from dcvc_b200.sequence import run_job
    h, w, n = 72, 104, 9
    frames = _planes(n, 13)
    _, fixed_log = run_job(nets["intra"], nets["hts"], frames, h, w, 30, 30, frame_delay=8)
    rc = RateController(200.0, fps=30.0)
    data, log = run_job(nets["intra"], nets["hts"], frames, h, w, 30, 30, frame_delay=8, rate_control=rc)
    assert set(log) == set(fixed_log)
    assert sum(u["bytes"] for u in rc.history) == len(data)
    assert log["ave_all_frame_bpp"] == pytest.approx(8 * len(data) / (n * h * w), rel=1e-12)
