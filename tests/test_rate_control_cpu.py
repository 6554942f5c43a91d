"""Rate estimate and rate control without a GPU.

* dcvc_rans_cost_table against a float64 restatement, on the golden CDF tables;
* the size formula of dcvc_estimate_bits (the table sum + 4 flush bytes per rANS stream + 4 per offset word) against
  the real coder's stream length, for Laplacian symbols with escapes, every ec_parallel and several z QP offsets;
* RateController against fake estimators with a known R(QP);
* the sequence driver: unchanged without a controller, each unit's QP from the controller with one;
* the small cases of tests/test_rate_control_gpu.py on the emulated runtime (tests/test_host_dry_run.py)."""
import ctypes as C
import io
import math
import os
import pickle

import numpy as np
import pytest

from test_host_dry_run import dry  # noqa: F401  (session fixture: the relinked library + the runtime shim)
from test_stream_sequence import _FakeIntra, _FakeVideo, _Pic

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def lib():
    from dcvc_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        from dcvc_b200.build import build
        build()
    return _lib.load()


def _cost_table(lib, cdf, lengths):
    cdf = np.ascontiguousarray(cdf, dtype=np.int32)
    lengths = np.ascontiguousarray(lengths, dtype=np.int32)
    out = np.zeros(cdf.shape, dtype=np.uint32)
    assert lib.dcvc_rans_cost_table(cdf.ctypes.data, lengths.ctypes.data, cdf.shape[0], cdf.shape[1],
                                    out.ctypes.data_as(C.c_void_p)) == 0
    return out


@pytest.mark.parametrize("name", ["gaussian_cdf", "bitest_cdf"])
def test_cost_table_matches_a_float64_restatement(lib, name):
    g = np.load(os.path.join(GOLD, name + ".npz"))
    cdf, lengths = g["quantized_cdf"], g["cdf_length"]
    table = _cost_table(lib, cdf, lengths).astype(np.int64)
    for r in range(cdf.shape[0]):
        n = lengths[r] - 1                       # symbols 0 .. max_value
        freq = np.diff(cdf[r, : n + 1].astype(np.float64))
        want = 65536.0 * (16.0 - np.log2(freq))
        assert np.all(np.abs(table[r, :n] - want) <= 1.0), r
        assert np.all(table[r, n:] == 0)


def _np_bits_q16(sym, rows, cost, maxv):
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
    c = cost[rows, np.where(esc, mv, value)] + np.where(esc, 2 * 65536 * (n_digits // 3 + 1 + n_digits), 0)
    return int(c.sum())


def _estimated_bytes(q16, ec):
    n_off = ec // 2 - 1 + ec % 2
    return -(-q16 // (8 << 16)) + 4 * ec + 4 * n_off


# The coder's state has finite precision, so what it spends drifts from the ideal code length by a small fraction of
# the stream; on top of that each rANS stream's flush holds up to 1 byte more or less than its share of the bits.
# The error model is |estimate - stream length| <= MEASURED_MAX_RELATIVE_ERROR * length + 1 byte per stream, with the
# relative part the largest observed below (2.08e-4, at 2 M symbols of a peaked distribution).  The GPU tests allow twice
# this model.
MEASURED_MAX_RELATIVE_ERROR = 2.1e-4


def test_size_formula_against_the_real_coder(lib):
    from test_cpu_parity import _Rans

    from dcvc_b200.entropy import bit_estimator_cdf_tables, gaussian_cdf_tables
    from dcvc_b200.spec import dmci_spec, synth_state_dict
    sd = synth_state_dict({k: v for k, v in dmci_spec().items() if k.startswith("bit_estimator_z.")}, 0)
    zc, zl = bit_estimator_cdf_tables(sd["bit_estimator_z.h"], sd["bit_estimator_z.b"], sd["bit_estimator_z.a"])
    yc, yl = gaussian_cdf_tables()
    coder = _Rans(lib, zc, zl, yc, yl)
    ycost, ymaxv = _cost_table(lib, yc, yl).astype(np.int64), (np.asarray(yl) - 2).astype(np.int64)
    zcost, zmaxv = _cost_table(lib, zc, zl).astype(np.int64), (np.asarray(zl) - 2).astype(np.int64)
    rng = np.random.default_rng(5)
    # (symbols per y step, ec_parallel, largest Laplacian scale, share of far escapes): every ec_parallel with escapes,
    # then unit sizes up to 1080p HT-S (~2 M y symbols) with peaked and wide distributions
    cases = [(ec * 32768 // 4 + int(rng.integers(0, 4000)), ec, 6.0, 0.002) for ec in range(1, 9)]
    cases += [(n, min(8, max(1, 4 * n // 32768)), smax, 0.0) for n in (30000, 130000, 500000) for smax in (0.5, 2.0, 6.0)]
    worst_rel, worst_stream, n_escapes = 0.0, 0, 0
    for i, (n, ec, smax, far) in enumerate(cases):
        qp = (0, 17, 40, 63)[i % 4]
        ys = []
        for _ in range(4):
            rows = rng.integers(0, yc.shape[0], n)
            scale = 0.1 + smax * rows / yc.shape[0]
            sym = np.clip(np.round(rng.laplace(0, scale)), -127, 127).astype(np.int64)
            big = rng.random(n) < far                       # far escapes: several bypass digits
            sym[big] = rng.choice([-120, -60, 60, 127], big.sum())
            ys.append(((sym.astype(np.int16) << 8) | rows.astype(np.int16)).astype(np.int16))
        z = np.clip(np.round(rng.laplace(0, 2.5, 128 * 60)), -64, 63).astype(np.int8)
        y_all = np.concatenate(ys)
        y_rows = y_all.astype(np.int64) & 0xff
        y_sym = (y_all.astype(np.int64) >> 8).astype(np.int8)
        n_escapes += int(np.sum(np.abs(y_sym.astype(np.int64)) * 2 >= ymaxv[y_rows]))
        q16 = _np_bits_q16(y_sym, y_rows, ycost, ymaxv)
        q16 += _np_bits_q16(z, np.arange(z.size) % 128 + qp * 128, zcost, zmaxv)
        stream = coder.encode(ys, z, qp, ec)
        err = abs(_estimated_bytes(q16, ec) - stream.size)
        worst_rel = max(worst_rel, max(0, err - ec) / stream.size)
        worst_stream = max(worst_stream, -(-err // ec))
    print(f"[rate] largest |estimate - stream|: {worst_rel:.2e} of the stream beyond 1 byte per rANS stream; "
          f"{worst_stream} bytes per stream ({n_escapes} escapes)")
    assert n_escapes > 0
    assert worst_rel <= MEASURED_MAX_RELATIVE_ERROR


# ------------------------------------------------------------------------------------------------ controller
def _fake(scale, slope=0.02, bump=None):
    """bytes(qp) = scale * exp(slope * qp), optionally with a non-monotone bump"""
    calls = []

    def est(qps):
        calls.append(list(qps))
        out = []
        for q in qps:
            b = scale * math.exp(slope * q)
            if bump and q in bump:
                b *= bump[q]
            out.append(int(b))
        return out
    return est, calls


def _run(rc, n_units=64, count=1, intra_every=None, scale_i=20000.0, scale_p=4000.0, **kw):
    total = 0
    for u in range(n_units):
        intra = u == 0 or (intra_every and u % intra_every == 0)
        est, _ = _fake(scale_i if intra else scale_p * count, **kw)     # a chunk of `count` pictures
        qp = rc.choose(u * count, count, bool(intra), est)
        actual = est([qp])[0] + 7                    # the unit header
        rc.update(actual)
        total += actual
    return total


@pytest.mark.parametrize("count", [1, 8])
def test_controller_reaches_a_reachable_target(count):
    from dcvc_b200.rate_control import RateController
    fps = 30.0
    n_units = 64
    target_kbps = 8 * 4000 * math.exp(0.02 * 35) * fps / 1000          # P units at about q 35
    rc = RateController(target_kbps, fps=fps)
    total = _run(rc, n_units, count)
    achieved = total * 8 / (n_units * count / fps) / 1000
    assert abs(achieved / target_kbps - 1) <= 0.02, (achieved, target_kbps)


def test_controller_respects_bounds_and_trials():
    from dcvc_b200.rate_control import RateController
    rc = RateController(500.0, qp_min=10, qp_max=50, max_trials=3)
    _run(rc, 40, intra_every=16)
    for h in rc.history:
        assert 10 <= h["qp"] <= 50 and len(h["tried"]) <= 3
        assert all(10 <= q <= 50 for q, _ in h["tried"])


@pytest.mark.parametrize("target_kbps,bound", [(1.0, 0), (1e7, 63)])
def test_controller_saturates_on_unreachable_targets(target_kbps, bound):
    from dcvc_b200.rate_control import RateController
    rc = RateController(target_kbps)
    _run(rc, 20, intra_every=8)
    assert all(h["qp"] == bound for h in rc.history[1:])


def test_controller_survives_flat_and_non_monotone_rates():
    from dcvc_b200.rate_control import RateController
    rc = RateController(1000.0)
    _run(rc, 30, slope=0.0)
    assert all(0 <= h["qp"] <= 63 for h in rc.history)
    rc = RateController(8 * 4000 * math.exp(0.02 * 30) * 30 / 1000)
    total = _run(rc, 64, bump={q: 1.3 if q % 2 else 0.8 for q in range(64)})
    assert all(0 <= h["qp"] <= 63 for h in rc.history) and total > 0


def test_controller_is_deterministic():
    from dcvc_b200.rate_control import RateController
    a, b = RateController(700.0), RateController(700.0)
    _run(a, 40, intra_every=10)
    _run(b, 40, intra_every=10)
    assert a.history == b.history


def test_controller_rejects_bad_settings():
    from dcvc_b200.rate_control import RateController
    for kw in ({"target_kbps": 0}, {"target_kbps": 10, "qp_min": 40, "qp_max": 30}, {"target_kbps": 10, "max_trials": 0}):
        with pytest.raises(ValueError):
            RateController(**kw)


# ------------------------------------------------------------------------------------------------ sequence driver
class _EstIntra(_FakeIntra):
    def estimate_bits(self, x, qps, padding_b, padding_r):
        return [{"bytes": 1000 + 40 * q} for q in qps]

    def compress(self, x, qp, padding_b, padding_r):
        out = super().compress(x, qp, padding_b, padding_r)
        out["bit_stream"] = pickle.dumps((x, b"\0" * (40 * qp)))
        return out

    def decompress(self, bit_stream, sps, qp, ec_part):
        return {"x_hat": pickle.loads(bit_stream)[0]}


class _EstVideo(_FakeVideo):
    def estimate_bits(self, x, qps, reset, padding_b, padding_r):
        return [{"bytes": 300 + 10 * q} for q in qps]


def _frames(n, H=36, W=52, seed=1):
    rng = np.random.default_rng(seed)
    return [(rng.integers(0, 256, (H, W), dtype=np.uint8), rng.integers(0, 256, (H // 2, W // 2), dtype=np.uint8),
             rng.integers(0, 256, (H // 2, W // 2), dtype=np.uint8)) for _ in range(n)]


def test_sequence_without_rate_control_is_unchanged():
    from dcvc_b200 import stream
    from dcvc_b200.sequence import SequenceEncoder, frame_schedule
    H, W, delay, n = 36, 52, 8, 19
    frames = _frames(n)
    to_model = lambda group, d: [_Pic(g) for g in group]    # noqa: E731
    log = []
    data = SequenceEncoder(_FakeIntra(log), _FakeVideo(log, delay), H, W, 21, 33, frame_delay=delay, reset_interval=8,
                           to_model=to_model, rate_control=None).encode(frames)
    out = io.BytesIO()
    stream.write_sps(out, {"sps_id": 0, "height": H, "width": W})
    for u in frame_schedule(n, delay, -1, 8):
        group = frames[u.first:u.first + u.count]
        if not u.is_intra:
            group = group + [group[-1]] * (delay - len(group))
        bs = pickle.dumps([_Pic(g) for g in group])
        stream.write_ip(out, u.is_intra, 0, 21 if u.is_intra else 33, 1 if u.is_intra else 3, u.reset_feature_memory, bs)
    assert data == out.getvalue()


def test_sequence_takes_each_unit_qp_from_the_controller():
    from dcvc_b200 import stream
    from dcvc_b200.rate_control import RateController
    from dcvc_b200.sequence import SequenceDecoder, SequenceEncoder
    H, W, delay, n = 36, 52, 8, 25
    frames = _frames(n, seed=2)
    to_model = lambda group, d: [_Pic(g) for g in group]    # noqa: E731
    rc = RateController(150.0, fps=30.0)
    log = []
    enc = SequenceEncoder(_EstIntra(log), _EstVideo(log, delay), H, W, 0, 0, frame_delay=delay, to_model=to_model,
                          rate_control=rc)
    data = enc.encode(frames)
    assert [h["qp"] for h in rc.history] == [e[1] for e in log if e[0].endswith("compress")]
    assert sum(h["bytes"] for h in rc.history) == len(data) and sum(enc.bits) == 8 * len(data)
    f, qps = io.BytesIO(data), []
    while f.tell() < len(data):
        hd = stream.read_header(f)
        if hd["nal_type"] == stream.NalType.NAL_SPS:
            stream.read_sps_remaining(f, hd["sps_id"])
            continue
        qps.append(stream.read_ip_remaining(f)[0])
    assert qps == [h["qp"] for h in rc.history]
    from_model = lambda x, h, w: (x[0] if isinstance(x, list) else x).planes      # noqa: E731
    out = list(SequenceDecoder(_EstIntra([]), _FakeVideo([], delay), frame_delay=delay, from_model=from_model).decode(data, n))
    assert all(all(np.array_equal(p, q) for p, q in zip(a, b)) for a, b in zip(out, frames))


# ------------------------------------------------------------------------------------------------ under emulation
def test_gpu_rate_tests_run_under_emulation(dry, tmp_path):  # noqa: F811
    """model mirrors -> proxies -> dcvc_estimate_bits -> the rate kernel's host restatement and the codecs' estimate
    wiring: exact sums, sizes against compress, and no state change between units.  The shim of the dry fixture plus
    tests/cpp/cuda_emu_rate.cpp, which adds the rate kernel to the emulated kernels by wrapping their lookup."""
    import shutil
    import subprocess
    import sys
    shim = str(tmp_path / "libdryshim_rate.so")
    wrap = "-Wl," + ",".join(f"--wrap=emu_{f}" for f in ("lookup", "num_args", "arg_size", "run"))
    subprocess.run([shutil.which("g++"), "-O2", "-shared", "-fPIC", "-std=c++17", "-I/usr/local/cuda/include",
                    os.path.join(ROOT, "tests/cpp/cuda_dry_shim.cpp"), os.path.join(ROOT, "tests/cpp/cuda_emu_kernels.cpp"),
                    os.path.join(ROOT, "tests/cpp/cuda_emu_rate.cpp"), wrap, "-o", shim], check=True, capture_output=True)
    env = dry.env(True)
    env["LD_PRELOAD"] = shim
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests/dry_pytest_runner.py"), dry.lib,
                        "tests/test_rate_control_gpu.py", "-q", "-x", "-k",
                        "small or (change_nothing and (intra or ld or hts))"],
                       env=env, capture_output=True, text=True, timeout=3000, cwd=ROOT)
    tail = r.stdout[-3000:] + r.stderr[-2000:]
    assert r.returncode == 0 and " passed" in r.stdout and " failed" not in r.stdout, tail
