"""Generates tests/golden/*.npz|json by importing the REFERENCE itself (python modules from
/root/reference, rANS built from its sources into oracle/_ref).  Run in the authoring container:

    python tests/golden/make_golden.py

The reference ships no golden vectors of its own (SURVEY.md §8c), so these fixtures are what pins
the oracle (oracle/dmci_oracle.py, oracle/ops_ref.py) and the host-side mirrors (dcvc_b200/spec.py,
dcvc_b200/entropy.py, the product rANS coder).  Weights are never stored: they are regenerated from
dcvc_b200.spec.synth_state_dict(seed).
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, "/root/reference")
from oracle.build_ref import build_ref, OUT_DIR  # noqa: E402

build_ref()
sys.path.insert(0, OUT_DIR)

from src.models.image_model import DMCI  # noqa: E402  (reference)
from src.models.entropy_models import BitEstimator, EntropyCoder, GaussianEncoder  # noqa: E402
import MLCodec_extensions_cpp as ref_rans  # noqa: E402

from dcvc_b200.spec import dmci_spec, synth_state_dict  # noqa: E402


def synth_frame(h, w, seed, channels=3):
    """band-limited noise frame in [-0.5, 0.5], fp16-representable (SURVEY.md §8d recipe, 4:4:4)"""
    rng = np.random.default_rng(seed)
    x = rng.random((1, channels, h + 4, w + 4)).astype(np.float32)
    t = torch.from_numpy(x)
    t = torch.nn.functional.avg_pool2d(t, 5, 1)
    t = (t - t.mean()) / t.std() * 0.18
    return t.clamp(-0.5, 0.5).half().float()


def make_ld():
    """6. low-delay model: layout + a 4-frame forward sequence (state carried, reset on frame 1), seed 2"""
    from src.models.video_model_ld import DMC as DMC_LD
    from dcvc_b200.spec import ld_spec
    p = DMC_LD()
    with open(os.path.join(HERE, "ld_state_dict_layout.json"), "w") as f:
        json.dump({k: list(v.shape) for k, v in p.state_dict().items()}, f, indent=0, sort_keys=True)
    p.load_state_dict(synth_state_dict(ld_spec(), 2), strict=True)
    p.eval()
    ref0 = synth_frame(64, 64, 700)
    out = {"ref_frame": ref0.numpy()}
    with torch.inference_mode():
        p.clear_dpb()
        p.ref_feature = torch.nn.functional.pixel_unshuffle(ref0, 8)
        for c, reset in enumerate([False, True, False, False]):
            x = synth_frame(64, 64, 800 + c)
            qp = 10 + 15 * c
            r = p.forward_one_frame(x, torch.tensor([qp]), reset_feature_memory=reset)
            out[f"x{c}"] = x.numpy()
            out[f"qp{c}"] = np.int32(qp)
            out[f"x_hat{c}"] = r["x_hat"].numpy()
            out[f"ref_feature{c}"] = p.ref_feature.numpy()
    np.savez_compressed(os.path.join(HERE, "ld_forward_64x64.npz"), **out)


def make_htl():
    """7. HT-L: layout + a 3-chunk forward sequence (state carried, reset on chunk 1), seed 3"""
    from src.models.video_model_ht import DMC as DMC_HT
    from src.utils.common import ModelStructure
    from dcvc_b200.spec import htl_spec
    p = DMC_HT(ModelStructure.HTL)
    with open(os.path.join(HERE, "htl_state_dict_layout.json"), "w") as f:
        json.dump({k: list(v.shape) for k, v in p.state_dict().items()}, f, indent=0, sort_keys=True)
    p.load_state_dict(synth_state_dict(htl_spec(), 3), strict=True)
    p.eval()
    ref0 = synth_frame(64, 64, 710)
    out = {"ref_frame": ref0.numpy()}
    with torch.inference_mode():
        p.clear_dpb()
        p.ref_feature = torch.nn.functional.pixel_unshuffle(ref0, 8)
        for c, reset in enumerate([False, True, False]):
            x = synth_frame(64, 64, 810 + c, channels=24)
            qp = 12 + 20 * c
            r = p.forward_one_frame(x, torch.tensor([qp]), reset_feature_memory=reset)
            out[f"x{c}"] = x.numpy()
            out[f"qp{c}"] = np.int32(qp)
            out[f"x_hat{c}"] = torch.cat(r["x_hat"], 1).numpy()
            out[f"ref_feature{c}"] = p.ref_feature.numpy()
    np.savez_compressed(os.path.join(HERE, "htl_forward_64x64.npz"), **out)


def container_payload(n, seed):
    return np.random.default_rng(seed).integers(0, 256, n, dtype=np.uint8).tobytes()


def container_script(seed):
    """a deterministic series of container writes shared by the golden and the test: ["sps", id, h, w] and
    ["ip", is_i, sps_id, qp, ec_parallel, reset, payload_len, payload_seed]; lengths sit on the varint boundaries"""
    rng = np.random.default_rng(seed)
    ops = []
    sizes = [(1080, 1920), (64, 64), (2160, 3840), (120, 17000)]
    lengths = [0, 1, 100, 127, 128, 16383, 16384, 70000]
    for i, (h, w) in enumerate(sizes):
        ops.append(["sps", i, h, w])
        for j in range(4):
            ops.append(["ip", bool(rng.integers(0, 2)), i, int(rng.integers(0, 64)), int(rng.integers(1, 9)),
                        int(rng.integers(0, 2)), lengths[(2 * i + j) % len(lengths)], 100 * i + j])
    return ops


def make_stream():
    """byte stream the reference's own container helpers produce for container_script(7): length, sha256, head"""
    import hashlib
    import io
    from src.utils.stream_helper import write_ip, write_sps  # reference
    ops = container_script(7)
    f = io.BytesIO()
    for op in ops:
        if op[0] == "sps":
            write_sps(f, {"sps_id": op[1], "height": op[2], "width": op[3]})
        else:
            write_ip(f, op[1], op[2], op[3], op[4], op[5], container_payload(op[6], op[7]))
    data = f.getvalue()
    with open(os.path.join(HERE, "stream_container.json"), "w") as out:
        json.dump({"ops": ops, "length": len(data), "sha256": hashlib.sha256(data).hexdigest(), "head_hex": data[:512].hex()}, out)


def container_random_ops(seed=11):
    """random container writes (ids 0..15, heights / widths / payloads across the varint widths), same format as
    container_script"""
    rng = np.random.default_rng(seed)
    ops = []
    for i in range(16):
        ops.append(["sps", i, int(rng.integers(1, 1 << 14)), int(rng.integers(1, 1 << 20))])
        ops.append(["ip", bool(i & 1), i, int(rng.integers(0, 256)), int(rng.integers(0, 128)), int(rng.integers(0, 2)),
                    int(rng.integers(0, 40000)), i])
    return ops


UINT_ADAPTIVE_VALUES = (0, 1, 127, 128, 16383, 16384, (1 << 30) - 1)


def make_stream_random():
    """the reference's container helpers on container_random_ops(11): stream length / sha256, and the bytes of
    write_uint_adaptive for values on the varint boundaries"""
    import hashlib
    import io
    from src.utils.stream_helper import write_ip, write_sps, write_uint_adaptive  # reference
    ops = container_random_ops(11)
    f = io.BytesIO()
    for op in ops:
        if op[0] == "sps":
            write_sps(f, {"sps_id": op[1], "height": op[2], "width": op[3]})
        else:
            write_ip(f, op[1], op[2], op[3], op[4], op[5], container_payload(op[6], op[7]))
    data = f.getvalue()
    uint = {}
    for v in UINT_ADAPTIVE_VALUES:
        b = io.BytesIO()
        n = write_uint_adaptive(b, v)
        uint[str(v)] = {"returned": n, "hex": b.getvalue().hex()}
    with open(os.path.join(HERE, "stream_container_random.json"), "w") as out:
        json.dump({"ops": ops, "length": len(data), "sha256": hashlib.sha256(data).hexdigest(),
                   "uint_adaptive": uint}, out)


def main():
    torch.manual_seed(0)
    torch.set_num_threads(8)
    if "--only-stream" in sys.argv:   # adds the bitstream-container fixtures without regenerating the others
        make_stream()
        make_stream_random()
        print("container golden fixture written to", HERE)
        return
    if "--only-htl" in sys.argv:   # adds the HT-L fixtures without regenerating the others
        make_htl()
        print("HT-L golden fixtures written to", HERE)
        return
    if "--only-ld" in sys.argv:   # adds the LD fixtures without regenerating the others
        make_ld()
        print("LD golden fixtures written to", HERE)
        return
    # 1. state_dict layout of the reference model
    m = DMCI()
    layout = {k: list(v.shape) for k, v in m.state_dict().items()}
    with open(os.path.join(HERE, "dmci_state_dict_layout.json"), "w") as f:
        json.dump(layout, f, indent=0, sort_keys=True)

    # 2. Gaussian CDF table (deterministic) and a seeded factorised-z table
    ec = EntropyCoder()
    ge = GaussianEncoder()
    ge.update(ec, skip_thres=0.15)
    q, l = ge.get_cdf_info()
    np.savez_compressed(os.path.join(HERE, "gaussian_cdf.npz"), quantized_cdf=q, cdf_length=l)
    be = BitEstimator(4, 16)
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        be.h.copy_(torch.randn(be.h.shape, generator=g) * 0.6 + 0.4)
        be.b.copy_(torch.randn(be.b.shape, generator=g) * 0.5)
        be.a.copy_(torch.randn(be.a.shape, generator=g) * 0.5)
    be.update(ec)
    q, l = be.get_cdf_info()
    np.savez_compressed(os.path.join(HERE, "bitest_cdf.npz"), h=be.h.detach().numpy(), b=be.b.detach().numpy(),
                        a=be.a.detach().numpy(), quantized_cdf=q, cdf_length=l)

    # 3. reference forward_one_frame on synthetic weights (seed 0), 64x64 and 128x64
    sd = synth_state_dict(dmci_spec(), 0)
    m.load_state_dict(sd, strict=True)
    m.eval()
    for (h, w, qp) in [(64, 64, 0), (64, 64, 32), (128, 64, 63)]:
        x = synth_frame(h, w, 1234 + qp)
        with torch.inference_mode():
            # replicate the internals we want to pin in addition to x_hat
            res = m.forward_one_frame(x, torch.tensor([qp]))
            q_enc = m.index_select_dim0(m.q_scale_enc, torch.tensor([qp]))
            y = m.enc(x, q_enc)
            z = m.hyper_enc(y)
        np.savez_compressed(os.path.join(HERE, f"dmci_forward_{h}x{w}_qp{qp}.npz"),
                            x=x.numpy(), x_hat=res["x_hat"].numpy(), y=y.numpy(), z=z.numpy(),
                            bits_y=res["bits_y"].numpy(), bits_z=res["bits_z"].numpy())

    # 4. reference rANS streams for seeded symbols
    m.update(0.15)
    zc, zl = m.bit_estimator_z.get_cdf_info()
    yc, yl = m.gaussian_encoder.get_cdf_info()
    enc = ref_rans.RansEncoder()
    enc.set_cdf(zc, zl, 0)
    enc.set_cdf(yc, yl, 1)
    out = {}
    rng = np.random.default_rng(77)
    for n_par, n_y, n_z in [(1, 5000, 640), (2, 70000, 1280), (3, 100001, 2560), (4, 40000, 128 * 7), (5, 170000, 1280),
                            (8, 270000, 65280), (1, 0, 128), (2, 3, 128)]:
        # symbols: mostly small, a few escapes; rows random
        def make_y(n):
            sym = np.rint(rng.standard_normal(n) * rng.choice([0.3, 1.5, 6.0, 40.0], n, p=[0.5, 0.3, 0.15, 0.05]))
            sym = np.clip(sym, -128, 127).astype(np.int32)
            row = rng.integers(0, 128, n).astype(np.int32)
            return ((sym << 8) + row).astype(np.int16)
        ys = [make_y(n_y // (k + 1)) for k in range(4)]
        z = np.clip(np.rint(rng.standard_normal(n_z) * 3), -64, 63).astype(np.int8)
        qp = int(rng.integers(0, 64))
        enc.reset()
        enc.set_entropy_coder_parallel(n_par)
        for k in (3, 2, 1, 0):
            enc.encode_y(ys[k])
        enc.encode_z(z, qp * 128, 128)
        enc.flush()
        stream = np.asarray(enc.get_encoded_stream()).copy()
        key = f"p{n_par}_y{n_y}_z{n_z}"
        for k in range(4):
            out[f"{key}_y{k}"] = ys[k]
        out[f"{key}_z"] = z
        out[f"{key}_qp"] = np.int32(qp)
        out[f"{key}_stream"] = stream
    np.savez_compressed(os.path.join(HERE, "rans_streams.npz"), **out)

    # 5. HT-S: layout + a 3-chunk forward sequence (state carried, reset on chunk 1) on synthetic weights (seed 1)
    from src.models.video_model_ht import DMC
    from src.utils.common import ModelStructure
    from dcvc_b200.spec import hts_spec
    p = DMC(ModelStructure.HTS)
    with open(os.path.join(HERE, "hts_state_dict_layout.json"), "w") as f:
        json.dump({k: list(v.shape) for k, v in p.state_dict().items()}, f, indent=0, sort_keys=True)
    p.load_state_dict(synth_state_dict(hts_spec(), 1), strict=True)
    p.eval()
    ref0 = synth_frame(64, 64, 500)
    out = {"ref_frame": ref0.numpy()}
    with torch.inference_mode():
        p.clear_dpb()
        p.ref_feature = torch.nn.functional.pixel_unshuffle(ref0, 8)
        for c, reset in enumerate([False, True, False]):
            x = synth_frame(64, 64, 600 + c, channels=24)
            r = p.forward_one_frame(x, torch.tensor([20 + c]), reset_feature_memory=reset)
            out[f"x{c}"] = x.numpy()
            out[f"x_hat{c}"] = torch.cat(r["x_hat"], 1).numpy()
            out[f"ref_feature{c}"] = p.ref_feature.numpy()
    np.savez_compressed(os.path.join(HERE, "hts_forward_64x64.npz"), **out)
    make_ld()
    make_htl()
    print("golden fixtures written to", HERE)


if __name__ == "__main__":
    main()
