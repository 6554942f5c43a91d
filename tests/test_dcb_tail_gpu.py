"""dcb_tail — dc.3 -> ffn.0 -> ffn.2 (-> next dc.0) of a DepthConvBlock as one CTA-pair kernel — against
(a) the fp32 oracle of the same four ops (oracle/ops_ref.py, the restatement of layers.py:152-159 that pins the per-op
kernels) and (b) the per-op pw_gemm kernels on the device, which round to fp16 at exactly the same three places
(o, t1', y): the fused kernel must agree with them to fp16 rounding of fp32 sums."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _rand(gen, *shape, scale=1.0):
    return ((torch.rand(*shape, generator=gen) - 0.5) * 2 * scale).half().float()


def _nhwc(x):
    return x[0].permute(1, 2, 0).contiguous().half().cuda()


def _nchw(t):
    return t.permute(2, 0, 1).unsqueeze(0)


# (H, W, C, inner, inner_next, shortcut, q)
CASES = [
    (16, 16, 128, 128, 128, False, False),     # one pair tile, one chunk per phase
    (16, 16, 384, 384, 384, False, False),     # the Intra P8 block shape, M = 256
    (17, 30, 384, 384, 0, True, True),         # ragged M = 510 (second CTA's last rows out of range), no phase 4
    (32, 40, 256, 128, 256, False, False),     # dcb2-style narrow inner width
    (68, 120, 512, 512, 512, False, False),    # P16 prior blocks: O fills 256 TMEM columns, P = 128 KB
    (136, 240, 384, 384, 384, True, False),    # 1080p P8: 128 pair tiles over 74 pairs (two tiles per pair, tail tile half empty)
    (136, 240, 384, 384, 0, False, True),
]


def _make(gen, H, W, C, inner, inner_n):
    d = {}
    d["t2"] = _rand(gen, 1, inner, H, W)
    d["x"] = _rand(gen, 1, C, H, W)
    d["w3"] = _rand(gen, C, inner, 1, 1, scale=inner ** -0.5)
    d["b3"] = _rand(gen, C, scale=0.1)
    d["wf0"] = _rand(gen, 4 * inner, C, 1, 1, scale=C ** -0.5)
    d["bf0"] = _rand(gen, 4 * inner, scale=0.1)
    d["wf2"] = _rand(gen, C, inner, 1, 1, scale=inner ** -0.5)
    d["bf2"] = _rand(gen, C, scale=0.1)
    if inner_n:
        d["w0n"] = _rand(gen, inner_n, C, 1, 1, scale=C ** -0.5)
        d["b0n"] = _rand(gen, inner_n, scale=0.1)
    return d


def _oracle(d, shortcut, qs, inner_n):
    from oracle import ops_ref
    h16 = lambda t: t.half().float()  # noqa: E731  (the kernels store o, t1', y as fp16)
    o = h16(ops_ref.conv1x1(d["t2"], d["w3"], d["b3"], res1=d["x"]))
    t1 = h16(ops_ref.conv1x1(o, d["wf0"], d["bf0"], act=True, chunk_add=True))
    y = h16(ops_ref.conv1x1(t1, d["wf2"], d["bf2"], res1=o, res2=d["x"] if shortcut else None, q=qs))
    t1n = h16(ops_ref.conv1x1(y, d["w0n"], d["b0n"], act=True)) if inner_n else None
    return y, t1n


def _per_op(d, H, W, C, inner, inner_n, shortcut, qs):
    from dcvc_b200 import ops
    dev = dict(device="cuda", dtype=torch.float16)
    x, t2 = _nhwc(d["x"]), _nhwc(d["t2"])
    o = torch.zeros(H, W, C, **dev)
    t1 = torch.zeros(H, W, inner, **dev)
    y = torch.zeros(H, W, C, **dev)
    pw = lambda w: ops.pack_weight(ops.GEMM_PW, w)  # noqa: E731
    ops.gemm(ops.GEMM_PW, t2, pw(d["w3"]), C, o, bias=d["b3"].half().cuda(), res1=x)
    ops.gemm(ops.GEMM_PW, o, pw(d["wf0"]), 4 * inner, t1, bias=d["bf0"].half().cuda(), act=ops.ACT_WSILU, chunk_add=True)
    ops.gemm(ops.GEMM_PW, t1, pw(d["wf2"]), C, y, bias=d["bf2"].half().cuda(), res1=o, res2=x if shortcut else None,
             qscale=qs.half().cuda() if qs is not None else None)
    t1n = None
    if inner_n:
        t1n = torch.zeros(H, W, inner_n, **dev)
        ops.gemm(ops.GEMM_PW, y, pw(d["w0n"]), inner_n, t1n, bias=d["b0n"].half().cuda(), act=ops.ACT_WSILU)
    return y, t1n


def _fused(d, H, W, C, inner, inner_n, shortcut, qs, y_out=None, t2_in=None, x_is_y=False):
    from dcvc_b200 import ops
    dev = dict(device="cuda", dtype=torch.float16)
    g = lambda k: d[k].half().cuda().reshape(d[k].shape[0], -1).contiguous() if k in d else None  # noqa: E731
    y = y_out if y_out is not None else torch.zeros(H, W, C, **dev)
    t1n = torch.zeros(H, W, inner_n, **dev) if inner_n else None
    ok = ops.dcb_tail(t2_in if t2_in is not None else _nhwc(d["t2"]), y if x_is_y else _nhwc(d["x"]), y, g("w3"), g("b3"), g("wf0"), g("bf0"),
                      g("wf2"), g("bf2"), t1n=t1n, w0n=g("w0n"), b0n=g("b0n"),
                      qscale=qs.half().cuda() if qs is not None else None, shortcut=shortcut)
    assert ok, "shape must be eligible for the fused kernel"
    torch.cuda.synchronize()
    return y, t1n


def _cmp(name, got, ref, rel, abs_):
    got, ref = got.float().cpu(), ref.float().cpu()
    err = (got - ref).abs()
    bad = (err > abs_ + rel * ref.abs()).sum().item()
    assert bad == 0, f"{name}: {bad} / {err.numel()} mismatches, max err {err.max().item():.5f}"


@pytest.mark.parametrize("H,W,C,inner,inner_n,shortcut,q", CASES)
def test_dcb_tail_matches_oracle_and_per_op_kernels(H, W, C, inner, inner_n, shortcut, q):
    gen = torch.Generator().manual_seed(H * 131 + W * 7 + C + inner)
    d = _make(gen, H, W, C, inner, inner_n)
    qs = (torch.rand(C, generator=gen) + 0.5).half().float() if q else None
    y_f, t_f = _fused(d, H, W, C, inner, inner_n, shortcut, qs)
    y_o, t_o = _oracle(d, shortcut, qs, inner_n)
    # three chained fp16 roundings: a flipped rounding of o or t1' moves y by ~1 fp16 ulp of its magnitude
    _cmp("y vs oracle", _nchw(y_f), y_o, 6e-3, 4e-3)
    if inner_n:
        _cmp("t1n vs oracle", _nchw(t_f), t_o, 6e-3, 4e-3)
    y_p, t_p = _per_op(d, H, W, C, inner, inner_n, shortcut, qs)
    torch.cuda.synchronize()
    _cmp("y vs per-op kernels", y_f, y_p, 2e-3, 2e-3)
    if inner_n:
        _cmp("t1n vs per-op kernels", t_f, t_p, 2e-3, 2e-3)
    same = (y_f == y_p).float().mean().item()
    print(f"[dcb_tail] {H}x{W} C={C} inner={inner}: y bit-identical to the per-op kernels in {100 * same:.3f} % of the elements")


@pytest.mark.parametrize("H,W,C,inner,inner_n,pairs", [(68, 120, 512, 512, 512, 4), (136, 240, 384, 384, 384, 8), (68, 120, 256, 128, 256, 3),
                                                      (135, 240, 512, 512, 512, 0)])
def test_dcb_tail_many_tiles_per_pair_in_place(H, W, C, inner, inner_n, pairs, monkeypatch):
    """several tiles per CTA pair (4K pictures; here forced with the debug cap on the grid) with y overwriting x, the way
    CodecBase::dcb runs the blocks of a network: bit-identical to the per-op kernels, run after run"""
    if pairs:
        monkeypatch.setenv("DCVC_B200_DT_MAXPAIRS", str(pairs))
    gen = torch.Generator().manual_seed(H + W + C)
    d = _make(gen, H, W, C, inner, inner_n)
    y_p, t_p = _per_op(d, H, W, C, inner, inner_n, True, None)
    torch.cuda.synchronize()
    for rep in range(3):
        xy = _nhwc(d["x"]).clone()
        y_f, t_f = _fused(d, H, W, C, inner, inner_n, True, None, y_out=xy, x_is_y=True)
        assert torch.equal(y_f, y_p), f"rep {rep}: y differs in {(y_f != y_p).sum().item()} elements"
        assert torch.equal(t_f, t_p), f"rep {rep}: t1n differs in {(t_f != t_p).sum().item()} elements"


def test_dcb_tail_pitched_views_and_in_place_output():
    """t2 is a channel slice of a wider buffer; y overwrites x in place (what CodecBase::dcb does: the block output lands in
    the block input's buffer)."""
    from dcvc_b200 import ops
    H, W, C, inner = 24, 40, 256, 256
    gen = torch.Generator().manual_seed(99)
    d = _make(gen, H, W, C, inner, 0)
    wide = torch.zeros(H, W, 2 * inner, device="cuda", dtype=torch.float16)
    wide[..., inner:] = _nhwc(d["t2"])
    xbuf = _nhwc(d["x"]).clone()
    g = lambda k: d[k].half().cuda().reshape(d[k].shape[0], -1).contiguous()  # noqa: E731
    assert ops.dcb_tail(wide[..., inner:], xbuf, xbuf, g("w3"), g("b3"), g("wf0"), g("bf0"), g("wf2"), g("bf2"), shortcut=True)
    torch.cuda.synchronize()
    y_o, _ = _oracle(d, True, None, 0)
    _cmp("in-place y vs oracle", _nchw(xbuf), y_o, 6e-3, 4e-3)


def test_dcb_tail_declines_unsupported_shapes():
    from dcvc_b200 import ops
    H, W, C, inner = 8, 8, 192, 192          # C % 128 != 0
    gen = torch.Generator().manual_seed(5)
    d = _make(gen, H, W, C, inner, 0)
    g = lambda k: d[k].half().cuda().reshape(d[k].shape[0], -1).contiguous()  # noqa: E731
    y = torch.zeros(H, W, C, device="cuda", dtype=torch.float16)
    assert ops.dcb_tail(_nhwc(d["t2"]), _nhwc(d["x"]), y, g("w3"), g("b3"), g("wf0"), g("bf0"), g("wf2"), g("bf2")) is False


def _reference_layers():
    """the reference's own src/layers/layers.py (the byte-code oracle/build_ref.py emits into oracle/_ref/py)"""
    import sys
    from oracle.build_ref import py_surface_root
    root = py_surface_root()
    if root is None:
        return None
    if root not in sys.path:
        sys.path.insert(0, root)
    from src.layers import layers
    return layers


@pytest.mark.parametrize("H,W,C,dcb2,shortcut", [(68, 120, 384, False, False), (136, 240, 384, False, True), (68, 120, 512, True, False)])
def test_whole_depth_conv_block_against_the_reference_module(H, W, C, dcb2, shortcut):
    """One DepthConvBlock end to end — dc.0 (pw_gemm) -> depthwise 3x3 (dw3x3) -> fused tail (dcb_tail) — against the
    REFERENCE's own nn.Module (src/layers/layers.py:134-159) evaluated in fp32 on the CPU with the same fp16 weights.
    Error budget: the block stores five fp16 tensors on the way (t1, t2, o, t1', y); each rounding moves a value by at most
    half an fp16 ulp of its magnitude (2^-11 relative) and the following 1x1 convolutions average such errors down, so the
    output stays within a few ulps: asserted 8 ulp (2^-10 x 8 of max(|y|, 1/4)) for every element, 2 ulp for 99.9 % of them."""
    layers = _reference_layers()
    if layers is None:
        pytest.skip("reference layers module not available")
    from dcvc_b200 import ops
    torch.manual_seed(H + C)
    blk = layers.DepthConvBlock(C, C, dcb2=dcb2, shortcut=shortcut).eval()
    with torch.no_grad():
        for prm in blk.parameters():
            prm.copy_((prm * 1.0).half().float())
    inner = blk.dc[0].out_channels
    x = _rand(torch.Generator().manual_seed(5), 1, C, H, W, scale=0.5)
    with torch.no_grad():
        ref = blk(x)
    dev = dict(device="cuda", dtype=torch.float16)
    w2 = lambda conv: conv.weight.detach().half().cuda().reshape(conv.out_channels, -1).contiguous()  # noqa: E731
    b2 = lambda conv: conv.bias.detach().half().cuda()  # noqa: E731
    xg = _nhwc(x)
    t1 = torch.zeros(H, W, inner, **dev)
    t2 = torch.zeros(H, W, inner, **dev)
    y = torch.zeros(H, W, C, **dev)
    ops.gemm(ops.GEMM_PW, xg, w2(blk.dc[0]), inner, t1, bias=b2(blk.dc[0]), act=ops.ACT_WSILU)
    # depthwise 3x3: weights [9][C]; its bias is folded into dc.3's bias by the codecs (W3 . b_dw + b3), do the same here
    wdw = blk.dc[2].weight.detach().reshape(inner, 9).t().contiguous().half().cuda()
    ops.dw3x3(t1, wdw, t2)
    b3 = (blk.dc[3].weight.detach().reshape(C, inner).double() @ blk.dc[2].bias.detach().double() + blk.dc[3].bias.detach().double()).float().half().cuda()
    assert ops.dcb_tail(t2, xg, y, w2(blk.dc[3]), b3, w2(blk.ffn[0]), b2(blk.ffn[0]), w2(blk.ffn[2]), b2(blk.ffn[2]), shortcut=shortcut)
    torch.cuda.synchronize()
    got = _nchw(y).float().cpu()
    ulp = (2.0 ** -10) * torch.clamp(ref.abs(), min=0.25)
    err = (got - ref).abs() / ulp
    print(f"[block parity] C={C} inner={inner} shortcut={shortcut}: max {err.max().item():.2f} ulp, "
          f"99.9 % within {torch.quantile(err.flatten()[:2_000_000], 0.999).item():.2f} ulp, mean {err.mean().item():.3f} ulp")
    assert err.max().item() <= 8.0
    assert (err <= 2.0).float().mean().item() >= 0.999
