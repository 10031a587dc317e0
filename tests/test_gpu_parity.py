"""GPU parity tests (run with ``-m gpu`` on a B200): our sm_100a kernels, called through the C ABI,
against the CPU oracle (oracle/oracle.c) and against what the reference's own kernels computed on the same seeded
inputs (tests/golden/ref_kernels, see tests/ref_golden.py).

Tolerance: max|d|/max|ref| <= 1e-4 and allclose(rtol=1e-4, atol=1e-4*rms(ref)) -- the contract in
BASELINE.json's north_star ("fp32 outputs matching the reference kernels within 1e-4 rel").
"""
import os

import numpy as np
import pytest
import torch

from oracle import cpu as orc
from oracle import ref as oref
import ref_golden as refk
from util import assert_close, rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-4


def _f2():
    import flownet2_b200
    return flownet2_b200


def _randn(shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).float()


# ------------------------------------------------------------------------------------------------
# Correlation
# ------------------------------------------------------------------------------------------------
CORR_CASES = [
    # (pad, k, md, s1, s2), (B, C, H, W), expected path (1 = TMA-tiled, 0 = generic)
    ((20, 1, 20, 1, 2), (1, 256, 48, 64), 2),     # BASELINE cfg1 (tensor-core forward)
    ((20, 1, 20, 1, 2), (2, 64, 10, 36), 2),      # tc: ragged tiles (Hc=5, Wc=18)
    ((20, 1, 20, 1, 2), (1, 128, 2, 2), 2),       # tc: a single class pixel per class
    ((20, 1, 20, 1, 2), (1, 192, 30, 70), 2),     # tc: 3 k-blocks, Wc=35 odd
    ((21, 1, 21, 1, 2), (1, 64, 12, 20), 2),      # tc: md=21 -> dr=10, pad == md
    ((20, 1, 20, 1, 2), (2, 20, 13, 192), 1),     # odd H, C % 8 != 0, 1.5 tiles wide
    ((20, 1, 20, 1, 2), (1, 3, 5, 8), 1),         # tiny: W < tile, H < row quad
    ((20, 1, 20, 1, 2), (1, 64, 9, 260), 1),      # 3 tiles wide, ragged last tile (odd H -> FMA path)
    ((24, 1, 20, 1, 2), (1, 16, 10, 32), 1),      # pad > md (output larger than input), tiled
    ((16, 1, 20, 1, 2), (1, 16, 14, 32), 1),      # pad < md (output smaller), tiled
    ((22, 1, 20, 1, 2), (1, 16, 10, 32), 0),      # (md - pad) % 4 != 0 -> generic (TMA start alignment)
    ((4, 1, 4, 1, 2), (2, 7, 9, 12), 1),          # (s2, dr) = (2, 2)
    ((8, 1, 8, 1, 2), (1, 9, 11, 16), 1),         # (2, 4)
    ((4, 1, 4, 1, 1), (1, 5, 8, 16), 1),          # (1, 4)
    ((3, 1, 3, 1, 1), (1, 5, 8, 8), 0),           # (1, 3): odd halo -> generic
    ((5, 1, 5, 1, 2), (1, 6, 8, 8), 1),           # md % s2 != 0 -> dr = 2
    ((4, 3, 4, 1, 2), (1, 6, 10, 12), 0),         # kernel_size 3 -> generic
    ((4, 1, 4, 1, 2), (1, 6, 9, 11), 0),          # W % 4 != 0 -> generic
    ((3, 1, 4, 1, 2), (1, 6, 9, 12), 0),          # (pad-md) odd -> oW % 4 != 0 -> generic
    ((6, 1, 6, 1, 3), (1, 4, 9, 12), 0),          # stride2 = 3 -> generic
]


@pytest.mark.parametrize("params,shape,path", CORR_CASES)
def test_correlation_vs_oracle(params, shape, path):
    f = _f2()
    pad, k, md, s1, s2 = params
    B, C, H, W = shape
    assert f._lib.LIB.fn2b200_correlation_path(C, H, W, pad, k, md, s1, s2) == path
    a, b = _randn(shape, 10), _randn(shape, 11)
    out = f.functional.correlation_forward(a.cuda(), b.cuda(), pad, k, md, s1, s2)
    ref = orc.correlation_forward(a.numpy(), b.numpy(), pad, k, md, s1, s2)
    assert_close(out.cpu().numpy(), ref, TOL, "corr fwd %s %s" % (params, shape))
    go = _randn(ref.shape, 12)
    g1, g2 = f.functional.correlation_backward(a.cuda(), b.cuda(), go.cuda(), pad, k, md, s1, s2)
    r1, r2 = orc.correlation_backward(a.numpy(), b.numpy(), go.numpy(), pad, k, md, s1, s2)
    assert_close(g1.cpu().numpy(), r1, TOL, "corr gI1 %s %s" % (params, shape))
    assert_close(g2.cpu().numpy(), r2, TOL, "corr gI2 %s %s" % (params, shape))


def test_correlation_tc_matches_fma_path(monkeypatch):
    """The tensor-core forward (bf16 hi/lo split) against the FP32-FMA forward on the same input."""
    f = _f2()
    a, b = _randn((2, 256, 24, 40), 50).cuda(), _randn((2, 256, 24, 40), 51).cuda()
    out_tc = f.functional.correlation_forward(a, b, 20, 1, 20, 1, 2)
    monkeypatch.setenv("FN2B200_CORR_FWD", "fma")
    assert f._lib.LIB.fn2b200_correlation_path(256, 24, 40, 20, 1, 20, 1, 2) == 1
    out_fma = f.functional.correlation_forward(a, b, 20, 1, 20, 1, 2)
    monkeypatch.delenv("FN2B200_CORR_FWD")
    assert f._lib.LIB.fn2b200_correlation_path(256, 24, 40, 20, 1, 20, 1, 2) == 2
    e = rel_err(out_tc.cpu().numpy(), out_fma.cpu().numpy())
    assert 0 < e < 5e-5, e          # different arithmetic (not bit-identical), far inside 1e-4
    go = _randn(tuple(out_fma.shape), 52).cuda()
    g1_tc, g2_tc = f.functional.correlation_backward(a, b, go, 20, 1, 20, 1, 2)
    monkeypatch.setenv("FN2B200_CORR_BWD", "fma")
    g1_fma, g2_fma = f.functional.correlation_backward(a, b, go, 20, 1, 20, 1, 2)
    monkeypatch.delenv("FN2B200_CORR_BWD")
    e1, e2 = rel_err(g1_tc.cpu().numpy(), g1_fma.cpu().numpy()), rel_err(g2_tc.cpu().numpy(), g2_fma.cpu().numpy())
    assert 0 < e1 < 5e-5 and 0 < e2 < 5e-5, (e1, e2)
    only1, none2 = f.functional.correlation_backward(a, b, go, 20, 1, 20, 1, 2, need2=False)
    assert none2 is None and rel_err(only1.cpu().numpy(), g1_fma.cpu().numpy()) < 5e-5
    # one launch computes both gradients (tiles [0, n) and [n, 2n)); each half on its own must give the same bits
    none1, only2 = f.functional.correlation_backward(a, b, go, 20, 1, 20, 1, 2, need1=False)
    assert none1 is None and torch.equal(only2, g2_tc) and torch.equal(only1, g1_tc)
    # badly scaled inputs: the hi/lo split must not lose the small operand
    out_tc = f.functional.correlation_forward(a * 1e-3, b * 3e4, 20, 1, 20, 1, 2)
    assert rel_err(out_tc.cpu().numpy(), (out_fma * 30.0).cpu().numpy()) < 5e-5


def test_correlation_tc_partial_last_round_and_producer_counts(monkeypatch):
    """160 tiles on 148 SMs: the forward deals the 12 tiles of the last, partial round out unit by unit, the
    backward runs 320 tiles in one launch.  Checked against the oracle; the number of TMA producer warps
    (FN2B200_TC_NP) must not change a single bit."""
    f = _f2()
    shape = (5, 64, 32, 128)                       # 5 x 4 classes x (16/8) x (64/16) = 160 tiles
    prm = (20, 1, 20, 1, 2)
    assert f._lib.LIB.fn2b200_correlation_path(shape[1], shape[2], shape[3], *prm) == 2
    a, b = _randn(shape, 70), _randn(shape, 71)
    out = f.functional.correlation_forward(a.cuda(), b.cuda(), *prm)
    go = _randn(tuple(out.shape), 72)
    g1, g2 = f.functional.correlation_backward(a.cuda(), b.cuda(), go.cuda(), *prm)
    assert_close(out.cpu().numpy(), orc.correlation_forward(a.numpy(), b.numpy(), *prm), TOL, "corr fwd tail")
    r1, r2 = orc.correlation_backward(a.numpy(), b.numpy(), go.numpy(), *prm)
    assert_close(g1.cpu().numpy(), r1, TOL, "corr gI1 tail")
    assert_close(g2.cpu().numpy(), r2, TOL, "corr gI2 tail")
    for np_ in ("1", "2"):
        monkeypatch.setenv("FN2B200_TC_NP", np_)
        o2 = f.functional.correlation_forward(a.cuda(), b.cuda(), *prm)
        h1, h2 = f.functional.correlation_backward(a.cuda(), b.cuda(), go.cuda(), *prm)
        assert torch.equal(o2, out) and torch.equal(h1, g1) and torch.equal(h2, g2), np_
    monkeypatch.delenv("FN2B200_TC_NP")


def test_correlation_tc_more_than_65535_rows(monkeypatch):
    """B * H > 65535: the split prepass carries (sample, row) in grid x (ADVICE r1: grid z was capped at 65535 and the
    default tensor-core path failed with 'invalid configuration').  Checked against the FP32-FMA kernels."""
    f = _f2()
    shape = (1200, 64, 56, 16)                          # 67200 rows
    assert f._lib.LIB.fn2b200_correlation_path(shape[1], shape[2], shape[3], 20, 1, 20, 1, 2) == 2
    g = torch.Generator(device="cuda").manual_seed(3)
    a = torch.randn(*shape, device="cuda", generator=g)
    b = torch.randn(*shape, device="cuda", generator=g)
    out = f.functional.correlation_forward(a, b, 20, 1, 20, 1, 2)
    monkeypatch.setenv("FN2B200_CORR_FWD", "fma")
    ref = f.functional.correlation_forward(a, b, 20, 1, 20, 1, 2)
    monkeypatch.delenv("FN2B200_CORR_FWD")
    assert rel_err(out.cpu().numpy(), ref.cpu().numpy()) < 5e-5
    n = 1199
    o1 = orc.correlation_forward(a[n:n + 1].cpu().numpy(), b[n:n + 1].cpu().numpy(), 20, 1, 20, 1, 2)
    assert_close(out[n:n + 1].cpu().numpy(), o1, TOL, "last sample of 1200")


def test_correlation_stride1_2_forward_only():
    f = _f2()
    a, b = _randn((1, 4, 12, 13), 1), _randn((1, 4, 12, 13), 2)
    out = f.functional.correlation_forward(a.cuda(), b.cuda(), 2, 1, 4, 2, 2)
    assert_close(out.cpu().numpy(), orc.correlation_forward(a.numpy(), b.numpy(), 2, 1, 4, 2, 2), TOL, "corr s1=2")
    with pytest.raises(RuntimeError, match="stride1"):
        f.functional.correlation_backward(a.cuda(), b.cuda(), out, 2, 1, 4, 2, 2)


def test_correlation_known_answers_gpu():
    f = _f2()
    ones = torch.ones(1, 5, 8, 8, device="cuda")
    out = f.Correlation(4, 1, 4, 1, 2, 1)(ones, ones)
    assert out.shape == (1, 25, 8, 8)
    assert torch.allclose(out[0, 12], torch.ones(8, 8, device="cuda"))
    assert float(out[0, 0, 0, 0]) == 0.0 and abs(float(out[0, 0, 4, 4]) - 1.0) < 1e-6
    f1 = _randn((1, 16, 16, 16), 3)
    f2 = torch.roll(f1, (2, -4), dims=(2, 3))
    out = f.Correlation(4, 1, 4, 1, 2, 1)(f1.cuda(), f2.cuda())
    assert int(out[0, :, 8, 8].argmax()) == (1 + 2) * 5 + (-2 + 2)


def test_correlation_autograd_module_and_noncontiguous():
    """Module API + autograd plumbing; inputs/grad_output non-contiguous (the reference assumes
    contiguity silently, SURVEY C-2; we accept a superset)."""
    f = _f2()
    base1 = _randn((2, 8, 12, 32), 5).cuda()
    base2 = _randn((2, 8, 12, 32), 6).cuda()
    a = base1.transpose(2, 3).contiguous().transpose(2, 3).requires_grad_()   # non-contiguous view
    b = base2.clone().requires_grad_()
    mod = f.Correlation(pad_size=20, kernel_size=1, max_displacement=20, stride1=1, stride2=2, corr_multiply=1)
    out = mod(a, b)
    go = _randn(tuple(out.shape), 7).cuda()
    out.backward(go.transpose(2, 3).contiguous().transpose(2, 3))
    r1, r2 = orc.correlation_backward(base1.cpu().numpy(), base2.cpu().numpy(), go.cpu().numpy(), 20, 1, 20, 1, 2)
    assert_close(a.grad.cpu().numpy(), r1, TOL, "autograd gI1")
    assert_close(b.grad.cpu().numpy(), r2, TOL, "autograd gI2")
    # only one input requires grad -> the other gradient is skipped
    a2 = base1.clone().requires_grad_()
    f.Correlation(20, 1, 20, 1, 2, 1)(a2, base2).backward(go)
    assert_close(a2.grad.cpu().numpy(), r1, TOL, "autograd gI1 only")


def test_correlation_autograd_tensor_core_path_reuses_workspace():
    """C % 64 == 0 -> tensor-core forward AND backward through the autograd Function; the backward
    reuses the forward's hi/lo workspace; a second backward-capable call after an in-place input
    update must not reuse stale copies."""
    f = _f2()
    a0, b0 = _randn((1, 64, 12, 20), 60), _randn((1, 64, 12, 20), 61)
    a, b = a0.cuda().requires_grad_(), b0.cuda().requires_grad_()
    out = f.Correlation(20, 1, 20, 1, 2, 1)(a, b)
    go = _randn(tuple(out.shape), 62)
    out.backward(go.cuda())
    r1, r2 = orc.correlation_backward(a0.numpy(), b0.numpy(), go.numpy(), 20, 1, 20, 1, 2)
    assert_close(a.grad.cpu().numpy(), r1, TOL, "tc autograd gI1")
    assert_close(b.grad.cpu().numpy(), r2, TOL, "tc autograd gI2")
    # functional API: stale workspace (input modified in place after the forward) is detected
    x, y = a0.cuda(), b0.cuda()
    _, ws = f.functional.correlation_forward(x, y, 20, 1, 20, 1, 2, return_workspace=True)
    assert ws is not None
    y.mul_(2.0)
    g1, _ = f.functional.correlation_backward(x, y, go.cuda(), 20, 1, 20, 1, 2, workspace=ws)
    assert_close(g1.cpu().numpy(), 2.0 * r1, TOL, "stale workspace must be ignored")
    with torch.no_grad():
        assert f.Correlation(20, 1, 20, 1, 2, 1)(x, y).shape == out.shape


def test_correlation_side_stream():
    f = _f2()
    a, b = _randn((1, 32, 16, 64), 8).cuda(), _randn((1, 32, 16, 64), 9).cuda()
    ref = orc.correlation_forward(a.cpu().numpy(), b.cpu().numpy(), 20, 1, 20, 1, 2)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        out = f.functional.correlation_forward(a, b, 20, 1, 20, 1, 2)
    s.synchronize()
    assert_close(out.cpu().numpy(), ref, TOL, "corr on side stream")


def test_correlation_full_size_cfg2_samples_and_linearity():
    """BASELINE cfg2 [8,256,112,256]: two whole samples against the oracle + size-independent properties."""
    f = _f2()
    shape = (8, 256, 112, 256)
    g = torch.Generator(device="cuda").manual_seed(0)
    a = torch.randn(*shape, device="cuda", generator=g)
    b = torch.randn(*shape, device="cuda", generator=g)
    out = f.functional.correlation_forward(a, b, 20, 1, 20, 1, 2)
    assert out.shape == (8, 441, 112, 256) and bool(torch.isfinite(out).all())
    for n in (0, 7):
        ref = orc.correlation_forward(a[n:n + 1].cpu().numpy(), b[n:n + 1].cpu().numpy(), 20, 1, 20, 1, 2)
        assert_close(out[n:n + 1].cpu().numpy(), ref, TOL, "cfg2 fwd sample %d" % n)
    # linearity in input1 and symmetry under swapping inputs + negating displacements
    out2 = f.functional.correlation_forward(a * 2.0, b, 20, 1, 20, 1, 2)
    assert rel_err(out2.cpu().numpy(), (out * 2.0).cpu().numpy()) < 1e-6
    del out2
    sw = f.functional.correlation_forward(b[:1], a[:1], 20, 1, 20, 1, 2)          # out'(d, p) = out(-d, p + d)
    d = 441 // 2 + 21 * 3 + 5                                                     # tj = 3, ti = 5
    dneg = 441 // 2 - 21 * 3 - 5
    lhs = sw[0, dneg, 6:100, 10:240]
    rhs = out[0, d, 0:94, 0:230]
    assert rel_err(lhs.cpu().numpy(), rhs.cpu().numpy()) < 1e-5
    go = torch.randn(out.shape, device="cuda", generator=g)
    g1, g2 = f.functional.correlation_backward(a, b, go, 20, 1, 20, 1, 2)
    n = 3
    r1, r2 = orc.correlation_backward(a[n:n + 1].cpu().numpy(), b[n:n + 1].cpu().numpy(), go[n:n + 1].cpu().numpy(),
                                      20, 1, 20, 1, 2)
    assert_close(g1[n:n + 1].cpu().numpy(), r1, TOL, "cfg2 gI1 sample %d" % n)
    assert_close(g2[n:n + 1].cpu().numpy(), r2, TOL, "cfg2 gI2 sample %d" % n)
    # adjoint identity: <corr(a,b), go> == <a, gI1> == <b, gI2>  (bilinear form)
    s0 = float((out.double() * go.double()).sum())
    s1 = float((a.double() * g1.double()).sum())
    s2 = float((b.double() * g2.double()).sum())
    assert abs(s0 - s1) <= 1e-4 * abs(s0) + 1e-3 and abs(s0 - s2) <= 1e-4 * abs(s0) + 1e-3


# ------------------------------------------------------------------------------------------------
# Resample2d
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape,sigma,C", [((2, 9, 13), 4.0, 3), ((1, 16, 20), 64.0, 3), ((2, 7, 5), 1.0, 2),
                                           ((1, 8, 12), 3.0, 5), ((1, 12, 12), 0.0, 1)])
def test_resample2d_vs_oracle(shape, sigma, C):
    f = _f2()
    B, H, W = shape
    g = torch.Generator().manual_seed(21)
    img = torch.rand(B, C, H, W, generator=g)
    flow = torch.randn(B, 2, H, W, generator=g) * sigma
    go = torch.randn(B, C, H, W, generator=g)
    out = f.functional.resample2d_forward(img.cuda(), flow.cuda())
    assert_close(out.cpu().numpy(), orc.resample2d_forward(img.numpy(), flow.numpy()), TOL, "resample fwd")
    near = f.functional.resample2d_forward(img.cuda(), flow.cuda(), 1, False)
    assert np.array_equal(near.cpu().numpy(), orc.resample2d_forward(img.numpy(), flow.numpy(), 1, False))
    g1, g2 = f.functional.resample2d_backward(img.cuda(), flow.cuda(), go.cuda())
    r1, r2 = orc.resample2d_backward(img.numpy(), flow.numpy(), go.numpy())
    assert_close(g1.cpu().numpy(), r1, TOL, "resample gImg")
    assert_close(g2.cpu().numpy(), r2, TOL, "resample gFlow")


@pytest.mark.parametrize("shape,sigma,C", [((2, 40, 72), 4.0, 3), ((1, 33, 52), 64.0, 3), ((2, 64, 128), 2.0, 2),
                                           ((1, 70, 200), 9.0, 1), ((1, 36, 64), 30.0, 3), ((1, 96, 256), 0.3, 3),
                                           ((1, 21, 45), 5.0, 5), ((2, 19, 30), 3.0, 3)])
def test_resample2d_kernel_families_vs_oracle(shape, sigma, C, monkeypatch):
    """Every Resample2d kernel family on the same inputs: 2-D tiles (default; PY = 1, 2, 4 rows per thread; both scatter
    flavours of the backward: vector reductions into the interleaved scratch, planar scalar reductions) and round 1's
    row kernels; partial tiles on both axes, C = 1, 2, 3 and the runtime-C path (5).
    Forward and flow gradient must agree bit for bit across families (same arithmetic); the image gradient (atomic
    order differs) within 1e-5 plus 2^-20 of the sum of |terms| a pixel collects; everything against the oracle within
    the 1e-4 contract."""
    f = _f2()
    F2 = f.functional
    B, H, W = shape
    g = torch.Generator().manual_seed(23)
    img = torch.rand(B, C, H, W, generator=g)
    flow = torch.randn(B, 2, H, W, generator=g) * sigma
    go = torch.randn(B, C, H, W, generator=g)
    imd, fld, god = img.cuda(), flow.cuda(), go.cuda()
    ref = orc.resample2d_forward(img.numpy(), flow.numpy())
    r1, r2 = orc.resample2d_backward(img.numpy(), flow.numpy(), go.numpy())
    r1_abs, _ = orc.resample2d_backward(img.numpy(), flow.numpy(), np.abs(go.numpy()))    # per pixel: sum of |terms|
    huge = flow.clone()
    huge[0, :, 0, 0] = float("nan")                      # NaN flow: taps clamp to (0, 0), NaN weights -> NaN out, no fault
    huge[0, 0, 1, 1] = 3e9                               # saturating float->int conversion (UB in the C oracle)
    huge[0, 1, 2, 2] = -float("inf")
    hud = huge.cuda()
    base = {}
    envs = [("tile", {}), ("tile py1", {"FN2B200_RS_PY": "1"}), ("tile py2 planar", {"FN2B200_RS_PY": "2", "FN2B200_RS_BWD": "planar"}),
            ("tile py4 planar", {"FN2B200_RS_BWD": "planar"}), ("row", {"FN2B200_RESAMPLE": "row"})]
    for name, env in envs:
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        out = F2.resample2d_forward(imd, fld)
        g1, g2 = F2.resample2d_backward(imd, fld, god)
        of = F2.resample2d_backward(imd, fld, god, need1=False)
        oi = F2.resample2d_backward(imd, fld, god, need2=False)
        oh = torch.nan_to_num(F2.resample2d_forward(imd, hud), nan=-1.0)
        for k in env:
            monkeypatch.delenv(k)
        assert_close(out.cpu().numpy(), ref, TOL, name + ": resample fwd")
        assert_close(g1.cpu().numpy(), r1, TOL, name + ": resample gImg")
        assert_close(g2.cpu().numpy(), r2, TOL, name + ": resample gFlow")
        assert of[0] is None and torch.equal(of[1], g2), name
        assert oi[1] is None
        assert_close(oi[0].cpu().numpy(), r1, TOL, name + ": resample gImg only")
        if not base:
            base = dict(out=out, g1=g1, g2=g2, oh=oh)
            assert bool((oh[0, :, 0, 0] == -1.0).all())
        else:
            d = (out - base["out"]).abs().max().item()
            assert torch.equal(out, base["out"]), "%s: forward differs from the tile kernel by %.3e" % (name, d)
            assert torch.equal(g2, base["g2"]), name + ": flow gradient differs"
            assert torch.equal(oh, base["oh"]), name + ": NaN / inf / huge flows handled differently"
            # a border pixel collecting hundreds of clamped taps can sum to far less than its terms: reordering those
            # float32 atomic adds moves the result by roundoff of the sum of |terms|, not of the result
            gi, gb = g1.cpu().numpy(), base["g1"].cpu().numpy()
            assert rel_err(gi, gb) <= 1e-5, name + ": image gradient vs tile kernel"
            rms = float(np.sqrt(np.mean(gb.astype(np.float64) ** 2)))
            excess = np.abs(gi - gb) - (1e-5 * (np.abs(gb) + rms) + 2.0 ** -20 * r1_abs)
            assert (excess <= 0).all(), "%s: image gradient vs tile kernel: %d pixels off by up to %.3e more than allowed" % (
                name, int((excess > 0).sum()), float(excess.max()))


def test_resample2d_shim_accumulates_into_caller_zeroed_gradient():
    """B1 convention (resample2d.py:31-32): gradInput1 arrives zero-filled and the kernel accumulates into it."""
    f = _f2()
    g = torch.Generator().manual_seed(24)
    img, flow = torch.rand(1, 3, 32, 64, generator=g).cuda(), (torch.randn(1, 2, 32, 64, generator=g) * 3).cuda()
    go = torch.randn(1, 3, 32, 64, generator=g).cuda()
    base = torch.full_like(img, 0.5)
    g1, _ = f.functional.resample2d_backward(img, flow, go, out1=base.clone(), zero_out1=False)
    ref, _ = f.functional.resample2d_backward(img, flow, go)
    assert_close((g1 - 0.5).cpu().numpy(), ref.cpu().numpy(), 1e-5, "accumulate into caller buffer")


@pytest.mark.parametrize("mode", ["bilinear", "nearest"])
def test_resample2d_with_fused_flow_upsample(mode):
    """SURVEY 8(f)-3 (models.py:130-133): Resample2d reading a quarter-resolution flow; against the oracle's
    upsample4 + resample2d composition and against torch's nn.Upsample feeding our own Resample2d."""
    f = _f2()
    g = torch.Generator().manual_seed(25)
    img = torch.rand(2, 3, 48, 80, generator=g)
    lr = torch.randn(2, 2, 12, 20, generator=g) * 0.4
    out = f.functional.resample2d_forward_up(img.cuda(), lr.cuda(), mode, 20.0)
    up = orc.upsample4(lr.numpy(), 1 if mode == "bilinear" else 2, 20.0)
    assert_close(out.cpu().numpy(), orc.resample2d_forward(img.numpy(), up), TOL, "resample_up vs oracle")
    t_up = torch.nn.Upsample(scale_factor=4, mode=mode)(lr.cuda() * 20.0)
    assert_close(out.cpu().numpy(), f.functional.resample2d_forward(img.cuda(), t_up).cpu().numpy(), TOL, "resample_up vs torch upsample")
    with pytest.raises(RuntimeError, match="does not match"):
        f.functional.resample2d_forward_up(img.cuda(), lr[:, :, :11].contiguous().cuda(), mode, 20.0)


def test_warp_concat_forward_vs_oracle_composition():
    """SURVEY 8(f)-1 (models.py:130-138): one kernel for upsample -> warp -> diff -> channel-norm -> concat."""
    f = _f2()
    g = torch.Generator().manual_seed(26)
    x = torch.rand(2, 6, 48, 80, generator=g) - 0.5
    flow = torch.randn(2, 2, 48, 80, generator=g) * 5
    cat = f.functional.warp_concat_forward(x.cuda(), flow.cuda(), flow_div=20.0)
    assert cat.shape == (2, 12, 48, 80)
    ref = orc.warp_concat_forward(x.numpy(), flow.numpy(), flow_div=20.0)
    assert np.array_equal(cat[:, :6].cpu().numpy(), x.numpy())
    assert_close(cat.cpu().numpy(), ref, TOL, "warp_concat (models.py:138 layout)")
    for c0, c1, what in ((6, 9, "warped"), (9, 11, "flow/div"), (11, 12, "diff norm")):
        assert_close(cat[:, c0:c1].cpu().numpy(), ref[:, c0:c1], TOL, "warp_concat " + what)
    # the fusion-stage layout (models.py:154-174): quarter-resolution flow, nearest upsample, x / div_flow folded in,
    # flow + flow norm + diff norm into chosen channels of an 11-channel buffer; img0 copied, warped not written
    lr = torch.randn(2, 2, 12, 20, generator=g) * 8
    buf = torch.full((2, 11, 48, 80), 7.0).cuda()
    f.functional.warp_concat_forward(x.cuda(), lr.cuda(), upsample="nearest", flow_mul=1.0 / 20.0, out=buf, ch_x=0, n_x=3,
                                     ch_warped=-1, ch_flow=3, flow_div=1.0, ch_flow_norm=7, ch_diff_norm=9)
    ref = orc.warp_concat_forward(x.numpy(), lr.numpy(), upsample_mode=2, flow_mul=1.0 / 20.0, cat_channels=11, ch_x=0, n_x=3,
                                  ch_warped=-1, ch_flow=3, flow_div=1.0, ch_flow_norm=7, ch_diff_norm=9)
    got = buf.cpu().numpy()
    for ch in (5, 6, 8, 10):
        assert (got[:, ch] == 7.0).all()                  # channels nobody owns are left alone
        ref[:, ch] = 7.0
    assert_close(got, ref, TOL, "warp_concat fusion-stage layout")
    # strided x (a channel slice of a larger tensor) and the bilinear-upsample variant
    big = torch.rand(2, 8, 48, 80, generator=g).cuda()
    xs = big[:, 1:7]
    cat = f.functional.warp_concat_forward(xs, lr.cuda(), upsample="bilinear", flow_mul=20.0, flow_div=20.0)
    ref = orc.warp_concat_forward(xs.cpu().numpy(), lr.numpy(), upsample_mode=1, flow_mul=20.0, flow_div=20.0)
    assert_close(cat.cpu().numpy(), ref, TOL, "warp_concat strided x + bilinear upsample")
    with pytest.raises(RuntimeError, match="overlap"):
        f.functional.warp_concat_forward(x.cuda(), flow.cuda(), ch_warped=4)


def test_warp_concat_backward_vs_oracle_and_unfused_autograd():
    """The fused backward (one kernel + the scratch transpose) against the oracle's composition of the reference
    modules' backward passes, and against torch autograd through the unfused chain of our drop-in modules."""
    from flownet2_b200 import fused
    f = _f2()
    g = torch.Generator().manual_seed(27)
    x0 = torch.rand(2, 6, 40, 72, generator=g) - 0.5
    fl0 = torch.randn(2, 2, 40, 72, generator=g) * 4
    gc = torch.randn(2, 12, 40, 72, generator=g)
    x, fl = x0.cuda().requires_grad_(), fl0.cuda().requires_grad_()
    cat = fused.WarpConcat(20.0)(x, fl)
    cat.backward(gc.cuda())
    rx, rf = orc.warp_concat_backward(x0.numpy(), fl0.numpy(), gc.numpy(), flow_div=20.0)
    assert_close(x.grad.cpu().numpy(), rx, TOL, "warp_concat grad_x")
    assert_close(fl.grad.cpu().numpy(), rf, TOL, "warp_concat grad_flow")
    x2, fl2 = x0.cuda().requires_grad_(), fl0.cuda().requires_grad_()
    warped = f.Resample2d()(x2[:, 3:], fl2)
    chain = torch.cat((x2, warped, fl2 / 20.0, f.ChannelNorm()(x2[:, :3] - warped)), dim=1)
    assert rel_err(cat.detach().cpu().numpy(), chain.detach().cpu().numpy()) < 1e-6
    chain.backward(gc.cuda())
    assert_close(x.grad.cpu().numpy(), x2.grad.cpu().numpy(), 1e-5, "fused vs unfused autograd grad_x")
    assert_close(fl.grad.cpu().numpy(), fl2.grad.cpu().numpy(), 1e-5, "fused vs unfused autograd grad_flow")
    # fusion-stage layout with a flow-norm channel, functional API
    gc11 = torch.randn(2, 11, 40, 72, generator=g)
    kw = dict(flow_div=1.0, ch_x=0, n_x=3, ch_warped=-1, ch_flow=3, ch_flow_norm=7, ch_diff_norm=9)
    gx, gf = f.functional.warp_concat_backward(x0.cuda(), fl0.cuda(), gc11.cuda(), **kw)
    rx, rf = orc.warp_concat_backward(x0.numpy(), fl0.numpy(), gc11.numpy(), **kw)
    assert_close(gx.cpu().numpy(), rx, TOL, "warp_concat grad_x (fusion layout)")
    assert_close(gf.cpu().numpy(), rf, TOL, "warp_concat grad_flow (fusion layout)")


def test_resample2d_strided_image_slice_and_module():
    """FlowNet2 passes x[:,3:,:,:] (non-contiguous, models.py:133); no .contiguous() copy needed."""
    f = _f2()
    g = torch.Generator().manual_seed(22)
    x = torch.rand(2, 6, 16, 24, generator=g).cuda()
    flow = (torch.randn(2, 2, 16, 24, generator=g) * 5).cuda().requires_grad_()
    img = x[:, 3:, :, :].requires_grad_()
    assert not img.is_contiguous()
    out = f.Resample2d()(img, flow)
    ref = orc.resample2d_forward(x[:, 3:].contiguous().cpu().numpy(), flow.detach().cpu().numpy())
    assert_close(out.detach().cpu().numpy(), ref, TOL, "resample strided fwd")
    go = torch.randn(out.shape, generator=g).cuda()
    out.backward(go)
    r1, r2 = orc.resample2d_backward(x[:, 3:].contiguous().cpu().numpy(), flow.detach().cpu().numpy(), go.cpu().numpy())
    assert_close(img.grad.cpu().numpy(), r1, TOL, "resample strided gImg")
    assert_close(flow.grad.cpu().numpy(), r2, TOL, "resample strided gFlow")
    with pytest.raises(RuntimeError, match="kernel_size"):
        f.Resample2d(kernel_size=2)(x[:, :3].contiguous(), flow.detach())


def test_resample2d_full_size_properties():
    """cfg3 shapes [8,3,448,1024]: identity under zero flow, shifted copy under integer flow,
    and one sample against the oracle."""
    f = _f2()
    g = torch.Generator(device="cuda").manual_seed(0)
    img = torch.rand(8, 3, 448, 1024, device="cuda", generator=g)
    zero = torch.zeros(8, 2, 448, 1024, device="cuda")
    assert torch.equal(f.functional.resample2d_forward(img, zero), img)
    sh = zero.clone()
    sh[:, 0] = 3.0
    sh[:, 1] = -2.0
    out = f.functional.resample2d_forward(img, sh)
    assert torch.equal(out[:, :, 2:, :-3], img[:, :, :-2, 3:])
    flow = torch.randn(8, 2, 448, 1024, device="cuda", generator=g) * 4
    out = f.functional.resample2d_forward(img, flow)
    ref = orc.resample2d_forward(img[5:6].cpu().numpy(), flow[5:6].cpu().numpy())
    assert_close(out[5:6].cpu().numpy(), ref, TOL, "cfg3 resample fwd sample 5")
    go = torch.randn(8, 3, 448, 1024, device="cuda", generator=g)
    g1, g2 = f.functional.resample2d_backward(img, flow, go)
    r1, r2 = orc.resample2d_backward(img[5:6].cpu().numpy(), flow[5:6].cpu().numpy(), go[5:6].cpu().numpy())
    assert_close(g1[5:6].cpu().numpy(), r1, TOL, "cfg3 resample gImg sample 5")
    assert_close(g2[5:6].cpu().numpy(), r2, TOL, "cfg3 resample gFlow sample 5")
    # mass conservation of the scatter: sum(gImg) == sum(go)  (bilinear weights sum to 1)
    assert abs(float(g1.double().sum()) - float(go.double().sum())) < 1e-3 * float(go.double().abs().sum()) ** 0.5 + 1.0


def test_resample2d_full_size_sigma64_border_clamps():
    """cfg3 with sigma = 64 px (SURVEY 8d): more than half of the taps clamp to the border; fwd and bwd vs oracle."""
    f = _f2()
    g = torch.Generator(device="cuda").manual_seed(1)
    img = torch.rand(8, 3, 448, 1024, device="cuda", generator=g)
    flow = torch.randn(8, 2, 448, 1024, device="cuda", generator=g) * 64
    go = torch.randn(8, 3, 448, 1024, device="cuda", generator=g)
    xf = torch.arange(1024, device="cuda").view(1, 1, 1024) + flow[:, 0]
    yf = torch.arange(448, device="cuda").view(1, 448, 1) + flow[:, 1]
    oob = ((xf < 0) | (xf > 1023) | (yf < 0) | (yf > 447)).float().mean().item()
    assert oob > 0.15, oob
    out = f.functional.resample2d_forward(img, flow)
    g1, g2 = f.functional.resample2d_backward(img, flow, go)
    n = 6
    i_, f_, g_ = img[n:n + 1].cpu().numpy(), flow[n:n + 1].cpu().numpy(), go[n:n + 1].cpu().numpy()
    assert_close(out[n:n + 1].cpu().numpy(), orc.resample2d_forward(i_, f_), TOL, "cfg3 sigma64 fwd")
    r1, r2 = orc.resample2d_backward(i_, f_, g_)
    assert_close(g1[n:n + 1].cpu().numpy(), r1, TOL, "cfg3 sigma64 gImg")
    assert_close(g2[n:n + 1].cpu().numpy(), r2, TOL, "cfg3 sigma64 gFlow")
    assert abs(float(g1.double().sum()) - float(go.double().sum())) < 1e-3 * float(go.double().abs().sum()) ** 0.5 + 1.0


def test_warp_concat_full_size():
    """[8,6,448,1024] + quarter-resolution flow: one sample against the oracle composition (models.py:130-138)."""
    f = _f2()
    g = torch.Generator(device="cuda").manual_seed(2)
    x = torch.rand(8, 6, 448, 1024, device="cuda", generator=g) - 0.5
    lr = torch.randn(8, 2, 112, 256, device="cuda", generator=g) * 0.3
    cat = f.functional.warp_concat_forward(x, lr, upsample="bilinear", flow_mul=20.0, flow_div=20.0)
    n = 4
    ref = orc.warp_concat_forward(x[n:n + 1].cpu().numpy(), lr[n:n + 1].cpu().numpy(), upsample_mode=1, flow_mul=20.0, flow_div=20.0)
    assert_close(cat[n:n + 1].cpu().numpy(), ref, TOL, "warp_concat full size")
    # unfused chain through the individual modules gives the same tensor
    up = torch.nn.Upsample(scale_factor=4, mode="bilinear")(lr * 20.0)
    warped = f.Resample2d()(x[:, 3:], up)
    chain = torch.cat((x, warped, up / 20.0, f.ChannelNorm()(x[:, :3] - warped)), dim=1)
    assert rel_err(cat.cpu().numpy(), chain.cpu().numpy()) < 1e-5


# ------------------------------------------------------------------------------------------------
# ChannelNorm
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(2, 3, 8, 12), (1, 2, 7, 9), (1, 1, 4, 4), (2, 5, 6, 10), (1, 7, 3, 3),
                                   (8, 3, 448, 1024), (8, 2, 448, 1024)])
def test_channelnorm_vs_oracle(shape):
    f = _f2()
    x = _randn(shape, 31)
    x[0, :, 0, 0] = 0.0                                # exact-zero pixel: gradient must be 0 (N-1)
    mod = f.ChannelNorm()
    xc = x.cuda().requires_grad_()
    out = mod(xc)
    ref = orc.channelnorm_forward(x.numpy())
    assert_close(out.detach().cpu().numpy(), ref, 1e-6, "cnorm fwd")
    go = _randn(tuple(out.shape), 32)
    out.backward(go.cuda())
    assert_close(xc.grad.cpu().numpy(), orc.channelnorm_backward(x.numpy(), ref, go.numpy()), 1e-5, "cnorm bwd")
    assert float(xc.grad[0, :, 0, 0].abs().max()) == 0.0


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("shape", [(1, 3, 8, 8), (2, 3, 7, 9), (2, 2, 16, 24)])
def test_channelnorm_16bit_native(dtype, shape):
    """--fp16 mode feeds ChannelNorm half tensors (models.py:39 is not wrapped in tofp32); the reference
    dispatches its kernels on half (channelnorm_kernel.cu:111,152): storage 16-bit, arithmetic fp32."""
    f = _f2()
    x = _randn(shape, 33).cuda().to(dtype).requires_grad_()
    out = f.ChannelNorm()(x)
    assert out.dtype == dtype
    ref = x.detach().float().pow(2).sum(1, keepdim=True).sqrt()
    tol = 2e-3 if dtype == torch.float16 else 1.6e-2
    assert torch.allclose(out.float(), ref, atol=tol, rtol=tol)
    go = _randn(tuple(out.shape), 34).cuda().to(dtype)
    out.backward(go)
    gref = go.float() * x.detach().float() / (out.detach().float() + 1e-9)
    assert x.grad.dtype == dtype and torch.allclose(x.grad.float(), gref, atol=4 * tol, rtol=4 * tol)


# ------------------------------------------------------------------------------------------------
# Against the reference's own kernels (their stored outputs) and through the reference's Python wrappers
# ------------------------------------------------------------------------------------------------
def test_host_pipeline_matches_resident_results():
    """flownet2_b200.hostpipe.HostPipeline: 5 steps with different host inputs through 2 buffer slots give, for
    every step, exactly what the resident call gives (stream / event ordering of slot reuse)."""
    f = _f2()
    prm = (20, 1, 20, 1, 2)
    shape = (2, 64, 16, 32)
    D, oH, oW = f.functional.correlation_out_shape(shape[1], shape[2], shape[3], *prm)
    oshape = (shape[0], D, oH, oW)
    pipe = f.hostpipe.HostPipeline([shape, shape, oshape], [oshape, shape, shape], "cuda:0", depth=2)

    def compute(din, dout):
        _, ws = f.functional.correlation_forward(din[0], din[1], *prm, 1, out=dout[0], return_workspace=True)
        f.functional.correlation_backward(din[0], din[1], din[2], *prm, 1, out1=dout[1], out2=dout[2], workspace=ws)

    steps = []
    for i in range(5):
        hin = [_randn(shape, 100 + i).pin_memory(), _randn(shape, 200 + i).pin_memory(), _randn(oshape, 300 + i).pin_memory()]
        hout = [torch.empty(oshape).pin_memory(), torch.empty(shape).pin_memory(), torch.empty(shape).pin_memory()]
        pipe.submit(compute, hin, hout)
        steps.append((hin, hout))
    pipe.drain()
    torch.cuda.synchronize()
    for hin, hout in steps:
        a, b, go = (t.cuda() for t in hin)
        out = f.functional.correlation_forward(a, b, *prm, 1)
        g1, g2 = f.functional.correlation_backward(a, b, go, *prm, 1)
        assert torch.equal(hout[0], out.cpu()) and torch.equal(hout[1], g1.cpu()) and torch.equal(hout[2], g2.cpu())
    with pytest.raises(RuntimeError):
        pipe.submit(compute, [torch.empty(shape)] * 2 + [torch.empty(oshape)], steps[0][1])   # not pinned


@pytest.mark.parametrize("shape", [(1, 256, 48, 64), (2, 20, 13, 36)])
def test_correlation_vs_reference_kernels(shape):
    f = _f2()
    G = refk.Golden(refk.case_name("correlation", shape))
    a, b = refk.correlation_inputs(shape)
    out = f.functional.correlation_forward(a.cuda(), b.cuda(), 20, 1, 20, 1, 2)
    go = refk.correlation_grad_output(tuple(out.shape))
    G.check_inputs(input1=a, input2=b, grad_output=go)
    assert_close(G.pick("output", out), G["output"], TOL, "ours vs reference kernel fwd")
    assert_close(G.pick("output", orc.correlation_forward(a.numpy(), b.numpy(), 20, 1, 20, 1, 2)), G["output"], 1e-5,
                 "oracle vs reference kernel fwd")
    g1, g2 = f.functional.correlation_backward(a.cuda(), b.cuda(), go.cuda(), 20, 1, 20, 1, 2)
    assert_close(G.pick("grad_input1", g1), G["grad_input1"], TOL, "ours vs reference kernel gI1")
    assert_close(G.pick("grad_input2", g2), G["grad_input2"], TOL, "ours vs reference kernel gI2")


def test_resample_channelnorm_vs_reference_kernels():
    f = _f2()
    G = refk.Golden("resample2d_channelnorm")
    inputs = refk.resample_channelnorm_inputs()
    G.check_inputs(**dict(zip(("img", "flow", "grad_output", "x", "grad_norm"), inputs)))
    img, flow, go, x, gon = (t.cuda() for t in inputs)
    assert_close(G.pick("resample2d_output", f.functional.resample2d_forward(img, flow)), G["resample2d_output"], TOL,
                 "resample fwd vs ref")
    g1, g2 = f.functional.resample2d_backward(img, flow, go)
    assert_close(G.pick("resample2d_grad_input1", g1), G["resample2d_grad_input1"], TOL, "resample gImg vs ref")
    assert_close(G.pick("resample2d_grad_input2", g2), G["resample2d_grad_input2"], TOL, "resample gFlow vs ref")
    o = f.functional.channelnorm_forward(x)
    assert_close(G.pick("channelnorm_output", o), G["channelnorm_output"], 1e-6, "cnorm fwd vs ref")
    assert_close(G.pick("channelnorm_grad_input1", f.functional.channelnorm_backward(x, o, gon)), G["channelnorm_grad_input1"],
                 1e-5, "cnorm bwd vs ref")


@pytest.mark.parametrize("shape", [(2, 3, 16, 24), (1, 2, 7, 9), (2, 3, 64, 128)])
def test_channelnorm_half_vs_reference_half_kernels(shape):
    """SURVEY 8(f)-4: our fp16 ChannelNorm kernels (8 pixels per thread, fwd and bwd; scalar kernels for ragged sizes)
    against the reference's OWN half dispatch (channelnorm_kernel.cu:111,152).  The forward
    reproduces the reference's arithmetic exactly (squares rounded to half, fp32 accumulation): bit-identical.  The
    backward's divide is fp32 here and double there before the single rounding to half: at most 1 half ulp apart."""
    f = _f2()
    G = refk.Golden(refk.case_name("channelnorm_half", shape))
    x, go = refk.channelnorm_half_inputs(shape)
    G.check_inputs(input1=x, grad_output=go)
    x, go = x.cuda(), go.cuda()
    o = f.functional.channelnorm_forward(x)
    assert o.dtype == torch.float16 and np.array_equal(G.pick("output", o), G["output"])
    gi = f.functional.channelnorm_backward(x, o, go)
    assert gi.dtype == torch.float16
    rgi = torch.from_numpy(G["grad_input1"]).float()
    d = (torch.from_numpy(G.pick("grad_input1", gi)).float() - rgi).abs()
    ulp = torch.maximum(rgi.abs(), torch.tensor(6.1e-5)) * 2.0 ** -10
    assert bool((d <= ulp).all()), float((d / ulp).max())
    assert float((d > 0).float().mean()) < 0.01


def _run_pybind_child(*args):
    """The compiled pybind modules are exercised in a CHILD interpreter: pybind11 caches extension modules by name, so
    they cannot share a process with the reference's own correlation_cuda / resample2d_cuda / channelnorm_cuda."""
    import os
    import subprocess
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, os.path.join(here, "pybind_child.py")] + list(args), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and r.stdout.strip().splitlines()[-1].startswith("OK"), (r.stdout[-2000:], r.stderr[-3000:])
    return r.stdout.strip().splitlines()[-1]


def test_pybind_extension_modules_under_reference_wrappers():
    """The compiled correlation_cuda / resample2d_cuda / channelnorm_cuda modules called with the reference's exact
    calling convention (empty `input1.new()` outputs for correlation, pre-zeroed outputs for the other two), through the
    reference's own correlation.py wrapper incl. its autograd worker thread, against the oracle (tests/pybind_child.py)."""
    _run_pybind_child("ops")


needs_models = pytest.mark.skipif(not (oref.available() and oref.python_tree_available()),
                                  reason="reference python tree / extensions not installed under baseline/_ref, oracle/_ref")


def _build_ref_model(name, level):
    """Instantiate the UNMODIFIED reference models.<name> on top of (a) the reference kernels,
    (b) our B1 extension shims, (c) our B2 layer modules."""
    import sys
    from types import SimpleNamespace
    from flownet2_b200 import compat
    compat.uninstall()
    if level == "ref":
        oref.install_reference_extensions()
    else:
        compat.install(level)
    models = oref.import_reference_models(fresh=True)
    torch.manual_seed(0)
    net = getattr(models, name)(SimpleNamespace(rgb_max=255.0, fp16=False)).cuda().eval()
    return net


@needs_models
@pytest.mark.parametrize("name", ["FlowNet2C", "FlowNet2"])
def test_unmodified_reference_models_run_on_our_layers(name):
    """SURVEY 8(b): models.py's stacks load our layers unchanged -- B1 (Python *_cuda shims), B1p (compiled pybind
    *_cuda modules under the reference's own wrappers) and B2 (our modules) -- and agree with the reference kernels on
    identical weights/inputs."""
    torch.backends.cudnn.deterministic = True
    torch.backends.cudnn.benchmark = False
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    g = torch.Generator().manual_seed(5)
    x = (torch.rand(1, 3, 2, 128, 192, generator=g) * 255.0).cuda()
    outs = {}
    for level in ("ref", "B1", "B2"):
        net = _build_ref_model(name, level)
        with torch.no_grad():
            outs[level] = net(x).float().cpu().numpy()
        kinds = {type(m).__module__ for m in net.modules() if type(m).__name__ in ("Correlation", "Resample2d", "ChannelNorm")}
        if level == "B2":
            assert all(k.startswith("flownet2_b200") for k in kinds), kinds
        else:
            assert all(k.startswith("networks.") for k in kinds), kinds
        del net
    from flownet2_b200 import compat
    compat.uninstall()
    assert np.isfinite(outs["ref"]).all()
    assert rel_err(outs["B1"], outs["ref"]) < 1e-3, rel_err(outs["B1"], outs["ref"])
    # B1p (compiled pybind modules under the reference's wrappers) in a child interpreter: == B1 bit for bit, ~ref
    import tempfile
    with tempfile.TemporaryDirectory() as td:
        np.save(os.path.join(td, "x.npy"), x.cpu().numpy())
        np.save(os.path.join(td, "ref.npy"), outs["ref"])
        _run_pybind_child("model", name, os.path.join(td, "x.npy"), os.path.join(td, "ref.npy"))
    assert rel_err(outs["B2"], outs["ref"]) < 1e-3, rel_err(outs["B2"], outs["ref"])


@needs_models
@pytest.mark.parametrize("name", ["FlowNet2C", "FlowNet2"])
def test_full_size_output_flow_agreement(name):
    """SURVEY 8(d) cfg4 / cfg5 at the stated configuration: 448x1024, bs 8, random xavier weights (seed 0), U(0,255)
    input, deterministic cuDNN with TF32 off -- the output flow of the unmodified models.py on our layers (B2) and
    through the fused forwards (flownet2_b200.fused) against the same network on the reference's own kernels."""
    from flownet2_b200 import compat, fused
    torch.backends.cudnn.deterministic = True
    torch.backends.cudnn.benchmark = False
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    g = torch.Generator().manual_seed(0)
    x = (torch.rand(8, 3, 2, 448, 1024, generator=g) * 255.0).cuda()
    net = _build_ref_model(name, "ref")
    with torch.no_grad():
        ref = net(x).float().cpu().numpy()
    del net
    torch.cuda.empty_cache()
    net = _build_ref_model(name, "B2")
    n0 = _f2().functional.launch_count()
    with torch.no_grad():
        ours = net(x).float().cpu().numpy()
    n1 = _f2().functional.launch_count()
    fz = fused.fused_forward(net, x).float().cpu().numpy()
    n2 = _f2().functional.launch_count()
    del net
    compat.uninstall()
    torch.cuda.empty_cache()
    assert ref.shape == (8, 2, 448, 1024) and np.isfinite(ref).all()
    assert n1 > n0 and 0 < n2 - n1 < n1 - n0 or name == "FlowNet2C"      # the fused graph launches fewer of our kernels
    assert rel_err(ours, ref) < 1e-3, rel_err(ours, ref)
    assert rel_err(fz, ref) < 1e-3, rel_err(fz, ref)
    assert rel_err(fz, ours) < 1e-3, rel_err(fz, ours)


def test_correlation_forward_cat_leaky_epilogue():
    """SURVEY 8(f)-2 (FlowNetC.py:86-92): LeakyReLU(0.1)(corr) written into channels 32.. of a 473-channel buffer,
    on all three kernel families, against torch's cat(leaky_relu(our plain forward)) and the oracle."""
    f = _f2()
    for shape, prm in (((2, 64, 12, 20), (20, 1, 20, 1, 2)),        # tensor cores
                       ((1, 20, 13, 64), (20, 1, 20, 1, 2)),        # TMA-tiled FMA
                       ((1, 6, 10, 12), (4, 3, 4, 1, 2))):          # generic
        a, b = _randn(shape, 80).cuda(), _randn(shape, 81).cuda()
        D, oH, oW = f.functional.correlation_out_shape(shape[1], shape[2], shape[3], *prm)
        cat = torch.full((shape[0], 32 + D + 3, oH, oW), 5.0).cuda()
        f.functional.correlation_forward_cat(a, b, cat, 32, 0.1, *prm)
        plain = f.functional.correlation_forward(a, b, *prm)
        assert torch.equal(cat[:, 32:32 + D], torch.nn.functional.leaky_relu(plain, 0.1))
        assert (cat[:, :32] == 5.0).all() and (cat[:, 32 + D:] == 5.0).all()
        ref = orc.correlation_forward(a.cpu().numpy(), b.cpu().numpy(), *prm)
        assert_close(cat[:, 32:32 + D].cpu().numpy(), np.where(ref > 0, ref, ref * np.float32(0.1)), TOL, "corr cat leaky")
        cat2 = torch.empty((shape[0], D, oH, oW)).cuda()
        f.functional.correlation_forward_cat(a, b, cat2, 0, 1.0, *prm)
        assert torch.equal(cat2, plain)
    with pytest.raises(RuntimeError, match="do not fit"):
        f.functional.correlation_forward_cat(a, b, cat2, 1, 0.1, *prm)


@needs_models
@pytest.mark.parametrize("name", ["FlowNet2C", "FlowNet2"])
def test_fused_forwards_match_unfused_models(name):
    """flownet2_b200.fused on the unmodified reference network object vs its own forward() on the drop-in modules."""
    from flownet2_b200 import compat, fused
    torch.backends.cudnn.deterministic = True
    torch.backends.cudnn.benchmark = False
    torch.backends.cudnn.allow_tf32 = False
    g = torch.Generator().manual_seed(6)
    x = (torch.rand(2, 3, 2, 128, 192, generator=g) * 255.0).cuda()
    net = _build_ref_model(name, "B2")
    with torch.no_grad():
        base = net(x)
    fz = fused.fused_forward(net, x)
    compat.uninstall()
    assert fz.shape == base.shape
    assert rel_err(fz.cpu().numpy(), base.cpu().numpy()) < 1e-4, rel_err(fz.cpu().numpy(), base.cpu().numpy())
