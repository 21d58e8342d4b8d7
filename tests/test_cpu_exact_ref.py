"""The exact references of tests/exact_ref.py against torch's own float64 convolutions, the operand families against
the exactness criterion, and the comparator's reports.  CPU only."""
import pytest
import torch
import torch.nn.functional as F

import exact_ref as X

F64 = torch.float64


def _nchw(t):
    return t.permute(0, 3, 1, 2)


def _nhwc(t):
    return t.permute(0, 2, 3, 1)


# (N, H, W, Ci, Co, R, stride, pad): stride 1 and 2, 1x1, odd and even maps
GEOMS = [(2, 7, 5, 3, 4, 3, 1, 1), (3, 9, 6, 2, 5, 3, 2, 1), (2, 8, 7, 4, 3, 1, 2, 0), (1, 5, 5, 3, 2, 1, 1, 0),
         (2, 6, 9, 3, 3, 3, 2, 1)]


@pytest.mark.parametrize("N,H,W,Ci,Co,R,stride,pad", GEOMS)
def test_conv_refs_match_torch(N, H, W, Ci, Co, R, stride, pad):
    g = torch.Generator().manual_seed(N * 100 + H * 10 + W)
    x = torch.randn(N, H, W, Ci, generator=g, dtype=F64)
    w = torch.randn(Co, Ci, R, R, generator=g, dtype=F64)
    y = F.conv2d(_nchw(x), w, stride=stride, padding=pad)
    assert torch.allclose(X.conv_fwd_ref(x, w, stride, pad), _nhwc(y), rtol=1e-12, atol=1e-12)
    dy = torch.randn(y.shape, generator=g, dtype=F64)
    dx = torch.nn.grad.conv2d_input(_nchw(x).shape, w, dy, stride=stride, padding=pad)
    assert torch.allclose(X.conv_dgrad_ref(_nhwc(dy), w, H, W, stride, pad), _nhwc(dx), rtol=1e-12, atol=1e-12)
    dw = torch.nn.grad.conv2d_weight(_nchw(x), w.shape, dy, stride=stride, padding=pad)
    assert torch.allclose(X.conv_wgrad_ref(x, _nhwc(dy), R, R, stride, pad), dw, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("H,W", [(7, 5), (6, 6)])
def test_dgrad_add_modes(H, W):
    g = torch.Generator().manual_seed(H * W)
    N, Ci, Co = 2, 3, 4
    w = torch.randn(Co, Ci, 3, 3, generator=g, dtype=F64)
    Ho, Wo = (H + 1) // 2, (W + 1) // 2        # 3x3 / s2 / pad 1
    dy = torch.randn(N, Ho, Wo, Co, generator=g, dtype=F64)
    base = X.conv_dgrad_ref(dy, w, H, W, 2, 1)
    res = torch.randn(N, H, W, Ci, generator=g, dtype=F64)
    assert torch.equal(X.conv_dgrad_ref(dy, w, H, W, 2, 1, res, 1), base + res)
    # mode 2: the compact 1x1 / s2 downsample gradient lands at even pixels, exactly like conv2d_input of that branch
    d_cd = torch.randn(N, Ho, Wo, Co, generator=g, dtype=F64)
    wd = torch.randn(Co, Ci, 1, 1, generator=g, dtype=F64)
    gd = torch.nn.grad.conv2d_input((N, Ci, H, W), wd, _nchw(d_cd), stride=2, padding=0)
    comp = X.conv_dgrad_ref(d_cd, wd, Ho, Wo, 1, 0)
    got = X.conv_dgrad_ref(dy, w, H, W, 2, 1, comp, 2)
    assert torch.allclose(got, base + _nhwc(gd), rtol=1e-12, atol=1e-12)
    odd = torch.zeros(N, H, W, Ci, dtype=F64)
    odd[:, 0::2, 0::2] = comp
    assert torch.equal(X.conv_dgrad_ref(dy, w, H, W, 2, 1, comp, 2), base + odd)


@pytest.mark.parametrize("C,H,W", [(1, 13, 9), (3, 10, 11)])
def test_stem_refs_through_space_to_depth(C, H, W):
    """The 7x7 / s2 stem equals a 4x4 / s1 convolution over the space-to-depth input (the form the kernel computes),
    and the references equal torch's."""
    g = torch.Generator().manual_seed(C * H * W)
    N = 2
    x = torch.randn(N, C, H, W, generator=g, dtype=F64)
    w = torch.randn(64, C, 7, 7, generator=g, dtype=F64)
    y = F.conv2d(x, w, stride=2, padding=3)
    Ho, Wo = y.shape[2:]
    assert torch.allclose(X.stem_fwd_ref(x, w), _nhwc(y), rtol=1e-12, atol=1e-12)
    x16 = X.space_to_depth_ref(x, Ho + 3, Wo + 3)
    w8 = torch.zeros(64, C, 8, 8, dtype=F64)        # tap r = 2 t + dy of the 4x4 kernel; r = 7 is zero
    w8[:, :, :7, :7] = w
    w4 = torch.zeros(64, 16, 4, 4, dtype=F64)
    for dy in range(2):
        for dx in range(2):
            k = (dy * 2 + dx) * C
            w4[:, k:k + C] = w8[:, :, dy::2, dx::2]
    s2d = X.conv_fwd_ref(x16, w4, 1, 0)
    assert torch.allclose(s2d[:, :Ho, :Wo], _nhwc(y), rtol=1e-12, atol=1e-12)
    dy_ = torch.randn(y.shape, generator=g, dtype=F64)
    dw = torch.nn.grad.conv2d_weight(x, w.shape, dy_, stride=2, padding=3)
    assert torch.allclose(X.stem_wgrad_ref(x, _nhwc(dy_)), dw, rtol=1e-12, atol=1e-12)


def test_film_refs():
    g = torch.Generator().manual_seed(3)
    B, D, ZB = 3, 8, 16
    a, v = X.mantissa_dense((B, D), 1), X.mantissa_dense((B, D), 2)
    Z = X.film_outer_ref(a, v, 3, ZB)
    assert torch.equal(Z[:, 9:].float(), torch.zeros(D * D, ZB - 9))
    assert Z[2 * D + 5, B + 1].item() == (a[1, 2] * a[1, 5]).to(torch.bfloat16).item()
    G = torch.randn(D * D, 2 * B, generator=g, dtype=F64).to(torch.bfloat16)
    x = torch.randn(B, D, generator=g, dtype=F64)
    full = X.film_contract_ref(G, B, x, 0, D)
    Gm = G[:, B:].double().reshape(D, D, B)
    want = torch.einsum("ijb,bj->bi", Gm, x) + torch.einsum("ijb,bi->bj", Gm, x)
    assert torch.allclose(full, want, rtol=1e-12, atol=1e-12)
    parts = X.film_contract_ref(G[:4 * D], B, x, 0, 4) + X.film_contract_ref(G[4 * D:], B, x, 4, 4)
    assert torch.allclose(parts, full, rtol=1e-12, atol=1e-12)


# ---------------------------------------------------------------------------------- families and criterion
def test_families_satisfy_the_criterion():
    N, H, W, Ci, Co = 3, 9, 7, 64, 64
    x = X.ternary((N, H, W, Ci), 0.5, 1)
    w = X.ternary((Co, Ci, 3, 3), 16 / (9 * Ci * 0.5), 2)
    assert set(x.unique().tolist()) <= {-1.0, 0.0, 1.0}
    X.check_operands("I", [(x, X.Q_I), (w, X.Q_I)])
    X.check_criterion("I fwd", X.conv_fwd_ref(x.abs(), w.abs(), 1, 1), 2 * X.Q_I)
    xm = X.mantissa_dense((N, H, W, Ci), 3)
    assert torch.equal(xm.to(torch.bfloat16).float(), xm)
    a = xm.abs()
    assert float(a.min()) >= 0.25 and float(a.max()) < 4
    wm = X.conv_weights_sparse(Co, Ci, 3, 3, 16, 4)
    assert int((wm != 0).reshape(Co, -1).sum(1).max()) <= 16
    assert bool(((wm != 0).sum((0, 1)) > 0).all()), "every tap carries a weight"
    X.check_operands("M", [(xm, X.Q_DENSE), (wm, X.Q_SPARSE)])
    X.check_criterion("M fwd", X.conv_fwd_ref(xm.abs(), wm.abs(), 1, 1), X.Q_DENSE + X.Q_SPARSE)
    dy = X.sparse_rows(Co, N * H * W, 16, 5, must=X.special_pixels(N, H, W)).t().reshape(N, H, W, Co)
    X.check_criterion("M wgrad", X.conv_wgrad_ref(xm.abs(), dy.abs(), 3, 3, 1, 1), X.Q_DENSE + X.Q_SPARSE)
    assert set(X.special_pixels(N, H, W)) >= {0, N * H * W - 1, H * W - 1, H * W}


def test_criterion_rejects_a_violating_draw():
    x = torch.full((1, 4, 4, 64), 3.0)                  # integers, but far too many large terms
    w = torch.full((64, 64, 3, 3), 1024.0)
    with pytest.raises(AssertionError, match="violates the exactness criterion"):
        X.check_criterion("bad", X.conv_fwd_ref(x.abs(), w.abs(), 1, 1), 0)
    with pytest.raises(AssertionError, match="not a multiple"):
        X.check_operands("bad", [(torch.tensor([0.5, 1.0]), 0)])
    with pytest.raises(AssertionError, match="not representable in fp32"):
        X.bf16_ref(torch.tensor([1.0 + 2.0 ** -40], dtype=F64))
    with pytest.raises(AssertionError, match="exact in bf16"):
        X.bf16_ref(torch.tensor([257.0, 259.0, 1.0], dtype=F64))


# ---------------------------------------------------------------------------------- comparator
def test_comparator_reports_one_unit_change():
    ref = torch.arange(2 * 3 * 4 * 5, dtype=torch.float32).reshape(2, 3, 4, 5).to(torch.bfloat16)
    got = ref.clone()
    got[1, 2, 0, 3] += 1
    n, first, worst = X.mismatches(got, ref)
    assert (n, first, worst) == (1, (1, 2, 0, 3), (1, 2, 0, 3))
    with pytest.raises(AssertionError, match=r"1 of 120 elements differ; first at \(1, 2, 0, 3\)"):
        X.check_bits("t", got, ref)


def test_comparator_reports_nan_as_worst():
    ref = torch.zeros(3, 4)
    got = ref.clone()
    got[0, 1] = 5.0
    got[2, 3] = float("nan")
    n, first, worst = X.mismatches(got, ref)
    assert (n, first, worst) == (2, (0, 1), (2, 3))


def test_comparator_signed_zero_is_equal():
    ref = torch.zeros(2, 2, dtype=torch.bfloat16)
    got = ref.clone()
    got[1, 0] = -0.0
    assert got.view(torch.int16)[1, 0].item() != 0
    assert X.mismatches(got, ref) == (0, None, None)
    X.check_bits("t", got, ref)
    got[0, 1] = 2.0 ** -133     # one unit in the last place at zero: a subnormal bf16
    assert X.mismatches(got, ref)[:2] == (1, (0, 1))
