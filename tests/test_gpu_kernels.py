"""Per-kernel parity of the C-ABI ops against plain PyTorch fp32 references of the same op,
on bf16-rounded operands (the kernels compute bf16 x bf16 -> fp32).  GPU only."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _ops():
    from gdl_b200 import ops
    ops.init()
    return ops


def nhwc(x_nchw):  # fp32 NCHW -> bf16 NHWC contiguous
    return x_nchw.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)


def nchw(x_nhwc):  # bf16 NHWC -> fp32 NCHW
    return x_nhwc.float().permute(0, 3, 1, 2).contiguous()


def rel_err(a, b):
    return ((a - b).norm() / (b.norm() + 1e-12)).item()


CONV_CASES = [
    # N, H, W, Ci, Co, R, stride, pad
    (2, 14, 14, 64, 64, 3, 1, 1),
    (2, 13, 9, 64, 128, 3, 2, 1),
    (3, 9, 6, 256, 512, 3, 1, 1),
    (2, 12, 10, 64, 128, 1, 2, 0),
    (1, 33, 24, 128, 128, 3, 1, 1),
    (4, 17, 12, 128, 256, 3, 2, 1),
    (2, 7, 7, 512, 512, 3, 1, 1),
    (5, 56, 56, 64, 64, 3, 1, 1),
    (3, 7, 5, 128, 256, 1, 1, 0),
    (6, 28, 28, 128, 128, 3, 1, 1),
    (3, 65, 47, 64, 64, 3, 1, 1),
    (5, 14, 14, 128, 256, 3, 2, 1),
    (40, 9, 6, 512, 512, 3, 1, 1),
    (40, 56, 56, 64, 64, 3, 1, 1),   # >= 148 items of 256 pixels: the resident-weights variant of conv_flat
    (64, 28, 28, 128, 128, 3, 1, 1), # >= 148 items with 128-channel tiles: the CTA-pair kernel (cta_group::2), fwd + dgrad
    (48, 56, 56, 64, 128, 3, 2, 1),  # CTA-pair kernel, stride-2 forward through the four parity planes
    (96, 28, 28, 128, 256, 3, 2, 1), # CTA-pair kernel, stride-2 forward and the four-class stride-2 data gradient
    (96, 28, 28, 128, 256, 1, 2, 0), # CTA-pair kernel, 1x1 stride-2 forward (strided view)
    (192, 14, 14, 128, 256, 1, 1, 0),# CTA-pair kernel, 1x1 data gradient on the compact grid
    (47, 28, 28, 128, 128, 3, 1, 1), # CTA-pair kernel with an ODD number of 256-pixel tiles (the last pair's peer is padding)
    (24, 14, 14, 256, 256, 3, 1, 1), # CTA-pair weight gradient (two ci tiles per cluster), band stages
    (9, 17, 12, 256, 512, 3, 2, 1),  # CTA-pair weight gradient through the four parity planes
    (12, 14, 14, 256, 512, 1, 2, 0), # CTA-pair weight gradient, 1x1 stride 2
    # KineticSound / VGGSound audio (129x626 spectrogram, stem 65x313) at the per-GPU batch N = 64
    (64, 33, 157, 64, 64, 3, 1, 1),
    (64, 33, 157, 64, 128, 3, 2, 1),
    (64, 33, 157, 64, 128, 1, 2, 0),
    (64, 17, 79, 128, 128, 3, 1, 1),
    (64, 17, 79, 128, 256, 3, 2, 1),
    (64, 9, 40, 256, 512, 3, 2, 1),
    (768, 56, 56, 64, 64, 3, 1, 1),  # visual layer 1 at the benchmark's B = 256 (3 frames per clip)
]


def _mk(N, H, W, Ci, Co, R, stride, pad, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(N, Ci, H, W, device="cuda", generator=g)
    w = torch.randn(Co, Ci, R, R, device="cuda", generator=g) * (2.0 / (Ci * R * R)) ** 0.5
    xb = x.to(torch.bfloat16).float()
    wb = w.to(torch.bfloat16).float()
    return xb, wb


@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_fwd(case):
    ops = _ops()
    N, H, W, Ci, Co, R, stride, pad = case
    xb, wb = _mk(*case)
    d = ops.conv_desc(N, H, W, Ci, Co, R, R, stride, pad)
    Kp = ops.conv_packed_k(d)
    wp = torch.empty(Co, Kp, device="cuda", dtype=torch.bfloat16)
    ops.conv_pack_weights(d, Ci, wb, wp, None)
    y = torch.full((N, d.Ho, d.Wo, Co), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.conv_fwd(d, nhwc(xb), wp, y)
    torch.cuda.synchronize()
    ref = F.conv2d(xb, wb, stride=stride, padding=pad)
    assert torch.isfinite(y.float()).all()
    assert rel_err(nchw(y), ref) < 6e-3, rel_err(nchw(y), ref)


@pytest.mark.parametrize("case", [c for c in CONV_CASES if c[3] % 64 == 0])
@pytest.mark.parametrize("use_res,relu", [(0, 1), (1, 1), (0, 0)])
def test_conv_fwd_bias_act(case, use_res, relu):
    """Eval-mode fused unit (gdl_conv_fwd_bias_act): y = [relu](conv(x, w * scale[co]) + bias[co] [+ res]) with the
    scale folded into the packed weights by the multi-tensor pack (gdl_pack_entry.scale) — against conv2d +
    eval-mode batch_norm-style affine in torch fp32."""
    ops = _ops()
    N, H, W, Ci, Co, R, stride, pad = case
    xb, wb = _mk(*case)
    g = torch.Generator(device="cuda").manual_seed(7)
    scale = torch.rand(Co, device="cuda", generator=g) + 0.5
    bias = torch.randn(Co, device="cuda", generator=g)
    d = ops.conv_desc(N, H, W, Ci, Co, R, R, stride, pad)
    Kp = ops.conv_packed_k(d)
    wp = torch.zeros(Co, Kp, device="cuda", dtype=torch.bfloat16)
    table = ops.make_pack_table([(wb, wp, None, Co, Ci, Ci, R, R, Kp, scale)], torch.device("cuda"))
    ops.conv_pack_weights_multi(*table)
    res = torch.randn(N, d.Ho, d.Wo, Co, device="cuda", generator=g).to(torch.bfloat16) if use_res else None
    y = torch.full((N, d.Ho, d.Wo, Co), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.conv_fwd_bias_act(d, nhwc(xb), wp, bias, res, relu, y)
    torch.cuda.synchronize()
    wf = (wb * scale.view(-1, 1, 1, 1)).to(torch.bfloat16).float()   # the fold rounds w * scale to bf16
    ref = F.conv2d(xb, wf, stride=stride, padding=pad) + bias.view(1, -1, 1, 1)
    if use_res:
        ref = ref + nchw(res)
    if relu:
        ref = torch.relu(ref)
    assert torch.isfinite(y.float()).all()
    assert rel_err(nchw(y), ref) < 6e-3, rel_err(nchw(y), ref)


@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_fwd_fused_bn_statistics(case):
    """gdl_conv_fwd_stats: the partial sums from the conv epilogue give the same BN statistics as a
    separate pass over the stored bf16 output."""
    ops = _ops()
    N, H, W, Ci, Co, R, stride, pad = case
    xb, wb = _mk(*case)
    d = ops.conv_desc(N, H, W, Ci, Co, R, R, stride, pad)
    wp = torch.empty(Co, ops.conv_packed_k(d), device="cuda", dtype=torch.bfloat16)
    ops.conv_pack_weights(d, Ci, wb, wp, None)
    y = torch.empty(N, d.Ho, d.Wo, Co, device="cuda", dtype=torch.bfloat16)
    P = N * d.Ho * d.Wo
    partial = torch.full((ops.bn_partial_floats(P, Co),), float("nan"), device="cuda")
    old = ops.set_fused_stats_min_k(0)
    try:
        rows = ops.conv_fwd_stats(d, nhwc(xb), wp, y, partial)
    finally:
        ops.set_fused_stats_min_k(old)
    ref = F.conv2d(xb, wb, stride=stride, padding=pad)
    assert rel_err(nchw(y), ref) < 6e-3
    if rows == 0:
        pytest.skip("shape served by a kernel without fused statistics")
    gamma, beta = torch.rand(Co, device="cuda") + 0.5, torch.randn(Co, device="cuda")
    outs = []
    for fused in (True, False):
        rm, rv = torch.zeros(Co, device="cuda"), torch.ones(Co, device="cuda")
        mean, invstd, scale, shift = (torch.empty(Co, device="cuda") for _ in range(4))
        if fused:
            ops.bn_stats_finalize(partial, rows, P, Co, gamma, beta, 1e-5, 0.1, rm, rv, mean, invstd, scale, shift)
        else:
            p2 = torch.empty_like(partial)
            ops.bn_stats(y, P, Co, p2, gamma, beta, 1e-5, 0.1, rm, rv, mean, invstd, scale, shift)
        outs.append((mean, invstd, scale, shift, rm, rv))
    torch.cuda.synchronize()
    for a, b in zip(*outs):
        assert torch.allclose(a, b, rtol=2e-5, atol=2e-6), (a - b).abs().max()


def test_pack_weights_multi_equals_single():
    ops = _ops()
    g = torch.Generator(device="cuda").manual_seed(31)
    entries, singles = [], []
    for (Co, Ci, R) in ((64, 64, 3), (128, 64, 3), (128, 64, 1), (256, 256, 3), (512, 256, 1)):
        d = ops.conv_desc(2, 8, 8, Ci, Co, R, R, 1, R // 2)
        Kp = ops.conv_packed_k(d)
        w = torch.randn(Co, Ci, R, R, device="cuda", generator=g)
        wp1, wT1 = torch.zeros(Co, Kp, device="cuda", dtype=torch.bfloat16), torch.zeros(Ci, R * R * Co, device="cuda", dtype=torch.bfloat16)
        ops.conv_pack_weights(d, Ci, w, wp1, wT1)
        wp2, wT2 = torch.zeros_like(wp1), torch.zeros_like(wT1)
        entries.append((w, wp2, wT2, Co, Ci, Ci, R, R, Kp))
        singles.append((wp1, wT1, wp2, wT2))
    ops.conv_pack_weights_multi(*ops.make_pack_table(entries, torch.device("cuda")))
    torch.cuda.synchronize()
    for wp1, wT1, wp2, wT2 in singles:
        assert torch.equal(wp1, wp2) and torch.equal(wT1, wT2)


@pytest.mark.parametrize("ci_real,H,W", [(3, 37, 29), (1, 41, 30), (3, 224, 224)])
def test_conv_fwd_stem(ci_real, H, W):
    ops = _ops()
    N, Co, R, stride, pad = 2, 64, 7, 2, 3
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(N, ci_real, H, W, device="cuda", generator=g).to(torch.bfloat16).float()
    w = (torch.randn(Co, ci_real, R, R, device="cuda", generator=g) * 0.1).to(torch.bfloat16).float()
    d = ops.conv_desc(N, H, W, 8, Co, R, R, stride, pad)
    Kp = ops.conv_packed_k(d)
    assert Kp == 448
    wp = torch.empty(Co, Kp, device="cuda", dtype=torch.bfloat16)
    ops.conv_pack_weights(d, ci_real, w, wp, None)
    x8 = torch.zeros(N, H, W, 8, device="cuda", dtype=torch.bfloat16)
    x8[..., :ci_real] = x.permute(0, 2, 3, 1).to(torch.bfloat16)
    y = torch.empty(N, d.Ho, d.Wo, Co, device="cuda", dtype=torch.bfloat16)
    ops.conv_fwd(d, x8, wp, y)
    torch.cuda.synchronize()
    ref = F.conv2d(x, w, stride=stride, padding=pad)
    assert rel_err(nchw(y), ref) < 6e-3

    # wgrad of the stem
    dy = torch.randn(N, Co, d.Ho, d.Wo, device="cuda", generator=g).to(torch.bfloat16).float()
    ws = torch.empty(ops.conv_wgrad_workspace_bytes(d) // 4, device="cuda", dtype=torch.float32)
    dw = torch.full((Co, ci_real, R, R), float("nan"), device="cuda")
    ops.conv_wgrad(d, ci_real, x8, nhwc(dy), dw, ws)
    torch.cuda.synchronize()
    ref_dw = torch.nn.grad.conv2d_weight(x, w.shape, dy, stride=stride, padding=pad)
    assert rel_err(dw, ref_dw) < 2e-3, rel_err(dw, ref_dw)


@pytest.mark.parametrize("ci_real,T,H,W", [(3, 2, 37, 29), (1, 1, 41, 30), (3, 3, 224, 224), (1, 1, 257, 188),
                                            (1, 1, 129, 626)])
def test_stem_space_to_depth(ci_real, T, H, W):
    """7x7/s2 stem as a 4x4/s1 space-to-depth implicit GEMM: layout + fwd + wgrad vs torch."""
    ops = _ops()
    B, Co = 2, 64
    N = B * T
    g = torch.Generator(device="cuda").manual_seed(11)
    src = torch.randn(B, ci_real, T, H, W, device="cuda", generator=g)
    w = (torch.randn(Co, ci_real, 7, 7, device="cuda", generator=g) * 0.1).to(torch.bfloat16).float()
    Ho, Wo, Hp, Wp = ops.stem_geometry(H, W)
    x16 = torch.full((N, Hp, Wp, 16), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.stem_layout(src, x16, B, ci_real, T, H, W)
    wp = torch.empty(Co, 256, device="cuda", dtype=torch.bfloat16)
    ops.stem_pack_weights(w, wp, ci_real)
    y = torch.full((N, Ho, Wo, Co), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.stem_fwd(x16, wp, y, N, H, W, ci_real)
    torch.cuda.synchronize()
    x = src.permute(0, 2, 1, 3, 4).reshape(N, ci_real, H, W).to(torch.bfloat16).float()
    ref = F.conv2d(x, w, stride=2, padding=3)
    assert torch.isfinite(x16.float()).all() and torch.isfinite(y.float()).all()
    assert rel_err(nchw(y), ref) < 6e-3, rel_err(nchw(y), ref)
    # BatchNorm statistics from the stem's epilogue == a separate pass over the stored output (and the same output)
    P = N * Ho * Wo
    partial = torch.full((ops.bn_partial_floats(P, Co),), float("nan"), device="cuda")
    y2 = torch.full_like(y, float("nan"))
    rows = ops.stem_fwd_stats(x16, wp, y2, N, H, W, ci_real, partial)
    assert rows > 0 and torch.equal(y, y2)
    gamma, beta = torch.rand(Co, device="cuda") + 0.5, torch.randn(Co, device="cuda")
    outs = []
    for fused in (True, False):
        rm, rv = torch.zeros(Co, device="cuda"), torch.ones(Co, device="cuda")
        mean, invstd, scale, shift = (torch.empty(Co, device="cuda") for _ in range(4))
        if fused:
            ops.bn_stats_finalize(partial, rows, P, Co, gamma, beta, 1e-5, 0.1, rm, rv, mean, invstd, scale, shift)
        else:
            ops.bn_stats(y, P, Co, torch.empty_like(partial), gamma, beta, 1e-5, 0.1, rm, rv, mean, invstd, scale, shift)
        outs.append((mean, invstd, scale, shift, rm, rv))
    torch.cuda.synchronize()
    for a, b in zip(*outs):
        assert torch.allclose(a, b, rtol=2e-5, atol=2e-6), (a - b).abs().max()
    dy = torch.randn(N, Co, Ho, Wo, device="cuda", generator=g).to(torch.bfloat16).float()
    ws = torch.empty(ops.stem_wgrad_workspace_bytes(N, H, W) // 4, device="cuda")
    dw = torch.full((Co, ci_real, 7, 7), float("nan"), device="cuda")
    ops.stem_wgrad(x16, nhwc(dy), dw, ci_real, N, H, W, ws)
    torch.cuda.synchronize()
    ref_dw = torch.nn.grad.conv2d_weight(x, w.shape, dy, stride=2, padding=3)
    assert rel_err(dw, ref_dw) < 2e-3, rel_err(dw, ref_dw)
    dw2 = torch.empty_like(dw)
    ops.stem_wgrad(x16, nhwc(dy), dw2, ci_real, N, H, W, ws)
    assert torch.equal(dw, dw2)


@pytest.mark.parametrize("case", CONV_CASES)
@pytest.mark.parametrize("add_mode", [0, 1])
def test_conv_dgrad(case, add_mode):
    ops = _ops()
    N, H, W, Ci, Co, R, stride, pad = case
    xb, wb = _mk(*case)
    d = ops.conv_desc(N, H, W, Ci, Co, R, R, stride, pad)
    g = torch.Generator(device="cuda").manual_seed(2)
    dy = torch.randn(N, Co, d.Ho, d.Wo, device="cuda", generator=g).to(torch.bfloat16).float()
    Kp = ops.conv_packed_k(d)
    wp = torch.empty(Co, Kp, device="cuda", dtype=torch.bfloat16)
    wT = torch.zeros(Ci, R * R * Co, device="cuda", dtype=torch.bfloat16)
    ops.conv_pack_weights(d, Ci, wb, wp, wT)
    dx = torch.full((N, H, W, Ci), float("nan"), device="cuda", dtype=torch.bfloat16)
    add = None
    if add_mode == 1:
        add = torch.randn(N, H, W, Ci, device="cuda", generator=g).to(torch.bfloat16)
    ops.conv_dgrad(d, nhwc(dy), wT, dx, add, add_mode)
    torch.cuda.synchronize()
    ref = torch.nn.grad.conv2d_input(xb.shape, wb, dy, stride=stride, padding=pad)
    if add is not None:
        ref = ref + nchw(add)
    assert torch.isfinite(dx.float()).all()
    assert rel_err(nchw(dx), ref) < 6e-3, rel_err(nchw(dx), ref)


@pytest.mark.parametrize("geom", [(2, 13, 9, 64, 128), (96, 28, 28, 128, 256)])  # the second: CTA-pair kernel
def test_conv_dgrad_add_compact(geom):
    """add_mode 2: gradient of the 1x1/s2 downsample branch added at even pixels."""
    ops = _ops()
    N, H, W, Ci, Co = geom
    case = (N, H, W, Ci, Co, 3, 2, 1)
    xb, wb = _mk(*case)
    d = ops.conv_desc(N, H, W, Ci, Co, 3, 3, 2, 1)
    g = torch.Generator(device="cuda").manual_seed(3)
    dy = torch.randn(N, Co, d.Ho, d.Wo, device="cuda", generator=g).to(torch.bfloat16).float()
    wp = torch.empty(Co, ops.conv_packed_k(d), device="cuda", dtype=torch.bfloat16)
    wT = torch.zeros(Ci, 9 * Co, device="cuda", dtype=torch.bfloat16)
    ops.conv_pack_weights(d, Ci, wb, wp, wT)
    Hc, Wc = (H + 1) // 2, (W + 1) // 2
    add = torch.randn(N, Hc, Wc, Ci, device="cuda", generator=g).to(torch.bfloat16)
    dx = torch.empty(N, H, W, Ci, device="cuda", dtype=torch.bfloat16)
    ops.conv_dgrad(d, nhwc(dy), wT, dx, add, 2)
    torch.cuda.synchronize()
    ref = torch.nn.grad.conv2d_input(xb.shape, wb, dy, stride=2, padding=1)
    up = torch.zeros_like(ref)
    up[:, :, ::2, ::2] = nchw(add)
    assert rel_err(nchw(dx), ref + up) < 6e-3


# includes the two >= 148-item cases: one-wave split-K, co-major partials and the group-parallel reduction at full grid
@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_wgrad(case):
    ops = _ops()
    N, H, W, Ci, Co, R, stride, pad = case
    xb, wb = _mk(*case)
    d = ops.conv_desc(N, H, W, Ci, Co, R, R, stride, pad)
    g = torch.Generator(device="cuda").manual_seed(4)
    dy = torch.randn(N, Co, d.Ho, d.Wo, device="cuda", generator=g).to(torch.bfloat16).float()
    ws = torch.empty(ops.conv_wgrad_workspace_bytes(d) // 4, device="cuda", dtype=torch.float32)
    dw = torch.full((Co, Ci, R, R), float("nan"), device="cuda")
    ops.conv_wgrad(d, Ci, nhwc(xb), nhwc(dy), dw, ws)
    torch.cuda.synchronize()
    ref = torch.nn.grad.conv2d_weight(xb, wb.shape, dy, stride=stride, padding=pad)
    assert torch.isfinite(dw).all()
    assert rel_err(dw, ref) < 2e-3, rel_err(dw, ref)
    # determinism: bitwise identical on a second run
    dw2 = torch.empty_like(dw)
    ops.conv_wgrad(d, Ci, nhwc(xb), nhwc(dy), dw2, ws)
    torch.cuda.synchronize()
    assert torch.equal(dw, dw2)


def test_layout():
    ops = _ops()
    B, Cc, T, H, W = 3, 3, 2, 10, 7
    src = torch.randn(B, Cc, T, H, W, device="cuda")
    dst = torch.empty(B * T, H, W, 8, device="cuda", dtype=torch.bfloat16)
    ops.layout_ncthw_to_nhwc8(src, dst, B, Cc, T, H, W)
    ref = src.permute(0, 2, 3, 4, 1).reshape(B * T, H, W, Cc).to(torch.bfloat16)
    assert torch.equal(dst[..., :Cc], ref)
    assert (dst[..., Cc:] == 0).all()


@pytest.mark.parametrize("P,Cc", [(1000, 64), (777, 128), (50000, 256), (98, 512), (300000, 64)])
@pytest.mark.parametrize("relu,use_res", [(1, 0), (1, 1), (0, 0)])
def test_bn_fwd_bwd(P, Cc, relu, use_res):
    ops = _ops()
    g = torch.Generator(device="cuda").manual_seed(5)
    x = (torch.randn(P, Cc, device="cuda", generator=g) * 2 + 0.5).to(torch.bfloat16)
    res = torch.randn(P, Cc, device="cuda", generator=g).to(torch.bfloat16) if use_res else None
    gamma = torch.rand(Cc, device="cuda", generator=g) + 0.5
    beta = torch.randn(Cc, device="cuda", generator=g) * 0.1
    rm = torch.zeros(Cc, device="cuda")
    rv = torch.ones(Cc, device="cuda")
    partial = torch.empty(ops.bn_partial_floats(P, Cc), device="cuda")
    mean, invstd, scale, shift = (torch.empty(Cc, device="cuda") for _ in range(4))
    ops.bn_stats(x, P, Cc, partial, gamma, beta, 1e-5, 0.1, rm, rv, mean, invstd, scale, shift)
    y = torch.empty_like(x)
    ops.bn_apply(x, res, y, P, Cc, scale, shift, relu)
    torch.cuda.synchronize()

    xf = x.float().requires_grad_(True)
    gref = gamma.clone().requires_grad_(True)
    bref = beta.clone().requires_grad_(True)
    rm2, rv2 = torch.zeros(Cc, device="cuda"), torch.ones(Cc, device="cuda")
    z = F.batch_norm(xf, rm2, rv2, gref, bref, True, 0.1, 1e-5)
    if use_res:
        z = z + res.float()
    yr = F.relu(z) if relu else z
    assert torch.allclose(mean, xf.detach().mean(0), atol=1e-4, rtol=1e-4)
    assert torch.allclose(rm, rm2, atol=1e-5, rtol=1e-4)
    assert torch.allclose(rv, rv2, atol=1e-5, rtol=1e-4)
    assert rel_err(y.float(), yr.detach()) < 5e-3

    dy = torch.randn(P, Cc, device="cuda", generator=g).to(torch.bfloat16)
    # use OUR y for the relu mask in the reference too (mask parity is tested above)
    mask = (y.float() > 0).float() if relu else torch.ones_like(y.float())
    (z * mask).backward(dy.float())
    dz = torch.empty_like(dy)
    dx = torch.empty_like(dy)
    dgamma, dbeta = torch.empty(Cc, device="cuda"), torch.empty(Cc, device="cuda")
    ops.bn_bwd(dy, y, x, dz if relu else None, dx, P, Cc, gamma, mean, invstd, partial, dgamma, dbeta, relu)
    torch.cuda.synchronize()
    assert rel_err(dgamma, gref.grad) < 2e-3
    assert rel_err(dbeta, bref.grad) < 2e-3
    assert rel_err(dx.float(), xf.grad) < 8e-3
    if relu:
        assert torch.equal(dz.float(), dy.float() * mask)


@pytest.mark.parametrize("N,H,W,Cc", [(2, 129, 94, 64), (3, 112, 112, 64), (1, 7, 9, 64)])
def test_maxpool(N, H, W, Cc):
    ops = _ops()
    g = torch.Generator(device="cuda").manual_seed(6)
    x = torch.relu(torch.randn(N, Cc, H, W, device="cuda", generator=g)).to(torch.bfloat16)
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    xn = x.permute(0, 2, 3, 1).contiguous()
    y = torch.empty(N, Ho, Wo, Cc, device="cuda", dtype=torch.bfloat16)
    am = torch.empty(N, Ho, Wo, Cc, device="cuda", dtype=torch.uint8)
    ops.maxpool_fwd(xn, y, am, N, H, W, Cc, Ho, Wo)
    xf = x.float().requires_grad_(True)
    yr = F.max_pool2d(xf, 3, 2, 1)
    assert torch.equal(nchw(y), yr.detach())
    dy = torch.randn(N, Cc, Ho, Wo, device="cuda", generator=g).to(torch.bfloat16)
    yr.backward(dy.float())
    dx = torch.empty(N, H, W, Cc, device="cuda", dtype=torch.bfloat16)
    ops.maxpool_bwd(nhwc(dy.float()), am, dx, N, H, W, Cc, Ho, Wo)
    torch.cuda.synchronize()
    # ties between equal positive bf16 values may route differently from cuDNN; compare sums and bulk
    assert rel_err(nchw(dx), xf.grad) < 2e-2
    assert abs(nchw(dx).sum().item() - xf.grad.sum().item()) < 1e-1 * (1 + abs(xf.grad.sum().item()))


@pytest.mark.parametrize("P,Cc", [(1000, 64), (50000, 256), (98, 512)])
def test_bn_bwd_nores_matches_masked_path(P, Cc):
    """BN+ReLU backward with the mask recomputed from x == the path that reads y and writes dz."""
    ops = _ops()
    g = torch.Generator(device="cuda").manual_seed(15)
    x = (torch.randn(P, Cc, device="cuda", generator=g) * 2 + 0.5).to(torch.bfloat16)
    gamma = torch.rand(Cc, device="cuda", generator=g) + 0.5
    beta = torch.randn(Cc, device="cuda", generator=g) * 0.1
    partial = torch.empty(ops.bn_partial_floats(P, Cc), device="cuda")
    mean, invstd, scale, shift = (torch.empty(Cc, device="cuda") for _ in range(4))
    ops.bn_stats(x, P, Cc, partial, gamma, beta, 1e-5, 0.1, None, None, mean, invstd, scale, shift)
    y = torch.empty_like(x)
    ops.bn_apply(x, None, y, P, Cc, scale, shift, 1)
    dy = torch.randn(P, Cc, device="cuda", generator=g).to(torch.bfloat16)
    dz, dx1, dx2 = torch.empty_like(dy), torch.empty_like(dy), torch.empty_like(dy)
    dg1, db1, dg2, db2 = (torch.empty(Cc, device="cuda") for _ in range(4))
    ops.bn_bwd(dy, y, x, dz, dx1, P, Cc, gamma, mean, invstd, partial, dg1, db1, 1)
    ops.bn_bwd_nores(dy, x, dx2, P, Cc, gamma, mean, invstd, scale, shift, partial, dg2, db2)
    torch.cuda.synchronize()
    assert torch.equal(dg1, dg2) and torch.equal(db1, db2)
    assert torch.equal(dx1, dx2)


@pytest.mark.parametrize("N,H,W", [(2, 129, 94), (3, 112, 112), (1, 7, 9), (2, 65, 313)])
def test_stem_tail_fused_matches_unfused(N, H, W):
    """bn_relu_maxpool_fwd/bwd == bn_apply + maxpool_fwd and maxpool_bwd + bn_bwd, bit for bit."""
    ops = _ops()
    Cc = 64
    g = torch.Generator(device="cuda").manual_seed(16)
    P = N * H * W
    x = (torch.randn(N, H, W, Cc, device="cuda", generator=g) * 2 + 0.3).to(torch.bfloat16)
    gamma = torch.rand(Cc, device="cuda", generator=g) + 0.5
    beta = torch.randn(Cc, device="cuda", generator=g) * 0.1
    partial = torch.empty(ops.bn_partial_floats(P, Cc), device="cuda")
    mean, invstd, scale, shift = (torch.empty(Cc, device="cuda") for _ in range(4))
    ops.bn_stats(x, P, Cc, partial, gamma, beta, 1e-5, 0.1, None, None, mean, invstd, scale, shift)
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    y0 = torch.empty_like(x)
    ops.bn_apply(x, None, y0, P, Cc, scale, shift, 1)
    y1 = torch.empty(N, Ho, Wo, Cc, device="cuda", dtype=torch.bfloat16)
    am1 = torch.empty(N, Ho, Wo, Cc, device="cuda", dtype=torch.uint8)
    ops.maxpool_fwd(y0, y1, am1, N, H, W, Cc, Ho, Wo)
    y2, am2, xm = torch.empty_like(y1), torch.empty_like(am1), torch.empty_like(y1)
    ops.bn_relu_maxpool_fwd(x, scale, shift, y2, am2, xm, N, H, W, Cc, Ho, Wo)
    torch.cuda.synchronize()
    assert torch.equal(y1, y2) and torch.equal(am1, am2)
    # xmax is the conv output at the arg-max: BN+ReLU of it reproduces the pooled map
    assert torch.equal(torch.relu(torch.addcmul(shift, xm.float(), scale)).to(torch.bfloat16), y2)
    gp = torch.randn(N, Ho, Wo, Cc, device="cuda", generator=g).to(torch.bfloat16)
    g0 = torch.empty_like(x)
    ops.maxpool_bwd(gp, am1, g0, N, H, W, Cc, Ho, Wo)
    dx1, dx2 = torch.empty_like(x), torch.empty_like(x)
    dg1, db1, dg2, db2 = (torch.empty(Cc, device="cuda") for _ in range(4))
    ops.bn_bwd(g0, y0, x, g0, dx1, P, Cc, gamma, mean, invstd, partial, dg1, db1, 1)
    for xmax in (None, xm):  # sums over the stem grid, or over the pooled grid through the saved arg-max values
        ops.bn_relu_maxpool_bwd(gp, am2, xmax, x, dx2, N, H, W, Cc, Ho, Wo, gamma, mean, invstd, scale, shift,
                                partial, dg2, db2)
        torch.cuda.synchronize()
        # same per-pixel values; the channel sums are accumulated in a different (fixed) order, and on the
        # pooled grid without the bf16 rounding of pixels hit by two windows
        tol = 1e-5 if xmax is None else 2e-3
        assert rel_err(dg2, dg1) < tol and rel_err(db2, db1) < tol, (rel_err(dg2, dg1), rel_err(db2, db1))
        assert rel_err(dx2.float(), dx1.float()) < 2e-3
    dx3, dg3, db3 = torch.empty_like(x), torch.empty_like(dg2), torch.empty_like(db2)
    ops.bn_relu_maxpool_bwd(gp, am2, xm, x, dx3, N, H, W, Cc, Ho, Wo, gamma, mean, invstd, scale, shift, partial,
                            dg3, db3)
    torch.cuda.synchronize()
    assert torch.equal(dg2, dg3) and torch.equal(db2, db3) and torch.equal(dx2, dx3)  # deterministic


@pytest.mark.parametrize("M,N,K", [(1024, 128, 64), (4096, 512, 256), (2048, 64, 512)])
def test_gemm_nt_bf16(M, N, K):
    ops = _ops()
    g = torch.Generator(device="cuda").manual_seed(21)
    lda = K + 64
    A = torch.randn(M, lda, device="cuda", generator=g).to(torch.bfloat16)
    Bm = torch.randn(N, K, device="cuda", generator=g).to(torch.bfloat16)
    Cm = torch.full((M, N), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.gemm_nt_bf16(A, lda, Bm, Cm, M, N, K)
    torch.cuda.synchronize()
    ref = A[:, :K].float() @ Bm.float().t()
    assert rel_err(Cm.float(), ref) < 6e-3


@pytest.mark.parametrize("M,N,K", [(128, 128, 4096), (384, 512, 16384), (64, 128, 2048)])
def test_gemm_tn_f32(M, N, K):
    ops = _ops()
    g = torch.Generator(device="cuda").manual_seed(22)
    At = torch.randn(K, M, device="cuda", generator=g).to(torch.bfloat16)
    Bt = torch.randn(K, N, device="cuda", generator=g).to(torch.bfloat16)
    bias = torch.randn(N, device="cuda", generator=g)
    ws = torch.empty(ops.gemm_tn_workspace_bytes(M, N, K) // 4, device="cuda")
    Cm = torch.full((M, N), float("nan"), device="cuda")
    ops.gemm_tn_f32(At, Bt, bias, Cm, M, N, K, ws)
    torch.cuda.synchronize()
    ref = At.float().t() @ Bt.float() + bias
    assert rel_err(Cm, ref) < 2e-3
    C2 = torch.empty_like(Cm)
    ops.gemm_tn_f32(At, Bt, bias, C2, M, N, K, ws)
    torch.cuda.synchronize()
    assert torch.equal(Cm, C2)


def test_film_fn_matches_torch():
    """FilmFn (outer product -> Linear(262144 -> 512)) forward and backward vs plain torch."""
    from gdl_b200.film import FilmFn
    _ops()
    B, D = 5, 512
    g = torch.Generator(device="cuda").manual_seed(23)
    x = torch.randn(B, D, device="cuda", generator=g, requires_grad=True)
    y = torch.randn(B, D, device="cuda", generator=g, requires_grad=True)
    W = (torch.randn(D, D * D, device="cuda", generator=g) * 0.002).requires_grad_(True)
    b = torch.randn(D, device="cuda", generator=g).requires_grad_(True)
    h = FilmFn.apply(x, y, W, b)
    dh = torch.randn(B, D, device="cuda", generator=g)
    gx, gy, gW, gb = torch.autograd.grad(h, (x, y, W, b), dh)
    z = torch.bmm(x.detach().unsqueeze(2), y.detach().unsqueeze(1)).flatten(1)
    x2, y2 = x.detach().clone().requires_grad_(True), y.detach().clone().requires_grad_(True)
    W2, b2 = W.detach().clone().requires_grad_(True), b.detach().clone().requires_grad_(True)
    h2 = torch.nn.functional.linear(torch.bmm(x2.unsqueeze(2), y2.unsqueeze(1)).flatten(1), W2, b2)
    rx, ry, rW, rb = torch.autograd.grad(h2, (x2, y2, W2, b2), dh)
    assert rel_err(h, h2.detach()) < 6e-3
    assert rel_err(gx, rx) < 1e-2 and rel_err(gy, ry) < 1e-2
    assert rel_err(gW, rW) < 1e-2 and rel_err(gb, rb) < 1e-5
    del z


def test_gap():
    ops = _ops()
    B, G, Cc = 5, 147, 512
    x = torch.randn(B, G, Cc, device="cuda").to(torch.bfloat16)
    out = torch.empty(B, Cc, device="cuda")
    ops.gap_fwd(x, out, B, G, Cc)
    assert torch.allclose(out, x.float().mean(1), atol=1e-5, rtol=1e-5)
    dout = torch.randn(B, Cc, device="cuda")
    dx = torch.empty_like(x)
    ops.gap_bwd(dout, dx, B, G, Cc)
    ref = (dout / G).to(torch.bfloat16)[:, None, :].expand(B, G, Cc)
    assert torch.equal(dx, ref)


@pytest.mark.parametrize("B,In,Out", [(7, 512, 6), (64, 512, 512), (33, 1024, 309)])
def test_linear(B, In, Out):
    ops = _ops()
    x = torch.randn(B, In, device="cuda", requires_grad=True)
    W = (torch.randn(Out, In, device="cuda") * 0.05).requires_grad_(True)
    b = torch.randn(Out, device="cuda", requires_grad=True)
    y = torch.empty(B, Out, device="cuda")
    ops.linear_fwd(x.detach(), W.detach(), b.detach(), y, B, In, Out)
    yr = F.linear(x.double(), W.double(), b.double())
    assert torch.allclose(y.double(), yr, atol=1e-4, rtol=1e-4)
    dy = torch.randn(B, Out, device="cuda")
    yr.backward(dy.double())
    dx, dW, db = torch.empty_like(x), torch.empty_like(W), torch.empty_like(b)
    ops.linear_bwd(dy, x.detach(), W.detach(), dx, dW, db, B, In, Out)
    assert torch.allclose(dx, x.grad, atol=1e-4, rtol=1e-4)
    assert torch.allclose(dW, W.grad, atol=1e-4, rtol=1e-4)
    assert torch.allclose(db, b.grad, atol=1e-4, rtol=1e-4)


@pytest.mark.parametrize("kind", [0, 1])
@pytest.mark.parametrize("B,n", [(16, 6), (37, 34), (64, 309), (256, 6), (64, 34)])
def test_dgl_head_linear(kind, B, n):
    """Fused head vs an autograd restatement of reference fusion_modules.py:22-30,51-59 +
    main_dgl.py:102-122 (two backward passes with the fusion grads wiped in between)."""
    ops = _ops()
    D, alpha = 512, 4.0
    g = torch.Generator(device="cuda").manual_seed(7)
    a = torch.randn(B, D, device="cuda", generator=g).double().requires_grad_(True)
    v = torch.randn(B, D, device="cuda", generator=g).double().requires_grad_(True)
    labels = torch.randint(0, n, (B,), device="cuda", generator=g)
    if kind == 0:
        W = (torch.randn(n, 2 * D, device="cuda", generator=g) * 0.05).double().requires_grad_(True)
        bx = torch.randn(n, device="cuda", generator=g).double().requires_grad_(True)
        out = F.linear(torch.cat((a, v), 1).detach(), W, bx)
        xo = F.linear(torch.cat((a, torch.zeros_like(v)), 1), W, bx)
        yo = F.linear(torch.cat((torch.zeros_like(a), v), 1), W, bx)
        params = [W, bx]
    else:
        Wx = (torch.randn(n, D, device="cuda", generator=g) * 0.05).double().requires_grad_(True)
        Wy = (torch.randn(n, D, device="cuda", generator=g) * 0.05).double().requires_grad_(True)
        bx = torch.randn(n, device="cuda", generator=g).double().requires_grad_(True)
        by = torch.randn(n, device="cuda", generator=g).double().requires_grad_(True)
        xo, yo = F.linear(a, Wx, bx), F.linear(v, Wy, by)
        out = F.linear(a.detach(), Wx, bx) + F.linear(v.detach(), Wy, by)
        params = [Wx, Wy, bx, by]
    Lf, La, Lv = (F.cross_entropy(t, labels) for t in (out, xo, yo))
    ((La + Lv) * alpha).backward(retain_graph=True)
    for p in params:
        p.grad = None
    Lf.backward()

    f32 = lambda t: t.detach().float().contiguous()
    logits = torch.empty(3, B, n, device="cuda")
    losses = torch.empty(3, device="cuda")
    da, dv = torch.empty(B, D, device="cuda"), torch.empty(B, D, device="cuda")
    scratch = torch.empty(ops.head_scratch_floats(B, n), device="cuda")
    if kind == 0:
        Wf, bf = f32(W), f32(bx)
        dW, db = torch.empty_like(Wf), torch.empty_like(bf)
        ops.dgl_head_linear(0, f32(a), f32(v), Wf.data_ptr(), Wf.data_ptr() + 4 * D, 2 * D, bf, None, labels,
                            alpha, 1.0 / B, logits, losses, da, dv, dW.data_ptr(), dW.data_ptr() + 4 * D,
                            2 * D, db, None, scratch, B, D, n)
        got = [dW, db]
    else:
        Wxf, Wyf, bxf, byf = f32(Wx), f32(Wy), f32(bx), f32(by)
        dWx, dWy, dbx, dby = (torch.empty_like(t) for t in (Wxf, Wyf, bxf, byf))
        ops.dgl_head_linear(1, f32(a), f32(v), Wxf.data_ptr(), Wyf.data_ptr(), D, bxf, byf, labels, alpha,
                            1.0 / B, logits, losses, da, dv, dWx.data_ptr(), dWy.data_ptr(), D, dbx, dby,
                            scratch, B, D, n)
        got = [dWx, dWy, dbx, dby]
    torch.cuda.synchronize()
    tol = dict(atol=2e-5, rtol=2e-4)
    assert torch.allclose(logits[0].double(), out.detach(), **tol)
    assert torch.allclose(logits[1].double(), xo.detach(), **tol)
    assert torch.allclose(logits[2].double(), yo.detach(), **tol)
    assert torch.allclose(losses.double(), torch.stack([Lf, La, Lv]).detach(), **tol)
    assert torch.allclose(da.double(), a.grad, **tol)
    assert torch.allclose(dv.double(), v.grad, **tol)
    for gt, p in zip(got, params):
        assert torch.allclose(gt.double(), p.grad, **tol)


@pytest.mark.parametrize("B,n", [(8, 6), (37, 34), (16, 309), (256, 6), (64, 34)])
def test_dgl_head_gated_fused(B, n):
    """Fused GatedFusion_DGL head vs an fp64 autograd restatement of reference fusion_modules.py:230-250 +
    main_dgl.py:102-122 (two backward passes, fusion-module gradients wiped in between): logits, losses, the
    encoder-facing gradients da / dv, fc_out's gradients from Lf; fc_x / fc_y get none."""
    ops = _ops()
    D, alpha = 512, 4.0
    g = torch.Generator(device="cuda").manual_seed(9)
    rnd = lambda *s: torch.randn(*s, device="cuda", generator=g)
    a = rnd(B, D).abs().double().requires_grad_(True)
    v = rnd(B, D).abs().double().requires_grad_(True)
    labels = torch.randint(0, n, (B,), device="cuda", generator=g)
    Wx, Wy = (rnd(D, D) * 0.05).double().requires_grad_(True), (rnd(D, D) * 0.05).double().requires_grad_(True)
    bx, by = (rnd(D) * 0.1).double().requires_grad_(True), (rnd(D) * 0.1).double().requires_grad_(True)
    Wo, bo = (rnd(n, D) * 0.05).double().requires_grad_(True), (rnd(n) * 0.1).double().requires_grad_(True)
    hx, hy = F.linear(a, Wx, bx), F.linear(v, Wy, by)
    out = F.linear(torch.sigmoid(hx.detach()) * hy.detach(), Wo, bo)
    xo = F.linear(torch.sigmoid(hx) * hx, Wo, bo)
    yo = F.linear(torch.sigmoid(hy) * hy, Wo, bo)
    Lf, La, Lv = (F.cross_entropy(t, labels) for t in (out, xo, yo))
    params = [Wx, Wy, bx, by, Wo, bo]
    ((La + Lv) * alpha).backward(retain_graph=True)
    for p in params:
        p.grad = None                      # the reference wipes every fusion-module gradient (main_dgl.py:114-119)
    Lf.backward()
    assert Wx.grad is None and Wy.grad is None  # Lf sees hx / hy detached: fc_x / fc_y are never trained

    f32 = lambda t: t.detach().float().contiguous()
    logits = torch.empty(3, B, n, device="cuda")
    losses = torch.empty(3, device="cuda")
    da, dv = torch.empty(B, D, device="cuda"), torch.empty(B, D, device="cuda")
    dWo, dbo = torch.empty(n, D, device="cuda"), torch.empty(n, device="cuda")
    scratch = torch.empty(ops.gated_head_scratch_floats(B, n), device="cuda")
    ops.dgl_head_gated(f32(a), f32(v), f32(Wx), f32(bx), f32(Wy), f32(by), f32(Wo), f32(bo), labels, alpha, 1.0 / B,
                       logits, losses, da, dv, dWo, dbo, scratch, B, D, n)
    torch.cuda.synchronize()
    tol = dict(atol=2e-5, rtol=2e-4)
    for got, ref in ((logits[0], out), (logits[1], xo), (logits[2], yo), (da, a.grad), (dv, v.grad), (dWo, Wo.grad),
                     (dbo, bo.grad)):
        assert torch.allclose(got.double(), ref.detach(), **tol)
    assert torch.allclose(losses.double(), torch.stack([Lf, La, Lv]).detach(), **tol)


def test_softmax_ce_and_gated():
    ops = _ops()
    B, n = 19, 34
    z = torch.randn(B, n, device="cuda", requires_grad=True)
    labels = torch.randint(0, n, (B,), device="cuda")
    loss = torch.empty(1, device="cuda")
    dz = torch.empty(B, n, device="cuda")
    scratch = torch.empty(B, device="cuda")
    ops.softmax_ce(z.detach(), labels, 1.0 / B, 4.0 / B, loss, dz, scratch, B, n)
    Lr = F.cross_entropy(z, labels)
    (Lr * 4.0).backward()
    assert torch.allclose(loss[0], Lr.detach(), atol=1e-5, rtol=1e-5)
    assert torch.allclose(dz, z.grad, atol=1e-6, rtol=1e-4)

    hx = torch.randn(B, 512, device="cuda", requires_grad=True)
    hy = torch.randn(B, 512, device="cuda", requires_grad=True)
    mo, mx, my = (torch.empty(B, 512, device="cuda") for _ in range(3))
    ops.gated_fwd(hx.detach(), hy.detach(), mo, mx, my)
    rx, ry = torch.sigmoid(hx) * hx, torch.sigmoid(hy) * hy
    assert torch.allclose(mo, (torch.sigmoid(hx) * hy).detach(), atol=1e-6, rtol=1e-5)
    assert torch.allclose(mx, rx.detach(), atol=1e-6, rtol=1e-5)
    gx, gy = torch.randn_like(hx), torch.randn_like(hy)
    (rx * gx + ry * gy).sum().backward()
    dhx, dhy = torch.empty_like(gx), torch.empty_like(gy)
    ops.gated_bwd(hx.detach(), hy.detach(), gx, gy, dhx, dhy)
    assert torch.allclose(dhx, hx.grad, atol=1e-5, rtol=1e-4)
    assert torch.allclose(dhy, hy.grad, atol=1e-5, rtol=1e-4)


def test_grad_stats_and_sgd():
    ops = _ops()
    sizes = [(64, 3, 7, 7), (64,), (64,), (128, 64, 3, 3), (6, 1024), (6,), (100003,)]
    groups = [0, 0, 1, 1, 2, 2, 1]
    pad = lambda n: (n + 63) // 64 * 64
    offs, total = [], 0
    for s in sizes:
        offs.append(total)
        total += pad(int(torch.tensor(s).prod()))
    g = torch.Generator(device="cuda").manual_seed(8)
    grad = torch.zeros(total, device="cuda")
    param = torch.zeros(total, device="cuda")
    grads, params = [], []
    for s, o in zip(sizes, offs):
        n = int(torch.tensor(s).prod())
        grad[o:o + n] = torch.randn(n, device="cuda", generator=g) * 3
        param[o:o + n] = torch.randn(n, device="cuda", generator=g)
        grads.append(grad[o:o + n].clone().view(s))
        params.append(param[o:o + n].clone().view(s).requires_grad_(True))
    seg_end = torch.tensor([o + pad(int(torch.tensor(s).prod())) for s, o in zip(sizes, offs)],
                           device="cuda", dtype=torch.int64)
    seg_group = torch.tensor(groups, device="cuda", dtype=torch.int32)
    seg_inv = torch.tensor([1.0 / int(torch.tensor(s).prod()) for s in sizes], device="cuda")
    scratch = torch.empty(ops.optim_scratch_floats(total, len(sizes)), device="cuda")
    stats = torch.empty(4, device="cuda")
    ops.grad_stats(grad, total, seg_end, seg_group, seg_inv, len(sizes), 40.0, scratch, stats)
    buf = torch.zeros(total, device="cuda")
    p0 = param.clone()
    for step in range(2):
        ops.sgd_momentum(param, grad, buf, total, 0.01, 0.9, 1e-4, step == 0, stats)
        if step == 0:
            stats[1] = 1.0  # second step: grads already clipped
    torch.cuda.synchronize()

    for p, gr in zip(params, grads):
        p.grad = gr.clone()
    norm = torch.nn.utils.clip_grad_norm_(params, 40.0, 2)
    opt = torch.optim.SGD(params, lr=0.01, momentum=0.9, weight_decay=1e-4)
    a_sum = sum(p.grad.abs().mean().item() for p, gg in zip(params, groups) if gg == 0)
    v_sum = sum(p.grad.abs().mean().item() for p, gg in zip(params, groups) if gg == 1)
    opt.step()
    opt.step()
    assert abs(stats[0].item() - norm.item()) < 1e-3 * norm.item()
    # stats[2], stats[3] were computed before we overwrote stats[1]
    assert abs(stats[2].item() - a_sum) < 1e-4 * (1 + a_sum)
    assert abs(stats[3].item() - v_sum) < 1e-4 * (1 + v_sum)
    for p, s, o in zip(params, sizes, offs):
        n = p.numel()
        assert torch.allclose(param[o:o + n].view(s), p.detach(), atol=1e-6, rtol=1e-5)
        assert torch.allclose(grad[o:o + n].view(s), p.grad, atol=1e-6, rtol=1e-5)
    assert p0.shape == param.shape


def test_generic_gather_kernels():
    """The generic (cp.async im2col gather) forward / data-gradient / weight-gradient kernels are the library's
    fallback for geometries outside the flat-window TMA kernels; GDL_FLAT=0 GDL_WFLAT=0 (read once per process)
    routes every convolution to them, so the same parity cases are re-run in a subprocess with those switches."""
    import os
    import subprocess
    import sys
    import time
    env = dict(os.environ, GDL_FLAT="0", GDL_WFLAT="0")
    t0 = time.monotonic()
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-m", "gpu", "--no-header", "-x",
                        "-p", "no:cacheprovider", "-k",
                        "(test_conv_fwd or test_conv_dgrad or test_conv_wgrad) and not bias_act and not statistics"],
                       env=env, capture_output=True, text=True, timeout=600)
    print("generic gather kernels: %.0f s of the 600 s timeout" % (time.monotonic() - t0))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert " passed" in r.stdout
