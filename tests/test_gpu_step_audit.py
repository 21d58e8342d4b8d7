"""Layer-by-layer audit of the full-size training forward, and the BatchNorm / stem-tail / FiLM kernels at the
geometries, sweep directions and call sequences the training step uses.  GPU only.

The whole-step parity tests either take the forward on trust (teacher forcing) or compare losses and gradient
norms loosely, and relative L2 does not see one wrong 128-pixel tile of a 2.4 M-pixel map.  Here every tensor the
real step stored is checked against a reference computed from the stored input of the same layer, element by
element, with bounds derived from the compute type:
  - convolutions (bf16 operands, fp32 accumulation, bf16 output): |got - ref| <= 2^-8 |ref| + 1e-3 rms(ref), the
    first term the output rounding, the second the fp32 accumulation order over K <= 4608;
  - element-wise outputs (fmaf + add + relu, rounded once): bit-exact against torch's addcmul, which rounds like
    fmaf; an element one bf16 ulp off is counted and reported, anything further off fails;
  - BatchNorm statistics: mean within 1e-5 std of its channel, invstd within 1e-4 relative;
  - reductions (dgamma, dbeta, pooled features): 1e-5 of the sum of absolute values of the terms, the error
    bound of an fp32 sum of a few hundred sequential terms per thread.
References are fp32 with TF32 off (convolutions) or fp64 (everything else), from operands taken as exact."""
import gc
import threading
from types import SimpleNamespace

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

BF = torch.bfloat16
ULP = 2.0 ** -8
EPS, MOMENTUM = 1e-5, 0.1

# (P, C) of the BatchNorm units of the residual blocks, layers 1..4: CREMA-D at B = 256 (the benchmark) and
# KineticSound at B = 64 (the per-GPU batch of G = 512 on eight GPUs); audio N = B, visual N = 3 B frames.
# test_step_forward_audit checks this list against the units of the engines it builds.
UNIT_GEOMS = {
    ("CREMAD", "audio"): [(256 * 65 * 47, 64), (256 * 33 * 24, 128), (256 * 17 * 12, 256), (256 * 9 * 6, 512)],
    ("CREMAD", "visual"): [(768 * 56 * 56, 64), (768 * 28 * 28, 128), (768 * 14 * 14, 256), (768 * 7 * 7, 512)],
    ("KineticSound", "audio"): [(64 * 33 * 157, 64), (64 * 17 * 79, 128), (64 * 9 * 40, 256), (64 * 5 * 20, 512)],
    ("KineticSound", "visual"): [(192 * 56 * 56, 64), (192 * 28 * 28, 128), (192 * 14 * 14, 256), (192 * 7 * 7, 512)],
}
# (N, H, W) of the stem conv outputs the stem tail (BN + ReLU + max-pool) runs on, same configurations
STEM_TAILS = {
    ("CREMAD", "audio"): (256, 129, 94),
    ("CREMAD", "visual"): (768, 112, 112),
    ("KineticSound", "audio"): (64, 65, 313),
    ("KineticSound", "visual"): (192, 112, 112),
}
AUDIT_CONFIGS = [("CREMAD", 256), ("KineticSound", 64)]


@pytest.fixture(autouse=True)
def ops():
    """The library, exact fp32 references (no TF32), and the sweep hint back at 0 after every test."""
    from gdl_b200 import ops as _ops
    _ops.init()
    saved = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        yield _ops
    finally:
        _ops.sweep(0)
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved
        assert _ops._sweep_state.get(threading.get_ident(), 0) == 0


def _free():
    gc.collect()
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------- comparison helpers
def _at(t, k):
    """Multi-index of flat index k of tensor t."""
    idx = []
    for s in reversed(t.shape):
        idx.append(k % s)
        k //= s
    return tuple(reversed(idx))


def _finite(name, got):
    bad = ~torch.isfinite(got.float())
    if bool(bad.any()):
        k = int(bad.flatten().nonzero()[0])
        raise AssertionError("%s: %d non-finite elements, first at %s" % (name, int(bad.sum()), _at(got, k)))


def check_bound(name, got, ref, bound):
    """|got - ref| <= bound element-wise (bound broadcasts against ref); names the worst element."""
    _finite(name, got)
    err = (got.double() - ref.double()).abs()
    excess = (err - bound).flatten()
    k = int(excess.argmax())
    if excess[k] > 0:
        b = torch.broadcast_to(bound, ref.shape).flatten()[k]
        raise AssertionError("%s: %d elements out of bound; worst at %s: got %r ref %r bound %.3g" % (
            name, int((excess > 0).sum()), _at(ref, k), got.flatten()[k].item(), ref.flatten()[k].item(), b.item()))


def check_conv(name, got, ref):
    """bf16 output of bf16 x bf16 -> fp32 accumulation: per element 2^-8 |ref| + 1e-3 rms(ref), and relative L2."""
    ref = ref.float()
    rms = ref.double().pow(2).mean().sqrt().item()
    check_bound(name, got.float(), ref, ref.abs() * ULP + 1e-3 * rms)
    rel = ((got.float() - ref).double().norm() / (ref.double().norm() + 1e-30)).item()
    assert rel < 6e-3, "%s: relative L2 %.3g" % (name, rel)


def check_exact(name, got, ref, ulps=None):
    """Bit-exact bf16 (values: -0 == +0).  Elements exactly one ulp off are counted in `ulps` (name -> count) and
    allowed up to 1e-4 of the tensor; any other difference fails.  Returns the one-ulp count."""
    assert got.shape == ref.shape and got.dtype == ref.dtype, (name, got.shape, ref.shape, got.dtype, ref.dtype)
    diff = (got.float() != ref.float()).flatten()   # NaN in got (a stale or unwritten element) differs
    if not bool(diff.any()):
        return 0
    gi = got.flatten().view(torch.int16)[diff].int()
    ri = ref.flatten().view(torch.int16)[diff].int()
    one = ((gi - ri).abs() == 1) & ((gi < 0) == (ri < 0)) & torch.isfinite(got.flatten()[diff].float())
    n1 = int(one.sum())
    if n1 < int(diff.sum()):
        k = int(diff.nonzero()[(~one).nonzero()[0]])
        raise AssertionError("%s: %d elements differ by more than one bf16 ulp; first at %s: got %r ref %r" % (
            name, int(diff.sum()) - n1, _at(got, k), got.flatten()[k].item(), ref.flatten()[k].item()))
    print("%s: %d elements one bf16 ulp off" % (name, n1))
    if ulps is not None:
        ulps[name] = n1
    assert n1 <= 1e-4 * got.numel(), "%s: %d elements one ulp off" % (name, n1)
    return n1


def rel_l2(a, b):
    return ((a.double() - b.double()).norm() / (b.double().norm() + 1e-300)).item()


# ---------------------------------------------------------------------------------- references
def space_to_depth(x, Hp, Wp):
    """fp32 [N, C, H, W] -> the stem's bf16 input [N, Hp, Wp, 16]: channel (dy*2 + dx)*C + c of pixel (p, q) is
    x[c, 2p + dy - 3, 2q + dx - 3] (zero outside the image and in the channels past 4 C)."""
    N, C, H, W = x.shape
    pad = x.new_zeros(N, C, 2 * Hp, 2 * Wp)
    pad[:, :, 3:3 + H, 3:3 + W] = x
    out = x.new_zeros(N, Hp, Wp, 16)
    for dy in range(2):
        for dx in range(2):
            k = (dy * 2 + dx) * C
            out[..., k:k + C] = pad[:, :, dy::2, dx::2].permute(0, 2, 3, 1)
    return out.to(BF)


def conv_nhwc(x, w, stride, pad, bias=None):
    """fp32 reference of a bf16 NHWC input and fp32 (already bf16-valued) OIHW weights -> fp32 NHWC."""
    y = F.conv2d(x.float().permute(0, 3, 1, 2), w.float(), stride=stride, padding=pad)
    y = y.permute(0, 2, 3, 1)
    return y if bias is None else y + bias


def bn_stats_ref(x, C):
    """fp64 batch mean and biased variance per channel of the bf16 [..., C] tensor x."""
    xd = x.reshape(-1, C).double()
    mean = xd.mean(0)
    var = (xd - mean).pow(2).mean(0)
    return mean, var, xd.shape[0]


def check_stats(name, x, C, mean, invstd, rm=None, rv=None, rm0=None, rv0=None, epilogue=False):
    """Kernel statistics of the stored bf16 tensor x against fp64; the running pair against the fp64 momentum
    update (unbiased variance) from the snapshot rm0 / rv0.
    epilogue=True: the kernel took the statistics from the fp32 conv outputs before their bf16 store.  Rounding adds
    noise of variance up to (2^-8 x)^2 / 3 per element (uniform within half an ulp), which matters in a channel whose
    |mean| >> std: the bounds add it, and 6 standard deviations of its sampling error on the mean and variance."""
    m, var, P = bn_stats_ref(x, C)
    std = var.sqrt()
    dm, dv = 0.0, 0.0
    if epilogue:
        noise = (x.reshape(-1, C).double() * ULP).pow(2).mean(0) / 3
        dm = 6 * (noise / P).sqrt()
        dv = noise + 12 * (var * noise / P).sqrt()
    check_bound(name + " mean", mean, m, 1e-5 * std + dm + 1e-30)
    ist = (var + EPS).rsqrt()
    check_bound(name + " invstd", invstd, ist, (1e-4 + 0.5 * dv / (var + EPS)) * ist)
    if rm is not None:
        rm_ref = (1 - MOMENTUM) * rm0.double() + MOMENTUM * m
        rv_ref = (1 - MOMENTUM) * rv0.double() + MOMENTUM * var * P / (P - 1)
        check_bound(name + " running_mean", rm, rm_ref, MOMENTUM * (1e-5 * std + dm) + 1e-6 * rm_ref.abs())
        check_bound(name + " running_var", rv, rv_ref, MOMENTUM * (2e-4 * var + dv) * P / (P - 1)
                    + 1e-6 * rv_ref.abs())


def check_affine(name, gamma, beta, mean, invstd, scale, shift):
    """scale = gamma * invstd, shift = beta - mean * scale from the kernel's own fp32 mean / invstd."""
    sc = gamma.double() * invstd.double()
    check_bound(name + " scale", scale, sc, 1e-6 * sc.abs())
    ms = mean.double() * scale.double()
    check_bound(name + " shift", shift, beta.double() - ms, 1e-6 * (beta.double().abs() + ms.abs()) + 1e-30)


def apply_ref(x, scale, shift, res=None, relu=True):
    """The BatchNorm apply as the kernel rounds it: fmaf(x, scale, shift) [+ res] [relu] -> bf16."""
    f = torch.addcmul(shift, x.float(), scale)
    if res is not None:
        f = f + res.float()
    return (torch.relu(f) if relu else f).to(BF)


def pool_taps(y, fill):
    """[9, N, Ho, Wo, C] values of the 3x3 / s2 / pad 1 windows of the NHWC tensor y, tap t = 3 r + s from the
    window's top-left pixel (2 ho - 1, 2 wo - 1); `fill` outside the image."""
    N, H, W, C = y.shape
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    p = y.new_full((N, H + 2, W + 2, C), fill)
    p[:, 1:H + 1, 1:W + 1] = y
    return torch.stack([p[:, r::2][:, :Ho][:, :, s::2][:, :, :Wo] for r in range(3) for s in range(3)])


def tail_fwd_ref(x, scale, shift):
    """pool_y = max_pool2d(3, 2, 1) of relu(addcmul(shift, x, scale)).bf16; arg-max = FIRST tap in scan order
    holding the window maximum; xmax = x at that tap."""
    taps = pool_taps(apply_ref(x, scale, shift).float(), float("-inf"))
    ymax = taps.max(0).values
    idx = torch.full(ymax.shape, 9, dtype=torch.uint8, device=x.device)
    for t in range(8, -1, -1):
        idx = torch.where(taps[t] == ymax, torch.full_like(idx, t), idx)
    del taps
    xt = pool_taps(x, 0.0)
    xmax = torch.gather(xt, 0, idx.long().unsqueeze(0)).squeeze(0)
    return ymax.to(BF), idx, xmax


def tail_scatter_ref(gpool, idx, H, W):
    """fp64 gradient wrt the stem-tail input: every window's gradient added at its arg-max pixel."""
    N, Ho, Wo, C = gpool.shape
    r, s = (idx.long() // 3), (idx.long() % 3)
    hh = 2 * torch.arange(Ho, device=gpool.device).view(1, Ho, 1, 1) - 1 + r
    ww = 2 * torch.arange(Wo, device=gpool.device).view(1, 1, Wo, 1) - 1 + s
    nn_ = torch.arange(N, device=gpool.device).view(N, 1, 1, 1)
    cc = torch.arange(C, device=gpool.device).view(1, 1, 1, C)
    flat = ((nn_ * H + hh) * W + ww) * C + cc
    g = torch.zeros(N * H * W * C, dtype=torch.float64, device=gpool.device)
    g.index_add_(0, flat.flatten(), gpool.double().flatten())
    return g.view(N, H, W, C)


def bn_bwd_ref(dz, x, gamma, mean, invstd):
    """fp64 BatchNorm backward (training statistics) given the kernel's mean / invstd: dbeta, dgamma, dx, and the
    sums of absolute values that bound an fp32 evaluation of the two reductions."""
    C = x.shape[-1]
    dz, x = dz.reshape(-1, C).double(), x.reshape(-1, C).double()
    P = dz.shape[0]
    m, ist, g = mean.double(), invstd.double(), gamma.double()
    xhat = (x - m) * ist
    dbeta = dz.sum(0)
    dgamma = (dz * xhat).sum(0)
    dx = g * ist * (dz - dbeta / P - xhat * (dgamma / P))
    abs_b = dz.abs().sum(0)
    abs_g = (dz.abs() * (x.abs() + m.abs())).sum(0) * ist
    return dbeta, dgamma, dx, abs_b, abs_g


def check_bn_bwd(name, dgamma, dbeta, dx, dz_ref, x, gamma, mean, invstd, dz_slack=None):
    """dgamma / dbeta within 1e-5 of the sums of |terms|; dx per element within 2^-8 |ref| + 2e-4 rms(ref).
    dz_slack: per-pixel |dz| the reference may differ by (the bf16 rounding of a pixel hit by several windows)."""
    rb, rg, rdx, abs_b, abs_g = bn_bwd_ref(dz_ref, x, gamma, mean, invstd)
    sb, sg, sdx = 0.0, 0.0, 0.0
    if dz_slack is not None:
        C = x.shape[-1]
        sl = dz_slack.reshape(-1, C)
        xhat = (x.reshape(-1, C).double() - mean.double()) * invstd.double()
        sb, sg = sl.sum(0), (sl * xhat.abs()).sum(0)
        sdx = (gamma.double() * invstd.double()) * sl
    check_bound(name + " dbeta", dbeta, rb, 1e-5 * abs_b + sb + 1e-30)
    check_bound(name + " dgamma", dgamma, rg, 1e-5 * abs_g + sg + 1e-30)
    rms = rdx.pow(2).mean().sqrt().item()
    check_bound(name + " dx", dx.reshape(rdx.shape), rdx, rdx.abs() * ULP + 2e-4 * rms + sdx)


# ---------------------------------------------------------------------------------- 1. in-situ audit of one step
def _encoder_input(name, spec, image):
    B = spec.shape[0]
    if name == "audio":
        return spec.unsqueeze(1).float()
    T = image.shape[2]
    return image.permute(0, 2, 1, 3, 4).reshape(B * T, 3, image.shape[3], image.shape[4]).float()


def _units_geoms(eng):
    return sorted({(u.P, u.C) for u in eng.units if u is not eng.stem})


def _audit_train(tag, eng, x_src, snap, ulps):
    s = eng.stem
    # stem input and conv
    x_ref = space_to_depth(x_src, s.Hp, s.Wp)
    assert torch.equal(eng.x_in, x_ref), "%s stem input: space-to-depth differs in %d elements" % (
        tag, int((eng.x_in.float() != x_ref.float()).sum()))
    xb = x_src.to(BF).float()
    w = snap[s.conv][0].to(BF).float()
    check_conv(tag + " conv1 (stem)", s.x, F.conv2d(xb, w, stride=2, padding=3).permute(0, 2, 3, 1))
    del xb, x_ref
    # stem BatchNorm and tail
    _, g0, b0, rm0, rv0 = snap[s.conv]
    check_stats(tag + " conv1 (stem)", s.x, 64, s.mean, s.invstd, s.bn.running_mean, s.bn.running_var, rm0, rv0,
                epilogue=True)
    check_affine(tag + " conv1 (stem)", g0, b0, s.mean, s.invstd, s.scale, s.shift)
    N = s.x.shape[0]
    for n0 in range(0, N, 64):   # image chunks: the visual tail's references stay at a few GB
        sl = slice(n0, min(N, n0 + 64))
        py, pi, pxm = tail_fwd_ref(s.x[sl], s.scale, s.shift)
        check_exact(tag + " stem tail pool_y", eng.pool_y[sl], py, ulps)
        bad = eng.pool_idx[sl] != pi
        assert not bool(bad.any()), "%s stem tail pool_idx: %d differ, first at %s" % (
            tag, int(bad.sum()), _at(pi, int(bad.flatten().nonzero()[0])))
        assert torch.equal(eng.pool_xmax[sl], pxm), tag + " stem tail pool_xmax"
        del py, pi, pxm
    # residual blocks
    inp = eng.pool_y
    for (u1, u2, ud) in eng.blocks:
        units = [(u1, inp, None, True)]
        if ud is not None:
            units.append((ud, inp, None, False))
        units.append((u2, u1.y, ud.y if ud is not None else inp, True))
        for u, src, res, relu in units:
            name = "%s %s" % (tag, u.name)
            w, g0, b0, rm0, rv0 = snap[u.conv]
            check_conv(name, u.x, conv_nhwc(src, w.to(BF).float(), u.conv.stride[0], u.conv.padding[0]))
            check_stats(name, u.x, u.C, u.mean, u.invstd, u.bn.running_mean, u.bn.running_var, rm0, rv0,
                        epilogue=True)
            check_affine(name, g0, b0, u.mean, u.invstd, u.scale, u.shift)
            check_exact(name + " y", u.y, apply_ref(u.x, u.scale, u.shift, res, relu), ulps)
        inp = u2.y
    return inp


def _audit_eval(tag, eng, x_src, ulps):
    """forward_eval: BatchNorm folded with the (post-step) running statistics, bf16(w * scale) weights, shift as
    the conv epilogue's bias (with the residual add and the ReLU)."""
    eng.forward_eval()
    torch.cuda.synchronize()
    for u in eng.units:
        gamma, beta, rm, rv = (t.detach().double() for t in (u.bn.weight, u.bn.bias, u.bn.running_mean,
                                                               u.bn.running_var))
        sc = gamma / (rv + u.bn.eps).sqrt()
        check_bound("%s eval %s scale" % (tag, u.name), u.scale_e, sc, 1e-6 * sc.abs())
        check_bound("%s eval %s shift" % (tag, u.name), u.shift_e, beta - rm * sc,
                    1e-6 * (beta.abs() + (rm * sc).abs()) + 1e-30)

    def wfold(u):
        return (u.conv.weight.detach() * u.scale_e.view(-1, 1, 1, 1)).to(BF).float()

    s = eng.stem
    xb = x_src.to(BF).float()
    check_conv(tag + " eval conv1 (stem)", s.x, F.conv2d(xb, wfold(s), stride=2, padding=3).permute(0, 2, 3, 1))
    del xb
    ones = torch.ones(64, device=s.x.device)
    N = s.x.shape[0]
    for n0 in range(0, N, 64):
        sl = slice(n0, min(N, n0 + 64))
        py, pi, _ = tail_fwd_ref(s.x[sl], ones, s.shift_e)
        check_exact(tag + " eval stem tail pool_y", eng.pool_y[sl], py, ulps)
        assert torch.equal(eng.pool_idx[sl], pi), tag + " eval stem tail pool_idx"
        del py, pi
    inp = eng.pool_y
    for (u1, u2, ud) in eng.blocks:
        units = [(u1, inp, None, True)]
        if ud is not None:
            units.append((ud, inp, None, False))
        units.append((u2, u1.y, ud.y if ud is not None else inp, True))
        for u, src, res, relu in units:
            c = conv_nhwc(src, wfold(u), u.conv.stride[0], u.conv.padding[0])
            ref = c + u.shift_e
            if res is not None:
                ref = ref + res.float()
            if relu:
                ref = torch.relu(ref)
            rms = c.double().pow(2).mean().sqrt().item()
            check_bound("%s eval %s y" % (tag, u.name), u.y.float(), ref, ref.abs() * ULP + 1e-3 * rms)
            assert rel_l2(u.y.float(), ref) < 6e-3, "%s eval %s y" % (tag, u.name)
            del c, ref
        inp = u2.y


@pytest.mark.parametrize("dataset,B", AUDIT_CONFIGS)
def test_step_forward_audit(dataset, B):
    """One real concat training step at full size; every stored forward tensor of both encoders is checked against
    a reference computed from the stored input of its own layer (the kernel at its real geometry, sweep direction,
    stream and buffer), then the eval-mode forward on the same engines."""
    from oracle.synth import make_batch
    from gdl_b200.shapes import HEAD_WIDTH, LABEL_MAX
    from test_gpu_step import build
    model, step = build("concat", dataset, B, dataset, lr=0.01)
    try:
        engines = {"audio": step.enc_a, "visual": step.enc_v}
        for name, eng in engines.items():
            assert _units_geoms(eng) == sorted(UNIT_GEOMS[(dataset, name)]), (name, _units_geoms(eng))
            s = eng.stem
            assert (s.N, s.Ho, s.Wo) == STEM_TAILS[(dataset, name)]
        snap = {}
        for eng in engines.values():
            for u in eng.units:
                bn = u.bn
                snap[u.conv] = tuple(t.detach().clone() for t in (u.conv.weight, bn.weight, bn.bias,
                                                                  bn.running_mean, bn.running_var))
        spec, image, label = make_batch(B, HEAD_WIDTH[dataset], dataset, seed=5, label_max=LABEL_MAX[dataset])
        spec, image, label = spec.cuda(), image.cuda(), label.cuda()
        step.step(spec, image, label)
        torch.cuda.synchronize()
        ulps = {}
        for name, eng in engines.items():
            x_src = _encoder_input(name, spec, image)
            fmap = _audit_train("%s %s" % (dataset, name), eng, x_src, snap, ulps)
            feat = step.a_feat if name == "audio" else step.v_feat
            f = fmap.reshape(B, -1, 512).double()
            check_bound("%s %s pooled features" % (dataset, name), feat, f.mean(1), 1e-5 * f.abs().mean(1) + 1e-30)
        for name, eng in engines.items():   # last: forward_eval overwrites stem.x, pool_y and every u.y
            _audit_eval("%s %s" % (dataset, name), eng, _encoder_input(name, spec, image), ulps)
        print("%s B=%d: elements one bf16 ulp off: %s" % (dataset, B, ulps or "none"))
    finally:
        del model, step
        _free()


# ---------------------------------------------------------------------------------- 2. BatchNorm in both sweeps
UNIT_CASES = sorted({g for v in UNIT_GEOMS.values() for g in v})
TAIL_CASES = sorted(set(STEM_TAILS.values()))
APPLY_MODES = [(1, 0), (1, 1), (0, 0)]   # (relu, residual): conv1, conv2, downsample


def _bn_inputs(P, C, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    r = lambda *s: torch.randn(*s, device="cuda", generator=g)
    return SimpleNamespace(
        x=(r(P, C) * 2 + 0.5).to(BF), res=r(P, C).to(BF), dy=r(P, C).to(BF),
        gamma=torch.rand(C, device="cuda", generator=g) + 0.5, beta=r(C) * 0.1,
        rm0=r(C) * 0.1, rv0=torch.rand(C, device="cuda", generator=g) + 0.5)


def _nan(*shape, dtype=torch.float32):
    return torch.full(shape, float("nan"), device="cuda", dtype=dtype)


def _run_bn(ops, t, P, C, sweep, stats=None):
    """Every BatchNorm kernel of a block unit with the sweep hint set, outputs pre-filled with NaN.  stats: the
    (mean, invstd, scale, shift) the apply and backward kernels use instead of this run's own bn_stats outputs."""
    o = SimpleNamespace()
    ops.sweep(sweep)
    try:
        partial = _nan(ops.bn_partial_floats(P, C))
        o.mean, o.invstd, o.scale, o.shift = (_nan(C) for _ in range(4))
        o.rm, o.rv = t.rm0.clone(), t.rv0.clone()
        ops.bn_stats(t.x, P, C, partial, t.gamma, t.beta, EPS, MOMENTUM, o.rm, o.rv, o.mean, o.invstd, o.scale,
                     o.shift)
        mean, invstd, scale, shift = stats or (o.mean, o.invstd, o.scale, o.shift)
        o.y = {}
        for relu, use_res in APPLY_MODES:
            o.y[(relu, use_res)] = _nan(P, C, dtype=BF)
            ops.bn_apply(t.x, t.res if use_res else None, o.y[(relu, use_res)], P, C, scale, shift, relu)
        o.dz, o.dx = _nan(P, C, dtype=BF), _nan(P, C, dtype=BF)      # conv2: mask from y, dz written
        o.dg, o.db = _nan(C), _nan(C)
        ops.bn_bwd(t.dy, o.y[(1, 1)], t.x, o.dz, o.dx, P, C, t.gamma, mean, invstd, partial, o.dg, o.db, 1)
        o.dx0, o.dg0, o.db0 = _nan(P, C, dtype=BF), _nan(C), _nan(C)  # downsample: no ReLU
        ops.bn_bwd(t.dy, None, t.x, None, o.dx0, P, C, t.gamma, mean, invstd, partial, o.dg0, o.db0, 0)
        o.dxn, o.dgn, o.dbn = _nan(P, C, dtype=BF), _nan(C), _nan(C)  # conv1: mask recomputed from x
        ops.bn_bwd_nores(t.dy, t.x, o.dxn, P, C, t.gamma, mean, invstd, scale, shift, partial, o.dgn, o.dbn)
    finally:
        ops.sweep(0)
    torch.cuda.synchronize()
    return o


@pytest.mark.parametrize("sweep", [0, 1])
@pytest.mark.parametrize("P,C", UNIT_CASES)
def test_bn_unit_kernels_at_step_geometry(ops, P, C, sweep):
    """bn_stats, bn_apply (three modes), bn_bwd (with and without ReLU) and bn_bwd_nores against fp64."""
    t = _bn_inputs(P, C, seed=P % 9973 + C)
    o = _run_bn(ops, t, P, C, sweep)
    tag = "P%d C%d sweep %d" % (P, C, sweep)
    check_stats(tag, t.x, C, o.mean, o.invstd, o.rm, o.rv, t.rm0, t.rv0)
    check_affine(tag, t.gamma, t.beta, o.mean, o.invstd, o.scale, o.shift)
    for (relu, use_res), y in o.y.items():
        check_exact("%s apply relu %d res %d" % (tag, relu, use_res), y,
                    apply_ref(t.x, o.scale, o.shift, t.res if use_res else None, relu))
    mask = o.y[(1, 1)].float() > 0
    dz = torch.where(mask, t.dy.float(), 0.0).to(BF)
    check_exact(tag + " bn_bwd dz", o.dz, dz)
    check_bn_bwd(tag + " bn_bwd", o.dg, o.db, o.dx, dz, t.x, t.gamma, o.mean, o.invstd)
    check_bn_bwd(tag + " bn_bwd no relu", o.dg0, o.db0, o.dx0, t.dy, t.x, t.gamma, o.mean, o.invstd)
    dzn = torch.where(torch.addcmul(o.shift, t.x.float(), o.scale) > 0, t.dy.float(), 0.0)
    check_bn_bwd(tag + " bn_bwd_nores", o.dgn, o.dbn, o.dxn, dzn, t.x, t.gamma, o.mean, o.invstd)


def _same_sums(name, a, b, abs_sum):
    check_bound(name, a, b.double(), 1e-5 * abs_sum + 1e-30)


def _same_up_to_ulp(name, a, b):
    """bf16 results of the same arithmetic on reductions that differ in the last fp32 bits: within one ulp, or
    1e-5 rms where the per-element terms cancel to near zero, and rarely different at all."""
    rms = a.double().pow(2).mean().sqrt()
    one_ulp = 2 * ULP * torch.maximum(a.double().abs(), b.double().abs())   # a bf16 ulp is at most 2^-7 |x|
    check_bound(name, b, a.double(), one_ulp + 1e-5 * rms)
    d = (a.float() != b.float())
    frac = d.float().mean().item()
    print("%s: %.3g of the elements one ulp apart" % (name, frac))
    assert frac <= 1e-3, (name, frac)


@pytest.mark.parametrize("P,C", UNIT_CASES)
def test_bn_unit_kernels_sweep_invariance(ops, P, C):
    """Element-wise outputs are bit-identical in both directions; reductions agree to fp32 reordering.  Both
    directions' apply and backward kernels get the statistics of the ascending run, so their inputs are identical."""
    t = _bn_inputs(P, C, seed=P % 9973 + C)
    o0 = _run_bn(ops, t, P, C, 0)
    o1 = _run_bn(ops, t, P, C, 1, stats=(o0.mean, o0.invstd, o0.scale, o0.shift))
    for k in o0.y:
        assert torch.equal(o0.y[k], o1.y[k]), ("bn_apply", k)
    assert torch.equal(o0.dz, o1.dz)
    absx = t.x.float().abs().sum(0).double()
    _same_sums("mean", o0.mean * P, o1.mean * P, absx)
    check_bound("invstd", o1.invstd, o0.invstd.double(), 1e-5 * o0.invstd.double())
    ady = t.dy.float().abs()
    axd = (t.x.float().abs() + o0.mean.abs()) * o0.invstd
    for a, b in ((o0.dg, o1.dg), (o0.dg0, o1.dg0), (o0.dgn, o1.dgn)):
        _same_sums("dgamma", a, b, (ady * axd).sum(0).double())
    for a, b in ((o0.db, o1.db), (o0.db0, o1.db0), (o0.dbn, o1.dbn)):
        _same_sums("dbeta", a, b, ady.sum(0).double())
    for k in ("dx", "dx0", "dxn"):
        _same_up_to_ulp(k, getattr(o0, k), getattr(o1, k))


def _tail_inputs(N, H, W, seed):
    C = 64
    g = torch.Generator(device="cuda").manual_seed(seed)
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    return SimpleNamespace(
        x=(torch.randn(N, H, W, C, device="cuda", generator=g) * 2 + 0.3).to(BF),
        gp=torch.randn(N, Ho, Wo, C, device="cuda", generator=g).to(BF),
        gamma=torch.rand(C, device="cuda", generator=g) + 0.5,
        beta=torch.randn(C, device="cuda", generator=g) * 0.1, Ho=Ho, Wo=Wo)


def _run_tail(ops, t, N, H, W, sweep):
    C, Ho, Wo, P = 64, t.Ho, t.Wo, N * H * W
    o = SimpleNamespace()
    partial = _nan(ops.bn_partial_floats(P, C))
    o.mean, o.invstd, o.scale, o.shift = (_nan(C) for _ in range(4))
    ops.bn_stats(t.x, P, C, partial, t.gamma, t.beta, EPS, MOMENTUM, None, None, o.mean, o.invstd, o.scale, o.shift)
    ops.sweep(sweep)
    try:
        o.y, o.idx, o.xm = _nan(N, Ho, Wo, C, dtype=BF), torch.full((N, Ho, Wo, C), 255, device="cuda",
                                                                     dtype=torch.uint8), _nan(N, Ho, Wo, C, dtype=BF)
        ops.bn_relu_maxpool_fwd(t.x, o.scale, o.shift, o.y, o.idx, o.xm, N, H, W, C, Ho, Wo)
        o.y2, o.idx2 = _nan(N, Ho, Wo, C, dtype=BF), torch.full_like(o.idx, 255)
        ops.bn_relu_maxpool_fwd(t.x, o.scale, o.shift, o.y2, o.idx2, None, N, H, W, C, Ho, Wo)
        o.bwd = {}
        for use_xmax in (True, False):
            dx, dg, db = _nan(N, H, W, C, dtype=BF), _nan(C), _nan(C)
            ops.bn_relu_maxpool_bwd(t.gp, o.idx, o.xm if use_xmax else None, t.x, dx, N, H, W, C, Ho, Wo, t.gamma,
                                    o.mean, o.invstd, o.scale, o.shift, partial, dg, db)
            o.bwd[use_xmax] = (dx, dg, db)
    finally:
        ops.sweep(0)
    torch.cuda.synchronize()
    return o


@pytest.mark.parametrize("sweep", [0, 1])
@pytest.mark.parametrize("N,H,W", TAIL_CASES)
def test_stem_tail_at_step_geometry(ops, N, H, W, sweep):
    """bn_relu_maxpool_fwd (with and without xmax) and _bwd (sums over the stem grid, or over the pooled grid
    through xmax) against max_pool2d of the rounded BN+ReLU output and an fp64 BatchNorm backward."""
    t = _tail_inputs(N, H, W, seed=N + H + W)
    o = _run_tail(ops, t, N, H, W, sweep)
    tag = "N%d %dx%d sweep %d" % (N, H, W, sweep)
    py, pi, pxm = tail_fwd_ref(t.x, o.scale, o.shift)
    for y, idx in ((o.y, o.idx), (o.y2, o.idx2)):
        check_exact(tag + " pool_y", y, py)
        bad = idx != pi
        assert not bool(bad.any()), "%s arg-max: %d differ, first at %s" % (
            tag, int(bad.sum()), _at(pi, int(bad.flatten().nonzero()[0])))
    assert torch.equal(o.xm, pxm), tag + " xmax"
    del py, pxm
    g = tail_scatter_ref(t.gp, pi, H, W)                   # exact per-pixel sum of the windows' gradients
    mask = torch.addcmul(o.shift, t.x.float(), o.scale) > 0
    dz = torch.where(mask, g, 0.0)
    del g
    # a pixel that is the arg-max of several windows: the kernels may round its summed gradient to bf16
    slack = (dz - dz.to(BF).double()).abs()
    for use_xmax, (dx, dg, db) in o.bwd.items():
        check_bn_bwd("%s bwd xmax %d" % (tag, use_xmax), dg, db, dx, dz, t.x, t.gamma, o.mean, o.invstd, slack)


@pytest.mark.parametrize("N,H,W", TAIL_CASES)
def test_stem_tail_sweep_invariance(ops, N, H, W):
    t = _tail_inputs(N, H, W, seed=N + H + W)
    o0, o1 = (_run_tail(ops, t, N, H, W, s) for s in (0, 1))
    for k in ("y", "idx", "xm", "y2", "idx2"):
        assert torch.equal(getattr(o0, k), getattr(o1, k)), k
    ag = t.gp.float().abs()
    for use_xmax in (True, False):
        (dx0, dg0, db0), (dx1, dg1, db1) = o0.bwd[use_xmax], o1.bwd[use_xmax]
        _same_sums("dbeta", db0, db1, ag.reshape(-1, 64).sum(0).double())
        axm = ((o0.xm.float().abs() + o0.mean.abs()) * o0.invstd).reshape(-1, 64)
        _same_sums("dgamma", dg0, dg1, (ag.reshape(-1, 64) * axm).sum(0).double())
        _same_up_to_ulp("dx xmax %d" % use_xmax, dx0, dx1)


# ---------------------------------------------------------------------------------- 4. the chunked FiLM head
def _film_ref(a, v, W1, b1, W2, b2, label, alpha, rounded, dH_in=None):
    """fp64 restatement of the FiLM_DGL routing (oracle.dgl_oracle.fusion_forward, film): Lf trains fc_out and fc
    (dW1, db1) from the detached a (x) v; the unimodal losses only produce dH_a, dH_v, which feed da / dv.
    rounded=True rounds where the kernels round: the outer products, W1t, dHfT, dHs and G to bf16.
    dH_in: the head's own fp32 [3, B, D] dH_f / dH_a / dH_v for the backward (the input of the bf16 casts)."""
    B, D = a.shape
    q = (lambda t: t.to(BF).double()) if rounded else (lambda t: t.double())
    outer = lambda x, y: (x[:, :, None] * y[:, None, :]).reshape(B, D * D)   # fp32 product, as the kernel forms it
    if rounded:
        Z = [q(outer(a, v)), q(outer(a, a)), q(outer(v, v))]
    else:
        a64, v64 = a.double(), v.double()
        Z = [outer(a64, v64), outer(a64, a64), outer(v64, v64)]
    W1q = q(W1)
    H = [z @ W1q.t() + b1.double() for z in Z]
    logits = [h @ W2.double().t() + b2.double() for h in H]
    onehot = F.one_hot(label, W2.shape[0]).double()
    losses, dl = [], []
    for i, lg in enumerate(logits):
        p = torch.softmax(lg, 1)
        losses.append(-(torch.log_softmax(lg, 1) * onehot).sum(1).mean())
        dl.append((p - onehot) / B * (1.0 if i == 0 else alpha))
    r = SimpleNamespace(H=torch.cat(H), logits=torch.stack(logits), losses=torch.stack(losses),
                        dH=torch.stack([d @ W2.double() for d in dl]))
    dH = r.dH if dH_in is None else dH_in.double()
    r.dW2, r.db2 = dl[0].t() @ H[0], dl[0].sum(0)
    r.db1 = dH[0].sum(0)
    r.dW1 = q(dH[0]).t() @ Z[0]
    del Z
    for name, dh, x in (("da", dH[1], a), ("dv", dH[2], v)):
        G = W1q.t() @ q(dh).t()                               # [F2, B]: bf16 output of the kernel's GEMM
        G = (G.to(BF).double() if rounded else G).view(D, D, B)   # [i, j, b]: feature i*D + j
        x64 = x.double()
        setattr(r, name, torch.einsum("ijb,bj->bi", G, x64) + torch.einsum("ijb,bi->bj", G, x64))
        G2, x2 = G.pow(2), x64.pow(2)                         # root sum of squares of the contraction's terms
        setattr(r, name + "_rss", (torch.einsum("ijb,bj->bi", G2, x2) + torch.einsum("ijb,bi->bj", G2, x2)).sqrt())
        del G, G2
    return r


def _check_rel(name, got, ref, tol):
    ref = ref.double()
    rel = rel_l2(got, ref)
    assert rel < tol, "%s: relative L2 %.3g > %g" % (name, rel, tol)
    rms = ref.pow(2).mean().sqrt()
    check_bound(name, got, ref, tol * (ref.abs() + rms))


@pytest.mark.parametrize("B,n", [(16, 6), (64, 34), (256, 6)])
def test_film_head_train_chunked(ops, B, n):
    """FilmHead.train (the fused step's FiLM head: chunked outer products, H accumulated with gemm_tn_f32_acc,
    dW1 windows through transpose_bf16_to_f32_window, film_contract_chunk with sum_mode, c0 = B and acc / rebuild)
    against the fp64 routing of the reference, once rounded where the kernels round and once unrounded."""
    from gdl_b200 import film
    from gdl_b200.film import D, F2, FC, FilmFn, FilmHead
    dev = torch.device("cuda")
    g = torch.Generator(device="cuda").manual_seed(B + n)
    r = lambda *s: torch.randn(*s, device="cuda", generator=g)
    fm = SimpleNamespace(fc=torch.nn.Linear(F2, D, device=dev), fc_out=torch.nn.Linear(D, n, device=dev))
    with torch.no_grad():
        fm.fc.weight.copy_(r(D, F2) * 2e-3)
        fm.fc.bias.copy_(r(D) * 0.1)
        fm.fc_out.weight.copy_(r(n, D) * 0.05)
        fm.fc_out.bias.copy_(r(n) * 0.1)
    for p in (fm.fc.weight, fm.fc.bias, fm.fc_out.weight, fm.fc_out.bias):
        p.grad = torch.full_like(p, float("nan"))
    head = FilmHead(fm, B, n, dev)
    alpha = 4.0
    a = torch.rand(B, D, device="cuda", generator=g)        # pooled ReLU features: non-negative
    v = torch.rand(B, D, device="cuda", generator=g)
    label = torch.randint(0, n, (B,), device="cuda", generator=g)
    st = SimpleNamespace(a_feat=a, v_feat=v, label_in=label, logits=_nan(3, B, n), losses=_nan(3),
                         da=_nan(B, D), dv=_nan(B, D), alpha=alpha, inv_batch=1.0 / B)
    head.train(st)
    torch.cuda.synchronize()
    W1, b1, W2, b2 = (t.detach() for t in (fm.fc.weight, fm.fc.bias, fm.fc_out.weight, fm.fc_out.bias))
    tag = "B%d n%d" % (B, n)

    # rounded tier: the backward starts from the head's stored fp32 dH, so a bf16 cast of it rounds the same way here
    ref = _film_ref(a, v, W1, b1, W2, b2, label, alpha, rounded=True, dH_in=head.dH)
    _check_rel(tag + " H", head.buf.H[:3 * B], ref.H, 1e-4)
    _check_rel(tag + " dH", head.dH, ref.dH, 1e-4)
    _check_rel(tag + " logits", st.logits, ref.logits, 1e-4)
    _check_rel(tag + " losses", st.losses, ref.losses, 1e-4)
    _check_rel(tag + " fc_out.weight grad", fm.fc_out.weight.grad, ref.dW2, 1e-4)
    _check_rel(tag + " fc_out.bias grad", fm.fc_out.bias.grad, ref.db2, 1e-4)
    _check_rel(tag + " fc.bias grad", fm.fc.bias.grad, ref.db1, 1e-4)
    for c in range(F2 // FC):   # one dW1 window per chunk: bf16 GEMM tile (K = B, fp32 accumulation)
        win = slice(c * FC, (c + 1) * FC)
        rw = ref.dW1[:, win]
        rms = rw.pow(2).mean().sqrt()
        check_bound("%s fc.weight grad window %d" % (tag, c), fm.fc.weight.grad[:, win], rw,
                    rw.abs() * ULP + 1e-3 * rms)
    # G is rounded to bf16 from fp32 sums in the kernel and from fp64 sums here: where the two straddle a rounding
    # boundary a term of the contraction moves by one ulp, at most 2^-7 of the terms' root sum of squares
    for name in ("da", "dv"):
        got, want = getattr(st, name), getattr(ref, name)
        assert rel_l2(got, want) < 1e-3, (tag, name, rel_l2(got, want))
        check_bound("%s %s" % (tag, name), got, want, 1e-3 * want.abs() + 2 * ULP * getattr(ref, name + "_rss"))
    del ref
    _free()

    ref = _film_ref(a, v, W1, b1, W2, b2, label, alpha, rounded=False)
    assert rel_l2(head.buf.H[:3 * B], ref.H) < 6e-3
    assert rel_l2(st.logits, ref.logits) < 6e-3 and rel_l2(st.losses, ref.losses) < 6e-3
    for name, got, want in (("fc.weight", fm.fc.weight.grad, ref.dW1), ("fc.bias", fm.fc.bias.grad, ref.db1),
                            ("fc_out.weight", fm.fc_out.weight.grad, ref.dW2), ("da", st.da, ref.da),
                            ("dv", st.dv, ref.dv)):
        assert rel_l2(got, want) < 1e-2, (tag, name, rel_l2(got, want))
    del ref
    _free()

    # the chunked forward == the whole-operand FilmFn forward, to fp32 reordering
    h = FilmFn.apply(a, v, W1, b1)
    torch.cuda.synchronize()
    Hc = head.buf.H[:B]
    zb = (a[:, :, None] * v[:, None, :]).reshape(B, F2).to(BF).double().abs()
    bound = 1e-5 * (zb @ W1.to(BF).double().abs().t() + b1.double().abs())
    del zb
    check_bound(tag + " chunked vs whole-operand H", Hc, h.double(), bound)
    assert film.CHUNK_I * D == FC
    del head, fm
    _free()
