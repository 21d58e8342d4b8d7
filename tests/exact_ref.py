"""Exact references for the convolution, stem and FiLM GEMM kernels (no GPU needed to import or run).

A reduction kernel is free to add its terms in any order: tile order, split-K split, CTA-pair half, chunk order.  A
tolerance wide enough for every order is about sqrt(n) looser than one term of an n-term sum, so it cannot see a
dropped partial or a wrong tap.  These helpers remove the tolerance instead, by drawing operands whose every partial
sum is exact in fp32.

Exactness criterion.  Let every element of operand A be an integer multiple of 2^qa and every element of B a multiple
of 2^qb.  If, for every output element, sum_k |a_k b_k| (plus |addend| for a fused residual or bias) is below
2^20 * 2^(qa + qb), every partial sum any summation order can form is a multiple of 2^(qa + qb) below 2^20 of them:
exact in fp32, whatever the order.  The kernel must then equal the float64 reference bit for bit (bf16 outputs: the
exact value rounded once, to nearest even, as __floats2bfloat162_rn does).  2^20 rather than 2^24 leaves 4 bits of
margin for the tensor core's internal alignment of a K group.  `check_criterion` asserts the bound from the same
float64 reference run on |A| and |B|; it is never assumed.

Two operand families satisfy it:
  I (integer)   entries in {-1, 0, +1}, the zero probability chosen per call: sees every index;
  M (mantissa)  the dense operand has all 8 bf16 significand bits random and exponents in [-2, 1]; the other operand is
                sparse powers of two +-2^k, k in [-3, 0], with at most ~16 nonzeros per output's reduction, placed at
                the first and last pixel, image seams, the last row and column and the last partial tile as well:
                catches mantissa and rounding-mode handling that integers cannot.

References are per-tap shifted views and float64 matmuls (no cuDNN, TF32 or im2col), chunked over images so a
visual layer-1 reference at N = 768 stays at a few GB.  Activations are NHWC, weights OIHW."""
import torch

BF = torch.bfloat16
F64 = torch.float64
EXACT_BITS = 20
Q_I = 0          # family I: integers
Q_DENSE = -9     # family M dense: (1 + m / 128) 2^e, e >= -2  ->  multiples of 2^-9
Q_SPARSE = -3    # family M sparse: +-2^k, k >= -3
IMG_CHUNK_ELEMS = 1 << 26   # float64 elements per reference chunk (512 MB)


# ---------------------------------------------------------------------------------- operand generators
def _gen(seed, device):
    return torch.Generator(device=device).manual_seed(int(seed))


def ternary(shape, p_nonzero, seed, device="cpu"):
    """Family I: +-1 with probability p_nonzero, else 0 (float32; exact in bf16)."""
    g = _gen(seed, device)
    u = torch.rand(shape, generator=g, device=device)
    s = torch.rand(shape, generator=g, device=device)
    return torch.where(u < p_nonzero, torch.where(s < 0.5, -1.0, 1.0), 0.0)


def mantissa_dense(shape, seed, device="cpu"):
    """Family M dense operand: +-(1 + m/128) 2^e, m uniform in 0..127, e uniform in [-2, 1] (bf16-exact float32)."""
    g = _gen(seed, device)
    m = torch.randint(0, 128, shape, generator=g, device=device).float()
    e = torch.randint(-2, 2, shape, generator=g, device=device).float()
    s = torch.randint(0, 2, shape, generator=g, device=device).float() * 2 - 1
    return s * (1 + m / 128) * torch.exp2(e)


def pow2_values(n, seed, device="cpu"):
    """n sparse-operand values +-2^k, k uniform in [-3, 0]."""
    g = _gen(seed, device)
    k = torch.randint(-3, 1, (n,), generator=g, device=device).float()
    s = torch.randint(0, 2, (n,), generator=g, device=device).float() * 2 - 1
    return s * torch.exp2(k)


def sparse_rows(rows, length, nnz, seed, device="cpu", must=()):
    """[rows, length] float32, each row with at most nnz nonzeros +-2^k.  `must`: positions (those inside the row) that
    are spread round-robin over the rows (each lands in at least one row when rows * nnz allows)."""
    g = _gen(seed, device)
    out = torch.zeros(rows, length, device=device)
    must = [int(m) for m in must if 0 <= int(m) < length]
    vals = pow2_values(rows * nnz, seed + 1, device).view(rows, nnz)
    for r in range(rows):
        pos = torch.randint(0, length, (nnz,), generator=g, device=device)
        forced = must[r::rows][:nnz]
        if forced:
            pos[:len(forced)] = torch.tensor(forced, device=device)
        out[r, pos] = vals[r, :len(pos)]   # a repeated position keeps one value: still at most nnz nonzeros
    return out


def special_pixels(N, H, W, tile=128):
    """Flat pixel indices (n*H + h)*W + w where kernels go wrong: first and last pixel, both sides of every image seam
    (first images only), the last row and column of the first and last image, and the last partial 128-pixel tile."""
    P = N * H * W
    s = {0, P - 1}
    for n in range(min(N, 4)):
        s.update({n * H * W, n * H * W + H * W - 1})
    for n in {0, N - 1}:
        base = n * H * W
        s.update(base + (H - 1) * W + w for w in range(0, W, max(1, W // 4)))
        s.update(base + h * W + W - 1 for h in range(0, H, max(1, H // 4)))
    s.update(range(P - 1, max(P - (P % tile or tile), 0) - 1, -max(1, (P % tile or tile) // 4)))
    return sorted(p for p in s if 0 <= p < P)


def conv_weights_sparse(Co, Ci, R, S, nnz, seed, device="cpu"):
    """Family M sparse weights: each output channel with at most nnz nonzero (ci, r, s), every tap used somewhere."""
    RS = R * S
    must = [(t * Ci + (t * 7) % Ci) for t in range(RS)]          # (tap, ci) flat: tap-major
    w = sparse_rows(Co, RS * Ci, nnz, seed, device, must=must)     # [Co][(r, s, ci)]
    return w.view(Co, R, S, Ci).permute(0, 3, 1, 2).contiguous()


# ---------------------------------------------------------------------------------- the criterion
def is_multiple(t, q):
    """Every element of t is an integer multiple of 2^q (checked in float64: scaling by a power of two is exact)."""
    x = t.double() * 2.0 ** (-q)
    return bool(torch.equal(x, torch.round(x)))


def check_criterion(name, abs_sum, q):
    """Assert that every output's sum of |terms| is below 2^20 * 2^q, so that every partial sum is exact in fp32.
    A draw that violates it is a bug of the test, not of the kernel: fail loudly."""
    m = float(abs_sum.max()) if abs_sum.numel() else 0.0
    lim = 2.0 ** (EXACT_BITS + q)
    if not m < lim:
        raise AssertionError("%s: operand draw violates the exactness criterion: max sum |terms| = %r >= 2^%d * 2^%d"
                             % (name, m, EXACT_BITS, q))
    return m


def check_operands(name, pairs):
    """pairs: [(tensor, q)]: every tensor is a multiple of its 2^q (else the criterion's premise is false)."""
    for i, (t, q) in enumerate(pairs):
        if not is_multiple(t, q):
            raise AssertionError("%s: operand %d is not a multiple of 2^%d" % (name, i, q))


def bf16_ref(ref, name="", min_exact=0.99):
    """The exact float64 result rounded once to bf16 (round to nearest even).  Asserts that the value is exact in fp32
    (so float64 -> fp32 -> bf16 rounds once) and that >= min_exact of the outputs are exact in bf16, so a single
    wrong term is visible and not rounded away."""
    f = ref.float()
    assert torch.equal(f.double(), ref), name + ": the exact result is not representable in fp32"
    b = f.to(BF)
    frac = (b.double() == ref).double().mean().item() if ref.numel() else 1.0
    assert frac >= min_exact, "%s: only %.4f of the reference outputs are exact in bf16" % (name, frac)
    return b


# ---------------------------------------------------------------------------------- comparator
def at(shape, k):
    """Multi-index of flat index k in a tensor of `shape`."""
    idx = []
    for s in reversed(shape):
        idx.append(k % s)
        k //= s
    return tuple(reversed(idx))


def mismatches(got, ref):
    """(count, first multi-index, worst multi-index) of the elements where got != ref as values (-0 == +0; NaN in got
    or ref differs from anything; the worst is a NaN if there is one, else the largest |got - ref|)."""
    assert tuple(got.shape) == tuple(ref.shape), (tuple(got.shape), tuple(ref.shape))
    g, r = got.double().flatten(), ref.double().flatten()
    bad = ~(g == r)
    n = int(bad.sum())
    if n == 0:
        return 0, None, None
    first = int(bad.nonzero()[0])
    err = (g - r).abs()
    err = torch.where(torch.isnan(err), torch.tensor(float("inf"), dtype=F64, device=err.device), err)
    err = torch.where(bad, err, torch.zeros_like(err))
    worst = int(err.argmax())
    return n, at(got.shape, first), at(got.shape, worst)


def check_bits(name, got, ref):
    """Bit-exact comparison (values; -0 == +0).  ref: the expected tensor in got's dtype."""
    assert got.dtype == ref.dtype, (name, got.dtype, ref.dtype)
    n, first, worst = mismatches(got, ref)
    if n:
        raise AssertionError("%s: %d of %d elements differ; first at %s: got %r ref %r; worst at %s: got %r ref %r" % (
            name, n, got.numel(), first, got[first].item(), ref[first].item(), worst, got[worst].item(),
            ref[worst].item()))


# ---------------------------------------------------------------------------------- float64 references
def _out_hw(H, W, R, S, stride, pad):
    return (H + 2 * pad - R) // stride + 1, (W + 2 * pad - S) // stride + 1


def _img_chunk(per_image_elems):
    return max(1, IMG_CHUNK_ELEMS // max(1, per_image_elems))


def _tap(xp, r, s, Ho, Wo, stride):
    return xp[:, r:r + stride * (Ho - 1) + 1:stride, s:s + stride * (Wo - 1) + 1:stride, :]


def _pad_nhwc(x, pad, Hp, Wp):
    N, H, W, C = x.shape
    xp = x.new_zeros(N, Hp, Wp, C)
    xp[:, pad:pad + H, pad:pad + W] = x
    return xp


def conv_fwd_ref(x, w, stride, pad, device=None):
    """y[n, ho, wo, co] = sum_{ci, r, s} x[n, ho*stride - pad + r, wo*stride - pad + s, ci] w[co, ci, r, s], float64.
    x NHWC (any float dtype), w OIHW.  The sum runs in float64 on `device` (default x's)."""
    dev = device or x.device
    N, H, W, Ci = x.shape
    Co, Ciw, R, S = w.shape
    assert Ciw == Ci, (Ciw, Ci)
    Ho, Wo = _out_hw(H, W, R, S, stride, pad)
    Hp, Wp = max(H + 2 * pad, stride * (Ho - 1) + R), max(W + 2 * pad, stride * (Wo - 1) + S)
    wt = w.to(dev, F64).permute(2, 3, 1, 0).contiguous()        # [R][S][Ci][Co]
    y = torch.empty(N, Ho, Wo, Co, dtype=F64, device=dev)
    nc = _img_chunk(Hp * Wp * Ci + Ho * Wo * (Ci + Co))
    for n0 in range(0, N, nc):
        xp = _pad_nhwc(x[n0:n0 + nc].to(dev, F64), pad, Hp, Wp)
        acc = torch.zeros(xp.shape[0], Ho, Wo, Co, dtype=F64, device=dev)
        for r in range(R):
            for s in range(S):
                acc += torch.matmul(_tap(xp, r, s, Ho, Wo, stride), wt[r, s])
        y[n0:n0 + nc] = acc
        del xp, acc
    return y


def conv_dgrad_ref(dy, w, Hi, Wi, stride, pad, add=None, add_mode=0, device=None):
    """dx[n, hi, wi, ci] = sum over the (ho, wo, r, s) with hi = ho*stride - pad + r ... of dy[n, ho, wo, co] w[co, ci,
    r, s], float64; add_mode 1 adds `add` (dx's shape), add_mode 2 adds `add` [N, ceil(Hi/2), ceil(Wi/2), Ci] at even
    (hi, wi) only (the compact-grid gradient of a 1x1 stride-2 downsample)."""
    dev = device or dy.device
    N, Ho, Wo, Co = dy.shape
    Cow, Ci, R, S = w.shape
    assert Cow == Co
    Hp, Wp = max(Hi + 2 * pad, stride * (Ho - 1) + R), max(Wi + 2 * pad, stride * (Wo - 1) + S)
    wt = w.to(dev, F64).permute(2, 3, 0, 1).contiguous()        # [R][S][Co][Ci]
    dx = torch.empty(N, Hi, Wi, Ci, dtype=F64, device=dev)
    nc = _img_chunk(Hp * Wp * Ci + Ho * Wo * (Ci + Co))
    for n0 in range(0, N, nc):
        g = dy[n0:n0 + nc].to(dev, F64)
        dxp = torch.zeros(g.shape[0], Hp, Wp, Ci, dtype=F64, device=dev)
        for r in range(R):
            for s in range(S):
                _tap(dxp, r, s, Ho, Wo, stride).add_(torch.matmul(g, wt[r, s]))
        dx[n0:n0 + nc] = dxp[:, pad:pad + Hi, pad:pad + Wi]
        del g, dxp
    if add_mode == 1:
        dx += add.to(dev, F64)
    elif add_mode == 2:
        assert add.shape == (N, (Hi + 1) // 2, (Wi + 1) // 2, Ci), add.shape
        dx[:, 0::2, 0::2] += add.to(dev, F64)
    else:
        assert add_mode == 0 and add is None
    return dx


def conv_wgrad_ref(x, dy, R, S, stride, pad, device=None):
    """dw[co, ci, r, s] = sum_{n, ho, wo} dy[n, ho, wo, co] x[n, ho*stride - pad + r, wo*stride - pad + s, ci]."""
    dev = device or x.device
    N, H, W, Ci = x.shape
    _, Ho, Wo, Co = dy.shape
    assert (Ho, Wo) == _out_hw(H, W, R, S, stride, pad)
    Hp, Wp = max(H + 2 * pad, stride * (Ho - 1) + R), max(W + 2 * pad, stride * (Wo - 1) + S)
    dw = torch.zeros(R, S, Co, Ci, dtype=F64, device=dev)
    nc = _img_chunk(Hp * Wp * Ci + Ho * Wo * (Ci + Co))
    for n0 in range(0, N, nc):
        xp = _pad_nhwc(x[n0:n0 + nc].to(dev, F64), pad, Hp, Wp)
        g = dy[n0:n0 + nc].to(dev, F64).reshape(-1, Co).t()
        for r in range(R):
            for s in range(S):
                dw[r, s] += torch.matmul(g, _tap(xp, r, s, Ho, Wo, stride).reshape(-1, Ci))
        del xp, g
    return dw.permute(2, 3, 0, 1).contiguous()


def space_to_depth_ref(x, Hp, Wp):
    """The stem input gdl_stem_layout writes: x [N, C, H, W] -> [N, Hp, Wp, 16], channel (dy*2 + dx)*C + c of pixel
    (p, q) = x[c, 2p + dy - 3, 2q + dx - 3] (zero outside the image and in the channels past 4 C)."""
    N, C, H, W = x.shape
    pad = x.new_zeros(N, C, 2 * Hp, 2 * Wp)
    pad[:, :, 3:3 + H, 3:3 + W] = x
    out = x.new_zeros(N, Hp, Wp, 16)
    for dy in range(2):
        for dx in range(2):
            k = (dy * 2 + dx) * C
            out[..., k:k + C] = pad[:, :, dy::2, dx::2].permute(0, 2, 3, 1)
    return out


def stem_fwd_ref(x, w, device=None):
    """The 7x7 / stride 2 / pad 3 stem: x [N, C, H, W] (the image before space-to-depth), w [64, C, 7, 7] -> NHWC."""
    return conv_fwd_ref(x.permute(0, 2, 3, 1), w, 2, 3, device)


def stem_wgrad_ref(x, dy, device=None):
    return conv_wgrad_ref(x.permute(0, 2, 3, 1), dy, 7, 7, 2, 3, device)


def gemm_ref(A, B, device=None):
    """C = A @ B in float64 (the FiLM GEMMs: gemm_tn C = At^T Bt, gemm_nt C = A B^T, the contractions)."""
    dev = device or A.device
    return torch.matmul(A.to(dev, F64), B.to(dev, F64))


def film_outer_ref(a, v, variants, ZB):
    """Zt [D*D][ZB] bf16: column var*B + b of row i*D + j = x_b[i] y_b[j] (variant 0 a (x) v, 1 a (x) a, 2 v (x) v),
    the fp32 product rounded once to bf16; columns >= variants*B zero."""
    B, D = a.shape
    pairs = [(a, v), (a, a), (v, v)][:variants]
    Z = torch.zeros(D * D, ZB, dtype=BF, device=a.device)
    for k, (x, y) in enumerate(pairs):
        p = (x.double()[:, :, None] * y.double()[:, None, :]).reshape(B, D * D)   # exact: <= 48 significand bits
        Z[:, k * B:(k + 1) * B] = p.float().t().to(BF)   # float: the fp32 product (exact for 24-bit operands' 8-bit
    return Z                                             # mantissas), then one RNE rounding to bf16


def film_contract_ref(G, c0, x, i0, ni):
    """Chunk part of the sum-mode contraction: G [ni*D][>= c0 + B] holds the rows (i - i0)*D + j.
    dx[b][k] = sum_j G[i=k, j] x[b][j] (k in the chunk) + sum_{i in chunk} G[i, j=k] x[b][i]; float64 [B][D]."""
    B, D = x.shape
    g = G[:, c0:c0 + B].double().reshape(ni, D, B)     # [i - i0][j][b]
    xd = x.double()
    out = torch.zeros(B, D, dtype=F64, device=x.device)
    out[:, i0:i0 + ni] += torch.einsum("ijb,bj->bi", g, xd)
    out += torch.einsum("ijb,bi->bj", g, xd[:, i0:i0 + ni])
    return out
