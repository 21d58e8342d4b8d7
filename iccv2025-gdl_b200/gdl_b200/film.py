"""FiLM_DGL head on the sm_100a kernels (reference models/fusion_modules.py:126-178).

`fc: Linear(512*512 -> 512)` applied to the outer products a (x) v (multimodal, detached features),
a (x) a and v (x) v (unimodal), then `fc_out`.  The outer products are materialised FEATURE-MAJOR in bf16
(Zt [262144][ZB], batch contiguous) next to a feature-major bf16 shadow of fc.weight (W1t [262144][512]),
so that the three big contractions are the library's two flat-window GEMMs (csrc/film.cu):

    H  [ZB, 512]     = Zt^T * W1t + b1              gemm_tn   (forward, all branches at once)
    dW1t[262144,512] = Zt[:, :B] * dH_f^T           gemm_nt   (Lf only: the unimodal head gradient is wiped)
    G  [262144, 2B]  = W1t * [dH_a; dH_v]^T         gemm_nt   (unimodal only: Lf saw detached features)

`FilmHead` is the fused-step path (step.DGLStep).  It never holds the 262144-row operands whole: the reduction
index f = i*512 + j is walked in CHUNKS of `CHUNK_I` = 128 values of i (65536 features).
Per chunk the outer products (100 MB at B = 256), the unimodal gradient G (67 MB) and the weight-gradient tile
(67 MB) live in three rolling buffers, instead of 403 + 268 + 268 MB held for the whole step; H accumulates over the
chunks (gemm_tn_f32 / gemm_tn_f32_acc), dW1 is written window by window, da / dv accumulate (film_contract_chunk).
Chunk order = summation order, fixed.  Measured at B = 256 (one B200, same box): 23.72 / 23.50 / 23.28 / 23.42 ms per
step for chunks of 64 / 128 / 256 / 512 (= whole operands) values of i: the price of never materialising the
operands is the second evaluation of the outer products in the backward loop (0.5 ms of kernel time).
`FilmFn` is the autograd bridge the drop-in module uses so the reference's own two-backward loop runs unmodified
(one outer product per call, whole operands).
"""
import torch

from . import ops

D = 512
F2 = D * D
CHUNK_I = 128  # values of the first outer-product index per chunk
FC = CHUNK_I * D        # features per chunk


def _ceil(x, m):
    return (x + m - 1) // m * m


class FilmBuffers:
    """Static buffers for `variants` outer products of batch B."""

    def __init__(self, B, variants, dev):
        self.B, self.variants = B, variants
        self.ZB = _ceil(variants * B, 128)            # columns of Zt = rows of H
        self.KB = _ceil(B, 64)                        # reduction length of the dW1 GEMM
        self.NG = _ceil(max(variants - 1, 1) * B, 64)  # columns of G (unimodal branches)
        bf = dict(device=dev, dtype=torch.bfloat16)
        self.Zt = torch.zeros(F2, self.ZB, **bf)
        self.W1t = torch.empty(F2, D, **bf)
        self.H = torch.empty(self.ZB, D, device=dev)
        self.ws = torch.empty(max(ops.gemm_tn_workspace_bytes(self.ZB, D, F2), 16) // 4, device=dev)
        self.dHfT = torch.empty(D, self.KB, **bf)
        self.dHs = torch.empty(self.NG, D, **bf)
        self.dW1t = torch.empty(F2, D, **bf)
        self.G = torch.empty(F2, self.NG, **bf)
        self.scratch = torch.empty(ops.film_scratch_floats(B, D), device=dev)

    def refresh(self, W1):
        """bf16 feature-major shadow of fc.weight (after every optimizer step)."""
        ops.transpose_f32_to_bf16(W1, self.W1t, D, F2)


class FilmChunkBuffers:
    """Rolling per-chunk operands of the fused FiLM head (3 variants of batch B)."""

    def __init__(self, B, dev):
        self.B = B
        self.ZB = _ceil(3 * B, 128)
        self.KB = _ceil(B, 64)
        self.NG = _ceil(2 * B, 64)
        bf = dict(device=dev, dtype=torch.bfloat16)
        self.Zt = torch.zeros(FC, self.ZB, **bf)       # outer products of the chunk, feature-major
        self.G = torch.empty(FC, self.NG, **bf)        # unimodal gradient wrt the chunk's features
        self.dW1t = torch.empty(FC, D, **bf)           # weight-gradient tile of the chunk
        self.W1t = torch.empty(F2, D, **bf)            # bf16 feature-major shadow of fc.weight (whole: it is a parameter)
        self.H = torch.empty(self.ZB, D, device=dev)
        self.ws = torch.empty(max(ops.gemm_tn_workspace_bytes(self.ZB, D, FC), 16) // 4, device=dev)
        self.dHfT = torch.empty(D, self.KB, **bf)
        self.dHs = torch.empty(self.NG, D, **bf)
        self.scratch = torch.empty(ops.film_scratch_floats(B, D), device=dev)    # a^T, v^T for the outer products
        self.scratch_a = torch.empty(ops.film_scratch_floats(B, D), device=dev)  # (a^T, a^T) / (v^T, v^T) for the
        self.scratch_v = torch.empty(ops.film_scratch_floats(B, D), device=dev)  # two contractions

    def refresh(self, W1):
        ops.transpose_f32_to_bf16(W1, self.W1t, D, F2)

    def forward(self, a, v, b1):
        """H = sum over chunks of Zt_c^T * W1t_c + b1  (rows: [a(x)v | a(x)a | v(x)v])."""
        B = self.B
        for c in range(D // CHUNK_I):
            ops.film_outer_chunk(a, v, self.Zt, B, D, self.ZB, 3, self.scratch, c * FC, FC)
            if c == 0:
                ops.gemm_tn_f32(self.Zt, self.W1t[:FC], b1, self.H, self.ZB, D, FC, self.ws)
            else:
                ops.gemm_tn_f32_acc(self.Zt, self.W1t[c * FC:(c + 1) * FC], self.H, self.ZB, D, FC, self.ws)


class FilmHead:
    """The FiLM head of heads.fusion_head: the fused training head, the eval head and the W1t shadow refresh."""

    def __init__(self, fm, B=None, n=None, dev=None):
        self.fm, self.B, self.n = fm, B, n
        if dev is None:
            return
        self.buf = FilmChunkBuffers(B, dev)
        z = lambda *s: torch.empty(*s, device=dev)
        self.dl = z(3, B, n)
        self.dH = z(3, B, D)   # dH_f, dH_a, dH_v
        self.sc = z(B)
        self.ones = torch.ones(B, 1, device=dev)
        self.a_pool, self.v_pool = z(B, D), z(B, D)  # pooled features of the eval head
        self.refresh_shadows()

    def trainable(self):
        fm = self.fm
        return [fm.fc.weight, fm.fc.bias, fm.fc_out.weight, fm.fc_out.bias]

    def refresh_shadows(self):
        self.buf.refresh(self.fm.fc.weight.data)

    def eval(self, ev, fa, Ga, fv, Gv):
        """Pooling (eval_head kind 3), the forward chunks, fc_out and the correct counts."""
        fm, b, B, n = self.fm, self.buf, self.B, self.n
        ops.eval_head(3, fa, Ga, fv, Gv, None, None, 0, None, None, None, None, 1, None, self.a_pool, self.v_pool,
                      None, None, B, n)
        b.forward(self.a_pool, self.v_pool, fm.fc.bias.data)
        for i in range(3):
            ops.linear_fwd(b.H[i * B:(i + 1) * B], fm.fc_out.weight.data, fm.fc_out.bias.data, ev.logits[i], B, D, n)
        ops.eval_count(ev.logits, ev.label_in, ev.counts, B, n)

    def train(self, st):
        """st: the DGLStep (features, labels, logits, losses, da/dv live there)."""
        fm, b, B, n = self.fm, self.buf, self.B, self.n
        W1, b1, W2, b2 = fm.fc.weight, fm.fc.bias, fm.fc_out.weight, fm.fc_out.bias
        b.forward(st.a_feat, st.v_feat, b1.data)
        for i in range(3):                                                       # logits: out, out_a, out_v
            ops.linear_fwd(b.H[i * B:(i + 1) * B], W2.data, b2.data, st.logits[i], B, D, n)
            gs = st.inv_batch if i == 0 else st.alpha * st.inv_batch
            ops.softmax_ce(st.logits[i], st.label_in, st.inv_batch, gs, st.losses[i:i + 1], self.dl[i], self.sc, B, n)
        # Lf -> fc_out (dW2, db2) and dH_f; the unimodal losses only produce dH_a, dH_v (head gradient wiped)
        ops.linear_bwd(self.dl[0], b.H[0:B], W2.data, self.dH[0], W2.grad, b2.grad, B, D, n)
        ops.linear_bwd(self.dl[1], None, W2.data, self.dH[1], None, None, B, D, n)
        ops.linear_bwd(self.dl[2], None, W2.data, self.dH[2], None, None, B, D, n)
        # db1 = sum_b dH_f  ==  the weight gradient of a Linear(1 -> 512) fed with ones
        ops.linear_bwd(self.dH[0], self.ones, None, None, b1.grad, None, B, 1, D)
        ops.cast_pad_bf16(self.dH[0], B, None, 0, D, D, True, b.dHfT, D, b.KB)
        ops.cast_pad_bf16(self.dH[1], B, self.dH[2], B, D, D, False, b.dHs, b.NG, D)
        # backward, chunk by chunk: the outer products again (L2-resident), dW1 window (Lf only), G tile and its
        # contraction with a / v (unimodal only)
        for c in range(D // CHUNK_I):
            ops.film_outer_chunk(st.a_feat, st.v_feat, b.Zt, B, D, b.ZB, 3, b.scratch, c * FC, FC)
            ops.gemm_nt_bf16(b.Zt, b.ZB, b.dHfT, b.dW1t, FC, D, b.KB)
            ops.transpose_bf16_to_f32_window(b.dW1t, W1.grad, D, FC, F2, c * FC)
            ops.gemm_nt_bf16(b.W1t[c * FC:(c + 1) * FC], D, b.dHs, b.G, FC, b.NG, D)
            ops.film_contract_chunk(b.G, b.NG, 0, st.a_feat, st.a_feat, st.da, None, B, D, True, b.scratch_a,
                                    c * CHUNK_I, CHUNK_I, c > 0, c == 0)
            ops.film_contract_chunk(b.G, b.NG, B, st.v_feat, st.v_feat, st.dv, None, B, D, True, b.scratch_v,
                                    c * CHUNK_I, CHUNK_I, c > 0, c == 0)


class FilmFn(torch.autograd.Function):
    """h[B,512] = fc(x (x) y): autograd bridge for the drop-in FiLM_DGL module (one outer product per call)."""

    @staticmethod
    def forward(ctx, x, y, W, b):
        x, y = x.contiguous().float(), y.contiguous().float()
        B = x.shape[0]
        buf = FilmBuffers(B, 1, x.device)
        buf.refresh(W.data)
        ops.film_outer(x, y, buf.Zt, B, D, buf.ZB, 1, buf.scratch)
        ops.gemm_tn_f32(buf.Zt, buf.W1t, b.data if b is not None else None, buf.H, buf.ZB, D, F2, buf.ws)
        ctx.save_for_backward(x, y, W, b)
        ctx.buf = buf
        return buf.H[:B].clone()

    @staticmethod
    def backward(ctx, dh):
        x, y, W, b = ctx.saved_tensors
        buf, B = ctx.buf, x.shape[0]
        dh = dh.contiguous().float()
        dx = dy = dW = db = None
        if ctx.needs_input_grad[2]:
            ops.cast_pad_bf16(dh, B, None, 0, D, D, True, buf.dHfT, D, buf.KB)
            ops.gemm_nt_bf16(buf.Zt, buf.ZB, buf.dHfT, buf.dW1t, F2, D, buf.KB)
            dW = torch.empty_like(W.data)
            ops.transpose_bf16_to_f32(buf.dW1t, dW, D, F2)
        if b is not None and ctx.needs_input_grad[3]:
            db = dh.sum(0)
        if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
            ops.cast_pad_bf16(dh, B, None, 0, D, D, False, buf.dHs, buf.NG, D)
            ops.gemm_nt_bf16(buf.W1t, D, buf.dHs, buf.G, F2, buf.NG, D)
            dx, dy = torch.empty_like(x), torch.empty_like(y)
            ops.film_contract(buf.G, buf.NG, 0, x, y, dx, dy, B, D, False, buf.scratch)
        return dx, dy, dW, db
