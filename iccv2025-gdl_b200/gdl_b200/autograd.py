"""Autograd-compatible execution mode (SURVEY.md §8b mode 1): torch.autograd.Function bridges
over the C-ABI so that the reference's OWN `train_epoch` (two backward calls with
retain_graph=True, `p.grad = None` wipes in between, main_dgl.py:108-122) runs unmodified on
top of the sm_100a kernels.  The heavy work (encoders, linears) runs in libgdl_b200.so; tiny
[B,n] glue (bias broadcast, the final add of two logit halves, sigmoid gates) is left to
torch autograd.  The throughput path is step.DGLStep, not this file.
"""
import torch

from . import ops


class _LinearFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, W, b, col0, cols):
        x = x.contiguous().float()
        B, In = x.shape
        Out = W.shape[0]
        y = torch.empty(B, Out, device=x.device, dtype=torch.float32)
        ops.linear_fwd(x, W.data_ptr() + 4 * col0, b, y, B, In, Out, ldw=W.shape[1])
        ctx.save_for_backward(x, W, b)
        ctx.col0 = col0
        return y

    @staticmethod
    def backward(ctx, dy):
        x, W, b = ctx.saved_tensors
        dy = dy.contiguous()
        B, In = x.shape
        Out = W.shape[0]
        dx = dW = db = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            ops.linear_bwd(dy, None, W.data_ptr() + 4 * ctx.col0, dx, None, None, B, In, Out, ldw=W.shape[1])
        if ctx.needs_input_grad[1]:
            dW = torch.zeros_like(W)
            db_t = torch.empty(Out, device=x.device) if (b is not None and ctx.needs_input_grad[2]) else None
            ops.linear_bwd(dy, x, None, None, dW.data_ptr() + 4 * ctx.col0, db_t, B, In, Out, lddw=W.shape[1])
            db = db_t
        elif b is not None and ctx.needs_input_grad[2]:
            db = dy.sum(0)
        return dx, dW, db, None, None


def linear(x, W, b, col0=0, cols=None):
    """y = x @ W[:, col0:col0+cols]^T + b through gdl_linear_fwd/bwd."""
    assert cols is None or cols == x.shape[1]
    return _LinearFn.apply(x, W, b, col0, cols)


def add_bias(z, b):
    return z + b


def gate(g, h):
    return torch.sigmoid(g) * h


def outer_linear(x, y, W, b):
    from .film import FilmFn
    return FilmFn.apply(x, y, W, b)


class _EncoderMapFn(torch.autograd.Function):
    """ResNet-18 encoder: input tensor -> layer4 map (fp32 NCHW view of the bf16 NHWC result)."""

    @staticmethod
    def forward(ctx, net, x8, eng, *params):
        feat = eng.forward(x8)
        ctx.net, ctx.eng, ctx.x8 = net, eng, x8
        ctx.params = params
        return feat.permute(0, 3, 1, 2).float()

    @staticmethod
    def backward(ctx, g):
        eng = ctx.eng
        eng.g_feat.copy_(g.permute(0, 2, 3, 1))
        outs = {p: torch.empty_like(p.data) for p in ctx.params}
        eng.grad_override = outs
        try:
            eng.backward(ctx.x8)
        finally:
            eng.grad_override = None
        return (None, None, None) + tuple(outs[p] for p in ctx.params)


def to_nhwc8(net, x):
    """Input tensor of the reference contract -> the encoder's bf16 space-to-depth stem input
    [N,Hp,Wp,16] via gdl_stem_layout (fuses the per-frame reshape of backbone.py:162-164)."""
    x = x.contiguous().float()
    if net.modality == 'visual':
        B, Cc, T, H, W = x.shape
    else:
        B, Cc, H, W = x.shape
        T = 1
    _, _, Hp, Wp = ops.stem_geometry(H, W)
    x16 = torch.empty(B * T, Hp, Wp, 16, device=x.device, dtype=torch.bfloat16)
    ops.stem_layout(x, x16, B, Cc, T, H, W)
    return x16, (B * T, H, W)


def encoder_map(net, x):
    x8, (N, H, W) = to_nhwc8(net, x)
    eng = net.engine(N, H, W)
    if not net.training:
        # eval: BatchNorm folded into the weights from the running statistics (re-folded only when they changed)
        with torch.no_grad():
            return eng.forward(x8, training=False).permute(0, 3, 1, 2).float()
    eng.repack()
    if not torch.is_grad_enabled():
        with torch.no_grad():
            feat = eng.forward(x8)
            return feat.permute(0, 3, 1, 2).float()
    params = eng.parameters()
    out = _EncoderMapFn.apply(net, x8, eng, *params)
    with torch.no_grad():
        for m in net.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.num_batches_tracked += 1
    return out
