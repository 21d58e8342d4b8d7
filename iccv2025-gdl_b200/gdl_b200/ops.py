"""Thin tensor-level wrappers over the C-ABI: borrow device pointers from torch tensors, pass
torch's current CUDA stream, check the status.  PyTorch is plumbing only (memory, streams);
every computation below runs in libgdl_b200.so.  No fallbacks.
"""
import ctypes as C
import functools
import threading

import torch

from . import _lib
from ._lib import ConvDesc, check

_initialised = set()

# Kernel-launch accounting (bench.py's "gpu_launches") and optional per-op CUDA-event timing
# (bench.py's roofline leg).  LAUNCHES counts kernels of libgdl_b200.so enqueued by this process.
LAUNCHES = 0
TIMING = None  # when a list: (name, start_event, end_event, work) is appended per op


def _op(name, kernels, work=None):
    """Decorator: count launches; when TIMING is a list, bracket the op with CUDA events on the
    launching stream.  work(*args) -> ("flops"|"bytes", amount) is the ALGORITHMIC work."""
    def deco(fn):
        @functools.wraps(fn)
        def wrapper(*args, **kw):
            global LAUNCHES
            LAUNCHES += kernels(*args, **kw) if callable(kernels) else kernels
            if TIMING is None:
                return fn(*args, **kw)
            st = torch.cuda.current_stream()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            out = fn(*args, **kw)
            e1.record(st)
            TIMING.append((name, e0, e1, work(*args, **kw) if work else None))
            return out
        return wrapper
    return deco


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "gdl ops need contiguous CUDA tensors"
    return C.c_void_p(t.data_ptr())


def _addr(t):
    """Raw device address; accepts a tensor, an int address or None."""
    if t is None:
        return None
    if isinstance(t, int):
        return C.c_void_p(t)
    return C.c_void_p(t.data_ptr())


def init(device=None):
    lib = _lib.load()
    dev = torch.cuda.current_device() if device is None else int(device)
    if dev not in _initialised:
        check(lib.gdl_init(dev), "gdl_init")
        _initialised.add(dev)
    return lib


# ---------------------------------------------------------------------------------- convolution
def conv_desc(N, Hi, Wi, Ci, Co, R, S, stride, pad):
    Ho = (Hi + 2 * pad - R) // stride + 1
    Wo = (Wi + 2 * pad - S) // stride + 1
    return ConvDesc(N, Hi, Wi, Ci, Ho, Wo, Co, R, S, stride, pad)


def conv_packed_k(d):
    return int(_lib.load().gdl_conv_packed_k(C.byref(d)))


def conv_wgrad_workspace_bytes(d):
    return int(_lib.load().gdl_conv_wgrad_workspace_bytes(C.byref(d)))


def _dstr(d):
    return "N%d %dx%d C%d->%d k%d s%d" % (d.N, d.Hi, d.Wi, d.Ci, d.Co, d.R, d.stride)


def conv_flops(d, ci_real=None):
    """Algorithmic FLOPs of one conv pass (fwd == dgrad == wgrad): 2*M*Co*R*S*Ci_real."""
    ci = ci_real if ci_real is not None else d.Ci
    return 2.0 * d.N * d.Ho * d.Wo * d.Co * d.R * d.S * ci


@_op("pack_weights", 1)
def conv_pack_weights(d, ci_real, w_oihw, w_packed, w_packed_T=None):
    check(_lib.load().gdl_conv_pack_weights(C.byref(d), ci_real, _ptr(w_oihw), _ptr(w_packed),
                                            _ptr(w_packed_T), _stream()), "gdl_conv_pack_weights")


def make_pack_table(entries, device):
    """entries: [(w_oihw, w_packed, w_packed_T or None, Co, Ci, ci_real, R, S, Kp[, scale or None])] ->
    (device table, n, total).  scale: fp32 [Co] folded into the rows (eval mode).
    The table holds raw device addresses: rebuild it if any tensor is re-allocated."""
    arr = (_lib.PackEntry * len(entries))()
    start = 0
    for e, ent in zip(arr, entries):
        w, wp, wT, Co, Ci, ci_real, R, S, Kp = ent[:9]
        scale = ent[9] if len(ent) > 9 else None
        e.w, e.wp, e.wT = w.data_ptr(), wp.data_ptr(), (wT.data_ptr() if wT is not None else None)
        e.scale = scale.data_ptr() if scale is not None else None
        e.Co, e.Ci, e.ci_real, e.R, e.S, e.Kp, e.start = Co, Ci, ci_real, R, S, Kp, start
        start += Co * Kp
    host = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8)
    # tiled kernel (coalesced through shared memory) when every entry is an unpadded block convolution
    tiled = all(e[4] == e[5] and e[4] % 64 == 0 and e[3] % 32 == 0 and e[8] == e[6] * e[7] * e[4] and e[6] * e[7] <= 9
                for e in entries)
    info = None
    if tiled:
        info = (max((e[3] // 32) * (e[4] // 64) for e in entries), max(e[6] * e[7] for e in entries))
    return host.to(device), len(entries), start, info


@_op("pack_weights", 1)
def conv_pack_weights_multi(table, n, total, tiled=None):
    """tiled = (max_tiles, max_rs) from make_pack_table selects the shared-memory tiled kernel."""
    if tiled is not None:
        check(_lib.load().gdl_conv_pack_weights_tiled(_ptr(table), n, tiled[0], tiled[1], _stream()),
              "gdl_conv_pack_weights_tiled")
    else:
        check(_lib.load().gdl_conv_pack_weights_multi(_ptr(table), n, total, _stream()), "gdl_conv_pack_weights_multi")


@_op("conv_fwd", 1, lambda d, x, w, y, ci_real=None: ("flops", conv_flops(d, ci_real), _dstr(d)))
def conv_fwd(d, x, w_packed, y, ci_real=None):
    check(_lib.load().gdl_conv_fwd(C.byref(d), _ptr(x), _ptr(w_packed), _ptr(y), _stream()),
          "gdl_conv_fwd")


@_op("conv_fwd", 1, lambda d, x, w, bias, res, relu, y: ("flops", conv_flops(d), _dstr(d)))
def conv_fwd_bias_act(d, x, w_packed, bias, res, relu, y):
    """Eval-mode fused unit: y = [relu](conv(x, w') + bias[co] [+ res]) with the BatchNorm scale folded into w'."""
    check(_lib.load().gdl_conv_fwd_bias_act(C.byref(d), _ptr(x), _ptr(w_packed), _ptr(bias), _ptr(res), int(relu),
                                            _ptr(y), _stream()), "gdl_conv_fwd_bias_act")


@_op("conv_fwd", 1, lambda d, x, w, y, partial, ci_real=None: ("flops", conv_flops(d, ci_real), _dstr(d)))
def conv_fwd_stats(d, x, w_packed, y, bn_partial, ci_real=None):
    """conv forward with the BatchNorm partial sums of y accumulated in the epilogue; returns the number of
    partial rows written (0: this shape has no fused statistics, run bn_stats on y)."""
    rows = C.c_int(0)
    check(_lib.load().gdl_conv_fwd_stats(C.byref(d), _ptr(x), _ptr(w_packed), _ptr(y), _ptr(bn_partial),
                                         C.byref(rows), _stream()), "gdl_conv_fwd_stats")
    return rows.value


_sweep_state = {}  # thread id -> last value handed to the (thread-local) C hint


def sweep(reverse):
    """Direction hint for the following conv / BN launches of this thread (gdl_set_sweep): reverse=1 walks the
    pixel range in descending order, so a pass that follows a forward-order producer starts on the part of the
    tensor that is still in L2.  Cached: the C call is made only when the setting changes."""
    reverse = 1 if reverse else 0
    tid = threading.get_ident()
    if _sweep_state.get(tid, 0) != reverse:
        _lib.load().gdl_set_sweep(reverse)
        _sweep_state[tid] = reverse


def set_fused_stats_min_k(k):
    """Enable the conv-epilogue BN statistics for convolutions with R*S*Ci >= k (k < 0: library default = every
    flat-window convolution).  Returns the previous setting."""
    return int(_lib.load().gdl_set_fused_stats_min_k(int(k)))


@_op("bn_stats", 1)
def bn_stats_finalize(partial, rows, P, Cc, gamma, beta, eps, momentum, running_mean, running_var, mean, invstd,
                      scale, shift):
    check(_lib.load().gdl_bn_stats_finalize(_ptr(partial), rows, P, Cc, _ptr(gamma), _ptr(beta), eps, momentum,
                                            _ptr(running_mean), _ptr(running_var), _ptr(mean), _ptr(invstd),
                                            _ptr(scale), _ptr(shift), _stream()), "gdl_bn_stats_finalize")


@_op("conv_dgrad", 1, lambda d, *a, **k: ("flops", conv_flops(d), _dstr(d)))
def conv_dgrad(d, dy, w_packed_T, dx, add_src=None, add_mode=0):
    check(_lib.load().gdl_conv_dgrad(C.byref(d), _ptr(dy), _ptr(w_packed_T), _ptr(dx),
                                     _ptr(add_src), add_mode, _stream()), "gdl_conv_dgrad")


@_op("conv_wgrad", 2, lambda d, ci_real, *a, **k: ("flops", conv_flops(d, ci_real), _dstr(d)))
def conv_wgrad(d, ci_real, x, dy, dw_oihw, workspace):
    check(_lib.load().gdl_conv_wgrad(C.byref(d), ci_real, _ptr(x), _ptr(dy), _ptr(dw_oihw),
                                     _ptr(workspace), workspace.numel() * workspace.element_size(),
                                     _stream()), "gdl_conv_wgrad")


# ---------------------------------------------------------------------------------- stems
def stem_geometry(H, W):
    ho, wo, hp, wp = C.c_int(), C.c_int(), C.c_int(), C.c_int()
    check(_lib.load().gdl_stem_geometry(H, W, C.byref(ho), C.byref(wo), C.byref(hp), C.byref(wp)),
          "gdl_stem_geometry")
    return ho.value, wo.value, hp.value, wp.value


def _stem_flops(N, H, W, Cc):
    ho, wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    return 2.0 * N * ho * wo * 64 * 49 * Cc


@_op("stem_layout", 1, lambda src, dst, B, Cc, T, H, W: ("bytes", B * T * H * W * 4.0 * Cc + dst.numel() * 2.0))
def stem_layout(src, dst, B, Cc, T, H, W):
    check(_lib.load().gdl_stem_layout(_ptr(src), _ptr(dst), B, Cc, T, H, W, _stream()), "gdl_stem_layout")


@_op("pack_weights", 1)
def stem_pack_weights(w_oihw, w_packed, Cc):
    check(_lib.load().gdl_stem_pack_weights(_ptr(w_oihw), _ptr(w_packed), Cc, _stream()), "gdl_stem_pack_weights")


@_op("pack_weights", 1)
def stem_pack_weights_scaled(w_oihw, scale64, w_packed, Cc):
    check(_lib.load().gdl_stem_pack_weights_scaled(_ptr(w_oihw), _ptr(scale64), _ptr(w_packed), Cc, _stream()),
          "gdl_stem_pack_weights_scaled")


@_op("conv_fwd", 1, lambda x16, w, y, N, H, W, Cc: ("flops", _stem_flops(N, H, W, Cc), "N%d %dx%d stem C%d s2d" % (N, H, W, Cc)))
def stem_fwd(x16, w_packed, y, N, H, W, Cc):
    check(_lib.load().gdl_stem_fwd(_ptr(x16), _ptr(w_packed), _ptr(y), N, H, W, _stream()), "gdl_stem_fwd")


@_op("conv_fwd", 1, lambda x16, w, y, N, H, W, Cc, partial: ("flops", _stem_flops(N, H, W, Cc), "N%d %dx%d stem C%d s2d" % (N, H, W, Cc)))
def stem_fwd_stats(x16, w_packed, y, N, H, W, Cc, bn_partial):
    """Stem forward with the BatchNorm partial sums of y formed in the epilogue; returns the number of partial rows."""
    rows = C.c_int(0)
    check(_lib.load().gdl_stem_fwd_stats(_ptr(x16), _ptr(w_packed), _ptr(y), N, H, W, _ptr(bn_partial), C.byref(rows),
                                         _stream()), "gdl_stem_fwd_stats")
    return rows.value


def stem_wgrad_workspace_bytes(N, H, W):
    return int(_lib.load().gdl_stem_wgrad_workspace_bytes(N, H, W))


@_op("conv_wgrad", 2, lambda x16, dy, dw, Cc, N, H, W, ws: ("flops", _stem_flops(N, H, W, Cc), "N%d %dx%d stem C%d s2d" % (N, H, W, Cc)))
def stem_wgrad(x16, dy, dw_oihw, Cc, N, H, W, workspace):
    check(_lib.load().gdl_stem_wgrad(_ptr(x16), _ptr(dy), _ptr(dw_oihw), Cc, N, H, W, _ptr(workspace),
                                     workspace.numel() * workspace.element_size(), _stream()), "gdl_stem_wgrad")


# ---------------------------------------------------------------------------------- elementwise
@_op("layout", 1, lambda src, dst, B, Cc, T, H, W: ("bytes", B * T * H * W * (4.0 * Cc + 16.0)))
def layout_ncthw_to_nhwc8(src, dst, B, Cc, T, H, W):
    check(_lib.load().gdl_layout_ncthw_to_nhwc8(_ptr(src), _ptr(dst), B, Cc, T, H, W, _stream()),
          "gdl_layout_ncthw_to_nhwc8")


def bn_partial_floats(P, Cc):
    return int(_lib.load().gdl_bn_partial_floats(P, Cc))


@_op("bn_stats", 2, lambda x, P, Cc, *a: ("bytes", 2.0 * P * Cc))
def bn_stats(x, P, Cc, partial, gamma, beta, eps, momentum, running_mean, running_var, mean,
             invstd, scale, shift):
    check(_lib.load().gdl_bn_stats(_ptr(x), P, Cc, _ptr(partial), _ptr(gamma), _ptr(beta), eps,
                                   momentum, _ptr(running_mean), _ptr(running_var), _ptr(mean),
                                   _ptr(invstd), _ptr(scale), _ptr(shift), _stream()), "gdl_bn_stats")


@_op("bn_eval_affine", 1)
def bn_eval_affine(gamma, beta, rm, rv, eps, scale, shift, Cc):
    check(_lib.load().gdl_bn_eval_affine(_ptr(gamma), _ptr(beta), _ptr(rm), _ptr(rv), eps, _ptr(scale),
                                         _ptr(shift), Cc, _stream()), "gdl_bn_eval_affine")


@_op("bn_apply", 1, lambda x, res, y, P, Cc, *a: ("bytes", (4.0 + (2.0 if res is not None else 0.0)) * P * Cc))
def bn_apply(x, res, y, P, Cc, scale, shift, relu):
    check(_lib.load().gdl_bn_apply(_ptr(x), _ptr(res), _ptr(y), P, Cc, _ptr(scale), _ptr(shift),
                                   int(relu), _stream()), "gdl_bn_apply")


@_op("bn_bwd", 3, lambda dy, y, x, dz, dx, P, Cc, *a: ("bytes", ((8.0 if a[-1] else 4.0) + 6.0) * P * Cc))
def bn_bwd(dy, y, x, dz, dx, P, Cc, gamma, mean, invstd, partial, dgamma, dbeta, relu):
    check(_lib.load().gdl_bn_bwd(_ptr(dy), _ptr(y), _ptr(x), _ptr(dz), _ptr(dx), P, Cc, _ptr(gamma),
                                 _ptr(mean), _ptr(invstd), _ptr(partial), _ptr(dgamma), _ptr(dbeta),
                                 int(relu), _stream()), "gdl_bn_bwd")


@_op("bn_bwd", 3, lambda dy, x, dx, P, Cc, *a: ("bytes", 10.0 * P * Cc))
def bn_bwd_nores(dy, x, dx, P, Cc, gamma, mean, invstd, scale, shift, partial, dgamma, dbeta):
    """BN+ReLU backward without a residual input: mask recomputed from x (no y read, no dz write)."""
    check(_lib.load().gdl_bn_bwd_nores(_ptr(dy), _ptr(x), _ptr(dx), P, Cc, _ptr(gamma), _ptr(mean), _ptr(invstd),
                                       _ptr(scale), _ptr(shift), _ptr(partial), _ptr(dgamma), _ptr(dbeta),
                                       _stream()), "gdl_bn_bwd_nores")


@_op("stem_tail_fwd", 1, lambda x, sc, sh, y, am, xm, N, H, W, Cc, Ho, Wo: ("bytes", N * Cc * (2.0 * H * W + (5.0 if xm is not None else 3.0) * Ho * Wo)))
def bn_relu_maxpool_fwd(x, scale, shift, y, argmax, xmax, N, H, W, Cc, Ho, Wo):
    check(_lib.load().gdl_bn_relu_maxpool_fwd(_ptr(x), _ptr(scale), _ptr(shift), _ptr(y), _ptr(argmax), _ptr(xmax),
                                              N, H, W, Cc, Ho, Wo, _stream()), "gdl_bn_relu_maxpool_fwd")


@_op("stem_tail_bwd", 3, lambda g, am, xm, x, dx, N, H, W, Cc, Ho, Wo, *a: ("bytes", N * Cc * ((4.0 if xm is not None else 6.0) * H * W + (7.0 if xm is not None else 6.0) * Ho * Wo)))
def bn_relu_maxpool_bwd(gpool, argmax, xmax, x, dx, N, H, W, Cc, Ho, Wo, gamma, mean, invstd, scale, shift, partial,
                        dgamma, dbeta):
    check(_lib.load().gdl_bn_relu_maxpool_bwd(_ptr(gpool), _ptr(argmax), _ptr(xmax), _ptr(x), _ptr(dx), N, H, W, Cc,
                                              Ho, Wo,
                                              _ptr(gamma), _ptr(mean), _ptr(invstd), _ptr(scale), _ptr(shift),
                                              _ptr(partial), _ptr(dgamma), _ptr(dbeta), _stream()),
          "gdl_bn_relu_maxpool_bwd")


def _pool_bytes(a, b, c, N, H, W, Cc, Ho, Wo):
    return ("bytes", N * Cc * (2.0 * H * W + 3.0 * Ho * Wo))


@_op("maxpool_fwd", 1, _pool_bytes)
def maxpool_fwd(x, y, argmax, N, H, W, Cc, Ho, Wo):
    check(_lib.load().gdl_maxpool_fwd(_ptr(x), _ptr(y), _ptr(argmax), N, H, W, Cc, Ho, Wo, _stream()),
          "gdl_maxpool_fwd")


@_op("maxpool_bwd", 1, _pool_bytes)
def maxpool_bwd(dy, argmax, dx, N, H, W, Cc, Ho, Wo):
    check(_lib.load().gdl_maxpool_bwd(_ptr(dy), _ptr(argmax), _ptr(dx), N, H, W, Cc, Ho, Wo, _stream()),
          "gdl_maxpool_bwd")


@_op("gap_fwd", 1, lambda x, out, B, G, Cc: ("bytes", 2.0 * B * G * Cc))
def gap_fwd(x, out, B, G, Cc):
    check(_lib.load().gdl_gap_fwd(_ptr(x), _ptr(out), B, G, Cc, _stream()), "gdl_gap_fwd")


@_op("gap_bwd", 1, lambda dout, dx, B, G, Cc: ("bytes", 2.0 * B * G * Cc))
def gap_bwd(dout, dx, B, G, Cc):
    check(_lib.load().gdl_gap_bwd(_ptr(dout), _ptr(dx), B, G, Cc, _stream()), "gdl_gap_bwd")


# ---------------------------------------------------------------------------------- heads
@_op("linear_fwd", 1)
def linear_fwd(x, W, b, y, B, In, Out, ldw=None):
    check(_lib.load().gdl_linear_fwd(_ptr(x), _addr(W), ldw or In, _ptr(b), _ptr(y), B, In, Out, _stream()),
          "gdl_linear_fwd")


@_op("linear_bwd", lambda dy, x, W, dx, dW, *a, **k: (dx is not None) + (dW is not None))
def linear_bwd(dy, x, W, dx, dW, db, B, In, Out, accumulate=False, ldw=None, lddw=None):
    check(_lib.load().gdl_linear_bwd(_ptr(dy), _ptr(x), _addr(W), ldw or In, _ptr(dx), _addr(dW),
                                     lddw or In, _ptr(db), B, In, Out, int(accumulate), _stream()),
          "gdl_linear_bwd")


def head_scratch_floats(B, n):
    return int(_lib.load().gdl_head_scratch_floats(B, n))


@_op("dgl_head", 2)
def dgl_head_linear(kind, a, v, Wx_ptr, Wy_ptr, ldw, bx, by, labels, alpha, inv_batch, logits, losses,
                    da, dv, dWx_ptr, dWy_ptr, lddw, dbx, dby, scratch, B, D, n):
    """Wx_ptr/Wy_ptr/dWx_ptr/dWy_ptr are raw integer device addresses (they may point into the
    middle of a tensor: concat's Wy = fc_out.weight + D)."""
    check(_lib.load().gdl_dgl_head_linear(kind, _ptr(a), _ptr(v), C.c_void_p(Wx_ptr), C.c_void_p(Wy_ptr),
                                          ldw, _ptr(bx), _ptr(by), _ptr(labels), alpha, inv_batch,
                                          _ptr(logits), _ptr(losses), _ptr(da), _ptr(dv),
                                          C.c_void_p(dWx_ptr), C.c_void_p(dWy_ptr), lddw, _ptr(dbx),
                                          _ptr(dby), _ptr(scratch), B, D, n, _stream()),
          "gdl_dgl_head_linear")


def gated_head_scratch_floats(B, n):
    return int(_lib.load().gdl_gated_head_scratch_floats(B, n))


@_op("dgl_head", 2)
def dgl_head_gated(a, v, Wx, bx, Wy, by, Wo, bo, labels, alpha, inv_batch, logits, losses, da, dv, dWo, dbo, scratch,
                   B, D, n):
    check(_lib.load().gdl_dgl_head_gated(_ptr(a), _ptr(v), _ptr(Wx), _ptr(bx), _ptr(Wy), _ptr(by), _ptr(Wo), _ptr(bo),
                                         _ptr(labels), alpha, inv_batch, _ptr(logits), _ptr(losses), _ptr(da), _ptr(dv),
                                         _ptr(dWo), _ptr(dbo), _ptr(scratch), B, D, n, _stream()), "gdl_dgl_head_gated")


EVAL_KINDS = {"concat": 0, "sum": 1, "gated": 2, "pool": 3}


def _eval_head_bytes(kind, fa, Ga, fv, Gv, Wx, Wy, ldw, bx, by, Wo, bo, x_gate, labels, a_out, v_out, logits, counts,
                     B, n):
    """Map reads (the weights are re-read from L2 by every CTA: counted once) + pooled / logit writes."""
    w = {0: n * 2 * 512, 1: n * 2 * 512, 2: 2 * 512 * 512 + n * 512, 3: 0}[kind]
    return ("bytes", 2.0 * B * (Ga + Gv) * 512 + 4.0 * w + (8.0 * B * 512 if a_out is not None else 0.0)
            + (12.0 * B * n if logits is not None else 0.0))


@_op("eval_head", 1, _eval_head_bytes)
def eval_head(kind, fa, Ga, fv, Gv, Wx, Wy, ldw, bx, by, Wo, bo, x_gate, labels, a_out, v_out, logits, counts, B, n):
    """Eval-mode head from the bf16 NHWC layer-4 maps (include/gdl_b200.h gdl_eval_head): pooling, the three logit
    sets of `kind` (EVAL_KINDS), their row arg-max, and `counts[h] += correct` when labels is given.
    Wx / Wy are raw integer device addresses or tensors (concat's Wy points into the middle of fc_out.weight)."""
    check(_lib.load().gdl_eval_head(kind, _ptr(fa), Ga, _ptr(fv), Gv, _addr(Wx), _addr(Wy), ldw, _ptr(bx), _ptr(by),
                                    _ptr(Wo), _ptr(bo), int(x_gate), _ptr(labels), _ptr(a_out), _ptr(v_out),
                                    _ptr(logits), _ptr(counts), B, n, _stream()), "gdl_eval_head")


@_op("eval_count", 1, lambda logits, labels, counts, B, n: ("bytes", 12.0 * B * n + 8.0 * B))
def eval_count(logits, labels, counts, B, n):
    """counts[h] += #rows of logits[h] ([3, B, n]) whose arg-max equals the label."""
    check(_lib.load().gdl_eval_count(_ptr(logits), _ptr(labels), _ptr(counts), B, n, _stream()), "gdl_eval_count")


@_op("eval_confusion", 1, lambda logits, labels, conf, out_of_range, B, n: ("bytes", 12.0 * B * n + 8.0 * B))
def eval_confusion(logits, labels, conf, out_of_range, B, n):
    """conf[h][label][pred] += 1 for the arg-max pred of every row of logits[h] ([3, B, n]) and its label (conf int64
    [3, n, n]); labels < 0 are skipped, labels >= n only add to out_of_range (int64 [1])."""
    check(_lib.load().gdl_eval_confusion(_ptr(logits), _ptr(labels), _ptr(conf), _ptr(out_of_range), B, n, _stream()),
          "gdl_eval_confusion")


@_op("eval_scores", 2, lambda logits, labels, store, store_labels, cursor, hits, overflow, B, n, k:
     ("bytes", 24.0 * B * n + 12.0 * B))
def eval_scores(logits, labels, store, store_labels, cursor, hits, overflow, B, n, k):
    """Append softmax(logits[h]) of the B rows of logits [3, B, n] class-major to store f32 [3, n, cap] at row
    cursor (int64 [1], advanced by B) and their labels to store_labels int32 [cap] (-1 outside 0..n-1); hits int64 [3]
    += the rows whose label ranks < k (NaN largest, ties to the lower index); labelled rows beyond cap only add to
    overflow (int64 [1])."""
    check(_lib.load().gdl_eval_scores(_ptr(logits), _ptr(labels), B, n, k, _ptr(store), _ptr(store_labels),
                                      store.shape[-1], _ptr(cursor), _ptr(hits), _ptr(overflow), _stream()),
          "gdl_eval_scores")


def eval_ap_workspace_bytes(cap, n):
    """Device workspace gdl_eval_ap needs for a store of cap rows (0 when a column sorts in shared memory)."""
    return int(_lib.load().gdl_eval_ap_workspace_bytes(cap, n))


@_op("eval_ap", 2, lambda store, store_labels, cursor, ap, support, nonfinite, workspace=None:
     ("bytes", 4.0 * store.numel() + 4.0 * store_labels.numel() * (store.shape[0] * store.shape[1] + 1)))
def eval_ap(store, store_labels, cursor, ap, support, nonfinite, workspace=None):
    """ap f64 [3, n] = the average precision of every (head, class) column of store f32 [3, n, cap] over its first
    min(cursor, cap) rows whose store_labels (int32 [cap]) are in 0..n-1 (NaN for a class without rows); support
    int64 [n] = rows per class; nonfinite int64 [1] = rows with a non-finite score.  workspace: uint8 of at least
    eval_ap_workspace_bytes(cap, n) bytes when that is not 0."""
    cap, n = store.shape[-1], store.shape[1]
    check(_lib.load().gdl_eval_ap(_ptr(store), _ptr(store_labels), _ptr(cursor), cap, n, _ptr(ap), _ptr(support),
                                  _ptr(nonfinite), _ptr(workspace), 0 if workspace is None else workspace.numel(),
                                  _stream()), "gdl_eval_ap")


@_op("softmax_ce", 2)
def softmax_ce(logits, labels, loss_scale, grad_scale, loss_out, dlogits, scratch, B, n):
    check(_lib.load().gdl_softmax_ce(_ptr(logits), _ptr(labels), loss_scale, grad_scale, _ptr(loss_out),
                                     _ptr(dlogits), _ptr(scratch), B, n, _stream()), "gdl_softmax_ce")


# ---------------------------------------------------------------------------------- FiLM head
@_op("gemm_nt", 1, lambda A, lda, Bm, Cm, M, N, K: ("flops", 2.0 * M * N * K))
def gemm_nt_bf16(A, lda, Bm, Cm, M, N, K):
    """C[M][N] bf16 = A[M][K] (row stride lda) * B[N][K]^T on the flat-window conv kernel."""
    check(_lib.load().gdl_gemm_nt_bf16(_addr(A), lda, _ptr(Bm), _ptr(Cm), M, N, K, _stream()), "gdl_gemm_nt_bf16")


def gemm_tn_workspace_bytes(M, N, K):
    return int(_lib.load().gdl_gemm_tn_workspace_bytes(M, N, K))


@_op("gemm_tn", 2, lambda At, Bt, bias, Cm, M, N, K, ws: ("flops", 2.0 * M * N * K))
def gemm_tn_f32(At, Bt, bias, Cm, M, N, K, ws):
    """C[M][N] f32 = At[K][M]^T * Bt[K][N] (+ bias) on the flat-window wgrad kernel (split-K)."""
    check(_lib.load().gdl_gemm_tn_f32(_ptr(At), _ptr(Bt), _ptr(bias), _ptr(Cm), M, N, K, _ptr(ws),
                                      ws.numel() * ws.element_size(), _stream()), "gdl_gemm_tn_f32")


@_op("gemm_tn", 2, lambda At, Bt, Cm, M, N, K, ws: ("flops", 2.0 * M * N * K))
def gemm_tn_f32_acc(At, Bt, Cm, M, N, K, ws):
    """C += At^T * Bt: a later K chunk of a reduction started by gemm_tn_f32."""
    check(_lib.load().gdl_gemm_tn_f32_acc(_ptr(At), _ptr(Bt), _ptr(Cm), M, N, K, _ptr(ws),
                                          ws.numel() * ws.element_size(), _stream()), "gdl_gemm_tn_f32_acc")


def film_scratch_floats(B, D):
    return int(_lib.load().gdl_film_scratch_floats(B, D))


@_op("film_outer", 2, lambda a, v, Zt, B, D, ZB, variants, scratch: ("bytes", 2.0 * D * D * ZB))
def film_outer(a, v, Zt, B, D, ZB, variants, scratch):
    check(_lib.load().gdl_film_outer(_ptr(a), _ptr(v), _ptr(Zt), B, D, ZB, variants, _ptr(scratch), _stream()),
          "gdl_film_outer")


@_op("film_outer", lambda a, v, Zt, B, D, ZB, variants, scratch, f0, nf: 2 if f0 == 0 else 1,
     lambda a, v, Zt, B, D, ZB, variants, scratch, f0, nf: ("bytes", 2.0 * nf * ZB))
def film_outer_chunk(a, v, Zt, B, D, ZB, variants, scratch, f0, nf):
    check(_lib.load().gdl_film_outer_chunk(_ptr(a), _ptr(v), _ptr(Zt), B, D, ZB, variants, _ptr(scratch), f0, nf,
                                           _stream()), "gdl_film_outer_chunk")


@_op("cast_pad", 1)
def cast_pad_bf16(src0, r0, src1, r1, cols, ld, transpose, dst, drows, dcols):
    check(_lib.load().gdl_cast_pad_bf16(_ptr(src0), r0, _ptr(src1), r1, cols, ld, int(transpose), _ptr(dst),
                                        drows, dcols, _stream()), "gdl_cast_pad_bf16")


@_op("film_contract", 2, lambda G, ldg, c0, x, y, dx, dy, B, D, sum_mode, scratch: ("bytes", 4.0 * D * D * B))
def film_contract(G, ldg, c0, x, y, dx, dy, B, D, sum_mode, scratch):
    check(_lib.load().gdl_film_contract(_ptr(G), ldg, c0, _ptr(x), _ptr(y), _ptr(dx), _ptr(dy), B, D,
                                        int(sum_mode), _ptr(scratch), _stream()), "gdl_film_contract")


@_op("film_contract", lambda G, ldg, c0, x, y, dx, dy, B, D, sum_mode, scratch, i0, ni, acc, rebuild: 2 if rebuild else 1,
     lambda G, ldg, c0, x, y, dx, dy, B, D, sum_mode, scratch, i0, ni, acc, rebuild: ("bytes", 4.0 * ni * D * B))
def film_contract_chunk(G, ldg, c0, x, y, dx, dy, B, D, sum_mode, scratch, i0, ni, acc, rebuild):
    check(_lib.load().gdl_film_contract_chunk(_ptr(G), ldg, c0, _ptr(x), _ptr(y), _ptr(dx), _ptr(dy), B, D,
                                              int(sum_mode), _ptr(scratch), i0, ni, int(acc), int(rebuild), _stream()),
          "gdl_film_contract_chunk")


@_op("transpose", 1, lambda src, dst, R, Cn, ldd, c0: ("bytes", 6.0 * R * Cn))
def transpose_bf16_to_f32_window(src, dst, R, Cn, ldd, c0):
    check(_lib.load().gdl_transpose_bf16_to_f32_window(_ptr(src), _ptr(dst), R, Cn, ldd, c0, _stream()),
          "gdl_transpose_bf16_to_f32_window")


@_op("transpose", 1, lambda src, dst, R, Cn: ("bytes", 6.0 * R * Cn))
def transpose_f32_to_bf16(src, dst, R, Cn):
    check(_lib.load().gdl_transpose_f32_to_bf16(_ptr(src), _ptr(dst), R, Cn, _stream()),
          "gdl_transpose_f32_to_bf16")


@_op("transpose", 1, lambda src, dst, R, Cn: ("bytes", 6.0 * R * Cn))
def transpose_bf16_to_f32(src, dst, R, Cn):
    check(_lib.load().gdl_transpose_bf16_to_f32(_ptr(src), _ptr(dst), R, Cn, _stream()),
          "gdl_transpose_bf16_to_f32")


@_op("gated_fwd", 1)
def gated_fwd(hx, hy, m_out, m_x, m_y):
    check(_lib.load().gdl_gated_fwd(_ptr(hx), _ptr(hy), _ptr(m_out), _ptr(m_x), _ptr(m_y), hx.numel(),
                                    _stream()), "gdl_gated_fwd")


@_op("gated_bwd", 1)
def gated_bwd(hx, hy, dm_x, dm_y, dhx, dhy):
    check(_lib.load().gdl_gated_bwd(_ptr(hx), _ptr(hy), _ptr(dm_x), _ptr(dm_y), _ptr(dhx), _ptr(dhy),
                                    hx.numel(), _stream()), "gdl_gated_bwd")


# ---------------------------------------------------------------------------------- optimizer
def optim_scratch_floats(numel, nseg):
    return int(_lib.load().gdl_optim_scratch_floats(numel, nseg))


@_op("grad_stats", 2, lambda grad, numel, *a: ("bytes", 4.0 * numel))
def grad_stats(grad, numel, seg_end, seg_group, seg_inv_numel, nseg, max_norm, scratch, stats):
    check(_lib.load().gdl_grad_stats(_ptr(grad), numel, _ptr(seg_end), _ptr(seg_group),
                                     _ptr(seg_inv_numel), nseg, max_norm, _ptr(scratch), _ptr(stats),
                                     _stream()), "gdl_grad_stats")


def _lr_dev(lr):
    """The device pointer of an lr held in device memory (a float64 CUDA tensor of one element), or None for a Python
    number (the host-lr entries)."""
    if not isinstance(lr, torch.Tensor):
        return None
    assert lr.is_cuda and lr.dtype == torch.float64 and lr.numel() == 1, "a device lr is one float64 on the GPU"
    return _ptr(lr)


# lr: a Python number, or a float64 CUDA tensor of one element that the update reads on the device (the *_lr_dev
# entries: a captured update then follows whatever the tensor holds when it is replayed)
@_op("sgd_momentum", 1, lambda param, grad, buf, numel, *a: ("bytes", 24.0 * numel))
def sgd_momentum(param, grad, buf, numel, lr, mu, wd, first_step, stats):
    lib, dev = _lib.load(), _lr_dev(lr)
    if dev is None:
        check(lib.gdl_sgd_momentum(_ptr(param), _ptr(grad), _ptr(buf), numel, lr, mu, wd, int(first_step),
                                   _ptr(stats), _stream()), "gdl_sgd_momentum")
    else:
        check(lib.gdl_sgd_momentum_lr_dev(_ptr(param), _ptr(grad), _ptr(buf), numel, dev, mu, wd, int(first_step),
                                          _ptr(stats), _stream()), "gdl_sgd_momentum_lr_dev")


# Adam / Adagrad: step_state is the int32 [3] device counter of include/gdl_b200.h (one launch advances it, one updates)
@_op("adam", 2, lambda param, grad, m, v, step_state, numel, *a: ("bytes", 32.0 * numel))
def adam(param, grad, exp_avg, exp_avg_sq, step_state, numel, lr, beta1, beta2, eps, wd, stats):
    lib, dev = _lib.load(), _lr_dev(lr)
    if dev is None:
        check(lib.gdl_adam(_ptr(param), _ptr(grad), _ptr(exp_avg), _ptr(exp_avg_sq), _ptr(step_state), numel, lr,
                           beta1, beta2, eps, wd, _ptr(stats), _stream()), "gdl_adam")
    else:
        check(lib.gdl_adam_lr_dev(_ptr(param), _ptr(grad), _ptr(exp_avg), _ptr(exp_avg_sq), _ptr(step_state), numel,
                                  dev, beta1, beta2, eps, wd, _ptr(stats), _stream()), "gdl_adam_lr_dev")


@_op("adagrad", 2, lambda param, grad, s, step_state, numel, *a: ("bytes", 24.0 * numel))
def adagrad(param, grad, state_sum, step_state, numel, lr, lr_decay, eps, wd, stats):
    lib, dev = _lib.load(), _lr_dev(lr)
    if dev is None:
        check(lib.gdl_adagrad(_ptr(param), _ptr(grad), _ptr(state_sum), _ptr(step_state), numel, lr, lr_decay, eps,
                              wd, _ptr(stats), _stream()), "gdl_adagrad")
    else:
        check(lib.gdl_adagrad_lr_dev(_ptr(param), _ptr(grad), _ptr(state_sum), _ptr(step_state), numel, dev,
                                     lr_decay, eps, wd, _ptr(stats), _stream()), "gdl_adagrad_lr_dev")


@_op("grad_accumulate", 1, lambda dst, src, numel, accumulate: ("bytes", (12.0 if accumulate else 8.0) * numel))
def grad_accumulate(dst, src, numel, accumulate):
    """dst[:numel] = src[:numel] (accumulate False) or dst[:numel] += src[:numel]."""
    check(_lib.load().gdl_grad_accumulate(_ptr(dst), _ptr(src), numel, int(accumulate), _stream()),
          "gdl_grad_accumulate")


# ---------------------------------------------------------------------------------- data pipeline
@_op("crop_resize_normalize", 2,
     lambda store, n, Hs, Ws, params, frames, T, S, mean, std, out, table: ("bytes", frames * 3.0 * S * S * 4.0))
def crop_resize_normalize(store, store_frames, Hs, Ws, params, frames, T, S, mean3, std3, out, table):
    """uint8 frame store + host-drawn crop boxes -> normalised fp32 [frames/T, 3, T, S, S] (datapipe.cu).
    mean3 / std3 are ctypes float[3] (host constants)."""
    check(_lib.load().gdl_crop_resize_normalize(_ptr(store), store_frames, Hs, Ws, _ptr(params), frames, T, S,
                                                C.cast(mean3, C.c_void_p), C.cast(std3, C.c_void_p), _ptr(out),
                                                _ptr(table), _stream()), "gdl_crop_resize_normalize")


@_op("log_stft", 1, lambda waves, stride, lens, params, B, L, n_fft, hop, pad, out: ("bytes", 4.0 * B * L + 4.0 * out.numel()))
def log_stft(waves, clip_stride, clip_len, params, B, L, n_fft, hop, pad_mode, out):
    check(_lib.load().gdl_log_stft(_ptr(waves), clip_stride, _ptr(clip_len), _ptr(params), B, L, n_fft, hop, pad_mode,
                                   _ptr(out), _stream()), "gdl_log_stft")
