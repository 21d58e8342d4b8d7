"""The fusion heads of the fused training and eval steps: `fusion_head(fm)` is the one place that tells the four
DGL heads apart.  Each head object provides

    trainable()           the parameters that receive a gradient from Lf (everything else stays grad-less)
    train(st)             the fused DGL head of a training step (step.DGLStep: features, labels, logits, losses, da/dv)
    eval(ev, fa, Ga, fv, Gv)  pooling of the bf16 layer-4 maps, the three logit sets and the correct counts
                          (step.EvalStep: labels, logits, counts)
    refresh_shadows()     re-derive the head's bf16 weight shadows from the fp32 parameters (FiLM only)

Constructed without a device (`fusion_head(fm)`) a head allocates nothing, so `trainable()` works on the CPU.
"""
import torch

from . import ops
from .film import FilmHead
from .fusion_modules import ConcatFusion_DGL, FiLM_DGL, GatedFusion_DGL, SumFusion_DGL

D = 512


class _LinearHead:
    """concat (kind 0: fc_out over [a | v]) and sum (kind 1: fc_x(a) + fc_y(v)): csrc/head.cu dgl_head_linear and
    the eval_head kinds 0 / 1.  _sides(): the (weight, first column, bias or None) that multiply a and v."""

    def __init__(self, fm, B=None, n=None, dev=None):
        self.fm = fm
        if dev is not None:
            self.scratch = torch.empty(ops.head_scratch_floats(B, n) + 64, device=dev)

    def _operands(self, grad):
        """(Wx address, Wy address, bx, by) of the parameters, or of their gradients."""
        (Wx, cx, bx), (Wy, cy, by) = self._sides()
        W = lambda w, c: (w.grad if grad else w).data_ptr() + 4 * c
        b = lambda t: None if t is None else (t.grad if grad else t.data)
        return W(Wx, cx), W(Wy, cy), b(bx), b(by)

    def train(self, st):
        Wx, Wy, bx, by = self._operands(False)
        dWx, dWy, dbx, dby = self._operands(True)
        ops.dgl_head_linear(self.kind, st.a_feat, st.v_feat, Wx, Wy, self.ldw, bx, by, st.label_in, st.alpha,
                            st.inv_batch, st.logits, st.losses, st.da, st.dv, dWx, dWy, self.ldw, dbx, dby,
                            self.scratch, st.B, D, st.n)

    def eval(self, ev, fa, Ga, fv, Gv):
        Wx, Wy, bx, by = self._operands(False)
        ops.eval_head(self.kind, fa, Ga, fv, Gv, Wx, Wy, self.ldw, bx, by, None, None, 1, ev.label_in, None, None,
                      ev.logits, ev.counts, ev.B, ev.n)

    def refresh_shadows(self):
        pass


class ConcatHead(_LinearHead):
    """reference fusion_modules.py:45-59; fc_auxi is never used."""
    kind, ldw = 0, 2 * D

    def _sides(self):
        W, b = self.fm.fc_out.weight, self.fm.fc_out.bias
        return (W, 0, b), (W, D, None)

    def trainable(self):
        return [self.fm.fc_out.weight, self.fm.fc_out.bias]


class SumHead(_LinearHead):
    """reference fusion_modules.py:16-30."""
    kind, ldw = 1, D

    def _sides(self):
        fm = self.fm
        return (fm.fc_x.weight, 0, fm.fc_x.bias), (fm.fc_y.weight, 0, fm.fc_y.bias)

    def trainable(self):
        return [self.fm.fc_x.weight, self.fm.fc_x.bias, self.fm.fc_y.weight, self.fm.fc_y.bias]


class GatedHead:
    """reference fusion_modules.py:230-250 with the DGL routing, one fused pass (csrc/head.cu
    dgl_gated_sample/param_kernel): fc_out <- Lf; a, v <- alpha*La/Lv through fc_out, the gates and fc_x / fc_y;
    fc_x / fc_y themselves get no gradient.  Training gates with x_gate=True; eval honours the module's x_gate."""

    def __init__(self, fm, B=None, n=None, dev=None):
        self.fm = fm
        if dev is not None:
            self.scratch = torch.empty(ops.gated_head_scratch_floats(B, n) + 64, device=dev)

    def trainable(self):
        return [self.fm.fc_out.weight, self.fm.fc_out.bias]

    def train(self, st):
        fm = self.fm
        Wo, bo = fm.fc_out.weight, fm.fc_out.bias
        ops.dgl_head_gated(st.a_feat, st.v_feat, fm.fc_x.weight.data, fm.fc_x.bias.data, fm.fc_y.weight.data,
                           fm.fc_y.bias.data, Wo.data, bo.data, st.label_in, st.alpha, st.inv_batch, st.logits,
                           st.losses, st.da, st.dv, Wo.grad, bo.grad, self.scratch, st.B, D, st.n)

    def eval(self, ev, fa, Ga, fv, Gv):
        fm = self.fm
        ops.eval_head(2, fa, Ga, fv, Gv, fm.fc_x.weight.data_ptr(), fm.fc_y.weight.data_ptr(), D, fm.fc_x.bias.data,
                      fm.fc_y.bias.data, fm.fc_out.weight.data, fm.fc_out.bias.data, fm.x_gate, ev.label_in, None,
                      None, ev.logits, ev.counts, ev.B, ev.n)

    def refresh_shadows(self):
        pass


def fusion_head(fm, B=None, n=None, dev=None):
    """The head object of fusion module `fm`, with the buffers of batch B and n classes on `dev` (none without)."""
    for cls, head in ((ConcatFusion_DGL, ConcatHead), (SumFusion_DGL, SumHead), (GatedFusion_DGL, GatedHead),
                      (FiLM_DGL, FilmHead)):
        if isinstance(fm, cls):
            return head(fm, B, n, dev)
    raise NotImplementedError('Incorrect fusion method: {}!'.format(type(fm).__name__))
