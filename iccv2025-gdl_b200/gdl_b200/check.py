"""FP32 check mode of the encoders (north_star: "losses within 1e-4 with an FP32-accumulate check mode").

`CheckEncoder` has the interface `step.DGLStep` uses of `engine.EncoderEngine`, but stores every activation in
fp32 (NCHW, the reference's own layout) and runs the CUDA-core fp64-accumulating kernels of csrc/check_fp32.cu on
the fp32 nn.Parameters directly.  It is selected explicitly (`DGLStep(..., check_fp32=True)` / `GDL_CHECK_FP32=1`),
never silently: the product path is the bf16 tcgen05 engine.  Everything around the encoders — input staging, the
fused DGL head, gradient truncation, clipping statistics, SGD-momentum, the arena, the all-reduce — is the SAME
code as the product path, so a free-running comparison of this mode against the fp32 reference checks the whole
step orchestration to fp32 accuracy (reference main_dgl.py:100-158, models/backbone.py:52-68,160-201).
"""
import ctypes as C

import torch

from . import _lib, ops
from ._lib import check


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _s():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _count(n=1):
    ops.LAUNCHES += n


class _Unit:
    """conv + BN (+ReLU) with fp32 saved tensors."""

    def __init__(self, eng, conv, bn, N, Hi, Wi, relu):
        Co, Ci, R, S = conv.weight.shape
        self.conv, self.bn, self.relu, self.ci = conv, bn, relu, Ci
        self.d = ops.conv_desc(N, Hi, Wi, Ci, Co, R, S, conv.stride[0], conv.padding[0])
        self.N, self.C, self.HW = N, Co, self.d.Ho * self.d.Wo
        dev = eng.device
        self.x = torch.empty(N, Co, self.d.Ho, self.d.Wo, device=dev)  # conv output
        self.y = torch.empty_like(self.x)                               # [relu](bn(x) [+ res])
        self.mean, self.invstd = torch.empty(Co, device=dev), torch.empty(Co, device=dev)

    def forward(self, inp, res=None, training=True, running=None):
        """running: the (mean, var) pair a training-mode forward updates (default: the module's own)."""
        lib, bn = _lib.load(), self.bn
        rm, rv = running if running is not None else (bn.running_mean, bn.running_var)
        check(lib.gdl_check_conv_fwd(C.byref(self.d), self.ci, _p(inp), _p(self.conv.weight.data), _p(self.x), _s()),
              "gdl_check_conv_fwd")
        check(lib.gdl_check_bn_fwd(_p(self.x), _p(res), _p(self.y), self.N, self.C, self.HW, _p(bn.weight.data),
                                   _p(bn.bias.data), bn.eps, bn.momentum, _p(rm), _p(rv),
                                   _p(self.mean), _p(self.invstd), int(self.relu), int(training), _s()),
              "gdl_check_bn_fwd")
        _count(2)
        return self.y

    def bn_backward(self, eng, dy, dz_out, dx):
        bn = self.bn
        check(_lib.load().gdl_check_bn_bwd(_p(dy), _p(self.y), _p(self.x), _p(dz_out), _p(dx), self.N, self.C, self.HW,
                                           _p(bn.weight.data), _p(self.mean), _p(self.invstd), _p(eng._grad(bn.weight)),
                                           _p(eng._grad(bn.bias)), int(self.relu), _s()), "gdl_check_bn_bwd")
        _count()

    def wgrad(self, eng, inp, d_c):
        check(_lib.load().gdl_check_conv_wgrad(C.byref(self.d), self.ci, _p(inp), _p(d_c), _p(eng._grad(self.conv.weight)),
                                               _s()), "gdl_check_conv_wgrad")
        _count()

    def dgrad(self, d_c, add, dx):
        check(_lib.load().gdl_check_conv_dgrad(C.byref(self.d), self.ci, _p(d_c), _p(self.conv.weight.data), _p(add), _p(dx),
                                               _s()), "gdl_check_conv_dgrad")
        _count()


class CheckEncoder:
    N_LATE_BLOCKS = 4
    grad_override = None

    def __init__(self, net, N, H, W, device, frames=1):
        """net: backbone.ResNet; N = B*frames images of H x W; the input is the fp32 batch itself
        ([B,H,W] spectrograms or [B,3,T,H,W] frames, folded here)."""
        ops.init()
        self.net, self.N, self.H, self.W, self.device, self.T = net, N, H, W, device, frames
        cin = net.conv1.weight.shape[1]
        self.cin = cin
        self.input_shape = (N, cin, H, W)
        self.stem = _Unit(self, net.conv1, net.bn1, N, H, W, True)
        H1, W1 = self.stem.d.Ho, self.stem.d.Wo
        self.Hp, self.Wp = (H1 - 1) // 2 + 1, (W1 - 1) // 2 + 1
        self.pool_y = torch.empty(N, 64, self.Hp, self.Wp, device=device)
        self.pool_idx = torch.empty(N, 64, self.Hp, self.Wp, device=device, dtype=torch.int32)
        self.units, self.blocks = [self.stem], []
        h, w = self.Hp, self.Wp
        for li in range(1, 5):
            for blk in getattr(net, "layer%d" % li):
                u1 = _Unit(self, blk.conv1, blk.bn1, N, h, w, True)
                u2 = _Unit(self, blk.conv2, blk.bn2, N, u1.d.Ho, u1.d.Wo, True)
                ud = None
                if blk.downsample is not None:
                    ud = _Unit(self, blk.downsample[0], blk.downsample[1], N, h, w, False)
                self.units += [u for u in (u1, u2, ud) if u is not None]
                self.blocks.append((u1, u2, ud))
                h, w = u1.d.Ho, u1.d.Wo
        self.Hf, self.Wf, self.Cf = h, w, 512
        self.g_feat = torch.empty(N, 512, h, w, device=device)
        self.folded = torch.empty(N, cin, H, W, device=device)  # private copy: the staging set may be refilled
        self.stats_sink = (torch.zeros(512, device=device), torch.zeros(512, device=device))  # see EncoderEngine

    # ---- interface shared with engine.EncoderEngine ------------------------------------------------------
    def repack(self):
        pass  # the fp32 parameters are the operands

    def _grad(self, p):
        if self.grad_override is not None:
            return self.grad_override[p]
        if p.grad is None:
            p.grad = torch.zeros_like(p.data)
        return p.grad

    def parameters(self):
        out = []
        for u in self.units:
            out += [u.conv.weight, u.bn.weight, u.bn.bias]
        return out

    def late_parameters(self):
        out = []
        for blk in self.blocks[len(self.blocks) - self.N_LATE_BLOCKS:]:
            for u in blk:
                if u is not None:
                    out += [u.conv.weight, u.bn.weight, u.bn.bias]
        return out

    def stage_input(self, src, B):
        """fp32 batch -> the encoder's own input buffer, frames folded into the batch (reference backbone.py:162-164;
        for the spectrograms C = T = 1 and this is a copy, main_dgl.py:100 unsqueeze(1).float())."""
        check(_lib.load().gdl_check_fold_frames(_p(src), _p(self.folded), B, self.cin, self.T, self.H, self.W, _s()),
              "gdl_check_fold_frames")
        _count()
        self.x_in = self.folded

    def forward(self, x_unused=None, training=True, own_stats=True):
        lib = _lib.load()
        run = None if own_stats else self.stats_sink
        s = self.stem
        y0 = s.forward(self.x_in, training=training, running=run)
        check(lib.gdl_check_maxpool_fwd(_p(y0), _p(self.pool_y), _p(self.pool_idx), self.N * 64, s.d.Ho, s.d.Wo, self.Hp,
                                        self.Wp, _s()), "gdl_check_maxpool_fwd")
        _count()
        u = self.pool_y
        for (u1, u2, ud) in self.blocks:
            y1 = u1.forward(u, training=training, running=run)
            ident = u if ud is None else ud.forward(u, training=training, running=run)
            u = u2.forward(y1, res=ident, training=training, running=run)
        return u

    def gap_fwd(self, feat, out, B):
        check(_lib.load().gdl_check_gap_fwd(_p(feat), _p(out), B, self.T, 512, self.Hf * self.Wf, _s()), "gdl_check_gap_fwd")
        _count()

    def gap_bwd(self, dout, B):
        check(_lib.load().gdl_check_gap_bwd(_p(dout), _p(self.g_feat), B, self.T, 512, self.Hf * self.Wf, _s()),
              "gdl_check_gap_bwd")
        _count()

    def backward(self, x_unused=None, part=None):
        chain = list(zip(reversed(self.blocks), reversed(self._block_inputs())))
        if part == 0:
            chain = chain[:self.N_LATE_BLOCKS]
        elif part == 1:
            chain = chain[self.N_LATE_BLOCKS:]
        g_out = self.g_feat if part != 1 else self._g_mid
        for (u1, u2, ud), in_t in chain:
            dz = torch.empty_like(u2.y)
            d_c2 = torch.empty_like(u2.x)
            u2.bn_backward(self, g_out, dz, d_c2)           # out = relu(bn2(c2) + identity)
            u2.wgrad(self, u1.y, d_c2)
            g_y1 = torch.empty_like(u1.y)
            u2.dgrad(d_c2, None, g_y1)
            d_c1 = torch.empty_like(u1.x)
            u1.bn_backward(self, g_y1, None, d_c1)
            u1.wgrad(self, in_t, d_c1)
            g_u = torch.empty_like(in_t)
            if ud is not None:
                d_cd = torch.empty_like(ud.x)
                ud.bn_backward(self, dz, None, d_cd)        # identity = bn_d(conv1x1_s2(u)), no relu
                ud.wgrad(self, in_t, d_cd)
                g_ds = torch.empty_like(in_t)
                ud.dgrad(d_cd, None, g_ds)
                u1.dgrad(d_c1, g_ds, g_u)
            else:
                u1.dgrad(d_c1, dz, g_u)
            g_out = g_u
        if part == 0:
            self._g_mid = g_out
            return
        s = self.stem
        g_y0 = torch.empty_like(s.y)
        check(_lib.load().gdl_check_maxpool_bwd(_p(g_out), _p(self.pool_idx), _p(g_y0), self.N * 64, s.d.Ho, s.d.Wo, self.Hp,
                                                self.Wp, _s()), "gdl_check_maxpool_bwd")
        _count()
        d_c0 = torch.empty_like(s.x)
        s.bn_backward(self, g_y0, None, d_c0)
        s.wgrad(self, self.x_in, d_c0)

    def _block_inputs(self):
        ins = [self.pool_y]
        for (u1, u2, ud) in self.blocks[:-1]:
            ins.append(u2.y)
        return ins
