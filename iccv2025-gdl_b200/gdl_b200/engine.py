"""EncoderEngine — runs one ResNet-18 modality encoder (reference models/backbone.py:160-201
forward, and its autograd backward) entirely through the sm_100a kernels of libgdl_b200.so.

The engine borrows the parameters of a `backbone.ResNet` module (fp32, reference names and
shapes), keeps bf16 packed shadows of the conv weights, and owns a static set of NHWC bf16
activation / gradient buffers for one input geometry, so a whole step is a fixed sequence of
kernel launches on fixed addresses (CUDA-graph capturable, no allocation inside the step).

Data layout in HBM:
  activations     bf16 NHWC  [N, H, W, C]                      (C = 64..512; stem input C = 8 padded)
  conv weights    fp32 OIHW master (the nn.Parameter)  +  bf16 [Co, Kp] (k = (r,s,ci)) for fwd/wgrad
                  +  bf16 [Ci, R*S*Co] (k = (r,s,co)) for dgrad
  BN              fp32 per-channel gamma/beta/running stats (nn.Parameter / buffers), fp32 batch
                  mean / invstd / fused scale+shift saved for backward
  gradients       activations bf16 NHWC; parameters fp32 written straight into p.grad storage
"""
import os

import torch

from . import ops


# Measured on B=256: no gain (24.05 vs 23.88 ms) — the two encoder streams already keep the GPU busy and the
# tensor-bound wgrads contend with the BN kernels for L2/HBM; kept as an option, off by default.
USE_WGRAD_STREAM = os.environ.get("GDL_WGRAD_STREAM", "0") != "0"

# Sweep directions (ops.sweep / gdl_set_sweep): every pass over a tensor larger than L2 leaves its LAST-touched
# part in the 126 MB L2, so the next pass over the same tensor should start there, i.e. run the other way.
#   0  every kernel ascending (the behaviour before this option)
#   1  BatchNorm passes alternate: statistics descending after the (ascending) conv, apply ascending; backward
#      reduce descending after the (ascending) dgrad, apply ascending
#   2  the convolutions alternate as well (conv1 of a block descending, conv2 ascending, BN passes in between)
SWEEP = int(os.environ.get("GDL_SWEEP", "1"))
APPLY_SWEEP = int(os.environ.get("GDL_APPLY_SWEEP", "1"))
STEM_STATS = int(os.environ.get("GDL_STEM_STATS", "1"))  # BatchNorm statistics of the stem from its epilogue


def note_writes(module):
    """Record that kernels changed `module`'s parameters or buffers behind torch's version counters (an optimizer
    update over the parameter arena, the BatchNorm running statistics of a training forward, a weight refresh).
    The eval-mode fold (EncoderEngine.fold_eval) and the FiLM eval shadow re-derive themselves when this count moves."""
    module._gdl_writes = getattr(module, "_gdl_writes", 0) + 1


def kernel_writes(module):
    return getattr(module, "_gdl_writes", 0)


class _Pool:
    """Static buffer planner: buffers are requested/released while the plan is built; a released
    buffer of the same size is reused by a later request (backward temporaries)."""

    def __init__(self, device):
        self.device = device
        self.free = {}
        self.total_bytes = 0

    def get(self, shape, dtype=torch.bfloat16):
        key = (tuple(shape), dtype)
        lst = self.free.get(key)
        if lst:
            return lst.pop()
        t = torch.empty(shape, device=self.device, dtype=dtype)
        self.total_bytes += t.numel() * t.element_size()
        return t

    def put(self, t):
        self.free.setdefault((tuple(t.shape), t.dtype), []).append(t)


class _ConvBN:
    """One conv + BatchNorm unit with its saved tensors."""

    def __init__(self, eng, name, conv, bn, N, Hi, Wi, ci_store, relu):
        w = conv.weight
        Co, ci_real, R, S = w.shape
        self.name = name
        self.conv, self.bn = conv, bn
        self.ci_real = ci_real
        self.relu = relu
        self.cdir = 0  # sweep direction of this unit's convolution (set by the engine for SWEEP == 2)
        self.d = ops.conv_desc(N, Hi, Wi, ci_store, Co, R, S, conv.stride[0], conv.padding[0])
        self.P = N * self.d.Ho * self.d.Wo
        self.C = Co
        dev = eng.device
        self.Kp = ops.conv_packed_k(self.d)
        self.wp = torch.zeros(Co, self.Kp, device=dev, dtype=torch.bfloat16)
        self.wT = None if ci_store == 8 else torch.zeros(ci_store, R * S * Co, device=dev, dtype=torch.bfloat16)
        self.x = torch.empty(N, self.d.Ho, self.d.Wo, Co, device=dev, dtype=torch.bfloat16)  # conv out
        self.y = torch.empty_like(self.x)                                                      # bn(+relu) out
        self.mean, self.invstd, self.scale, self.shift = (torch.empty(Co, device=dev) for _ in range(4))
        eng.max_wgrad_ws = max(eng.max_wgrad_ws, ops.conv_wgrad_workspace_bytes(self.d))
        eng.max_bn_partial = max(eng.max_bn_partial, ops.bn_partial_floats(self.P, Co))

    def repack(self):
        ops.conv_pack_weights(self.d, self.ci_real, self.conv.weight.data, self.wp, self.wT)

    def forward(self, eng, inp, res=None):
        """Training-mode unit (eval mode is EncoderEngine.forward_eval: BatchNorm folded into the conv)."""
        bn = self.bn
        c = self.cdir
        # batch statistics come out of the conv epilogue where the kernel supports it (no extra pass over x)
        ops.sweep(c)
        rows = ops.conv_fwd_stats(self.d, inp, self.wp, self.x, eng.bn_partial, self.ci_real)
        ops.sweep((not c) if SWEEP else 0)
        rm, rv = eng.running(bn)
        if rows:
            ops.bn_stats_finalize(eng.bn_partial, rows, self.P, self.C, bn.weight.data, bn.bias.data, bn.eps,
                                  bn.momentum, rm, rv, self.mean, self.invstd, self.scale, self.shift)
        else:
            ops.bn_stats(self.x, self.P, self.C, eng.bn_partial, bn.weight.data, bn.bias.data, bn.eps,
                         bn.momentum, rm, rv, self.mean, self.invstd, self.scale, self.shift)
        # with the statistics out of the conv epilogue the apply pass is the FIRST pass over x after the convolution: it
        # walks against the convolution's direction (starts on the tail that is still in L2) and leaves the head of y,
        # where the next convolution starts, in L2.  GDL_APPLY_SWEEP=0: the round-1 order (same direction).
        ops.sweep(((not c) if (rows and APPLY_SWEEP and SWEEP) else c))
        ops.bn_apply(self.x, res, self.y, self.P, self.C, self.scale, self.shift, self.relu)
        return self.y


class _StemBN(_ConvBN):
    """The 7x7/s2 stem + BN: space-to-depth implicit GEMM (csrc/conv_stem.cu)."""

    def __init__(self, eng, conv, bn, N, H, W):
        Co, ci_real, R, S = conv.weight.shape
        assert (Co, R, S) == (64, 7, 7) and conv.stride[0] == 2 and conv.padding[0] == 3
        self.name, self.conv, self.bn, self.ci_real, self.relu = "conv1", conv, bn, ci_real, True
        self.N, self.H, self.W = N, H, W
        self.d = ops.conv_desc(N, H, W, 8, 64, 7, 7, 2, 3)  # geometry only (Ho, Wo)
        self.Ho, self.Wo, self.Hp, self.Wp = ops.stem_geometry(H, W)
        assert (self.Ho, self.Wo) == (self.d.Ho, self.d.Wo)
        self.P, self.C = N * self.Ho * self.Wo, 64
        dev = eng.device
        self.wp = torch.zeros(64, 256, device=dev, dtype=torch.bfloat16)
        self.wT = None
        self.x = torch.empty(N, self.Ho, self.Wo, 64, device=dev, dtype=torch.bfloat16)
        self.y = None  # relu(bn(x)) is never materialised: the stem tail is fused with the max-pool
        self.mean, self.invstd, self.scale, self.shift = (torch.empty(64, device=dev) for _ in range(4))
        eng.max_wgrad_ws = max(eng.max_wgrad_ws, ops.stem_wgrad_workspace_bytes(N, H, W))
        eng.max_bn_partial = max(eng.max_bn_partial, ops.bn_partial_floats(self.P, 64))

    def repack(self):
        ops.stem_pack_weights(self.conv.weight.data, self.wp, self.ci_real)

    def forward(self, eng, x16, res=None):
        bn = self.bn
        rm, rv = eng.running(bn)
        if STEM_STATS:  # batch statistics out of the stem's epilogue: no separate pass over the largest activation
            rows = ops.stem_fwd_stats(x16, self.wp, self.x, self.N, self.H, self.W, self.ci_real, eng.bn_partial)
            ops.bn_stats_finalize(eng.bn_partial, rows, self.P, self.C, bn.weight.data, bn.bias.data, bn.eps,
                                  bn.momentum, rm, rv, self.mean, self.invstd, self.scale, self.shift)
            ops.sweep(1 if SWEEP else 0)
        else:
            ops.stem_fwd(x16, self.wp, self.x, self.N, self.H, self.W, self.ci_real)
            ops.sweep(1 if SWEEP else 0)
            ops.bn_stats(self.x, self.P, self.C, eng.bn_partial, bn.weight.data, bn.bias.data, bn.eps,
                         bn.momentum, rm, rv, self.mean, self.invstd, self.scale, self.shift)
        # BN-apply + ReLU + MaxPool(3,2,1) in one pass (reference backbone.py:104-106)
        ops.bn_relu_maxpool_fwd(self.x, self.scale, self.shift, eng.pool_y, eng.pool_idx, eng.pool_xmax,
                                self.N, self.Ho, self.Wo, 64, eng.Hp, eng.Wp)
        return eng.pool_y


class EncoderEngine:
    def __init__(self, net, N, H, W, device):
        """net: backbone.ResNet; N images of H x W (audio: N=B, visual: N=B*T)."""
        ops.init()
        self.net = net
        self.N, self.H, self.W = N, H, W
        self.device = device
        self.max_wgrad_ws = 0
        self.max_bn_partial = 0
        self.units = []
        self.blocks = []
        self.stem = _StemBN(self, net.conv1, net.bn1, N, H, W)
        self.units.append(self.stem)
        self.input_shape = (N, self.stem.Hp, self.stem.Wp, 16)  # space-to-depth bf16 input (gdl_stem_layout)
        H1, W1 = self.stem.d.Ho, self.stem.d.Wo
        self.Hp, self.Wp = (H1 - 1) // 2 + 1, (W1 - 1) // 2 + 1
        self.pool_y = torch.empty(N, self.Hp, self.Wp, 64, device=device, dtype=torch.bfloat16)
        self.pool_idx = torch.empty(N, self.Hp, self.Wp, 64, device=device, dtype=torch.uint8)
        self.pool_xmax = torch.empty(N, self.Hp, self.Wp, 64, device=device, dtype=torch.bfloat16)  # conv out at arg-max
        h, w, cin = self.Hp, self.Wp, 64
        for li in range(1, 5):
            layer = getattr(net, "layer%d" % li)
            for bi, blk in enumerate(layer):
                pre = "layer%d.%d." % (li, bi)
                u1 = self._unit(pre + "conv1", blk.conv1, blk.bn1, N, h, w, cin, True)
                u2 = self._unit(pre + "conv2", blk.conv2, blk.bn2, N, u1.d.Ho, u1.d.Wo, u1.C, True)
                ud = None
                if blk.downsample is not None:
                    ud = self._unit(pre + "downsample", blk.downsample[0], blk.downsample[1], N, h, w, cin, False)
                if SWEEP >= 2:  # the block input was written ascending (max-pool / previous bn2 apply)
                    u1.cdir = 1
                    if ud is not None:
                        ud.cdir = 1
                self.blocks.append((u1, u2, ud))
                h, w, cin = u1.d.Ho, u1.d.Wo, u1.C
        self.Hf, self.Wf, self.Cf = h, w, cin
        self.wgrad_ws = torch.empty(max(self.max_wgrad_ws, 16) // 4, device=device, dtype=torch.float32)
        self.bn_partial = torch.empty(self.max_bn_partial, device=device, dtype=torch.float32)
        self.wgrad_stream = torch.cuda.Stream(device) if USE_WGRAD_STREAM else None
        # running-statistics sink of a forward that must leave the modules' running buffers untouched (a replica
        # other than the first of a DGLStep with replicas > 1): the finalize kernels update this pair instead
        self.stats_sink = (torch.zeros(512, device=device), torch.zeros(512, device=device))
        self.own_stats = True
        self._readers = {}
        self._eval_key_folded = None
        self._plan_backward()
        self.repack()

    def _unit(self, name, conv, bn, N, Hi, Wi, ci_store, relu):
        u = _ConvBN(self, name, conv, bn, N, Hi, Wi, ci_store, relu)
        self.units.append(u)
        return u

    # ------------------------------------------------------------------ weights
    def repack(self):
        """Refresh the bf16 shadows from the fp32 masters (after every optimizer step): one multi-tensor
        launch for the 19 block convolutions + the stem's own packer."""
        note_writes(self.net)  # parameters / running statistics changed behind torch's version counters
        convs = [u for u in self.units if u is not self.stem]
        key = tuple(u.conv.weight.data_ptr() for u in convs)
        if getattr(self, "_pack_key", None) != key:  # the parameters moved (e.g. into the step's arena)
            entries = [(u.conv.weight.data, u.wp, u.wT, u.C, u.d.Ci, u.ci_real, u.d.R, u.d.S, u.Kp) for u in convs]
            self._pack_table = ops.make_pack_table(entries, self.device)
            self._pack_key = key
        self.stem.repack()
        ops.conv_pack_weights_multi(*self._pack_table)

    # ------------------------------------------------------------------ eval mode: BatchNorm folded into the conv
    def _eval_key(self):
        v = kernel_writes(self.net)
        for u in self.units:
            bn = u.bn
            v += (u.conv.weight._version + bn.weight._version + bn.bias._version + bn.running_mean._version
                  + bn.running_var._version)
        return (v, tuple(u.conv.weight.data_ptr() for u in self.units))

    def fold_eval(self):
        """model.eval() (reference valid(), main_dgl.py:186): every BatchNorm uses its running statistics, so
        conv -> BN is one affine map per output channel.  scale = gamma / sqrt(running_var + eps) is folded into
        separate bf16 shadows (w' = w * scale, one multi-tensor pack launch with gdl_pack_entry.scale), and
        shift = beta - running_mean * scale becomes the bias of the conv epilogue (gdl_conv_fwd_bias_act), together
        with the residual add and the ReLU: an eval unit is ONE kernel, no BatchNorm pass.  Re-folded only when a
        parameter / buffer changed (torch version counters + the module's count of kernel-side writes, note_writes).
        Runs outside any CUDA graph: a graph that captured forward_eval reads the fold's fixed-address buffers."""
        key = self._eval_key()
        if self._eval_key_folded == key:
            return
        dev = self.device
        if not hasattr(self.stem, "wp_e"):
            for u in self.units:
                u.wp_e = torch.zeros_like(u.wp)
                u.scale_e, u.shift_e = torch.empty(u.C, device=dev), torch.empty(u.C, device=dev)
            self.ones64 = torch.ones(64, device=dev)
        for u in self.units:
            bn = u.bn
            ops.bn_eval_affine(bn.weight.data, bn.bias.data, bn.running_mean, bn.running_var, bn.eps,
                               u.scale_e, u.shift_e, u.C)
        convs = [u for u in self.units if u is not self.stem]
        entries = [(u.conv.weight.data, u.wp_e, None, u.C, u.d.Ci, u.ci_real, u.d.R, u.d.S, u.Kp, u.scale_e) for u in convs]
        self._pack_table_eval = ops.make_pack_table(entries, dev)  # holds raw addresses: rebuilt with the fold
        s = self.stem
        ops.stem_pack_weights_scaled(s.conv.weight.data, s.scale_e, s.wp_e, s.ci_real)
        ops.conv_pack_weights_multi(*self._pack_table_eval)
        self._eval_key_folded = key

    def forward_eval(self, x16):
        """Eval-mode forward with folded BatchNorm: stem conv -> (+shift, ReLU, max-pool) -> 8 blocks of three fused
        conv kernels (reference backbone.py:52-68 with model.eval())."""
        self.fold_eval()
        s = self.stem
        ops.sweep(0)
        ops.stem_fwd(x16, s.wp_e, s.x, s.N, s.H, s.W, s.ci_real)
        ops.bn_relu_maxpool_fwd(s.x, self.ones64, s.shift_e, self.pool_y, self.pool_idx, None, s.N, s.Ho, s.Wo, 64,
                                self.Hp, self.Wp)
        u = self.pool_y
        for (u1, u2, ud) in self.blocks:
            ops.conv_fwd_bias_act(u1.d, u, u1.wp_e, u1.shift_e, None, 1, u1.y)
            ident = u
            if ud is not None:
                ops.conv_fwd_bias_act(ud.d, u, ud.wp_e, ud.shift_e, None, 0, ud.y)
                ident = ud.y
            ops.conv_fwd_bias_act(u2.d, u1.y, u2.wp_e, u2.shift_e, ident, 1, u2.y)
            u = u2.y
        return u

    # ------------------------------------------------------------------ forward
    def running(self, bn):
        """The running-statistics pair a training-mode forward updates: the module's own, or the sink."""
        return (bn.running_mean, bn.running_var) if self.own_stats else self.stats_sink

    def forward(self, x16, training=True, own_stats=True):
        """x16: bf16 space-to-depth input [N,Hp,Wp,16] -> bf16 [N,Hf,Wf,512] (the layer4 map,
        reference backbone.py:175-181).  training=False: eval mode, BatchNorm folded into the convolutions.
        own_stats=False: batch statistics as usual, but the BatchNorm running buffers stay bit-identical (the
        choice is fixed into a CUDA graph that captures the call)."""
        if not training:
            return self.forward_eval(x16)
        self.own_stats = own_stats
        s = self.stem
        u = s.forward(self, x16)  # stem conv + BN + ReLU + max-pool -> pool_y
        for (u1, u2, ud) in self.blocks:
            y1 = u1.forward(self, u)
            ident = u
            if ud is not None:
                ident = ud.forward(self, u)
            # bn2 + residual + relu (reference backbone.py:62-66)
            u = u2.forward(self, y1, res=ident)
        ops.sweep(0)
        return u

    # ------------------------------------------------------------------ backward
    def _plan_backward(self):
        """Assign the (reused) gradient buffers of every block once."""
        pool = _Pool(self.device)
        plan = []
        N = self.N
        g_out = pool.get((N, self.Hf, self.Wf, self.Cf))
        self.g_feat = g_out
        for (u1, u2, ud) in reversed(self.blocks):
            d_c2 = pool.get(u2.x.shape)
            g_y1 = pool.get(u1.y.shape)
            d_c1 = pool.get(u1.x.shape)
            in_shape = (N, u1.d.Hi, u1.d.Wi, u1.d.Ci)
            g_u = pool.get(in_shape)
            d_cd = g_ds = None
            if ud is not None:
                d_cd = pool.get(ud.x.shape)
                g_ds = pool.get((N, ud.d.Ho, ud.d.Wo, ud.d.Ci))
            plan.append(dict(g_out=g_out, d_c2=d_c2, g_y1=g_y1, d_c1=d_c1, g_u=g_u, d_cd=d_cd, g_ds=g_ds))
            # lifetimes: everything but g_u dies with the block; g_out dies too
            for t in (d_c2, g_y1, d_c1, d_cd, g_ds, g_out):
                if t is not None:
                    pool.put(t)
            g_out = g_u
        s = self.stem
        self.g_pool = g_out                      # grad wrt maxpool output
        self.d_c0 = pool.get(s.x.shape)          # grad wrt the stem conv output
        self.bwd_plan = plan
        self.grad_buffer_bytes = pool.total_bytes

    grad_override = None  # optional {param: tensor} destination map (autograd-compatible mode)

    def _grad(self, p):
        if self.grad_override is not None:
            return self.grad_override[p]
        if p.grad is None:
            p.grad = torch.zeros_like(p.data)
        return p.grad

    def parameters(self):
        """Encoder parameters in the order the backward writes them (units order)."""
        out = []
        for u in self.units:
            out += [u.conv.weight, u.bn.weight, u.bn.bias]
        return out

    def _bn_bwd(self, u, dy, dz, dx, relu):
        bn = u.bn
        ops.bn_bwd(dy, u.y, u.x, dz, dx, u.P, u.C, bn.weight.data, u.mean, u.invstd, self.bn_partial,
                   self._grad(bn.weight), self._grad(bn.bias), relu)

    # ------------------------------------------------------------------ weight-gradient side stream
    # A weight gradient only needs the BN-backward output d_c and a saved forward activation, and nothing in
    # the backward chain needs ITS result: all wgrads run on a side stream, concurrently with the dgrad -> BN
    # chain, so the tensor-bound wgrad kernels overlap the HBM-bound BN kernels.  d_c buffers are reused by
    # later blocks: before the chain overwrites one, it waits for the wgrad that still reads it.
    def _wgrad(self, fn, d_c):
        ws = self.wgrad_stream
        if ws is None:
            fn()
            return
        main = torch.cuda.current_stream()
        ws.wait_stream(main)              # d_c is complete
        with torch.cuda.stream(ws):
            fn()
            ev = torch.cuda.Event()
            ev.record(ws)
        self._readers[d_c.data_ptr()] = ev

    def _before_write(self, buf):
        ev = self._readers.pop(buf.data_ptr(), None)
        if ev is not None:
            torch.cuda.current_stream().wait_event(ev)

    N_LATE_BLOCKS = 4  # layer4 + layer3: 94 % of the encoder's parameters, the first gradients to be complete

    def late_parameters(self):
        """Parameters whose gradients are complete after backward(part=0) (layer3 + layer4)."""
        out = []
        for (u1, u2, ud) in self.blocks[len(self.blocks) - self.N_LATE_BLOCKS:]:
            for u in (u1, u2, ud):
                if u is not None:
                    out += [u.conv.weight, u.bn.weight, u.bn.bias]
        return out

    def backward(self, x16, part=None):
        """Consumes self.g_feat (grad wrt the layer4 map, bf16) and writes every parameter
        gradient of the encoder into p.grad (overwrite).  x16 is the stem input of the forward.
        part=None runs the whole backward; part=0 only layer4 + layer3 (after which the gradients of
        late_parameters() are final and their all-reduce can start), part=1 the rest (layer2, layer1, stem)."""
        self._readers = {}
        chain = list(zip(reversed(self.blocks), self.bwd_plan, reversed(self._block_inputs())))
        if part == 0:
            chain = chain[:self.N_LATE_BLOCKS]
        elif part == 1:
            chain = chain[self.N_LATE_BLOCKS:]
        for (u1, u2, ud), b, in_t in chain:
            g_out = b["g_out"]
            # out = relu(bn2(c2) + identity): dz = g_out * (out > 0), in place
            self._before_write(b["d_c2"])
            ops.sweep(1 if SWEEP else 0)      # g_out was written ascending: reduce descending, apply ascending
            self._bn_bwd(u2, g_out, g_out, b["d_c2"], True)
            self._wgrad(lambda: ops.conv_wgrad(u2.d, u2.ci_real, u1.y, b["d_c2"], self._grad(u2.conv.weight),
                                               self.wgrad_ws), b["d_c2"])
            ops.sweep(1 if SWEEP >= 2 else 0)
            ops.conv_dgrad(u2.d, b["d_c2"], u2.wT, b["g_y1"])
            ops.sweep(1 if SWEEP == 1 else 0)  # SWEEP 2: g_y1 was written descending -> reduce ascending
            # bn1 + relu has no residual input: mask recomputed from x, no y read / dz write
            self._before_write(b["d_c1"])
            ops.bn_bwd_nores(b["g_y1"], u1.x, b["d_c1"], u1.P, u1.C, u1.bn.weight.data, u1.mean, u1.invstd,
                             u1.scale, u1.shift, self.bn_partial, self._grad(u1.bn.weight), self._grad(u1.bn.bias))
            self._wgrad(lambda: ops.conv_wgrad(u1.d, u1.ci_real, in_t, b["d_c1"], self._grad(u1.conv.weight),
                                               self.wgrad_ws), b["d_c1"])
            if ud is not None:
                # identity = bn_d(conv1x1_s2(u)), no relu: its output gradient is dz (= g_out now)
                self._before_write(b["d_cd"])
                ops.sweep(1 if SWEEP else 0)
                self._bn_bwd(ud, g_out, None, b["d_cd"], False)
                ops.sweep(0)
                self._wgrad(lambda: ops.conv_wgrad(ud.d, ud.ci_real, in_t, b["d_cd"], self._grad(ud.conv.weight),
                                                   self.wgrad_ws), b["d_cd"])
                # 1x1 stride-2 dgrad on the compact grid, then folded into conv1's dgrad epilogue
                dc = ops.conv_desc(self.N, ud.d.Ho, ud.d.Wo, ud.d.Ci, ud.d.Co, 1, 1, 1, 0)
                ops.conv_dgrad(dc, b["d_cd"], ud.wT, b["g_ds"])
                ops.conv_dgrad(u1.d, b["d_c1"], u1.wT, b["g_u"], b["g_ds"], 2)
            else:
                ops.sweep(0)
                ops.conv_dgrad(u1.d, b["d_c1"], u1.wT, b["g_u"], g_out, 1)
        if part == 0:
            ops.sweep(0)
            if self.wgrad_stream is not None:
                torch.cuda.current_stream().wait_stream(self.wgrad_stream)
            self._readers = {}
            return
        s = self.stem
        ops.sweep(1 if SWEEP else 0)  # g_pool was written ascending by the last dgrad
        # max-pool scatter + ReLU mask + BN backward in one pair of passes over the stem conv output
        self._before_write(self.d_c0)
        ops.bn_relu_maxpool_bwd(self.g_pool, self.pool_idx, self.pool_xmax, s.x, self.d_c0, self.N, s.d.Ho, s.d.Wo,
                                64, self.Hp, self.Wp, s.bn.weight.data, s.mean, s.invstd, s.scale, s.shift, self.bn_partial,
                                self._grad(s.bn.weight), self._grad(s.bn.bias))
        self._wgrad(lambda: ops.stem_wgrad(x16, self.d_c0, self._grad(s.conv.weight), s.ci_real, self.N, self.H,
                                           self.W, self.wgrad_ws), self.d_c0)
        ops.sweep(0)
        if self.wgrad_stream is not None:
            torch.cuda.current_stream().wait_stream(self.wgrad_stream)  # join: every gradient is complete
        self._readers = {}

    def _block_inputs(self):
        ins = [self.pool_y]
        for (u1, u2, ud) in self.blocks[:-1]:
            ins.append(u2.y)
        return ins
