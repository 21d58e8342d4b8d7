"""DGLStep — the fused Disentangled-Gradient-Learning training step (SURVEY.md §8b mode 2).

One call = reference main_dgl.py:93-158 for one batch: H2D of (spec, image, label), both
ResNet-18 encoders forward, global average pooling, the fused DGL head (three logit sets,
three cross-entropies, truncated gradients), both encoder backwards, [gradient all-reduce],
clip_grad_norm_(40), the audio/visual gradient diagnostics, the optimizer update (SGD-momentum, Adam or Adagrad:
gdl_b200.optim.UpdateRule), and the refresh of
the bf16 weight shadows — as a fixed sequence of libgdl_b200.so kernels on two CUDA streams
(audio || visual), optionally captured into one CUDA graph.  The only device->host traffic is
one 7-float read (3 losses + norm, clip coefficient, 2 diagnostics) when the caller asks.

Gradient routing (the point of DGL, reference main_dgl.py:108-122):
    encoders  <- alpha * d(La + Lv)        (the multimodal head saw detached features)
    head      <- d(Lf)                     (the unimodal gradient of the head is wiped)
Parameters that never receive a gradient in the reference (ConcatFusion_DGL.fc_auxi,
GatedFusion_DGL.fc_x / fc_y — SURVEY.md §8a quirks 1-2) are left untouched: no weight decay,
no momentum, exactly like torch.optim.SGD skipping `grad is None`.
"""
import os

import torch

from . import ops, parallel
from .autograd import to_nhwc8  # noqa: F401  (re-export for callers)
from .basic_model import AVClassifier_DGL
from .fusion_modules import ConcatFusion_DGL, FiLM_DGL, GatedFusion_DGL, SumFusion_DGL
from .optim import UpdateRule

_SEG_ALIGN = 64  # floats; keeps every tensor 256-byte aligned inside the arenas

# Data parallel: all-reduce the gradients in two buckets, the first (layer3 + layer4 of both encoders, 94 % of
# the bytes) on NCCL's stream WHILE layer2 / layer1 / stem are still being back-propagated (SURVEY.md §8e,
# reference main_dgl.py:244 nn.DataParallel's reduce-add).  0 = one all-reduce after the whole backward.
AR_OVERLAP = os.environ.get("GDL_AR_OVERLAP", "1") != "0"

# The step is captured lazily (second step, and again when MultiStepLR changes lr) while a DataLoader's pin-memory
# thread may be calling cudaHostAlloc / cudaEventQuery: in the default "global" capture mode those calls from OTHER
# threads are illegal and can invalidate the capture; "thread_local" restricts the check to the capturing thread.
_CAPTURE_MODE = "thread_local"


def _pad(n):
    return (n + _SEG_ALIGN - 1) // _SEG_ALIGN * _SEG_ALIGN


def head_trainable(fm):
    """Head parameters that receive a gradient from Lf (everything else stays grad-less)."""
    if isinstance(fm, ConcatFusion_DGL):
        return [fm.fc_out.weight, fm.fc_out.bias]
    if isinstance(fm, SumFusion_DGL):
        return [fm.fc_x.weight, fm.fc_x.bias, fm.fc_y.weight, fm.fc_y.bias]
    if isinstance(fm, GatedFusion_DGL):
        return [fm.fc_out.weight, fm.fc_out.bias]
    if isinstance(fm, FiLM_DGL):
        return [fm.fc.weight, fm.fc.bias, fm.fc_out.weight, fm.fc_out.bias]
    raise NotImplementedError('Incorrect fusion method: {}!'.format(type(fm).__name__))


class ParamArena:
    """Flat fp32 arenas (parameters, gradients, optimizer state) with the nn.Parameters re-pointed to
    views, so clipping statistics, the update and the gradient all-reduce are single passes.
    Order: head | audio_net | visual_net  (groups 2, 0, 1 for the diagnostics).
    The optimizer state is that of `rule.kind` only (default SGD): `momentum`; Adam `exp_avg`, `exp_avg_sq`;
    Adagrad `sum`.  `state_buffers` pairs each with its key in torch's `optimizer.state[p]`."""

    def __init__(self, model, device, rule=None):
        groups = [(2, head_trainable(model.fusion_module)),
                  (0, list(model.audio_net.parameters())),
                  (1, list(model.visual_net.parameters()))]
        self.params, seg_end, seg_group, seg_inv = [], [], [], []
        off = 0
        self.offsets = []
        self.group_ranges = {}
        for gid, plist in groups:
            start = off
            for p in plist:
                self.params.append(p)
                self.offsets.append(off)
                off += _pad(p.numel())
                seg_end.append(off)
                seg_group.append(gid)
                seg_inv.append(1.0 / p.numel())
            self.group_ranges[gid] = (start, off)
        self.numel = off
        self.extra = 64  # tail slots all-reduced together with the gradients (3 losses)
        self.param = torch.zeros(off, device=device)
        self.grad = torch.zeros(off + self.extra, device=device)
        self.kind = rule.kind if rule is not None else "sgd"
        if self.kind == "sgd":
            self.momentum = torch.zeros(off, device=device)
            self.state_buffers = [("momentum_buffer", self.momentum)]
        elif self.kind == "adam":
            self.exp_avg = torch.zeros(off, device=device)
            self.exp_avg_sq = torch.zeros(off, device=device)
            self.state_buffers = [("exp_avg", self.exp_avg), ("exp_avg_sq", self.exp_avg_sq)]
        else:
            self.sum = torch.full((off,), rule.initial_accumulator_value, device=device)
            self.state_buffers = [("sum", self.sum)]
        # Adam / Adagrad step count t (torch's state['step']): one count for the whole arena, so every DGLStep on it
        # (an epoch's short tail batch has its own) continues it.  step_state[0] is the copy the update kernels advance
        # on the device (also under CUDA-graph replay), `steps` the host's, advanced by DGLStep.step; `step_tensors`
        # are the CPU tensors train.adopt_momentum put into optimizer.state[p]['step'], refreshed by sync_step_tensors.
        self.step_state = torch.zeros(3, device=device, dtype=torch.int32)
        self.steps = 0
        self.step_tensors = {}
        for p, o in zip(self.params, self.offsets):
            n = p.numel()
            self.param[o:o + n].copy_(p.data.reshape(-1))
            p.data = self.param[o:o + n].view(p.shape)
            p.grad = self.grad[o:o + n].view(p.shape)
        self.offset_of = {id(p): o for p, o in zip(self.params, self.offsets)}
        self.acc = None  # gradient sum of the earlier replicas of a step (DGLStep replicas > 1), see accumulator()
        self.nseg = len(seg_end)
        self.seg_end = torch.tensor(seg_end, device=device, dtype=torch.int64)
        self.seg_group = torch.tensor(seg_group, device=device, dtype=torch.int32)
        self.seg_inv = torch.tensor(seg_inv, device=device, dtype=torch.float32)
        self.scratch = torch.empty(ops.optim_scratch_floats(off, self.nseg), device=device)

    def owns(self, model, device):
        """True while every parameter of `model` still is the view into this arena that __init__ made (a
        `model.to(...)`, `load_state_dict(assign=True)` or a changed trainable set breaks that)."""
        groups = head_trainable(model.fusion_module) + list(model.audio_net.parameters()) + \
            list(model.visual_net.parameters())
        if self.param.device != device or len(groups) != len(self.params):
            return False
        base = self.param.data_ptr()
        return all(p is q and p.data.data_ptr() == base + 4 * o for p, q, o in zip(groups, self.params, self.offsets))

    def accumulator(self):
        """The fp32 arena (shape of `grad`, loss tail included) that sums the gradients of a step's replicas before
        the last one; allocated on first use, so a step with one replica per process costs no memory for it."""
        if self.acc is None:
            self.acc = torch.zeros_like(self.grad)
        return self.acc

    def set_steps(self, t):
        """Continue from step count t (a restored checkpoint)."""
        self.steps = int(t)
        self.step_state[0] = self.steps

    def sync_step_tensors(self):
        """Write the step count into the optimizer's state['step'] tensors, so optimizer.state_dict() carries it."""
        for t in self.step_tensors.values():
            t.fill_(float(self.steps))

    def late_split(self, gid, late_params):
        """Offset where the `late_params` of group gid start, checked to be exactly the tail of the group
        (module registration order: conv1, bn1, layer1 .. layer4)."""
        start, end = self.group_ranges[gid]
        cut = min(self.offset_of[id(p)] for p in late_params)
        tail = {id(p) for p, o in zip(self.params, self.offsets) if cut <= o < end}
        if tail != {id(p) for p in late_params} or not start < cut < end:
            raise RuntimeError("late parameters are not a contiguous tail of their arena group")
        return cut


class DGLStep:
    def __init__(self, model, batch_size, spec_hw, image_thw, alpha=4.0, lr=0.001, momentum=0.9,
                 weight_decay=1e-4, max_norm=40.0, world_size=1, process_group=None, use_graph=True, check_fp32=None,
                 rule=None, replicas=1):
        """model: AVClassifier_DGL on a CUDA device (possibly wrapped: `.module` is unwrapped).
        batch_size: rows of ONE replica (the BatchNorm batch); losses are means over batch_size*replicas*world_size.
        replicas: data-parallel replicas run one after another on this GPU per step (nn.DataParallel over
        replicas*world_size devices, reference main_dgl.py:244).  A step then takes replicas*batch_size rows; replica k
        trains on rows [k*batch_size, (k+1)*batch_size) with its own BatchNorm batch statistics, the gradients (and
        losses) of the replicas are summed on the device before the all-reduce, the clip and the update, and only
        replica 0 updates the BatchNorm running statistics (DataParallel's replica 0 aliases the module's buffers).
        rule: the update (gdl_b200.optim.UpdateRule, e.g. update_rule(torch_optimizer)); its lr, weight decay and
        momentum replace the three arguments of the same names.  Default: SGD with lr, momentum, weight_decay.
        check_fp32 (default: env GDL_CHECK_FP32): the FP32 check mode — the encoders store fp32 activations and run
        the CUDA-core fp64-accumulating kernels of csrc/check_fp32.cu (gdl_b200/check.py) instead of the bf16
        tcgen05 engine; head, truncation, clipping, SGD and the all-reduce are the product code.  For parity
        checks (north_star: losses within 1e-4), not for speed."""
        model = getattr(model, "module", model)
        if not isinstance(model, AVClassifier_DGL):
            raise TypeError("DGLStep needs a gdl_b200.AVClassifier_DGL")
        self.model = model
        dev = next(model.parameters()).device
        if dev.type != "cuda":
            raise RuntimeError("DGLStep runs on a B200 only (no CPU fallback)")
        ops.init()
        self.device = dev
        self.B = batch_size
        self.F_, self.Tt = spec_hw
        self.T, self.H, self.W = image_thw
        if rule is None:
            rule = UpdateRule("sgd", lr, weight_decay, momentum=momentum)
        self.rule = rule
        self.alpha, self.lr, self.mu, self.wd, self.max_norm = alpha, rule.lr, rule.momentum, rule.weight_decay, max_norm
        self.world_size, self.pg = world_size, process_group
        if replicas < 1:
            raise ValueError("replicas must be >= 1, got {}".format(replicas))
        self.replicas = R = replicas
        self.rows = R * batch_size  # rows of this process's share of a global batch
        self.inv_batch = 1.0 / (batch_size * R * world_size)
        self.n = model.n_classes
        self.use_graph = use_graph
        B, T = self.B, self.T

        # ONE arena per model: a second DGLStep of another batch geometry (an epoch's short tail batch) shares the
        # parameters, gradients and optimizer state of the first instead of re-allocating and copying them
        arena = getattr(model, "_gdl_arena", None)
        if arena is None or not arena.owns(model, dev) or arena.kind != rule.kind:
            arena = ParamArena(model, dev, rule)
            model._gdl_arena = arena
        self.arena = arena
        self.acc = arena.accumulator() if R > 1 else None
        if check_fp32 is None:
            check_fp32 = os.environ.get("GDL_CHECK_FP32", "0") != "0"
        self.check_fp32 = bool(check_fp32)
        if self.check_fp32:
            from .check import CheckEncoder
            self.enc_a = CheckEncoder(model.audio_net, B, self.F_, self.Tt, dev, frames=1)
            self.enc_v = CheckEncoder(model.visual_net, B * T, self.H, self.W, dev, frames=T)
            self.use_graph = use_graph = False  # the check engine allocates its backward temporaries per step
        else:
            self.enc_a = model.audio_net.engine(B, self.F_, self.Tt)
            self.enc_v = model.visual_net.engine(B * T, self.H, self.W)
        # Inputs: two staging sets (fp32 batch as the reference's DataLoader delivers it).  The layout kernels
        # read the current set OUTSIDE the captured graph and write the fixed-address bf16 stem inputs a8/v8, so
        # the next batch can be copied H2D on a side stream into the other set while this step computes.
        rows = self.rows
        self._stage = [(torch.zeros(rows, self.F_, self.Tt, device=dev), torch.zeros(rows, 3, T, self.H, self.W, device=dev),
                        torch.zeros(rows, device=dev, dtype=torch.int64)) for _ in range(2)]
        self._cur, self._pending = 0, None
        self._crop_params = None  # device copies of the crop-box tables (prefetch with a VisualPipeline)
        self._audio_params = None  # device copies of the {clip, start} tables (prefetch with an AudioPipeline)
        self.copy_stream = torch.cuda.Stream(dev)
        self._stage_ready = [torch.cuda.Event() for _ in range(2)]
        self._stage_free = [torch.cuda.Event() for _ in range(2)]
        self.label_in = torch.zeros(B, device=dev, dtype=torch.int64)  # fixed address: read inside the graph
        self.a8 = self.v8 = None
        if not self.check_fp32:
            self.a8 = torch.empty(self.enc_a.input_shape, device=dev, dtype=torch.bfloat16)  # space-to-depth
            self.v8 = torch.empty(self.enc_v.input_shape, device=dev, dtype=torch.bfloat16)
        D = 512
        self.a_feat, self.v_feat = torch.empty(B, D, device=dev), torch.empty(B, D, device=dev)
        self.da, self.dv = torch.empty(B, D, device=dev), torch.empty(B, D, device=dev)
        self.logits = torch.empty(3, B, self.n, device=dev)
        self.head_scratch = torch.empty(ops.head_scratch_floats(B, self.n) + 64, device=dev)
        self.stats = torch.zeros(8, device=dev)  # [0:3] losses Lf,La,Lv  [4:8] norm, coef, audio, visual
        self.losses = self.arena.grad[self.arena.numel:self.arena.numel + 3]
        self._bn_counters = [m.num_batches_tracked for m in model.modules()
                             if isinstance(m, torch.nn.BatchNorm2d)]
        self._init_head()
        # GDL_STREAM_PRIO: 0 = equal priorities, 1 = the visual encoder's stream (the long chain: 3x the audio work) is
        # high priority so its kernels' CTAs are placed first and the audio kernels fill the gaps, 2 = the reverse
        prio = int(os.environ.get("GDL_STREAM_PRIO", "1"))  # measured: 20.40 / 20.09 ms vs 20.48 / 20.40 ms per step, e2e +1.7 %
        self.stream_a = torch.cuda.Stream(dev, priority=-1 if prio == 2 else 0)
        self.stream_v = torch.cuda.Stream(dev, priority=-1 if prio == 1 else 0)
        self.steps_done = 0
        self.momentum_loaded = False  # set by train.adopt_momentum when a checkpoint's buffers were copied in
        self._graph = None
        self._graph_b = None
        self._graph_update = None
        self._graph_first = None  # replicas > 1: replica 0 (owns the running statistics), then acc <- grad
        self._graph_mid = None    # replicas > 2: replicas 1 .. R-2, acc += grad
        self._graph_lr = None
        self.launches_per_step = None
        # gradient buckets (views of the gradient arena; arena order: head | audio | visual)
        self.overlap = AR_OVERLAP and world_size > 1
        self._buckets = None
        if self.overlap:
            ar = self.arena
            cut_a = ar.late_split(0, self.enc_a.late_parameters())
            cut_v = ar.late_split(1, self.enc_v.late_parameters())
            self._buckets = parallel.gradient_buckets(ar.grad, cut_a, ar.group_ranges[0][1], cut_v)
        # the ranges grad += acc covers after the last replica (the arena + the 3 losses): all at once, or per bucket
        # just before that bucket's all-reduce
        end = self.arena.numel + 3
        if self.overlap:
            ea = self.arena.group_ranges[0][1]
            self._acc_ranges = {"late": [(cut_a, ea), (cut_v, end)], "early": [(0, cut_a), (ea, cut_v)]}
        else:
            self._acc_ranges = {"all": [(0, end)]}

    # ------------------------------------------------------------------ heads
    def _init_head(self):
        fm, B, n, dev = self.model.fusion_module, self.B, self.n, self.device
        self.film = None
        if isinstance(fm, GatedFusion_DGL):
            self.gated_scratch = torch.empty(ops.gated_head_scratch_floats(B, n) + 64, device=dev)
        elif isinstance(fm, FiLM_DGL):
            from .film import FilmHead
            self.film = FilmHead(fm, B, n, dev)

    def _head(self):
        fm, B, n, D = self.model.fusion_module, self.B, self.n, 512
        if isinstance(fm, ConcatFusion_DGL):
            W, b = fm.fc_out.weight, fm.fc_out.bias
            ops.dgl_head_linear(0, self.a_feat, self.v_feat, W.data_ptr(), W.data_ptr() + 4 * D, 2 * D,
                                b.data, None, self.label_in, self.alpha, self.inv_batch, self.logits,
                                self.losses, self.da, self.dv, W.grad.data_ptr(), W.grad.data_ptr() + 4 * D,
                                2 * D, b.grad, None, self.head_scratch, B, D, n)
        elif isinstance(fm, SumFusion_DGL):
            ops.dgl_head_linear(1, self.a_feat, self.v_feat, fm.fc_x.weight.data_ptr(),
                                fm.fc_y.weight.data_ptr(), D, fm.fc_x.bias.data, fm.fc_y.bias.data,
                                self.label_in, self.alpha, self.inv_batch, self.logits, self.losses,
                                self.da, self.dv, fm.fc_x.weight.grad.data_ptr(),
                                fm.fc_y.weight.grad.data_ptr(), D, fm.fc_x.bias.grad, fm.fc_y.bias.grad,
                                self.head_scratch, B, D, n)
        elif isinstance(fm, GatedFusion_DGL):
            self._head_gated(fm)
        else:
            self.film.run(self)

    def _head_gated(self, fm):
        """reference fusion_modules.py:230-250 with the DGL routing, one fused pass (csrc/head.cu
        dgl_gated_sample/param_kernel): fc_out <- Lf; a, v <- alpha*La/Lv through fc_out, the gates and fc_x / fc_y;
        fc_x / fc_y themselves get no gradient."""
        Wo, bo = fm.fc_out.weight, fm.fc_out.bias
        ops.dgl_head_gated(self.a_feat, self.v_feat, fm.fc_x.weight.data, fm.fc_x.bias.data, fm.fc_y.weight.data,
                           fm.fc_y.bias.data, Wo.data, bo.data, self.label_in, self.alpha, self.inv_batch, self.logits,
                           self.losses, self.da, self.dv, Wo.grad, bo.grad, self.gated_scratch, self.B, 512, self.n)

    # ------------------------------------------------------------------ the step
    @property
    def spec_in(self):
        return self._stage[self._cur][0]

    @property
    def image_in(self):
        return self._stage[self._cur][1]

    def _enqueue_inputs(self, k=0):
        """Eager, outside the graph: consume the prefetched batch if there is one (k = 0), then the per-frame
        reshape + fp32->bf16 space-to-depth layout of both modalities (reference backbone.py:162-164,
        main_dgl.py:100) of replica k's rows of the current staging set into the fixed-address stem inputs."""
        B, T = self.B, self.T
        main = torch.cuda.current_stream()
        if k == 0 and self._pending is not None:
            main.wait_event(self._stage_ready[self._pending])
            self._cur, self._pending = self._pending, None
        spec, image, label = (t[k * B:(k + 1) * B] for t in self._stage[self._cur])
        if self.check_fp32:
            self.enc_a.stage_input(spec, B)
            self.enc_v.stage_input(image, B)
        else:
            ops.stem_layout(spec, self.a8, B, 1, 1, self.F_, self.Tt)
            ops.stem_layout(image, self.v8, B, 3, T, self.H, self.W)
        self.label_in.copy_(label, non_blocking=True)
        if k == self.replicas - 1:
            self._stage_free[self._cur].record(main)

    def _enqueue(self, lr, first):
        """The last replica of the step (with replicas == 1 its only one), the all-reduce and the update."""
        if self.overlap:
            self._enqueue_last(part=0)
            works = self._allreduce_late()
            self._enqueue_last(part=1)
            self._allreduce_finish(works)
        else:
            self._enqueue_last()
            if self.world_size > 1:
                self._allreduce()
        self._enqueue_update(lr, first)

    def _enqueue_last(self, part=None):
        """Compute of the last replica; with replicas > 1 then grad += acc over the part's range (part 0: the late
        bucket, so its all-reduce carries the sum over the replicas)."""
        self._enqueue_compute(part, own_stats=self.replicas == 1)
        if self.replicas > 1:
            key = "all" if part is None else ("late", "early")[part]
            for a, b in self._acc_ranges[key]:
                ops.grad_accumulate(self.arena.grad[a:b], self.acc[a:b], b - a, True)

    def _enqueue_replica(self, k):
        """Replica k < replicas - 1: compute, then acc <- grad (k = 0) or acc += grad, over the arena + 3 losses.
        Only replica 0 updates the BatchNorm running statistics."""
        self._enqueue_compute(own_stats=k == 0)
        n = self.arena.numel + 3
        ops.grad_accumulate(self.acc, self.arena.grad, n, k > 0)

    def _enqueue_compute(self, part=None, own_stats=True):
        """Forward + head + backward on the current stream (+ the two encoder streams).
        part=0: forward, head and the backward of layer4 + layer3; part=1: the rest of the backward.
        own_stats=False: the forward leaves the BatchNorm running statistics untouched."""
        B, T = self.B, self.T
        main = torch.cuda.current_stream()
        sa, sv = self.stream_a, self.stream_v
        if part != 1:
            sa.wait_stream(main)
            sv.wait_stream(main)
            with torch.cuda.stream(sa):
                fa = self.enc_a.forward(self.a8, own_stats=own_stats)
                self._gap_fwd(self.enc_a, fa, self.a_feat, 1)
            with torch.cuda.stream(sv):
                fv = self.enc_v.forward(self.v8, own_stats=own_stats)
                self._gap_fwd(self.enc_v, fv, self.v_feat, T)
            main.wait_stream(sa)
            main.wait_stream(sv)
            self._head()
        sa.wait_stream(main)
        sv.wait_stream(main)
        with torch.cuda.stream(sa):
            if part != 1:
                self._gap_bwd(self.enc_a, self.da, 1)
            self.enc_a.backward(self.a8, part)
        with torch.cuda.stream(sv):
            if part != 1:
                self._gap_bwd(self.enc_v, self.dv, T)
            self.enc_v.backward(self.v8, part)
        main.wait_stream(sa)
        main.wait_stream(sv)

    def _gap_fwd(self, enc, feat, out, frames):
        """global average pool over (frames, h, w) (reference models/basic_model.py:73-82)."""
        if self.check_fp32:
            enc.gap_fwd(feat, out, self.B)
        else:
            ops.gap_fwd(feat, out, self.B, frames * enc.Hf * enc.Wf, 512)

    def _gap_bwd(self, enc, dout, frames):
        if self.check_fp32:
            enc.gap_bwd(dout, self.B)
        else:
            ops.gap_bwd(dout, enc.g_feat, self.B, frames * enc.Hf * enc.Wf, 512)

    def _allreduce(self):
        # each rank scaled its CE by 1/B_global, so a plain SUM reproduces the reference's
        # full-batch mean (DataParallel gathers logits, main_dgl.py:102-104); BN stays per replica.
        # The 3 losses ride in the tail of the gradient arena (one collective per step).
        torch.distributed.all_reduce(self.arena.grad, group=self.pg)

    def _allreduce_late(self):
        """Bucket 1 (layer3 + layer4 of both encoders + the losses): issued asynchronously — NCCL's stream waits
        for what the current stream has enqueued so far (the backward of those layers) and then runs beside
        the kernels enqueued next (the backward of layer2 / layer1 / stem)."""
        return parallel.allreduce_async(self._buckets["late"], self.pg)

    def _allreduce_finish(self, works):
        """Join bucket 1, then bucket 2 (head + the early layers, 6 % of the bytes) on the critical path."""
        parallel.allreduce_finish(works, self._buckets["early"], self.pg)

    def _enqueue_update(self, lr, first):
        """Clip statistics + diagnostics + optimizer update + bf16 shadow refresh (after the all-reduce)."""
        ar, r = self.arena, self.rule
        ops.grad_stats(ar.grad, ar.numel, ar.seg_end, ar.seg_group, ar.seg_inv, ar.nseg, self.max_norm,
                       ar.scratch, self.stats[4:8])
        if r.kind == "sgd":
            ops.sgd_momentum(ar.param, ar.grad, ar.momentum, ar.numel, lr, self.mu, self.wd,
                             first and not self.momentum_loaded, self.stats[4:8])
        elif r.kind == "adam":
            ops.adam(ar.param, ar.grad, ar.exp_avg, ar.exp_avg_sq, ar.step_state, ar.numel, lr, r.betas[0], r.betas[1],
                     r.eps, self.wd, self.stats[4:8])
        else:
            ops.adagrad(ar.param, ar.grad, ar.sum, ar.step_state, ar.numel, lr, r.lr_decay, r.eps, self.wd,
                        self.stats[4:8])
        self.enc_a.repack()
        self.enc_v.repack()
        if self.film is not None:
            self.film.refresh()
        self.stats[0:3].copy_(self.losses)
        torch._foreach_add_(self._bn_counters, 1)

    def refresh_shadows(self):
        """Re-derive the bf16 weight shadows of this step's engines from the fp32 parameters (after ANOTHER step of
        the same model — a different batch geometry — or a load_state_dict changed them)."""
        self.enc_a.repack()
        self.enc_v.repack()
        if self.film is not None:
            self.film.refresh()

    def load_inputs(self, spec, image, label):
        """Copy a batch (host or device tensors of the reference contract) into the current staging set,
        on the current stream (the synchronous path; see prefetch() for the overlapped one)."""
        self._pending = None
        for dst, src in zip(self._stage[self._cur], (spec, image, label)):
            if src.data_ptr() != dst.data_ptr():
                dst.copy_(src, non_blocking=True)

    def prefetch(self, spec, image, label, pipeline=None, audio_pipeline=None):
        """Start the H2D copy of the NEXT batch (pinned host tensors) on the copy stream into the staging
        set that the running step does not read; the next step() without arguments consumes it.  This is the
        pin_memory + non_blocking pattern of the reference's DataLoader (main_dgl.py:284-288,93-95) made
        explicit, so that PCIe traffic overlaps the previous step's kernels.

        pipeline: a datapipe.VisualPipeline — `image` is then the int32 [B*T, 6] table of host-drawn crop boxes
        (datapipe.draw_frame_params) and the fp32 frames are produced ON the device from the resident uint8
        frame store (bit-identical to the reference transform), so only the spectrograms and 24 bytes per frame
        cross PCIe.
        audio_pipeline: a datapipe.AudioPipeline — `spec` is then the int32 [B, 2] table {clip index, start sample}
        and the log-STFT spectrograms are computed on the device from the resident waveforms (gdl_log_stft)."""
        nxt = 1 - self._cur
        cs = self.copy_stream
        cs.wait_event(self._stage_free[nxt])  # the layout kernels that last read this set have run
        with torch.cuda.stream(cs):
            s_spec, s_image, s_label = self._stage[nxt]
            s_label.copy_(label, non_blocking=True)
            if audio_pipeline is None:
                s_spec.copy_(spec, non_blocking=True)
            else:
                if self._audio_params is None:
                    self._audio_params = [torch.empty(self.rows, 2, device=self.device, dtype=torch.int32)
                                          for _ in range(2)]
                self._audio_params[nxt].copy_(spec, non_blocking=True)
                audio_pipeline(self._audio_params[nxt], out=s_spec)
            if pipeline is None:
                s_image.copy_(image, non_blocking=True)
            else:
                if self._crop_params is None:
                    self._crop_params = [torch.empty(self.rows * self.T, 6, device=self.device, dtype=torch.int32)
                                         for _ in range(2)]
                self._crop_params[nxt].copy_(image, non_blocking=True)
                pipeline(self._crop_params[nxt], out=s_image)
            self._stage_ready[nxt].record(cs)
        self._pending = nxt

    def step(self, spec=None, image=None, label=None, lr=None):
        """Run one training step; returns the device tensor `stats` (8 floats, see __init__)."""
        if lr is not None:
            self.lr = lr
        if spec is not None:
            self.load_inputs(spec, image, label)
        first = self.steps_done == 0
        n0 = ops.LAUNCHES
        self._enqueue_inputs()
        if first or not self.use_graph:
            for k in range(1, self.replicas):
                self._enqueue_replica(k - 1)
                self._enqueue_inputs(k)
            self._enqueue(self.lr, first)
            self.launches_per_step = ops.LAUNCHES - n0  # kernels of libgdl_b200.so per (global) step
        else:
            if self._graph is None or self._graph_lr != self.lr:
                torch.cuda.synchronize()
                if self.world_size == 1:
                    self._graph = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(self._graph, capture_error_mode=_CAPTURE_MODE):
                        self._enqueue(self.lr, False)
                    self._graph_update = None
                else:
                    # NCCL stays outside the captured regions: graph(compute) -> all-reduce -> graph(update), or with
                    # the overlapped buckets graph(fwd + late bwd) -> [NCCL bucket 1 || graph(early bwd)] ->
                    # NCCL bucket 2 -> graph(update)
                    self._graph = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(self._graph, capture_error_mode=_CAPTURE_MODE):
                        self._enqueue_last(part=0 if self.overlap else None)
                    self._graph_b = None
                    if self.overlap:
                        self._graph_b = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(self._graph_b, capture_error_mode=_CAPTURE_MODE):
                            self._enqueue_last(part=1)
                    self._graph_update = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(self._graph_update, capture_error_mode=_CAPTURE_MODE):
                        self._enqueue_update(self.lr, False)
                # replicas before the last: one graph for replica 0, one shared by replicas 1 .. R-2 (the eager
                # input layout of the next replica runs between the replays)
                self._graph_first = self._graph_mid = None
                for k in range(min(self.replicas - 1, 2)):
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, capture_error_mode=_CAPTURE_MODE):
                        self._enqueue_replica(k)
                    if k == 0:
                        self._graph_first = g
                    else:
                        self._graph_mid = g
                self._graph_lr = self.lr
                # capture does not execute: the replays below run this step
            for k in range(1, self.replicas):
                (self._graph_first if k == 1 else self._graph_mid).replay()
                self._enqueue_inputs(k)
            self._graph.replay()
            if self._graph_b is not None:
                works = self._allreduce_late()
                self._graph_b.replay()
                self._allreduce_finish(works)
                self._graph_update.replay()
            elif self._graph_update is not None:
                self._allreduce()
                self._graph_update.replay()
        self.steps_done += 1
        self.arena.steps += 1
        return self.stats

    def read_stats(self):
        """One D2H copy: (Lf, La, Lv, grad_norm, clip_coef, audio_grad_sum, visual_grad_sum)."""
        s = self.stats.tolist()
        return s[0], s[1], s[2], s[4], s[5], s[6], s[7]
