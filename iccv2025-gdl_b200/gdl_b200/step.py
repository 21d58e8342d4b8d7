"""DGLStep — the fused Disentangled-Gradient-Learning training step (SURVEY.md §8b mode 2).

One call = reference main_dgl.py:93-158 for one batch: H2D of (spec, image, label), both
ResNet-18 encoders forward, global average pooling, the fused DGL head (three logit sets,
three cross-entropies, truncated gradients), both encoder backwards, [gradient all-reduce],
clip_grad_norm_(40), the audio/visual gradient diagnostics, the optimizer update (SGD-momentum, Adam or Adagrad:
gdl_b200.optim.UpdateRule), and the refresh of
the bf16 weight shadows — as a fixed sequence of libgdl_b200.so kernels on two CUDA streams
(audio || visual), schedule(), whose device segments are optionally replayed as CUDA graphs.  The only
device->host traffic is one 7-float read (3 losses + norm, clip coefficient, 2 diagnostics) when the caller asks.

Gradient routing (the point of DGL, reference main_dgl.py:108-122):
    encoders  <- alpha * d(La + Lv)        (the multimodal head saw detached features)
    head      <- d(Lf)                     (the unimodal gradient of the head is wiped)
Parameters that never receive a gradient in the reference (the concat head's fc_auxi,
the gated head's fc_x / fc_y — SURVEY.md §8a quirks 1-2) are left untouched: no weight decay,
no momentum, exactly like torch.optim.SGD skipping `grad is None`.
"""
import os

import torch

from . import ops, parallel
from .basic_model import AVClassifier_DGL
from .engine import kernel_writes, note_writes
from .heads import fusion_head
from .optim import UpdateRule

_SEG_ALIGN = 64  # floats; keeps every tensor 256-byte aligned inside the arenas

# Data parallel: all-reduce the gradients in two buckets, the first (layer3 + layer4 of both encoders, 94 % of
# the bytes) on NCCL's stream WHILE layer2 / layer1 / stem are still being back-propagated (SURVEY.md §8e,
# reference main_dgl.py:244 nn.DataParallel's reduce-add).  0 = one all-reduce after the whole backward.
AR_OVERLAP = os.environ.get("GDL_AR_OVERLAP", "1") != "0"

# The step is captured lazily (on its second step, once for its lifetime) while a DataLoader's pin-memory
# thread may be calling cudaHostAlloc / cudaEventQuery: in the default "global" capture mode those calls from OTHER
# threads are illegal and can invalidate the capture; "thread_local" restricts the check to the capturing thread.
_CAPTURE_MODE = "thread_local"


def _pad(n):
    return (n + _SEG_ALIGN - 1) // _SEG_ALIGN * _SEG_ALIGN


class GraphCache(dict):
    """CUDA graphs by key."""

    def capture(self, key, enqueue):
        """The graph of `key`; under a new key, first capture what enqueue() launches (capture does not execute it)."""
        if key not in self:
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, capture_error_mode=_CAPTURE_MODE):
                enqueue()
            self[key] = g
        return self[key]


# The segments of a global step: the DEVICE ones are capturable, the others (the stem layout of replica k's rows, the
# NCCL calls) always run eagerly.
DEVICE = ("replica0", "replica", "last", "update")


def schedule(replicas, world_size, overlap):
    """The global step (DESIGN.md §5) as an ordered list of (name, argument) segments:
        ("inputs", k)           eager: the stem layout of replica k's rows (k = 0 first consumes a prefetched batch)
        ("replica0", None)      replica 0's compute (it owns the BatchNorm running statistics), then acc <- grad
        ("replica", None)       replica 1 .. R-2: compute, then acc += grad
        ("last", part)          the last replica's compute, then grad += acc: whole (part None), or with the two
                                all-reduce buckets of `overlap` forward + layer4/layer3 backward (0) and the rest (1)
        ("allreduce", None), ("allreduce_late", None), ("allreduce_finish", None)     NCCL
        ("update", None)        clip statistics, diagnostics, optimizer update, bf16 shadow refresh"""
    seq = [("inputs", 0)]
    for k in range(1, replicas):
        seq += [("replica0" if k == 1 else "replica", None), ("inputs", k)]
    if overlap and world_size > 1:
        seq += [("last", 0), ("allreduce_late", None), ("last", 1), ("allreduce_finish", None)]
    else:
        seq += [("last", None)] + ([("allreduce", None)] if world_size > 1 else [])
    return seq + [("update", None)]


def graph_runs(seq):
    """`seq` cut into runs: an eager segment alone, or a maximal run of consecutive device segments, which a graph
    step replays as one CUDA graph cached under the run itself (so replicas 1 .. R-2 share one graph)."""
    runs = []
    for seg in seq:
        if seg[0] in DEVICE and runs and runs[-1][-1][0] in DEVICE:
            runs[-1] += (seg,)
        else:
            runs.append((seg,))
    return runs


class ParamArena:
    """Flat fp32 arenas (parameters, gradients, optimizer state) with the nn.Parameters re-pointed to
    views, so clipping statistics, the update and the gradient all-reduce are single passes.
    Order: head | audio_net | visual_net  (groups 2, 0, 1 for the diagnostics).
    The optimizer state is that of `rule.kind` only (default SGD): `momentum`; Adam `exp_avg`, `exp_avg_sq`;
    Adagrad `sum`.  `state_buffers` pairs each with its key in torch's `optimizer.state[p]`."""

    def __init__(self, model, device, rule=None):
        groups = [(2, fusion_head(model.fusion_module).trainable()),
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
        # the lr the update reads on the device (one float64): DGLStep.step writes it before every step, so a captured
        # update follows any lr schedule without re-capture
        self.lr = torch.zeros(1, device=device, dtype=torch.float64)
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
        groups = fusion_head(model.fusion_module).trainable() + list(model.audio_net.parameters()) + \
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


class InputStage:
    """Two device staging sets for batches of `rows` rows of the reference contract (fp32 spectrograms [rows, F, Tt],
    fp32 frames [rows, 3, T, H, W], int64 labels) and the copy stream that fills the set the running step does not
    read, so the H2D copy (or the device data pipeline) of the next batch overlaps the current batch's kernels.
    Shared by DGLStep (training) and EvalStep (validation)."""

    def __init__(self, device, rows, spec_hw, image_thw):
        F_, Tt = spec_hw
        T, H, W = image_thw
        self.device, self.rows, self.T = device, rows, T
        self.sets = [(torch.zeros(rows, F_, Tt, device=device), torch.zeros(rows, 3, T, H, W, device=device),
                      torch.zeros(rows, device=device, dtype=torch.int64)) for _ in range(2)]
        self.cur, self.pending = 0, None
        self.crop_params = None   # device copies of the crop-box tables (prefetch with a VisualPipeline)
        self.audio_params = None  # device copies of the {clip, start} tables (prefetch with an AudioPipeline)
        self.copy_stream = torch.cuda.Stream(device)
        self.ready = [torch.cuda.Event() for _ in range(2)]
        self.free = [torch.cuda.Event() for _ in range(2)]

    def stage_rows(self, k, parts, B, enc_a, enc_v, label_in):
        """Eager, on the current stream: rows [k*B, (k+1)*B) of the current set -> both encoders' stem inputs
        (stage_input) and `label_in`.  k = 0 first makes a prefetched batch the current set; after slice k = parts - 1
        the set is free for the next prefetch."""
        main = torch.cuda.current_stream()
        if k == 0 and self.pending is not None:
            main.wait_event(self.ready[self.pending])
            self.cur, self.pending = self.pending, None
        spec, image, label = (t[k * B:(k + 1) * B] for t in self.sets[self.cur])
        enc_a.stage_input(spec, B)
        enc_v.stage_input(image, B)
        label_in.copy_(label, non_blocking=True)
        if k == parts - 1:
            self.free[self.cur].record(main)

    def load(self, spec, image, label):
        """Copy a batch (host or device tensors) into the current set on the current stream."""
        self.pending = None
        for dst, src in zip(self.sets[self.cur], (spec, image, label)):
            if src.data_ptr() != dst.data_ptr():
                dst.copy_(src, non_blocking=True)

    def prefetch(self, spec, image, label, pipeline=None, audio_pipeline=None):
        """Start the copy of the next batch into the other set on the copy stream (see DGLStep.prefetch)."""
        nxt = 1 - self.cur
        cs = self.copy_stream
        cs.wait_event(self.free[nxt])  # the layout kernels that last read this set have run
        with torch.cuda.stream(cs):
            s_spec, s_image, s_label = self.sets[nxt]
            s_label.copy_(label, non_blocking=True)
            if audio_pipeline is None:
                s_spec.copy_(spec, non_blocking=True)
            else:
                if self.audio_params is None:
                    self.audio_params = [torch.empty(self.rows, 2, device=self.device, dtype=torch.int32)
                                         for _ in range(2)]
                self.audio_params[nxt].copy_(spec, non_blocking=True)
                audio_pipeline(self.audio_params[nxt], out=s_spec)
            if pipeline is None:
                s_image.copy_(image, non_blocking=True)
            else:
                if self.crop_params is None:
                    self.crop_params = [torch.empty(self.rows * self.T, 6, device=self.device, dtype=torch.int32)
                                        for _ in range(2)]
                self.crop_params[nxt].copy_(image, non_blocking=True)
                pipeline(self.crop_params[nxt], out=s_image)
            self.ready[nxt].record(cs)
        self.pending = nxt


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
        # read the current set OUTSIDE the captured graphs and write the encoders' fixed-address bf16 stem inputs, so
        # the next batch can be copied H2D on a side stream into the other set while this step computes.
        self.stage = InputStage(dev, self.rows, spec_hw, image_thw)
        self.label_in = torch.zeros(B, device=dev, dtype=torch.int64)  # fixed address: read inside the graph
        D = 512
        self.a_feat, self.v_feat = torch.empty(B, D, device=dev), torch.empty(B, D, device=dev)
        self.da, self.dv = torch.empty(B, D, device=dev), torch.empty(B, D, device=dev)
        self.logits = torch.empty(3, B, self.n, device=dev)
        self.stats = torch.zeros(8, device=dev)  # [0:3] losses Lf,La,Lv  [4:8] norm, coef, audio, visual
        self.losses = self.arena.grad[self.arena.numel:self.arena.numel + 3]
        self._bn_counters = [m.num_batches_tracked for m in model.modules()
                             if isinstance(m, torch.nn.BatchNorm2d)]
        self.head = fusion_head(model.fusion_module, B, self.n, dev)
        # GDL_STREAM_PRIO: 0 = equal priorities, 1 = the visual encoder's stream (the long chain: 3x the audio work) is
        # high priority so its kernels' CTAs are placed first and the audio kernels fill the gaps, 2 = the reverse
        prio = int(os.environ.get("GDL_STREAM_PRIO", "1"))  # measured: 20.40 / 20.09 ms vs 20.48 / 20.40 ms per step, e2e +1.7 %
        self.stream_a = torch.cuda.Stream(dev, priority=-1 if prio == 2 else 0)
        self.stream_v = torch.cuda.Stream(dev, priority=-1 if prio == 1 else 0)
        self.steps_done = 0
        self.momentum_loaded = False  # set by train.adopt_momentum when a checkpoint's buffers were copied in
        self.graphs = GraphCache()  # the device runs of the schedule, captured once
        self.launches_per_step = None
        # gradient buckets (views of the gradient arena; arena order: head | audio | visual)
        self.overlap = AR_OVERLAP and world_size > 1
        self._runs = graph_runs(schedule(R, world_size, self.overlap))
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

    # ------------------------------------------------------------------ the segments of schedule()
    def _enqueue(self, seg):
        """Enqueue one segment on the current stream (+ the two encoder streams).  Every segment reads the streams
        and the rest of the step's state when it is enqueued; the update reads the lr from the arena on the device."""
        name, arg = seg
        if name == "inputs":
            self.stage.stage_rows(arg, self.replicas, self.B, self.enc_a, self.enc_v, self.label_in)
        elif name in ("replica0", "replica"):
            self._enqueue_compute(own_stats=name == "replica0")
            ops.grad_accumulate(self.acc, self.arena.grad, self.arena.numel + 3, name == "replica")
        elif name == "last":
            self._enqueue_compute(arg, own_stats=self.replicas == 1)
            if self.replicas > 1:  # part 0: the late bucket, so its all-reduce carries the sum over the replicas
                for a, b in self._acc_ranges["all" if arg is None else ("late", "early")[arg]]:
                    ops.grad_accumulate(self.arena.grad[a:b], self.acc[a:b], b - a, True)
        elif name == "allreduce":
            # each rank scaled its CE by 1/B_global, so a plain SUM reproduces the reference's
            # full-batch mean (DataParallel gathers logits, main_dgl.py:102-104); BN stays per replica.
            # The 3 losses ride in the tail of the gradient arena (one collective per step).
            torch.distributed.all_reduce(self.arena.grad, group=self.pg)
        elif name == "allreduce_late":
            # bucket 1 (layer3 + layer4 of both encoders + the losses), asynchronously: NCCL's stream waits for what
            # the current stream has enqueued so far and then runs beside the backward of layer2 / layer1 / stem
            self._works = parallel.allreduce_async(self._buckets["late"], self.pg)
        elif name == "allreduce_finish":
            # join bucket 1, then bucket 2 (head + the early layers, 6 % of the bytes) on the critical path
            parallel.allreduce_finish(self._works, self._buckets["early"], self.pg)
        else:
            self._enqueue_update()

    def _enqueue_compute(self, part=None, own_stats=True):
        """Forward + head + backward on the current stream (+ the two encoder streams).
        part=0: forward, head and the backward of layer4 + layer3; part=1: the rest of the backward.
        own_stats=False: the forward leaves the BatchNorm running statistics untouched."""
        B = self.B
        main = torch.cuda.current_stream()
        sa, sv = self.stream_a, self.stream_v
        if part != 1:
            sa.wait_stream(main)
            sv.wait_stream(main)
            with torch.cuda.stream(sa):
                self.enc_a.gap_fwd(self.enc_a.forward(own_stats=own_stats), self.a_feat, B)
            with torch.cuda.stream(sv):
                self.enc_v.gap_fwd(self.enc_v.forward(own_stats=own_stats), self.v_feat, B)
            main.wait_stream(sa)
            main.wait_stream(sv)
            self.head.train(self)
        sa.wait_stream(main)
        sv.wait_stream(main)
        with torch.cuda.stream(sa):
            if part != 1:
                self.enc_a.gap_bwd(self.da, B)
            self.enc_a.backward(part=part)
        with torch.cuda.stream(sv):
            if part != 1:
                self.enc_v.gap_bwd(self.dv, B)
            self.enc_v.backward(part=part)
        main.wait_stream(sa)
        main.wait_stream(sv)

    def _enqueue_update(self):
        """Clip statistics + diagnostics + optimizer update + bf16 shadow refresh (after the all-reduce)."""
        ar, r, lr = self.arena, self.rule, self.arena.lr
        ops.grad_stats(ar.grad, ar.numel, ar.seg_end, ar.seg_group, ar.seg_inv, ar.nseg, self.max_norm,
                       ar.scratch, self.stats[4:8])
        if r.kind == "sgd":
            ops.sgd_momentum(ar.param, ar.grad, ar.momentum, ar.numel, lr, self.mu, self.wd,
                             self.steps_done == 0 and not self.momentum_loaded, self.stats[4:8])
        elif r.kind == "adam":
            ops.adam(ar.param, ar.grad, ar.exp_avg, ar.exp_avg_sq, ar.step_state, ar.numel, lr, r.betas[0], r.betas[1],
                     r.eps, self.wd, self.stats[4:8])
        else:
            ops.adagrad(ar.param, ar.grad, ar.sum, ar.step_state, ar.numel, lr, r.lr_decay, r.eps, self.wd,
                        self.stats[4:8])
        self.refresh_shadows()
        self.stats[0:3].copy_(self.losses)
        torch._foreach_add_(self._bn_counters, 1)

    def refresh_shadows(self):
        """Re-derive the bf16 weight shadows of this step's engines from the fp32 parameters (after ANOTHER step of
        the same model — a different batch geometry — or a load_state_dict changed them)."""
        self.enc_a.repack()
        self.enc_v.repack()
        self.head.refresh_shadows()

    def load_inputs(self, spec, image, label):
        """Copy a batch (host or device tensors of the reference contract) into the current staging set,
        on the current stream (the synchronous path; see prefetch() for the overlapped one)."""
        self.stage.load(spec, image, label)

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
        self.stage.prefetch(spec, image, label, pipeline, audio_pipeline)

    def step(self, spec=None, image=None, label=None, lr=None):
        """Run one training step at learning rate `lr` (default: the last one given, initially the rule's); returns
        the device tensor `stats` (8 floats, see __init__)."""
        if lr is not None:
            self.lr = lr
        # stream-ordered behind the previous step's update, which read the arena's lr
        self.arena.lr.fill_(self.lr)
        if spec is not None:
            self.load_inputs(spec, image, label)
        eager = self.steps_done == 0 or not self.use_graph
        if not eager:
            for run in self._runs:
                if run[0][0] in DEVICE:
                    self.graphs.capture(run, lambda run=run: [self._enqueue(seg) for seg in run])
            # capture does not execute: the replays below run this step
        n0 = ops.LAUNCHES
        for run in self._runs:
            if eager or run[0][0] not in DEVICE:
                for seg in run:
                    self._enqueue(seg)
            else:
                self.graphs[run].replay()
        if eager:
            self.launches_per_step = ops.LAUNCHES - n0  # kernels of libgdl_b200.so per (global) step
        self.steps_done += 1
        self.arena.steps += 1
        for m in (self.model.audio_net, self.model.visual_net, self.model.fusion_module):
            note_writes(m)  # the update and the running statistics changed on the device (graph replays included)
        return self.stats

    def read_stats(self):
        """One D2H copy: (Lf, La, Lv, grad_norm, clip_coef, audio_grad_sum, visual_grad_sum)."""
        s = self.stats.tolist()
        return s[0], s[1], s[2], s[4], s[5], s[6], s[7]


# ---------------------------------------------------------------------------------------------------- evaluation
def _eval_resources(model, rows, spec_hw, image_thw):
    """(b, audio engine, visual engine, head or None) that an EvalStep of `rows` rows runs on.  When a training step
    of this geometry has a per-replica batch b dividing `rows` (with --dp_replicas the step's rows are R_local * b),
    evaluation runs in sub-batches of b on the training step's own engines and head, so nothing is evicted or rebuilt
    and no second set of activation buffers (or FiLM weight shadow) is allocated.  Otherwise the modules' engine cache
    serves `rows`."""
    steps = list(getattr(model, "_gdl_steps", {}).values())
    cur = getattr(model, "_gdl_step", None)
    if cur is not None and cur not in steps:
        steps.append(cur)
    for st in sorted(steps, key=lambda st: -st.B):
        if (not st.check_fp32 and (st.F_, st.Tt) == tuple(spec_hw) and (st.T, st.H, st.W) == tuple(image_thw)
                and rows % st.B == 0):
            return st.B, st.enc_a, st.enc_v, st.head
    (F_, Tt), (T, H, W) = spec_hw, image_thw
    return rows, model.audio_net.engine(rows, F_, Tt), model.visual_net.engine(rows * T, H, W), None


def eval_counts(model, device):
    """The model's int64 [3] device counter of correct arg-maxes (out, out_a, out_v) that every EvalStep adds to."""
    c = getattr(model, "_gdl_eval_counts", None)
    if c is None or c.device != device:
        c = model._gdl_eval_counts = torch.zeros(3, device=device, dtype=torch.int64)
    return c


def eval_confusion(model, device):
    """The model's int64 [1 + 3 n n] device buffer of the per-class report (valid_report), allocated on first use:
    element 0 counts the rows whose label is >= n, the rest is the confusion matrices [3, n, n] (out, out_a, out_v;
    rows = true class, columns = arg-max) that an EvalStep adds to when run(report=True)."""
    c = getattr(model, "_gdl_eval_confusion", None)
    if c is None or c.device != device:
        n = model.n_classes
        c = model._gdl_eval_confusion = torch.zeros(1 + 3 * n * n, device=device, dtype=torch.int64)
    return c


class EvalScores:
    """The device buffers of valid_report(ap=True) for a model with n classes and room for `capacity` rows:
    store      f32 [3, n, capacity]: softmax scores, class-major (heads out, out_a, out_v), written by gdl_eval_scores
    labels     int32 [capacity]: the rows' labels (-1 outside 0..n-1)
    state      int64 [5]: cursor (rows appended so far), overflow (labelled rows that did not fit), hits [3] (top-k)
    ap, support, nonfinite   what gdl_eval_ap writes: f64 [3, n], int64 [n], int64 [1]
    workspace  gdl_eval_ap's sort workspace (None when a column sorts in shared memory)
    k          the top-k of the hits (set before a pass)"""

    def __init__(self, n, capacity, device):
        self.n, self.capacity = n, capacity
        self.store = torch.empty(3, n, capacity, device=device)
        self.labels = torch.full((capacity,), -1, dtype=torch.int32, device=device)
        self.state = torch.zeros(5, dtype=torch.int64, device=device)
        self.cursor, self.overflow, self.hits = self.state[0:1], self.state[1:2], self.state[2:5]
        self.ap = torch.empty(3, n, dtype=torch.float64, device=device)
        self.support = torch.empty(n, dtype=torch.int64, device=device)
        self.nonfinite = torch.empty(1, dtype=torch.int64, device=device)
        ws = ops.eval_ap_workspace_bytes(capacity, n)
        self.workspace = torch.empty(ws, dtype=torch.uint8, device=device) if ws else None
        self.k = min(5, n)
        self.gathered = None  # the store of every rank's rows (train.valid_report on a sharded loader)

    def graph_key(self):
        """What a captured gdl_eval_scores launch depends on."""
        return (self.store.data_ptr(), self.labels.data_ptr(), self.state.data_ptr(), self.capacity, self.k)

    def append(self, logits, labels, B):
        """gdl_eval_scores of logits [3, B, n] and labels [B]: append at the cursor, add the top-k hits."""
        ops.eval_scores(logits, labels, self.store, self.labels, self.cursor, self.hits, self.overflow, B, self.n,
                        self.k)

    def average_precision(self):
        """gdl_eval_ap over the appended rows into ap, support and nonfinite."""
        ops.eval_ap(self.store, self.labels, self.cursor, self.ap, self.support, self.nonfinite, self.workspace)


def eval_scores(model, device, capacity):
    """The model's EvalScores (the score store of valid_report(ap=True)), allocated on first use and re-allocated only
    when `capacity` rows do not fit in it."""
    sc = getattr(model, "_gdl_eval_scores", None)
    if sc is None or sc.store.device != device or sc.capacity < capacity:
        sc = model._gdl_eval_scores = None  # free the smaller store first
        sc = model._gdl_eval_scores = EvalScores(model.n_classes, max(int(capacity), 1), device)
    return sc


class EvalStep:
    """Eval-mode forward of AVClassifier_DGL for batches of `rows` rows (reference valid(), main_dgl.py:168-222, and
    `model(...)` in eval mode): stem layout of each sub-batch of b rows, both encoders with BatchNorm folded
    (EncoderEngine.forward_eval) on the audio and visual streams, then the eval head (gdl_eval_head: pooling, the
    three logit sets, arg-max and correct counts into `counts`; FiLM: pooling, the FiLM forward GEMMs, fc_out and
    gdl_eval_count).  Everything after the layout is one CUDA graph, captured on the second call and re-captured only
    when a head parameter moves or the gated head's x_gate flips.  The BatchNorm fold and the FiLM weight shadow are
    refreshed outside the graph, and only when a parameter or buffer changed.  The logits of the last sub-batch stay
    in `logits` [3, b, n].  run(report=True) appends gdl_eval_confusion (the per-class confusion matrices of
    eval_confusion) to the head; that variant is captured as a graph of its own, so the two alternate without
    re-capture and run(report=False) launches exactly what it would without the report.  run(scores=True) appends
    gdl_eval_scores (the softmax scores and top-k hits of the model's EvalScores, after the confusion matrices when
    both are asked for): one more graph variant, keyed by the store it writes."""

    def __init__(self, model, rows, spec_hw, image_thw, use_graph=True):
        model = getattr(model, "module", model)
        if not isinstance(model, AVClassifier_DGL):
            raise TypeError("EvalStep needs a gdl_b200.AVClassifier_DGL")
        dev = next(model.parameters()).device
        if dev.type != "cuda":
            raise RuntimeError("EvalStep runs on a B200 only (no CPU fallback)")
        ops.init()
        self.model, self.device, self.rows = model, dev, rows
        self.F_, self.Tt = spec_hw
        self.T, self.H, self.W = image_thw
        self.n = model.n_classes
        self.use_graph = use_graph
        self.B, self.enc_a, self.enc_v, head = _eval_resources(model, rows, spec_hw, image_thw)
        self.chunks = rows // self.B
        B = self.B
        self.stage = InputStage(dev, rows, spec_hw, image_thw)
        self.label_in = torch.full((B,), -1, dtype=torch.int64, device=dev)
        self.logits = torch.empty(3, B, self.n, device=dev)
        self.counts = eval_counts(model, dev)
        self.report, self.confusion, self.scores = False, None, None
        self.head = head if head is not None else fusion_head(model.fusion_module, B, self.n, dev)
        self._head_key = None
        self.stream_a, self.stream_v = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        self.calls = 0
        self.graphs = GraphCache()

    # ------------------------------------------------------------------ outside the graph
    def refresh(self):
        """Re-fold BatchNorm into the eval weight packs and re-derive the head's bf16 shadows, each only if its inputs
        changed since the last call (torch version counters + engine.note_writes counts)."""
        self.enc_a.fold_eval()
        self.enc_v.fold_eval()
        fm = self.model.fusion_module
        key = tuple((p.data_ptr(), p._version) for p in fm.parameters()) + (kernel_writes(fm),)
        if key != self._head_key:
            self.head.refresh_shadows()
            self._head_key = key

    # ------------------------------------------------------------------ the captured part
    def _enqueue(self):
        main = torch.cuda.current_stream()
        sa, sv = self.stream_a, self.stream_v
        sa.wait_stream(main)
        sv.wait_stream(main)
        with torch.cuda.stream(sa):
            fa = self.enc_a.forward_eval()
        with torch.cuda.stream(sv):
            fv = self.enc_v.forward_eval()
        main.wait_stream(sa)
        main.wait_stream(sv)
        self.head.eval(self, fa, self.enc_a.Hf * self.enc_a.Wf, fv, self.T * self.enc_v.Hf * self.enc_v.Wf)
        if self.report:
            c = self.confusion
            ops.eval_confusion(self.logits, self.label_in, c[1:], c[:1], self.B, self.n)
        if self.scores is not None:
            self.scores.append(self.logits, self.label_in, self.B)

    def _compute(self):
        """Eager the first time (and without graphs), a graph replay afterwards."""
        if not self.use_graph or self.calls == 0:
            self._enqueue()
            return
        fm = self.model.fusion_module
        base = tuple(p.data_ptr() for p in fm.parameters()) + (self.counts.data_ptr(), getattr(fm, "x_gate", None))
        key = (base, self.confusion.data_ptr() if self.report else None,
               self.scores.graph_key() if self.scores is not None else None)
        if key not in self.graphs:
            for k in [k for k in self.graphs if k[0] != base]:
                del self.graphs[k]  # a graph of moved parameters or another x_gate is never replayed again
        self.graphs.capture(key, self._enqueue).replay()

    def run(self, out=None, report=False, scores=False):
        """Evaluate the current (or just prefetched) batch: counts += correct arg-maxes of its rows.  out: optional
        f32 [3, rows, n] that receives the logits (out, out_a, out_v) of every row.  report: also add the rows to the
        model's confusion matrices (eval_confusion).  scores: also append the rows' softmax scores to the model's
        EvalScores (allocated beforehand by eval_scores) and add their top-k hits."""
        self.report = report
        if report:
            self.confusion = eval_confusion(self.model, self.device)
        self.scores = None
        if scores:
            self.scores = getattr(self.model, "_gdl_eval_scores", None)
            if self.scores is None or self.scores.store.device != self.device:
                raise RuntimeError("run(scores=True) appends to the store of step.eval_scores(model, device, "
                                   "capacity): allocate it first")
        self.refresh()
        for k in range(self.chunks):
            self.stage.stage_rows(k, self.chunks, self.B, self.enc_a, self.enc_v, self.label_in)
            self._compute()
            if out is not None:
                out[:, k * self.B:(k + 1) * self.B].copy_(self.logits)
        self.calls += 1

    def load_inputs(self, spec, image, label=None):
        """Synchronous input path: spec [rows, F, Tt] (or [rows, 1, F, Tt]), image [rows, 3, T, H, W], label [rows] or
        None (a label of -1 is never counted)."""
        if label is None:
            label = torch.full((self.rows,), -1, dtype=torch.int64, device=self.device)
        self.stage.load(spec.reshape(self.rows, self.F_, self.Tt), image, label)

    def prefetch(self, spec, image, label, pipeline=None, audio_pipeline=None):
        """Start the copy of the next batch on the copy stream (DGLStep.prefetch); the next run() consumes it."""
        self.stage.prefetch(spec, image, label, pipeline, audio_pipeline)


def get_eval_step(model, rows, spec_hw, image_thw):
    """The model's cached EvalStep for this geometry (two live entries: the full batch and a short tail batch).  The
    cache key includes the engines it runs on, so a training step created later is picked up."""
    model = getattr(model, "module", model)
    cache = getattr(model, "_gdl_evals", None)
    if cache is None:
        cache = model._gdl_evals = {}
    b, enc_a, enc_v, _ = _eval_resources(model, rows, spec_hw, image_thw)
    key = (rows, tuple(spec_hw), tuple(image_thw), b, id(enc_a), id(enc_v))
    ev = cache.pop(key, None)
    if ev is None:
        ev = EvalStep(model, rows, spec_hw, image_thw)
        while len(cache) >= 2:
            cache.pop(next(iter(cache)))
    cache[key] = ev  # most recently used last
    return ev


def eval_forward(model, audio, visual):
    """`model(audio, visual)` in eval mode: (out, a_out, v_out) of the EvalStep that valid() runs, bit for bit."""
    B = audio.shape[0]
    spec_hw, thw = tuple(audio.shape[-2:]), tuple(visual.shape[2:])
    ev = get_eval_step(model, B, spec_hw, thw)
    out = torch.empty(3, B, ev.n, device=ev.device)
    ev.load_inputs(audio.float(), visual.float())
    ev.run(out)
    return out[0], out[1], out[2]
