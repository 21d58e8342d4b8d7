"""Drop-ins for the reference's `train_epoch` (main_dgl.py:69-165) and `valid` (:168-222) with
the same signatures, return values, prints and CSV side effects, running on the fused DGLStep.

Differences that are invisible to the caller: the 123 per-step host syncs of the reference
(120 `.item()` for the diagnostics + 3 losses) become one 8-float D2H per LOG_EVERY steps
(the per-step values are kept in a device ring and flushed in order), and the optimizer passed
in is only read for its update rule, hyper-parameters and lr schedule (gdl_b200.optim.update_rule: SGD-momentum,
Adam or Adagrad; anything else raises) — the update itself is a fused kernel over the parameter arena (its state is
exposed through `optimizer.state[p]` — `momentum_buffer`, `exp_avg` / `exp_avg_sq` / `step`, `sum` / `step` — so
reference-format checkpoints still carry it).
"""
import csv

import torch

from .optim import update_rule
from .parallel import ChunkShardBatchSampler, broadcast_running_stats, replicas_per_rank
from .step import DGLStep, eval_counts, get_eval_step

LOG_EVERY = 100  # the reference prints every 100 steps (main_dgl.py:125,144)
GRAD_CSV = 'audio_visual_grad_vanilla.csv'  # main_dgl.py:148


def _pipeline_of(dataloader):
    """The dataset's device-side visual pipeline (datapipe.VisualPipeline), if it delivers crop boxes instead of
    pixels (synthetic.SyntheticCramedDevice); None for the reference contract (fp32 frames)."""
    return getattr(getattr(dataloader, "dataset", None), "device_pipeline", None)


def _audio_pipeline_of(dataloader):
    """The dataset's device-side audio pipeline (datapipe.AudioPipeline): items then carry {clip, start} instead of
    the spectrogram."""
    return getattr(getattr(dataloader, "dataset", None), "device_audio_pipeline", None)


def _geometry(spec, image, pipeline=None, audio_pipeline=None):
    """(spectrogram (F, Tt), frames (T, H, W)) of a batch as the loader delivers it."""
    thw = (pipeline.T, pipeline.S, pipeline.S) if pipeline is not None else tuple(image.shape[2:])
    spec_hw = (audio_pipeline.F, audio_pipeline.frames) if audio_pipeline is not None else tuple(spec.shape[1:])
    return spec_hw, thw


def _prefetch(step, batch, pipe, apipe):
    """Start the copy of `batch` into the step's (DGLStep or EvalStep) other staging set.  With the device pipelines
    batch[1] is the int32 [B, T, 6] table of host-drawn crop boxes, batch[0] {clip, start} with apipe."""
    if pipe is None:
        step.prefetch(*batch, audio_pipeline=apipe)
    else:
        step.prefetch(batch[0], batch[1].reshape(-1, 6), batch[2], pipeline=pipe, audio_pipeline=apipe)


def _world():
    return torch.distributed.get_world_size() if torch.distributed.is_available() and \
        torch.distributed.is_initialized() else 1


def _get_step(args, model, optimizer, spec, image, pipeline=None, audio_pipeline=None):
    inner = getattr(model, "module", model)
    B = spec.shape[0]
    spec_hw, thw = _geometry(spec, image, pipeline, audio_pipeline)
    world = _world()
    # args.dp_replicas (main_dgl.py --dp_replicas; 0 = one replica per process): R data-parallel replicas of
    # batch_size / R rows, R / world of them run one after another by each process (DGLStep replicas)
    replicas = getattr(args, 'dp_replicas', 0) or 0
    local = 1
    if replicas:
        local = replicas_per_rank(getattr(args, 'batch_size', B * world), replicas, world)
        if B % local:
            raise ValueError("a batch of {} rows does not split into {} replicas of equal size (a short last batch: "
                             "drop it, as the reference's loaders do)".format(B, local))
    key = (B, spec_hw, thw, local)
    # per-geometry cache (two entries: the full batch and an epoch's short tail batch when the loader does not drop it).
    # The steps share ONE parameter / gradient / momentum arena (DGLStep), so switching costs a weight-shadow refresh,
    # not a re-allocation, a momentum copy and a graph re-capture.
    steps = getattr(inner, "_gdl_steps", None)
    if steps is None:
        steps = inner._gdl_steps = {}
    last = getattr(inner, "_gdl_step_key", None)
    st = steps.get(key)
    if st is not None:
        if last != key:
            st.refresh_shadows()
            st.momentum_loaded = True  # the momentum arena is live: never torch's first-step `buf = g` again
        inner._gdl_step, inner._gdl_step_key = st, key
        return st
    rule = update_rule(optimizer)
    trained = any(s.steps_done > 0 for s in steps.values())
    st = DGLStep(inner, B // local, spec_hw, thw, alpha=args.alpha, rule=rule, max_norm=40.0,
                 world_size=world, process_group=torch.distributed.group.WORLD if world > 1 else None,
                 replicas=local)
    adopt_momentum(st.arena, optimizer, st)
    if trained:
        st.momentum_loaded = True
    if len(steps) >= 2:
        steps.pop(next(k for k in steps if k != last))
    steps[key] = st
    inner._gdl_step, inner._gdl_step_key = st, key
    return st


def adopt_momentum(arena, optimizer, step=None):
    """Checkpoint compatibility in both directions (reference main_dgl.py:396-412 saves `optimizer.state_dict()`):
    optimizer state already present in `optimizer.state` — loaded from a checkpoint by `optimizer.load_state_dict`,
    created by torch's Adagrad at construction (`sum` = initial_accumulator_value), or left by a previous DGLStep of
    another batch geometry — is copied INTO the arena buffers of the rule in use (SGD `momentum_buffer`, Adam
    `exp_avg` / `exp_avg_sq`, Adagrad `sum`), then `optimizer.state[p]` is re-pointed at the arena views so the next
    `optimizer.state_dict()` carries what the fused kernels maintain.  Returns whether anything was copied.
    SGD: when anything was adopted the step's first update must use `mu * buf + g` instead of torch's first-step
    `buf = g`.
    Adam / Adagrad: a `state['step']` the arena did not put there sets the arena's step count, which must then be
    the same for every arena parameter (ValueError otherwise; a parameter without state counts 0).  It is replaced by
    a CPU float tensor of the arena's, which `ParamArena.sync_step_tensors` (end of train_epoch) keeps current.
    Parameters outside the arena (never trained, e.g. concat's fc_auxi) keep whatever state torch gave them."""
    loaded, counts = False, set()
    for p, o in zip(arena.params, arena.offsets):
        state = optimizer.state[p]
        for key, buf in arena.state_buffers:
            view = buf[o:o + p.numel()].view(p.shape)
            old = state.get(key)
            if old is not None and old.data_ptr() != view.data_ptr():
                view.copy_(old)
                loaded = True
            state[key] = view
        if arena.kind != "sgd":
            t, own = state.get('step'), arena.step_tensors.get(id(p))
            if own is None or t is not own:
                counts.add(0 if t is None else int(t))
    if len(counts) > 1:
        raise ValueError("optimizer state holds different step counts {} for the parameters of one update; the fused "
                         "{} step keeps one count for all of them".format(sorted(counts), arena.kind))
    if counts:
        arena.set_steps(counts.pop())
        for p in arena.params:
            arena.step_tensors[id(p)] = optimizer.state[p]['step'] = torch.tensor(float(arena.steps))
    if loaded and step is not None:
        step.momentum_loaded = True
    return loaded


def train_epoch(args, epoch, model, device, dataloader, optimizer, scheduler, writer=None):
    if scheduler is not None:
        scheduler.step()  # stepped at epoch START like the reference (main_dgl.py:73-74)
    if epoch < 20:
        print(epoch, optimizer.param_groups[0]['lr'])
    model.train()
    print("Start training ... ")
    rank0 = not (torch.distributed.is_available() and torch.distributed.is_initialized()) or \
        torch.distributed.get_rank() == 0
    hist, pending, totals, nsteps = None, [], [0.0, 0.0, 0.0], 0

    def flush():
        if not pending:
            return
        rows = hist[:len(pending)].tolist()  # ONE D2H for up to LOG_EVERY steps
        if rank0:
            with open(GRAD_CSV, 'a', newline='') as f:
                w = csv.writer(f)
                for r in rows:
                    w.writerow([r[6], r[7]])
        for r in rows:
            totals[0] += r[0]
            totals[1] += r[1]
            totals[2] += r[2]
        del pending[:]

    # one batch of look-ahead: the H2D copy of batch k+1 (copy stream) overlaps the kernels of step k
    pipe, apipe = _pipeline_of(dataloader), _audio_pipeline_of(dataloader)
    it = iter(dataloader)
    nxt = next(it, None)
    st = None
    if nxt is not None:
        st = _get_step(args, model, optimizer, nxt[0], nxt[1], pipe, apipe)
        _prefetch(st, nxt, pipe, apipe)
    step_i = -1
    while nxt is not None:
        step_i += 1
        spec, image, label = nxt
        if hist is None:
            hist = torch.zeros(LOG_EVERY, 8, device=st.device)
        stats = st.step(lr=optimizer.param_groups[0]['lr'])
        nxt = next(it, None)
        if nxt is not None:
            st2 = _get_step(args, model, optimizer, nxt[0], nxt[1], pipe, apipe)
            if st2 is not st:  # geometry changed (last partial batch without drop_last): new engine
                st = st2
            _prefetch(st, nxt, pipe, apipe)
        hist[len(pending)].copy_(stats)
        pending.append(step_i)
        nsteps += 1
        if step_i % LOG_EVERY == 0:
            s = st.read_stats()
            print("unimodal_loss:", s[1] + s[2], "cls_loss:", s[0])
            print("grad:", s[5], s[6])
            print("unimodal", st.logits[1].abs().mean().item(), st.logits[2].abs().mean().item())
        if len(pending) == LOG_EVERY:
            flush()
    flush()
    if st is not None:
        st.arena.sync_step_tensors()  # optimizer.state[p]['step'] for the checkpoint main_dgl.py writes next
    n = max(len(dataloader), 1) if hasattr(dataloader, "__len__") else max(nsteps, 1)
    return totals[0] / n, totals[1] / n, totals[2] / n, 0.0, 0.0, 0.0, 0.0


def _sharded(dataloader):
    """True for a data-parallel test loader: one rank's contiguous shards of the global batches."""
    return _world() > 1 and isinstance(getattr(dataloader, "batch_sampler", None), ChunkShardBatchSampler)


def valid(args, model, device, dataloader):
    """reference main_dgl.py:168-222: eval-mode forward (BN running statistics), softmax,
    arg-max accuracy of the fused / audio / visual heads.  Runs on the cached EvalStep of the batch geometry (CUDA
    graph, the next batch prefetched on the copy stream); the correct counts accumulate on the device and are read
    once at the end.  `drop_last` behaviour is the loader's.
    A data-parallel test loader (parallel.ChunkShardBatchSampler: each rank evaluates its shard of every global batch)
    is evaluated like nn.DataParallel evaluates the reference's: every rank first takes rank 0's BatchNorm running
    statistics, and the counts are summed over the ranks, so every rank returns the accuracy over all the samples."""
    inner = getattr(model, "module", model)
    inner.args.drop = 0
    with torch.no_grad():
        model.eval()
        print(inner.args.drop)
        pipe, apipe = _pipeline_of(dataloader), _audio_pipeline_of(dataloader)
        sharded = _sharded(dataloader)
        if sharded:
            broadcast_running_stats(inner)
        counts = eval_counts(inner, next(inner.parameters()).device)
        counts.zero_()
        total = 0
        it = iter(dataloader)
        nxt = next(it, None)
        ev = None

        def get(batch):
            spec_hw, thw = _geometry(batch[0], batch[1], pipe, apipe)
            return get_eval_step(inner, batch[2].shape[0], spec_hw, thw)
        if nxt is not None:
            ev = get(nxt)
            _prefetch(ev, nxt, pipe, apipe)
        while nxt is not None:
            ev.run()
            total += ev.rows
            nxt = next(it, None)
            if nxt is not None:
                ev = get(nxt)
                _prefetch(ev, nxt, pipe, apipe)
        res = torch.cat([counts, torch.tensor([total], device=counts.device, dtype=torch.int64)])
        if sharded:
            torch.distributed.all_reduce(res)
        res = res.tolist()  # the one D2H of the evaluation
    inner.args.drop = 1
    n = max(res[3], 1)
    return res[0] / n, res[1] / n, res[2] / n
