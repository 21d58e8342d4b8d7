"""Drop-ins for the reference's `train_epoch` (main_dgl.py:69-165) and `valid` (:168-222) with
the same signatures, return values, prints and CSV side effects, running on the fused DGLStep.

Differences that are invisible to the caller: the 123 per-step host syncs of the reference
(120 `.item()` for the diagnostics + 3 losses) become one 8-float D2H per LOG_EVERY steps
(the per-step values are kept in a device ring and flushed in order), and the optimizer passed
in is only read for its update rule, hyper-parameters and lr schedule (gdl_b200.optim.update_rule: SGD-momentum,
Adam or Adagrad; anything else raises) — the update itself is a fused kernel over the parameter arena (its state is
exposed through `optimizer.state[p]` — `momentum_buffer`, `exp_avg` / `exp_avg_sq` / `step`, `sum` / `step` — so
reference-format checkpoints still carry it).
`valid_report` is an addition: `valid` plus the per-class confusion matrices of the three heads (EvalReport), and
with ap=True the per-class average precision, mAP and top-k accuracy of the three heads.
"""
import csv

import torch

from .optim import update_rule
from .parallel import ChunkShardBatchSampler, broadcast_running_stats, replicas_per_rank
from .step import DGLStep, EvalScores, eval_confusion, eval_counts, eval_scores, get_eval_step

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


def _evaluate(model, dataloader, report, topk=None):
    """The evaluation pass of valid() and valid_report() on the model's cached EvalSteps, with the reference's
    args.drop flips, print, eval() and no_grad.  Returns the CPU int64 tensor [counts (3), total] and, with `report`,
    then the out-of-range row count and the confusion matrices [3 n n] (step.eval_confusion), summed over the ranks of
    a sharded loader by one all-reduce after rank 0's BatchNorm statistics were broadcast.  With `topk` (an int) the
    pass also appends every row's softmax scores to the model's EvalScores, sized len(loader) x the first batch's rows,
    and the tensor goes on with [overflow, top-k hits (3), capacity, rows beyond it, total^2, capacity^2] (summed
    with the rest) and gdl_eval_ap's results: ap [3 n] (f64 bits), support [n], nonfinite.  A sharded loader's stores
    are gathered after the all-reduce and every rank computes the AP of all the rows."""
    inner = getattr(model, "module", model)
    inner.args.drop = 0
    with torch.no_grad():
        model.eval()
        print(inner.args.drop)
        pipe, apipe = _pipeline_of(dataloader), _audio_pipeline_of(dataloader)
        sharded = _sharded(dataloader)
        if sharded:
            broadcast_running_stats(inner)
        dev = next(inner.parameters()).device
        counts = eval_counts(inner, dev)
        counts.zero_()
        conf = eval_confusion(inner, dev).zero_() if report else None
        total = 0
        it = iter(dataloader)
        nxt = next(it, None)
        ev = None
        sc, capacity = None, 0
        if topk is not None:
            capacity = len(dataloader) * (nxt[2].shape[0] if nxt is not None else 0)
            sc = eval_scores(inner, dev, capacity)
            sc.state.zero_()
            sc.k = max(1, min(int(topk), inner.n_classes))

        def get(batch):
            spec_hw, thw = _geometry(batch[0], batch[1], pipe, apipe)
            return get_eval_step(inner, batch[2].shape[0], spec_hw, thw)
        if nxt is not None:
            ev = get(nxt)
            _prefetch(ev, nxt, pipe, apipe)
        while nxt is not None:
            ev.run(report=report, scores=sc is not None)
            total += ev.rows
            nxt = next(it, None)
            if nxt is not None:
                ev = get(nxt)
                _prefetch(ev, nxt, pipe, apipe)
        parts = [counts, torch.tensor([total], device=dev, dtype=torch.int64)] + ([conf] if report else [])
        if sc is not None:
            parts += [sc.state[1:], torch.tensor([capacity, max(total - capacity, 0), total * total, sc.capacity,
                                                  sc.capacity * sc.capacity], device=dev, dtype=torch.int64)]
        res = torch.cat(parts)
        if sharded:
            torch.distributed.all_reduce(res)
        if sc is not None:
            g = _gather_scores(sc, res, total) if sharded else sc
            if g is not None:
                g.average_precision()
                res = torch.cat([res, g.ap.view(-1).view(torch.int64), g.support, g.nonfinite])
        res = res.cpu()  # the one D2H of the evaluation
    inner.args.drop = 1
    return res


def _gather_scores(sc, res, rows):
    """Every rank's stored rows (all_gather_into_tensor of the score and label stores) in one EvalScores of W x rows
    rows, or None when the all-reduced tail of `res` shows that the ranks cannot be gathered: a rank ran out of store
    rows, or the ranks evaluated different numbers of rows or hold stores of different sizes (checked as
    sum^2 == W x sum of squares, so every rank takes the same decision).  ChunkShardBatchSampler with drop_last gives
    every rank the same rows."""
    W = torch.distributed.get_world_size()
    overflow = int(res[-9])
    _, beyond, rows_sq, caps, caps_sq = res[-5:].tolist()  # the only read before the gather
    total = int(res[3])
    if overflow or beyond or total * total != W * rows_sq or caps * caps != W * caps_sq:
        return None
    g = sc.gathered
    if g is None or g.capacity != max(W * rows, 1) or g.flat.numel() != W * sc.store.numel():
        g = sc.gathered = EvalScores(sc.n, max(W * rows, 1), sc.store.device)
        g.flat = torch.empty(W * sc.store.numel(), device=sc.store.device)
        g.flat_labels = torch.empty(W * sc.capacity, dtype=torch.int32, device=sc.store.device)
    torch.distributed.all_gather_into_tensor(g.flat, sc.store.view(-1))
    torch.distributed.all_gather_into_tensor(g.flat_labels, sc.labels)
    n, cap = sc.n, sc.capacity
    if rows:
        g.store.view(3, n, W, rows).copy_(g.flat.view(W, 3, n, cap)[..., :rows].permute(1, 2, 0, 3))
        g.labels.view(W, rows).copy_(g.flat_labels.view(W, cap)[:, :rows])
    g.cursor.fill_(W * rows)
    return g


def valid(args, model, device, dataloader):
    """reference main_dgl.py:168-222: eval-mode forward (BN running statistics), softmax,
    arg-max accuracy of the fused / audio / visual heads.  Runs on the cached EvalStep of the batch geometry (CUDA
    graph, the next batch prefetched on the copy stream); the correct counts accumulate on the device and are read
    once at the end.  `drop_last` behaviour is the loader's.
    A data-parallel test loader (parallel.ChunkShardBatchSampler: each rank evaluates its shard of every global batch)
    is evaluated like nn.DataParallel evaluates the reference's: every rank first takes rank 0's BatchNorm running
    statistics, and the counts are summed over the ranks, so every rank returns the accuracy over all the samples."""
    res = _evaluate(model, dataloader, False).tolist()
    n = max(res[3], 1)
    return res[0] / n, res[1] / n, res[2] / n


HEADS = ("out", "out_a", "out_v")


class EvalReport:
    """Per-class result of valid_report().
    confusion  CPU int64 [3, n, n]: heads (out, out_a, out_v), rows = true class, columns = arg-max
    total      evaluated rows (as valid() counts them)
    support    int64 [n]: rows per true class (the row sums, the same for every head)
    correct    int64 [3, n]: the diagonals
    acc, acc_a, acc_v   the traces over max(total, 1): what valid() returns for the same loader
    per_class  float64 [3, n]: correct / support, NaN for a class without samples
    With valid_report(ap=True) (None otherwise):
    ap         float64 [3, n]: average precision of every head and class on the softmax scores (sklearn's
               average_precision_score, ties included), NaN for a class without samples (sklearn gives 0.0 there)
    map, map_a, map_v   the mean AP over the classes with samples (NaN when there is none)
    k          the k of the top-k accuracy (5, or n when there are fewer classes)
    hits       int64 [3]: rows whose label ranks < k in each head's logits (the arg-max order)
    top5, top5_a, top5_v   hits / max(total, 1)
    nonfinite  rows with a non-finite score in some head (counted, not raised)"""

    def __init__(self, confusion, total, ap=None, hits=None, k=None, nonfinite=None):
        self.confusion = confusion
        self.total = int(total)
        self.n = confusion.shape[-1]
        self.support = confusion[0].sum(1)
        self.correct = confusion.diagonal(dim1=1, dim2=2).clone()
        hits_1 = self.correct.sum(1).tolist()
        den = max(self.total, 1)
        self.acc, self.acc_a, self.acc_v = hits_1[0] / den, hits_1[1] / den, hits_1[2] / den
        self.per_class = torch.where(self.support > 0, self.correct.double() / self.support.clamp(min=1).double(),
                                     torch.tensor(float("nan"), dtype=torch.float64))
        self.ap, self.hits, self.k = ap, hits, k
        self.nonfinite = None if nonfinite is None else int(nonfinite)
        self.map = self.map_a = self.map_v = self.top5 = self.top5_a = self.top5_v = None
        if ap is not None:
            present = self.support > 0
            m = [ap[h][present].mean().item() if bool(present.any()) else float("nan") for h in range(3)]
            self.map, self.map_a, self.map_v = m
            t = [int(x) / den for x in hits]
            self.top5, self.top5_a, self.top5_v = t

    def rows(self, epoch):
        """[epoch, head, class, support, correct, accuracy] for every head and class (accuracy 'nan' for an empty
        class): the rows of main_dgl.py --per_class's per-class CSV."""
        sup, cor, acc = self.support.tolist(), self.correct.tolist(), self.per_class.tolist()
        return [[epoch, HEADS[h], c, sup[c], cor[h][c], acc[h][c]] for h in range(3) for c in range(self.n)]

    def ap_rows(self, epoch):
        """Per head: [epoch, head, class, support, ap] for every class (ap nan for an empty class), then
        [epoch, head, 'mAP', classes with samples, map] and [epoch, head, 'top5', total, top-5 accuracy] (the label
        is 'top<k>'): the rows of main_dgl.py --ap's CSV."""
        if self.ap is None:
            raise ValueError("ap_rows() needs a report of valid_report(ap=True)")
        sup, ap = self.support.tolist(), self.ap.tolist()
        present = int((self.support > 0).sum())
        maps, tops = (self.map, self.map_a, self.map_v), (self.top5, self.top5_a, self.top5_v)
        out = []
        for h in range(3):
            out += [[epoch, HEADS[h], c, sup[c], ap[h][c]] for c in range(self.n)]
            out.append([epoch, HEADS[h], "mAP", present, maps[h]])
            out.append([epoch, HEADS[h], "top%d" % self.k, self.total, tops[h]])
        return out

    def table(self):
        """The per-class accuracies as text: one line per class, one column per head."""
        acc = self.per_class.tolist()
        lines = ["{:>5} {:>7} {:>8} {:>8} {:>8}".format("class", "support", *HEADS)]
        for c, sup in enumerate(self.support.tolist()):
            lines.append("{:>5} {:>7} {:>8.4f} {:>8.4f} {:>8.4f}".format(c, sup, acc[0][c], acc[1][c], acc[2][c]))
        return "\n".join(lines)

    def ap_table(self):
        """The per-class average precisions as text: one line per class, one column per head, then the mAP line."""
        ap = self.ap.tolist()
        lines = ["{:>5} {:>7} {:>8} {:>8} {:>8}".format("class", "support", *HEADS)]
        for c, sup in enumerate(self.support.tolist()):
            lines.append("{:>5} {:>7} {:>8.4f} {:>8.4f} {:>8.4f}".format(c, sup, ap[0][c], ap[1][c], ap[2][c]))
        lines.append("{:>5} {:>7} {:>8.4f} {:>8.4f} {:>8.4f}".format("mAP", int((self.support > 0).sum()), self.map,
                                                                     self.map_a, self.map_v))
        return "\n".join(lines)


def valid_report(args, model, device, dataloader, ap=False, topk=5):
    """valid() with the per-class confusion matrices of the three heads (EvalReport), counted on the device by
    gdl_eval_confusion in the same graph-captured pass and read with the counts in its one D2H (one all-reduce for a
    sharded loader).  Same args.drop flips, print and accuracies as valid().  Raises ValueError when a label is >= the
    head width (the reference fails with an IndexError on `num[label]`).
    ap=True: the same pass also appends every row's softmax scores to a device store (gdl_eval_scores, room for
    len(dataloader) x the first batch's rows) and counts the top-`topk` hits; gdl_eval_ap then computes the per-class
    average precision, read in the same D2H.  A sharded loader's stores are gathered so that every rank computes the
    AP of all the rows, bit for bit the same.  Raises ValueError for a loader without len(), for more rows than the
    store holds, and for a sharded loader whose ranks evaluated different numbers of rows."""
    if ap:
        try:
            len(dataloader)
        except TypeError:
            raise ValueError("valid_report(ap=True) sizes its score store as len(loader) x the first batch's rows; "
                             "{} has no len()".format(type(dataloader).__name__)) from None
    res = _evaluate(model, dataloader, True, topk if ap else None)
    n = getattr(model, "module", model).n_classes
    if int(res[4]):
        raise ValueError("{} evaluated rows have a label outside the {} classes of the heads (0..{})"
                         .format(int(res[4]), n, n - 1))
    base = 5 + 3 * n * n
    conf, total = res[5:base].view(3, n, n), int(res[3])
    if not ap:
        return EvalReport(conf, total)
    overflow, capacity, beyond = int(res[base]), int(res[base + 4]), int(res[base + 5])
    if overflow or beyond:
        raise ValueError("{} evaluated rows do not fit in the {} rows of the score store (len(loader) x the first "
                         "batch's rows{})".format(total, capacity, ", over all ranks" if _sharded(dataloader) else ""))
    if res.numel() == base + 9:
        raise ValueError("average precision over a sharded test loader needs the same number of rows on every rank "
                         "(ChunkShardBatchSampler with drop_last): {} rows over {} ranks"
                         .format(total, _world()))
    tail = res[base + 9:]
    k = max(1, min(int(topk), n))
    return EvalReport(conf, total, ap=tail[:3 * n].view(torch.float64).view(3, n).clone(),
                      hits=res[base + 1:base + 4].clone(), k=k, nonfinite=int(tail[-1]))
