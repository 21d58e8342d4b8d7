"""Average precision, mAP and top-k accuracy in validation (train.valid_report(ap=True), EvalStep.run(scores=True)) and
their kernels (csrc/eval.cu gdl_eval_scores, gdl_eval_ap).  GPU only."""
import argparse
import os
import warnings

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def make_model(fusion="concat", dataset="CREMAD"):
    import gdl_b200
    args = argparse.Namespace(dataset=dataset, fusion_method=fusion, modality="full", alpha=4.0, epochs=1, drop=0)
    gdl_b200.setup_seed(0)
    m = gdl_b200.AVClassifier_DGL(args)
    m.apply(gdl_b200.weight_init)
    return args, m.cuda()


def trained(fusion, shape, B, steps=3):
    from gdl_b200.step import DGLStep
    from oracle.synth import SHAPES, make_batch
    args, model = make_model(fusion)
    Fq, Tt, T, H, W = SHAPES[shape]
    st = DGLStep(model, B, (Fq, Tt), (T, H, W), lr=0.01, use_graph=False)
    for s in range(steps):
        st.step(*[t.cuda() for t in make_batch(B, 6, shape, seed=1 + s)])
    torch.cuda.synchronize()
    return args, model


def ap_numpy(scores, labels, n):
    """AP of every class column of scores [N, n] (rows with a label outside 0..n-1 dropped): (1 / P_c) times the sum
    over the positives i of TP(>= s_i) / N(>= s_i); NaN for a class without positives."""
    keep = (labels >= 0) & (labels < n)
    scores, labels = scores[keep], labels[keep]
    out = np.full(n, np.nan)
    for c in range(n):
        s = scores[:, c].astype(np.float64)
        pos = labels == c
        if not pos.any():
            continue
        all_sorted, pos_sorted, t = np.sort(s), np.sort(s[pos]), s[pos]
        out[c] = np.mean((len(t) - np.searchsorted(pos_sorted, t, "left")) /
                         (len(s) - np.searchsorted(all_sorted, t, "left")))
    return out


def ap_sklearn(scores, labels, n):
    """sklearn's average_precision_score(average=None) per class column of scores [N, n] over the rows with a label in
    0..n-1; NaN for a class without positives (sklearn returns 0.0 there)."""
    sk = pytest.importorskip("sklearn.metrics")
    keep = (labels >= 0) & (labels < n)
    s, y = np.asarray(scores, dtype=np.float64)[keep], labels[keep]
    out = np.full(n, np.nan)
    present = np.unique(y)
    if len(present):
        onehot = (y[:, None] == present[None, :]).astype(np.int64)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            out[present] = sk.average_precision_score(onehot, s[:, present], average=None)
    return out


def rank_hits(logits, labels, k):
    """int64 [3]: rows (label in 0..n-1) whose label ranks < k: #{j: z_j > z_y} + #{j < y: z_j == z_y}, NaN largest."""
    n = logits.shape[-1]
    keep = (labels >= 0) & (labels < n)
    z = logits[:, keep].double()
    y = labels[keep]
    zy = z.gather(2, y.view(1, -1, 1).expand(3, -1, 1))
    j = torch.arange(n, device=z.device).view(1, 1, n)
    nz, ny = z.isnan(), zy.isnan()
    greater = torch.where(ny, torch.zeros_like(nz), nz | (z > zy))
    equal = (nz & ny) | (z == zy)
    rank = (greater | (equal & (j < y.view(1, -1, 1)))).sum(2)
    return (rank < k).sum(1).cpu()


def softmax_ulps(got, ref):
    """max distance in units of the last place of ref (NaN must match NaN)."""
    got, ref = got.double().cpu().numpy(), ref.double().cpu().numpy()
    assert np.array_equal(np.isnan(got), np.isnan(ref))
    ok = ~np.isnan(ref)
    ulp = np.spacing(np.abs(ref[ok]).astype(np.float32)).astype(np.float64)
    return float(np.max(np.abs(got[ok] - ref[ok]) / ulp)) if ok.any() else 0.0


# ------------------------------------------------------------------------------------------------ gdl_eval_scores
@pytest.mark.parametrize("n", [6, 309])
def test_scores_kernel_softmax_class_major_cursor_and_overflow(n):
    from gdl_b200 import ops
    g = torch.Generator().manual_seed(n)
    B, cap, guard = 100, 250, 64
    batches = []
    for i in range(3):
        logits = 3 * torch.randn(3, B, n, generator=g)
        label = torch.randint(0, n, (B,), generator=g)
        label[10:15] = -1                       # padding rows: stored as -1, never counted
        label[15:17] = n                        # out of range: stored as -1
        logits[2, 20:23, n // 2] = float("nan")  # a NaN logit: the row's scores are NaN, as torch.softmax's
        label[90:] = -1 if i == 2 else label[90:]  # the padding rows beyond cap are not overflow
        batches.append((logits.cuda(), label.cuda()))
    store_buf = torch.full((guard + 3 * n * cap + guard,), 7.0, device="cuda")
    label_buf = torch.full((guard + cap + guard,), 77, dtype=torch.int32, device="cuda")
    state = torch.zeros(guard + 5 + guard, dtype=torch.int64, device="cuda")
    store, slabels = store_buf[guard:guard + 3 * n * cap].view(3, n, cap), label_buf[guard:guard + cap]
    cursor, overflow, hits = state[guard:guard + 1], state[guard + 1:guard + 2], state[guard + 2:guard + 5]
    for logits, label in batches:
        ops.eval_scores(logits, label, store, slabels, cursor, hits, overflow, B, n, min(5, n))
    torch.cuda.synchronize()
    assert int(cursor) == 3 * B
    # rows 200..249 of the third batch fit; its rows 50..89 are labelled and do not fit, 90..99 are padding
    assert int(overflow) == 40
    for i, (logits, label) in enumerate(batches):
        rows = min(B, cap - i * B)
        ref = torch.softmax(logits[:, :rows], -1).permute(0, 2, 1)  # [3, n, rows]
        assert softmax_ulps(store[:, :, i * B:i * B + rows], ref) <= 2.0
        lab = label[:rows].clone()
        lab[(lab < 0) | (lab >= n)] = -1
        assert torch.equal(slabels[i * B:i * B + rows].long(), lab)
    assert float((store_buf[:guard] - 7).abs().sum()) == 0 and float((store_buf[-guard:] - 7).abs().sum()) == 0
    assert bool((label_buf[:guard] == 77).all()) and bool((label_buf[-guard:] == 77).all())
    assert int(state[:guard].abs().sum()) == 0 and int(state[-guard:].abs().sum()) == 0
    ref_hits = sum(rank_hits(lg, lb, min(5, n)) for lg, lb in batches)
    assert hits.cpu().tolist() == ref_hits.tolist()


@pytest.mark.parametrize("n", [6, 34, 309])
@pytest.mark.parametrize("k", [1, 5])
def test_scores_kernel_topk_hits_with_ties_and_nan(n, k):
    from gdl_b200 import ops
    g = torch.Generator().manual_seed(7 * n + k)
    B = 300
    logits = torch.randn(3, B, n, generator=g)
    logits = torch.round(logits * 2) / 2                              # many ties everywhere
    label = torch.randint(0, n, (B,), generator=g)
    logits[:, 0:20, 1] = logits[:, 0:20, 0] = 50.0
    label[0:20:2] = 1                                                 # tied with a lower index: rank 1
    logits[:, 30:40, n // 3] = float("nan")                           # a NaN beats the label
    logits[:, 40:45, label[40:45]] = float("nan")                     # a NaN label logit
    logits[:, 45:47, 0] = float("nan")
    logits[1, 50:55] = 0.0                                            # a whole row ties
    label[60:63] = -1
    label[63] = n
    logits, label = logits.cuda(), label.cuda()
    store = torch.empty(3, n, B, device="cuda")
    slabels = torch.empty(B, dtype=torch.int32, device="cuda")
    state = torch.zeros(5, dtype=torch.int64, device="cuda")
    ops.eval_scores(logits, label, store, slabels, state[0:1], state[2:5], state[1:2], B, n, min(k, n))
    torch.cuda.synchronize()
    assert state[2:5].cpu().tolist() == rank_hits(logits, label, min(k, n)).tolist()
    if k == 1:  # top-1 is valid()'s count, row for row
        counts = torch.zeros(3, dtype=torch.int64, device="cuda")
        ops.eval_count(logits, label, counts, B, n)
        assert state[2:5].tolist() == counts.tolist()


def test_scores_and_ap_kernels_reject_bad_arguments():
    from gdl_b200 import _lib, ops
    from gdl_b200.step import EvalScores
    sc = EvalScores(6, 16, torch.device("cuda"))
    logits = torch.zeros(3, 4, 6, device="cuda")
    label = torch.zeros(4, dtype=torch.int64, device="cuda")
    for B, n, k in ((0, 6, 5), (4, 0, 1), (4, 6, 0), (4, 6, 7), (4, 513, 5)):
        with pytest.raises(_lib.GdlError):
            ops.eval_scores(logits, label, sc.store, sc.labels, sc.cursor, sc.hits, sc.overflow, B, n, k)
    big = EvalScores(6, 20000, torch.device("cuda"))
    assert big.workspace is not None
    with pytest.raises(_lib.GdlError):  # a long store without its workspace
        ops.eval_ap(big.store, big.labels, big.cursor, big.ap, big.support, big.nonfinite, None)
    torch.cuda.synchronize()
    assert int(sc.state.abs().sum()) == 0


# ------------------------------------------------------------------------------------------------ gdl_eval_ap
def _store(n, N, cap, seed, levels=0, nan_rows=0):
    """An EvalScores whose first N rows hold softmax-like scores (quantised to `levels` steps to force ties), labels
    with classes 0 and n - 1 empty, a few padding rows, and garbage beyond N; returns it with the CPU scores [N, n]
    and labels [N]."""
    from gdl_b200.step import EvalScores
    g = torch.Generator().manual_seed(seed)
    s = torch.softmax(2 * torch.randn(3, N, n, generator=g), -1)
    if levels:
        s = torch.round(s * levels) / levels
    label = torch.randint(1, max(n - 1, 2), (N,), generator=g) if n > 2 else torch.zeros(N, dtype=torch.int64)
    label[::97] = -1
    if nan_rows:
        idx = torch.randperm(N, generator=g)[:nan_rows]
        s[torch.randint(0, 3, (nan_rows,), generator=g), idx, torch.randint(0, n, (nan_rows,), generator=g)] = \
            float("nan")
    sc = EvalScores(n, cap, torch.device("cuda"))
    sc.store.fill_(0.5)
    sc.store[:, :, :N] = s.permute(0, 2, 1).cuda()
    sc.labels.fill_(0)
    sc.labels[:N] = label.to(torch.int32).cuda()
    sc.cursor.fill_(N)
    return sc, s, label


@pytest.mark.parametrize("n,N,levels", [(6, 1, 0), (6, 2, 0), (6, 1000, 16), (34, 3000, 0), (34, 3000, 64),
                                        (309, 15000, 0), (309, 15000, 1000), (400, 20000, 0),
                                        (6, 100_000, 0), (6, 100_000, 256)])
def test_ap_kernel_against_sklearn_and_row_order(n, N, levels):
    from gdl_b200 import ops
    sc, s, label = _store(n, N, N + 37, seed=n + N + levels, levels=levels)
    sc.average_precision()
    torch.cuda.synchronize()
    lab = label.numpy()
    for h in range(3):
        ref = ap_sklearn(s[h].numpy(), lab, n)
        got = sc.ap[h].cpu().numpy()
        assert np.array_equal(np.isnan(got), np.isnan(ref)), (h, got, ref)
        ok = ~np.isnan(ref)
        assert np.max(np.abs(got[ok] - ref[ok]), initial=0.0) <= 1e-12, (h, np.max(np.abs(got[ok] - ref[ok])))
    valid = (label >= 0) & (label < n)
    assert sc.support.cpu().tolist() == torch.bincount(label[valid], minlength=n).tolist()
    assert int(sc.nonfinite) == 0
    # the same rows in another order: bit-identical
    perm = torch.randperm(N, generator=torch.Generator().manual_seed(N))
    sc2, _, _ = _store(n, N, N + 37, seed=n + N + levels, levels=levels)
    sc2.store[:, :, :N] = sc.store[:, :, :N][:, :, perm.cuda()]
    sc2.labels[:N] = sc.labels[:N][perm.cuda()]
    ops.eval_ap(sc2.store, sc2.labels, sc2.cursor, sc2.ap, sc2.support, sc2.nonfinite, sc2.workspace)
    torch.cuda.synchronize()
    assert torch.equal(sc.ap.view(torch.int64), sc2.ap.view(torch.int64))
    assert torch.equal(sc.support, sc2.support)


def test_ap_kernel_with_nan_scores_against_numpy():
    n, N = 6, 5000
    sc, s, label = _store(n, N, N, seed=3, levels=32, nan_rows=300)
    sc.average_precision()
    torch.cuda.synchronize()
    valid = (label >= 0) & (label < n)
    bad = (~torch.isfinite(s)).any(2).any(0) & valid
    assert int(sc.nonfinite) == int(bad.sum()) > 0
    for h in range(3):
        ref = ap_numpy(torch.nan_to_num(s[h], nan=2.0).numpy(), label.numpy(), n)  # NaN above every probability
        got = sc.ap[h].cpu().numpy()
        assert np.array_equal(np.isnan(got), np.isnan(ref))
        ok = ~np.isnan(ref)
        assert np.max(np.abs(got[ok] - ref[ok])) <= 1e-12


# ------------------------------------------------------------------------------------------------ valid_report(ap=True)
def model_scores(model, batches):
    """softmax of the logits model(...) returns in eval mode for `batches` ([3, N, n] CPU) and the labels."""
    outs, labels = [], []
    model.eval()
    with torch.no_grad():
        for spec, image, label in batches:
            out = model(spec.cuda().unsqueeze(1).float(), image.cuda().float())
            outs.append(torch.stack(out).cpu())
            labels.append(label)
    return torch.cat(outs, 1), torch.cat(labels)


def check_against_model(rep, logits, labels, n, k=5):
    # torch's CUDA softmax (the CPU one rounds exp differently, which moves ties); the store holds the same scores
    scores = torch.softmax(logits.cuda(), -1).cpu()
    for h in range(3):
        ref = ap_sklearn(scores[h].numpy(), labels.numpy(), n)
        got = rep.ap[h].numpy()
        assert np.array_equal(np.isnan(got), np.isnan(ref)), (got, ref)
        ok = ~np.isnan(ref)
        assert np.max(np.abs(got[ok] - ref[ok]), initial=0.0) <= 1e-12
    assert rep.hits.tolist() == rank_hits(logits, labels, min(k, n)).tolist()
    present = rep.support > 0
    assert rep.map == rep.ap[0][present].mean().item() and rep.top5 == int(rep.hits[0]) / rep.total


@pytest.mark.parametrize("fusion,x_gate", [("concat", True), ("sum", True), ("gated", True), ("gated", False),
                                           ("film", True)])
@pytest.mark.parametrize("shape,B", [("tiny", 16), ("CREMAD", 4)])
def test_valid_report_ap_against_sklearn_on_the_softmax_of_model(fusion, x_gate, shape, B):
    from gdl_b200.train import valid, valid_report
    from oracle.synth import make_batch
    args, model = trained(fusion, shape, B)
    if fusion == "gated":
        model.fusion_module.x_gate = x_gate
    batches = [make_batch(B, 6, shape, seed=50 + i) for i in range(3)]
    dev = torch.device("cuda")
    rep = valid_report(args, model, dev, batches, ap=True)
    assert args.drop == 1 and not model.training
    plain = valid_report(args, model, dev, batches)
    acc = valid(args, model, dev, batches)
    n = model.n_classes
    assert torch.equal(rep.confusion, plain.confusion) and (rep.acc, rep.acc_a, rep.acc_v) == acc
    assert rep.ap.dtype == torch.float64 and rep.ap.shape == (3, n) and rep.k == 5 and rep.nonfinite == 0
    logits, labels = model_scores(model, batches)
    check_against_model(rep, logits, labels, n)
    assert rep.total == labels.numel()
    rep1 = valid_report(args, model, dev, batches, ap=True, topk=1)  # top-1 is the accuracy
    assert rep1.k == 1 and (rep1.top5, rep1.top5_a, rep1.top5_v) == acc
    assert torch.equal(rep1.ap.view(torch.int64), rep.ap.view(torch.int64))


@pytest.mark.parametrize("fusion", ["concat", "film"])
def test_scores_graph_replay_is_bit_identical_to_eager(fusion):
    from gdl_b200.step import EvalStep, eval_confusion, eval_counts, eval_scores
    from oracle.synth import SHAPES, make_batch
    args, model = trained(fusion, "tiny", 8, steps=1)
    model.eval()
    Fq, Tt, T, H, W = SHAPES["tiny"]
    dev = next(model.parameters()).device
    counts = eval_counts(model, dev)
    res = {}
    for use_graph in (False, True):
        ev = EvalStep(model, 16, (Fq, Tt), (T, H, W), use_graph=use_graph)
        counts.zero_()
        eval_confusion(model, dev).zero_()
        sc = eval_scores(model, dev, 48)
        sc.state.zero_()
        sc.store.zero_()
        for i in range(3):
            spec, image, label = make_batch(16, 6, "tiny", seed=70 + i)
            ev.load_inputs(spec, image, label)
            ev.run(report=True, scores=True)
        sc.average_precision()
        res[use_graph] = (counts.clone(), eval_confusion(model, dev).clone(), sc.store.clone(), sc.labels.clone(),
                          sc.state.clone(), sc.ap.view(torch.int64).clone())
        assert bool(ev.graphs) == use_graph
    for a, b in zip(res[False], res[True]):
        assert torch.equal(a, b)
    assert int(res[True][4][0]) == 48 and int(res[True][4][1]) == 0


def test_second_ap_epoch_captures_nothing_and_allocates_nothing():
    from gdl_b200.train import valid_report
    from oracle.synth import make_batch
    args, model = trained("concat", "tiny", 8, steps=1)
    test = [make_batch(8, 6, "tiny", seed=90 + s) for s in range(3)]
    dev = torch.device("cuda")
    first = valid_report(args, model, dev, test, ap=True)
    torch.cuda.synchronize()
    evs = dict(model._gdl_evals)
    graphs = [dict(e.graphs) for e in evs.values()]
    store = model._gdl_eval_scores.store
    mem = torch.cuda.memory_allocated()
    second = valid_report(args, model, dev, test, ap=True)
    torch.cuda.synchronize()
    assert dict(model._gdl_evals) == evs and [dict(e.graphs) for e in evs.values()] == graphs and all(graphs)
    assert model._gdl_eval_scores.store is store
    assert torch.cuda.memory_allocated() == mem
    assert torch.equal(first.ap.view(torch.int64), second.ap.view(torch.int64))
    assert torch.equal(first.hits, second.hits) and torch.equal(first.confusion, second.confusion)


def test_valid_report_and_ap_alternate_on_cached_graphs():
    from gdl_b200 import ops
    from gdl_b200.train import valid, valid_report
    from oracle.synth import make_batch
    args, model = trained("concat", "tiny", 8, steps=1)
    test = [make_batch(8, 6, "tiny", seed=100 + s) for s in range(3)]
    dev = torch.device("cuda")

    def launches(fn, **kw):
        torch.cuda.synchronize()
        n0 = ops.LAUNCHES
        r = fn(args, model, dev, test, **kw)
        torch.cuda.synchronize()
        return ops.LAUNCHES - n0, r

    launches(valid)
    n_before, acc_before = launches(valid)
    launches(valid_report)
    launches(valid_report, ap=True)
    (ev,) = model._gdl_evals.values()
    graphs = dict(ev.graphs)
    assert len(graphs) == 3 and sorted((k[1] is not None, k[2] is not None) for k in graphs) == \
        [(False, False), (True, False), (True, True)]
    n_ap, rep = launches(valid_report, ap=True)
    n_after, acc_after = launches(valid)
    n_rep, _ = launches(valid_report)
    launches(valid_report, ap=True)
    assert dict(ev.graphs) == graphs  # the same three graph objects: nothing re-captured
    assert acc_before == acc_after == (rep.acc, rep.acc_a, rep.acc_v)
    assert n_before == n_after == n_rep == 2 * len(test), (n_before, n_after, n_rep)  # stem layouts + replays
    assert n_ap == 2 * len(test) + 2, n_ap  # + gdl_eval_ap (nonfinite count + AP)


# ------------------------------------------------------------------------------------------------ other paths
def test_ap_with_two_replicas_runs_in_sub_batches(tmp_path):
    from gdl_b200.train import train_epoch, valid, valid_report
    from oracle.synth import make_batch
    args, model = make_model("concat")
    args.batch_size, args.dp_replicas = 8, 2
    opt = torch.optim.SGD(model.parameters(), lr=0.01, momentum=0.9, weight_decay=1e-4)
    train = [make_batch(8, 6, "tiny", seed=1 + s) for s in range(2)]
    test = [make_batch(8, 6, "tiny", seed=110 + s) for s in range(3)]
    dev = torch.device("cuda")
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        train_epoch(args, 0, model, dev, train, opt, None)
    finally:
        os.chdir(cwd)
    rep = valid_report(args, model, dev, test, ap=True)
    (ev,) = model._gdl_evals.values()
    assert ev.B == 4 and ev.chunks == 2
    logits, labels = model_scores(model, test)
    check_against_model(rep, logits, labels, model.n_classes)
    assert (rep.acc, rep.acc_a, rep.acc_v) == valid(args, model, dev, test)


def test_ap_device_pipeline_and_short_tail_batch():
    from torch.utils.data import DataLoader
    from gdl_b200.synthetic import SyntheticCramedDevice
    from gdl_b200.train import valid, valid_report
    args, model = make_model("concat")
    args.fps, args.use_video_frames = 2, 3
    ds = SyntheticCramedDevice(args, "test", 10)
    ds.attach_pipeline(torch.device("cuda"))
    loader = DataLoader(ds, batch_size=4, shuffle=False, num_workers=0, drop_last=False)  # 4, 4, 2: room for 12
    dev = torch.device("cuda")
    rep = valid_report(args, model, dev, loader, ap=True)
    outs, labels = [], []
    model.eval()
    with torch.no_grad():
        for params, boxes, label in loader:
            spec = ds.device_audio_pipeline(params.cuda())
            image = ds.device_pipeline(boxes.reshape(-1, 6).cuda())
            outs.append(torch.stack(model(spec.unsqueeze(1), image)).cpu())
            labels.append(label)
    assert rep.total == 10 and model._gdl_eval_scores.capacity == 12
    check_against_model(rep, torch.cat(outs, 1), torch.cat(labels), model.n_classes)
    assert (rep.acc, rep.acc_a, rep.acc_v) == valid(args, model, dev, loader)


def test_ap_value_errors_name_the_numbers():
    from gdl_b200.train import valid_report
    from oracle.synth import make_batch
    args, model = make_model("concat")
    dev = torch.device("cuda")
    test = [make_batch(8, 6, "tiny", seed=120 + s) for s in range(2)]
    with pytest.raises(ValueError) as e:
        valid_report(args, model, dev, iter(test), ap=True)
    assert "len()" in str(e.value)
    grows = [make_batch(4, 6, "tiny", seed=130), make_batch(8, 6, "tiny", seed=131)]  # room for 2 x 4 rows, 12 come
    with pytest.raises(ValueError) as e:
        valid_report(args, model, dev, grows, ap=True)
    assert "12 evaluated rows" in str(e.value) and "8 rows" in str(e.value), str(e.value)
    assert args.drop == 1
    rep = valid_report(args, model, dev, test, ap=True)  # and the next evaluation is fine
    assert rep.total == 16


def test_cli_ap_csv_and_eval_only_print(tmp_path, capsys):
    import csv
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import main_dgl
    ckpt = tmp_path / "ckpt"
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        main_dgl.main(["--train", "--ckpt_path", str(ckpt), "--audio_path", "synthetic", "--synthetic_len", "64",
                       "--batch_size", "8", "--epochs", "2", "--ap"])
        out = capsys.readouterr().out
        with open(ckpt / "CREMAD_full.csv", newline="") as f:
            accs = [[float(x) for x in r] for r in csv.reader(f)][1:]
        with open(ckpt / "CREMAD_full_ap.csv", newline="") as f:
            rows = list(csv.reader(f))
        assert not os.path.exists(ckpt / "CREMAD_full_per_class.csv")
        assert rows[0] == ["epoch", "head", "class", "support", "ap"]
        assert len(accs) == 2 and len(rows) == 1 + 2 * 3 * (6 + 2)
        lines = out.splitlines()
        maps = [i for i, ln in enumerate(lines) if ln.startswith("mAP: ")]
        assert len(maps) == 2 and all(lines[i - 1].startswith("Audio Acc:") for i in maps), out[-3000:]
        for e in range(2):
            mine = [r for r in rows[1:] if r[0] == str(e)]
            for h in ("out", "out_a", "out_v"):
                per = [r for r in mine if r[1] == h]
                cls = [float(r[4]) for r in per if r[2].isdigit() and int(r[3]) > 0]
                (m,) = [r for r in per if r[2] == "mAP"]
                assert abs(float(m[4]) - sum(cls) / len(cls)) <= 1e-12 and int(m[3]) == len(cls)
        # evaluation mode on a checkpoint of the same model layout
        import gdl_b200
        a = main_dgl.get_arguments(["--ckpt_path", "x"])
        gdl_b200.setup_seed(0)
        m = gdl_b200.AVClassifier_DGL(a)
        m.apply(gdl_b200.weight_init)
        path = tmp_path / "model.pth"
        torch.save({"modulation": a.modulation, "fusion": a.fusion_method,
                    "model": {"module." + k: v for k, v in m.state_dict().items()}}, path)
        main_dgl.main(["--ckpt_path", str(path), "--audio_path", "synthetic", "--synthetic_len", "64",
                       "--batch_size", "8", "--ap"])
        out = capsys.readouterr().out.splitlines()
        i = [j for j, ln in enumerate(out) if ln.startswith("Accuracy: ")][0]
        assert out[i + 1].startswith("mAP: ") and "Top-5 Acc: " in out[i + 1]
        assert out[i + 2].startswith("Per-class average precision") and out[i + 3].split()[0] == "class"
        assert out[i + 4 + 6].split()[0] == "mAP"
    finally:
        os.chdir(cwd)


def test_two_gpus_ap_shards():
    """torchrun, 2 ranks (tests/dist_ap_check.py)."""
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = os.path.join(os.path.dirname(__file__), "dist_ap_check.py")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29543", script],
                       capture_output=True, text=True, timeout=900)
    assert "DIST_AP_CHECK_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
