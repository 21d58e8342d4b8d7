"""Per-class validation (train.valid_report, EvalStep.run(report=True)) and its confusion kernel (csrc/eval.cu
gdl_eval_confusion).  GPU only."""
import argparse
import os

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


def confusion_of(preds, labels, n):
    """int64 [3, n, n] by torch.bincount: preds [3, N] arg-maxes, labels [N] (only 0 <= label < n count)."""
    keep = (labels >= 0) & (labels < n)
    conf = torch.zeros(3, n * n, dtype=torch.int64)
    for h in range(3):
        conf[h] = torch.bincount((labels[keep] * n + preds[h][keep]).cpu(), minlength=n * n)
    return conf.view(3, n, n)


def model_confusion(model, batches, n):
    """The confusion matrices of the logits model(...) returns in eval mode for `batches`."""
    preds, labels = [], []
    model.eval()
    with torch.no_grad():
        for spec, image, label in batches:
            out = model(spec.cuda().unsqueeze(1).float(), image.cuda().float())
            preds.append(torch.stack([o.argmax(1) for o in out]).cpu())
            labels.append(label)
    return confusion_of(torch.cat(preds, 1), torch.cat(labels), n)


# ------------------------------------------------------------------------------------------------ the kernel
@pytest.mark.parametrize("n", [6, 34, 309, 512])
def test_confusion_kernel_against_bincount_of_torch_argmax(n):
    from gdl_b200 import ops
    g = torch.Generator().manual_seed(n)
    B = 300
    logits = torch.randn(3, B, n, generator=g)
    logits[:, 0:20, 1] = logits[:, 0:20, 0] = 50.0                   # ties between columns 0 and 1
    logits[:, 20:30, n - 1] = logits[:, 20:30, n // 2] = 50.0        # ties between two inner columns
    logits[:, 30:40, n // 3] = float("nan")                           # a NaN is the largest value
    logits[:, 40:45, n - 1] = logits[:, 40:45, 0] = float("nan")      # two NaNs: the lowest index
    logits[1, 45:50] = 0.0                                            # a whole row ties
    label = torch.randint(0, n, (B,), generator=g)
    label[0:20:2] = 1
    label[50:60] = -1                                                 # padding rows: skipped
    label[60:63] = n                                                  # out of range: counted, never indexed
    label[63] = n + 1000
    logits, label = logits.cuda(), label.cuda()
    guard = 64
    buf = torch.zeros(guard + 1 + 3 * n * n + guard, dtype=torch.int64, device="cuda")
    oor, conf = buf[guard:guard + 1], buf[guard + 1:guard + 1 + 3 * n * n]
    ops.eval_confusion(logits, label, conf, oor, B, n)
    ops.eval_confusion(logits, label, conf, oor, B, n)  # it adds
    torch.cuda.synchronize()
    ref = confusion_of(logits.argmax(2), label, n)
    assert torch.equal(conf.view(3, n, n).cpu(), 2 * ref)
    assert int(oor) == 2 * 4
    assert int(buf[:guard].abs().sum()) == 0 and int(buf[-guard:].abs().sum()) == 0
    # the trace of every head's matrix is what the count kernel adds on the same logits
    counts = torch.zeros(3, dtype=torch.int64, device="cuda")
    ops.eval_count(logits, label, counts, B, n)
    assert [int(c) * 2 for c in counts] == [int(conf.view(3, n, n)[h].trace()) for h in range(3)]
    assert int(ref.sum()) == 3 * (B - 10 - 4)


def test_confusion_kernel_rejects_bad_arguments():
    from gdl_b200 import _lib, ops
    logits = torch.zeros(3, 4, 513, device="cuda")
    label = torch.zeros(4, dtype=torch.int64, device="cuda")
    conf = torch.zeros(3 * 513 * 513, dtype=torch.int64, device="cuda")
    oor = torch.zeros(1, dtype=torch.int64, device="cuda")
    for B, n in ((4, 513), (4, 0), (0, 6)):
        with pytest.raises(_lib.GdlError):
            ops.eval_confusion(logits, label, conf, oor, B, n)
    with pytest.raises(_lib.GdlError):
        ops.eval_confusion(logits, label, conf, None, 4, 6)
    torch.cuda.synchronize()
    assert int(conf.abs().sum()) == 0 and int(oor) == 0


# ------------------------------------------------------------------------------------------------ valid_report()
@pytest.mark.parametrize("fusion,x_gate", [("concat", True), ("sum", True), ("gated", True), ("gated", False),
                                           ("film", True)])
@pytest.mark.parametrize("shape,B", [("tiny", 16), ("CREMAD", 4)])
def test_valid_report_against_the_logits_of_model(fusion, x_gate, shape, B):
    from gdl_b200.train import valid, valid_report
    from oracle.synth import make_batch
    args, model = trained(fusion, shape, B)
    if fusion == "gated":
        model.fusion_module.x_gate = x_gate
    batches = [make_batch(B, 6, shape, seed=50 + i) for i in range(3)]
    dev = torch.device("cuda")
    rep = valid_report(args, model, dev, batches)
    assert args.drop == 1 and not model.training
    acc = valid(args, model, dev, batches)
    n = model.n_classes
    assert rep.confusion.device.type == "cpu" and rep.confusion.dtype == torch.int64
    assert rep.confusion.shape == (3, n, n)
    assert torch.equal(rep.confusion, model_confusion(model, batches, n))
    assert (rep.acc, rep.acc_a, rep.acc_v) == acc
    labels = torch.cat([b[2] for b in batches])
    assert rep.total == labels.numel()
    assert torch.equal(rep.support, torch.bincount(labels, minlength=n))
    empty = rep.support == 0
    assert bool(rep.per_class[:, empty].isnan().all()) and not bool(rep.per_class[:, ~empty].isnan().any())


# ------------------------------------------------------------------------------------------------ graphs and launches
@pytest.mark.parametrize("fusion", ["concat", "film"])
def test_report_graph_replay_is_bit_identical_to_eager(fusion):
    from gdl_b200.step import EvalStep, eval_confusion, eval_counts
    from oracle.synth import SHAPES, make_batch
    args, model = trained(fusion, "tiny", 8, steps=1)
    model.eval()
    Fq, Tt, T, H, W = SHAPES["tiny"]
    dev = next(model.parameters()).device  # cuda:0, the device the EvalStep keys its buffers by
    counts = eval_counts(model, dev)
    res = {}
    for use_graph in (False, True):
        ev = EvalStep(model, 16, (Fq, Tt), (T, H, W), use_graph=use_graph)
        counts.zero_()
        eval_confusion(model, dev).zero_()
        outs = []
        for i in range(3):
            spec, image, label = make_batch(16, 6, "tiny", seed=70 + i)
            ev.load_inputs(spec, image, label)
            out = torch.empty(3, 16, model.n_classes, device="cuda")
            ev.run(out, report=True)
            outs.append(out)
        res[use_graph] = (torch.stack(outs), counts.clone(), eval_confusion(model, dev).clone())
        assert bool(ev.graphs) == use_graph
    for a, b in zip(res[False], res[True]):
        assert torch.equal(a, b)
    assert int(res[True][2][1:].sum()) == 3 * 3 * 16


def test_second_report_epoch_captures_nothing_and_allocates_nothing():
    from gdl_b200.train import valid_report
    from oracle.synth import make_batch
    args, model = trained("concat", "tiny", 8, steps=1)
    test = [make_batch(8, 6, "tiny", seed=90 + s) for s in range(3)]
    dev = torch.device("cuda")
    first = valid_report(args, model, dev, test)
    torch.cuda.synchronize()
    evs = dict(model._gdl_evals)
    graphs = [dict(e.graphs) for e in evs.values()]
    mem = torch.cuda.memory_allocated()
    second = valid_report(args, model, dev, test)
    torch.cuda.synchronize()
    assert dict(model._gdl_evals) == evs and [dict(e.graphs) for e in evs.values()] == graphs and all(graphs)
    assert torch.cuda.memory_allocated() == mem
    assert torch.equal(first.confusion, second.confusion)


def test_valid_and_valid_report_alternate_on_two_cached_graphs():
    from gdl_b200 import ops
    from gdl_b200.train import valid, valid_report
    from oracle.synth import make_batch
    args, model = trained("concat", "tiny", 8, steps=1)
    test = [make_batch(8, 6, "tiny", seed=100 + s) for s in range(3)]
    dev = torch.device("cuda")

    def launches(fn):
        torch.cuda.synchronize()
        n0 = ops.LAUNCHES
        r = fn(args, model, dev, test)
        torch.cuda.synchronize()
        return ops.LAUNCHES - n0, r

    launches(valid)
    n_before, acc_before = launches(valid)
    launches(valid_report)
    (ev,) = model._gdl_evals.values()
    graphs = dict(ev.graphs)
    assert len(graphs) == 2 and sorted(k[1] is not None for k in graphs) == [False, True]
    n_rep, rep = launches(valid_report)
    n_after, acc_after = launches(valid)
    launches(valid_report)
    assert dict(ev.graphs) == graphs  # the same two graph objects: nothing re-captured
    assert acc_before == acc_after == (rep.acc, rep.acc_a, rep.acc_v)
    assert n_before == n_after == n_rep == 2 * len(test), (n_before, n_after, n_rep)  # stem layouts + replays


# ------------------------------------------------------------------------------------------------ other paths
def test_report_with_two_replicas_runs_in_sub_batches(tmp_path):
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
    rep = valid_report(args, model, dev, test)
    (ev,) = model._gdl_evals.values()
    assert ev.B == 4 and ev.chunks == 2 and ev.enc_a is model._gdl_step.enc_a
    assert torch.equal(rep.confusion, model_confusion(model, test, model.n_classes))
    assert (rep.acc, rep.acc_a, rep.acc_v) == valid(args, model, dev, test)


def test_report_device_pipeline_and_short_tail_batch():
    from torch.utils.data import DataLoader
    from gdl_b200.synthetic import SyntheticCramedDevice
    from gdl_b200.train import valid, valid_report
    args, model = make_model("concat")
    args.fps, args.use_video_frames = 2, 3
    ds = SyntheticCramedDevice(args, "test", 10)
    ds.attach_pipeline(torch.device("cuda"))
    loader = DataLoader(ds, batch_size=4, shuffle=False, num_workers=0, drop_last=False)  # 4, 4, 2
    dev = torch.device("cuda")
    rep = valid_report(args, model, dev, loader)
    preds, labels = [], []
    model.eval()
    with torch.no_grad():
        for params, boxes, label in loader:
            spec = ds.device_audio_pipeline(params.cuda())
            image = ds.device_pipeline(boxes.reshape(-1, 6).cuda())
            out = model(spec.unsqueeze(1), image)
            preds.append(torch.stack([o.argmax(1) for o in out]).cpu())
            labels.append(label)
    n = model.n_classes
    assert rep.total == 10 and int(rep.support.sum()) == 10
    assert torch.equal(rep.confusion, confusion_of(torch.cat(preds, 1), torch.cat(labels), n))
    assert (rep.acc, rep.acc_a, rep.acc_v) == valid(args, model, dev, loader)


def test_out_of_range_labels_raise_naming_the_width_and_the_rows():
    from gdl_b200.train import valid, valid_report
    from oracle.synth import make_batch
    args, model = make_model("concat")
    n = model.n_classes
    test = [make_batch(8, 6, "tiny", seed=120 + s) for s in range(2)]
    test[1][2][3] = n
    test[1][2][5] = n + 4
    dev = torch.device("cuda")
    with pytest.raises(ValueError) as e:
        valid_report(args, model, dev, test)
    msg = str(e.value)
    assert "2 evaluated rows" in msg and "{} classes".format(n) in msg, msg
    assert args.drop == 1
    valid(args, model, dev, test)  # valid() keeps the reference's counting: such a row is simply never correct


def test_cli_per_class_csv_agrees_with_the_accuracy_csv(tmp_path):
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
                       "--batch_size", "8", "--epochs", "2", "--per_class"])
    finally:
        os.chdir(cwd)
    with open(ckpt / "CREMAD_full.csv", newline="") as f:
        accs = [[float(x) for x in r] for r in csv.reader(f)][1:]  # after the run separator
    with open(ckpt / "CREMAD_full_per_class.csv", newline="") as f:
        rows = list(csv.reader(f))
    assert rows[0] == ["epoch", "head", "class", "support", "correct", "accuracy"]
    assert len(accs) == 2 and len(rows) == 1 + 2 * 3 * 6
    for e in range(2):
        mine = [r for r in rows[1:] if r[0] == str(e)]
        total = sum(int(r[3]) for r in mine if r[1] == "out")
        got = [sum(int(r[4]) for r in mine if r[1] == h) / total for h in ("out", "out_a", "out_v")]
        assert got == accs[e], (got, accs[e])


def test_two_gpus_report_shards():
    """torchrun, 2 ranks (tests/dist_report_check.py)."""
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = os.path.join(os.path.dirname(__file__), "dist_report_check.py")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29541", script],
                       capture_output=True, text=True, timeout=900)
    assert "DIST_REPORT_CHECK_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
