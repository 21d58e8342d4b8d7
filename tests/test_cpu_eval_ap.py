"""Average precision and top-k accuracy on the host side: a numpy restatement of the AP that gdl_eval_ap computes,
checked against sklearn (ties, empty classes); EvalReport's AP arithmetic and its `ap_rows`; the `--ap` flag's
default; a run without it writes no AP file; the C-ABI declarations.  No GPU."""
import argparse
import math
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


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
        all_sorted, pos_sorted = np.sort(s), np.sort(s[pos])
        t = s[pos]
        n_ge = len(s) - np.searchsorted(all_sorted, t, "left")
        tp_ge = len(t) - np.searchsorted(pos_sorted, t, "left")
        out[c] = np.mean(tp_ge / n_ge)
    return out


@pytest.mark.parametrize("n,N,levels", [(6, 2000, 8), (7, 2000, 3), (34, 500, 0), (5, 40, 2)])
def test_numpy_restatement_equals_sklearn_with_ties(n, N, levels):
    sk = pytest.importorskip("sklearn.metrics")
    rng = np.random.default_rng(n * 1000 + N)
    s = rng.random((N, n)).astype(np.float32)
    if levels:
        s = np.round(s * levels) / levels  # heavy ties
    labels = rng.integers(0, n, N)
    labels[labels == n - 1] = 0  # class n - 1 has no positives
    labels[:5] = -1              # padding rows
    got = ap_numpy(s, labels, n)
    keep = labels >= 0
    onehot = np.eye(n)[labels[keep]]
    with np.errstate(all="ignore"):
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ref = sk.average_precision_score(onehot, s[keep], average=None)
    assert math.isnan(got[n - 1]) and ref[n - 1] == 0.0  # the documented difference: NaN, not 0.0
    np.testing.assert_allclose(got[:n - 1], ref[:n - 1], rtol=0, atol=1e-12)


def _report(ap=True):
    from gdl_b200.train import EvalReport
    conf = torch.zeros(3, 4, 4, dtype=torch.int64)
    conf[0] = torch.tensor([[3, 1, 0, 0], [0, 2, 0, 1], [0, 0, 0, 0], [1, 0, 1, 2]])
    conf[1] = torch.tensor([[4, 0, 0, 0], [3, 0, 0, 0], [0, 0, 0, 0], [0, 0, 0, 4]])
    conf[2] = torch.tensor([[0, 0, 4, 0], [0, 3, 0, 0], [0, 0, 0, 0], [1, 1, 1, 1]])
    if not ap:
        return EvalReport(conf, 12)
    nan = float("nan")
    aps = torch.tensor([[0.5, 0.25, nan, 1.0], [1.0, 0.5, nan, 0.75], [0.125, 1.0, nan, 0.5]], dtype=torch.float64)
    return EvalReport(conf, 12, ap=aps, hits=torch.tensor([10, 9, 8]), k=4, nonfinite=1)


def test_report_map_and_topk_arithmetic():
    r = _report()
    assert (r.map, r.map_a, r.map_v) == ((0.5 + 0.25 + 1.0) / 3, (1.0 + 0.5 + 0.75) / 3, (0.125 + 1.0 + 0.5) / 3)
    assert (r.top5, r.top5_a, r.top5_v) == (10 / 12, 9 / 12, 8 / 12)
    assert r.k == 4 and r.nonfinite == 1
    assert (r.acc, r.acc_a, r.acc_v) == (7 / 12, 8 / 12, 4 / 12)  # the accuracies are untouched


def test_report_without_ap_has_none():
    r = _report(ap=False)
    for name in ("ap", "map", "map_a", "map_v", "top5", "top5_a", "top5_v", "k", "nonfinite"):
        assert getattr(r, name) is None, name
    with pytest.raises(ValueError):
        r.ap_rows(0)


def test_report_map_of_no_class_with_samples_is_nan():
    from gdl_b200.train import EvalReport
    r = EvalReport(torch.zeros(3, 6, 6, dtype=torch.int64), 0, ap=torch.full((3, 6), float("nan"), dtype=torch.float64),
                   hits=torch.zeros(3, dtype=torch.int64), k=5, nonfinite=0)
    assert math.isnan(r.map) and math.isnan(r.map_a) and math.isnan(r.map_v)
    assert (r.top5, r.top5_a, r.top5_v) == (0.0, 0.0, 0.0)


def test_ap_rows_and_table():
    r = _report()
    rows = r.ap_rows(3)
    assert len(rows) == 3 * (4 + 2)
    assert rows[0] == [3, "out", 0, 4, 0.5]
    assert rows[2][:4] == [3, "out", 2, 0] and math.isnan(rows[2][4])
    assert rows[4] == [3, "out", "mAP", 3, r.map]
    assert rows[5] == [3, "out", "top4", 12, 10 / 12]
    assert rows[6 + 3] == [3, "out_a", 3, 4, 0.75]
    assert rows[17] == [3, "out_v", "top4", 12, 8 / 12]
    lines = r.ap_table().splitlines()
    assert len(lines) == 1 + 4 + 1 and lines[3].split() == ["2", "0", "nan", "nan", "nan"]
    assert lines[-1].split()[:2] == ["mAP", "3"]
    assert str(r.rows(3)) == str(_report(ap=False).rows(3))  # the per-class accuracy rows do not change


def _main_dgl():
    sys.path.insert(0, ROOT)
    import main_dgl
    return main_dgl


def test_ap_flag_defaults_off():
    main_dgl = _main_dgl()
    assert main_dgl.get_arguments(["--ckpt_path", "x"]).ap is False
    assert main_dgl.get_arguments(["--ckpt_path", "x", "--ap"]).ap is True


def _args(tmp_path, per_class, ap):
    return argparse.Namespace(ckpt_path=str(tmp_path), dataset="VGGSound", modality="full", per_class=per_class, ap=ap)


def _patch(main_dgl, monkeypatch, calls):
    monkeypatch.setattr(main_dgl, "valid", lambda *a: calls.append("valid") or (0.5, 0.25, 0.125))
    monkeypatch.setattr(main_dgl, "valid_report", lambda *a, **kw: calls.append(("report", kw)) or _report(**kw))


def test_epoch_without_the_flag_writes_no_ap_file(tmp_path, monkeypatch):
    main_dgl = _main_dgl()
    calls = []
    _patch(main_dgl, monkeypatch, calls)
    assert main_dgl.evaluate_epoch(_args(tmp_path, False, False), None, None, None, 0, 0) == (0.5, 0.25, 0.125)
    main_dgl.evaluate_epoch(_args(tmp_path, True, False), None, None, None, 0, 0)
    assert calls == ["valid", ("report", {})]
    assert os.listdir(tmp_path) == ["VGGSound_full_per_class.csv"]


def test_epoch_with_the_flag_appends_ap_rows(tmp_path, monkeypatch):
    import csv
    main_dgl = _main_dgl()
    calls, reports = [], []
    _patch(main_dgl, monkeypatch, calls)
    args = _args(tmp_path, False, True)
    r = _report()
    assert main_dgl.evaluate_epoch(args, None, None, None, 0, 0, reports) == (r.acc, r.acc_a, r.acc_v)
    main_dgl.evaluate_epoch(args, None, None, None, 1, 0)
    main_dgl.evaluate_epoch(args, None, None, None, 2, 1)  # not rank 0: computes, writes nothing
    assert calls == [("report", {"ap": True})] * 3 and len(reports) == 1
    assert os.listdir(tmp_path) == ["VGGSound_full_ap.csv"]
    with open(tmp_path / "VGGSound_full_ap.csv", newline="") as f:
        rows = list(csv.reader(f))
    assert rows[0] == ["epoch", "head", "class", "support", "ap"]
    assert len(rows) == 1 + 2 * 18
    assert rows[1] == ["0", "out", "0", "4", "0.5"] and rows[3][:4] == ["0", "out", "2", "0"]
    assert rows[5] == ["0", "out", "mAP", "3", repr(r.map)]
    assert rows[19 + 17] == ["1", "out_v", "top4", "12", repr(8 / 12)]
    assert main_dgl.ap_line(r) == "mAP: {:.4f}, Audio mAP: {:.4f}, Visual mAP: {:.4f}, Top-4 Acc: {:.4f}".format(
        r.map, r.map_a, r.map_v, 10 / 12)


def test_ap_entry_points_are_declared_and_exported():
    from gdl_b200 import _lib, ops
    hdr = open(os.path.join(ROOT, "include", "gdl_b200.h")).read()
    for name, nargs in (("gdl_eval_scores", 12), ("gdl_eval_ap", 11), ("gdl_eval_ap_workspace_bytes", 2)):
        assert "{}(".format(name) in hdr, name
        assert len(_lib.SIGNATURES[name][1]) == nargs, name
        assert hasattr(_lib.load(), name), name
    assert "int gdl_eval_scores(" in hdr and "int gdl_eval_ap(" in hdr
    assert callable(ops.eval_scores) and callable(ops.eval_ap)
    # columns of up to 16384 rows sort in shared memory; longer ones in a workspace of 3 n 2^ceil(log2 cap) keys
    assert ops.eval_ap_workspace_bytes(16384, 309) == 0
    assert ops.eval_ap_workspace_bytes(16385, 6) == 3 * 6 * 32768 * 8
