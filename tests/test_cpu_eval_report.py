"""The per-class validation report on the host side: EvalReport's arithmetic, the per-class CSV rows of
`main_dgl.py --per_class`, the flag's default, and the C-ABI declaration of gdl_eval_confusion.  No GPU."""
import argparse
import csv
import math
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _report():
    from gdl_b200.train import EvalReport
    # 4 classes; class 2 has no sample; 11 labelled rows + 1 padded (label -1) row in the total
    conf = torch.zeros(3, 4, 4, dtype=torch.int64)
    conf[0] = torch.tensor([[3, 1, 0, 0], [0, 2, 0, 1], [0, 0, 0, 0], [1, 0, 1, 2]])
    conf[1] = torch.tensor([[4, 0, 0, 0], [3, 0, 0, 0], [0, 0, 0, 0], [0, 0, 0, 4]])
    conf[2] = torch.tensor([[0, 0, 4, 0], [0, 3, 0, 0], [0, 0, 0, 0], [1, 1, 1, 1]])
    return EvalReport(conf, 12)


def test_report_accuracies_come_from_the_traces_and_empty_classes_are_nan():
    r = _report()
    assert r.total == 12 and r.n == 4
    assert r.support.tolist() == [4, 3, 0, 4]
    assert r.correct.tolist() == [[3, 2, 0, 2], [4, 0, 0, 4], [0, 3, 0, 1]]
    assert (r.acc, r.acc_a, r.acc_v) == (7 / 12, 8 / 12, 4 / 12)
    assert r.per_class.dtype == torch.float64 and r.per_class.shape == (3, 4)
    for h in range(3):
        assert math.isnan(r.per_class[h, 2].item())  # no sample: NaN, not 0
        for c in (0, 1, 3):
            assert r.per_class[h, c].item() == r.correct[h, c].item() / r.support[c].item()
    assert r.per_class[1, 1].item() == 0.0  # a class with samples and no hit is 0


def test_report_of_an_empty_loader():
    from gdl_b200.train import EvalReport
    r = EvalReport(torch.zeros(3, 6, 6, dtype=torch.int64), 0)
    assert (r.acc, r.acc_a, r.acc_v) == (0.0, 0.0, 0.0)  # valid()'s max(total, 1)
    assert bool(r.per_class.isnan().all())


def test_report_rows_and_table():
    r = _report()
    rows = r.rows(7)
    assert len(rows) == 3 * 4
    assert rows[0] == [7, "out", 0, 4, 3, 0.75]
    assert rows[4 + 1] == [7, "out_a", 1, 3, 0, 0.0]
    assert rows[8 + 3] == [7, "out_v", 3, 4, 1, 0.25]
    assert math.isnan(rows[2][5]) and rows[2][:5] == [7, "out", 2, 0, 0]
    lines = r.table().splitlines()
    assert len(lines) == 1 + 4 and lines[0].split() == ["class", "support", "out", "out_a", "out_v"]
    assert lines[3].split() == ["2", "0", "nan", "nan", "nan"]
    assert lines[1].split() == ["0", "4", "0.7500", "1.0000", "0.0000"]


def _main_dgl():
    sys.path.insert(0, ROOT)
    import main_dgl
    return main_dgl


def test_per_class_flag_defaults_off():
    main_dgl = _main_dgl()
    assert main_dgl.get_arguments(["--ckpt_path", "x"]).per_class is False
    assert main_dgl.get_arguments(["--ckpt_path", "x", "--per_class"]).per_class is True


def _args(tmp_path, per_class):
    return argparse.Namespace(ckpt_path=str(tmp_path), dataset="CREMAD", modality="full", per_class=per_class)


def test_epoch_without_the_flag_runs_valid_and_writes_no_file(tmp_path, monkeypatch):
    main_dgl = _main_dgl()
    calls = []
    monkeypatch.setattr(main_dgl, "valid", lambda *a: calls.append("valid") or (0.5, 0.25, 0.125))
    monkeypatch.setattr(main_dgl, "valid_report", lambda *a: calls.append("report") or _report())
    got = main_dgl.evaluate_epoch(_args(tmp_path, False), None, None, None, 0, 0)
    assert got == (0.5, 0.25, 0.125) and calls == ["valid"]
    assert os.listdir(tmp_path) == []


def test_epoch_with_the_flag_appends_per_class_rows(tmp_path, monkeypatch):
    main_dgl = _main_dgl()
    calls = []
    monkeypatch.setattr(main_dgl, "valid", lambda *a: calls.append("valid") or (0.5, 0.25, 0.125))
    monkeypatch.setattr(main_dgl, "valid_report", lambda *a: calls.append("report") or _report())
    args = _args(tmp_path, True)
    r = _report()
    assert main_dgl.evaluate_epoch(args, None, None, None, 0, 0) == (r.acc, r.acc_a, r.acc_v)
    main_dgl.evaluate_epoch(args, None, None, None, 1, 0)
    main_dgl.evaluate_epoch(args, None, None, None, 2, 1)  # not rank 0: computes, writes nothing
    assert calls == ["report"] * 3
    assert os.listdir(tmp_path) == ["CREMAD_full_per_class.csv"]
    with open(tmp_path / "CREMAD_full_per_class.csv", newline="") as f:
        rows = list(csv.reader(f))
    assert rows[0] == ["epoch", "head", "class", "support", "correct", "accuracy"]
    assert len(rows) == 1 + 2 * 12
    assert rows[1] == ["0", "out", "0", "4", "3", "0.75"]
    assert rows[3] == ["0", "out", "2", "0", "0", "nan"]
    assert rows[13] == ["1", "out", "0", "4", "3", "0.75"]
    assert rows[24] == ["1", "out_v", "3", "4", "1", "0.25"]


def test_confusion_entry_point_is_declared_and_exported():
    from gdl_b200 import _lib, ops
    hdr = open(os.path.join(ROOT, "include", "gdl_b200.h")).read()
    assert "int gdl_eval_confusion(" in hdr
    assert len(_lib.SIGNATURES["gdl_eval_confusion"][1]) == 7  # logits, labels, conf, out_of_range, B, n, stream
    assert hasattr(_lib.load(), "gdl_eval_confusion")
    assert callable(ops.eval_confusion)
