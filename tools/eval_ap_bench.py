"""valid() against valid_report(ap=True) (the same pass plus gdl_eval_confusion and gdl_eval_scores per batch, then
one gdl_eval_ap) at the CREMA-D (n = 6) and VGGSound (n = 309) shapes, B = 256, concat and FiLM heads, one GPU.  An
evaluation is --batches test batches (60 x 256 = 15360 rows, about the VGGSound test set), cycled over --distinct
pinned host batches so that the host memory stays small.  Both run alternately (valid, ap, valid, ap, ...) in the same
process after a warm-up round that captures the graphs; the accuracies they return are printed side by side.  Also
times gdl_eval_ap alone over a full store with CUDA events.  Writes the report to --out (default
profiles/eval_ap_bench.txt):
python tools/eval_ap_bench.py"""
import argparse
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "iccv2025-gdl_b200"))
import gdl_b200  # noqa: E402
from gdl_b200 import ops  # noqa: E402
from gdl_b200.shapes import BATCH_SHAPES, LABEL_MAX, make_batch  # noqa: E402
from gdl_b200.step import EvalScores  # noqa: E402
from gdl_b200.train import valid, valid_report  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--batch", type=int, default=256)
ap.add_argument("--batches", type=int, default=60, help="test batches per evaluation")
ap.add_argument("--distinct", type=int, default=4, help="distinct pinned host batches the evaluation cycles over")
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--shapes", default="CREMAD,VGGSound")
ap.add_argument("--fusions", default="concat,film")
ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "eval_ap_bench.txt"))
cli = ap.parse_args()
ops.init()
lines = []


def say(s):
    print(s, flush=True)
    lines.append(s)


def query(field):
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=" + field, "--format=csv,noheader", "-i",
                               str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    except OSError:
        return "unknown"


def ap_ms(rows, n, reps=20):
    """Mean time of one gdl_eval_ap over a store of `rows` softmax rows with n classes (CUDA events)."""
    sc = EvalScores(n, rows, torch.device("cuda"))
    sc.store.copy_(torch.softmax(torch.randn(3, rows, n, device="cuda"), -1).permute(0, 2, 1))
    sc.labels.copy_(torch.randint(0, n, (rows,), device="cuda", dtype=torch.int32))
    sc.cursor.fill_(rows)
    for _ in range(3):
        sc.average_precision()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        sc.average_precision()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


say("# tools/eval_ap_bench.py: device %s, power limit %s, max SM clock %s; B = %d, %d test batches per evaluation "
    "(%d rows) cycled over %d pinned host batches, valid() / valid_report(ap=True) alternating for %d rounds after "
    "one warm-up round (median reported)" % (torch.cuda.get_device_name(), query("power.limit"),
                                             query("clocks.max.sm"), cli.batch, cli.batches, cli.batch * cli.batches,
                                             cli.distinct, cli.rounds))
dev = torch.device("cuda")
for shape in cli.shapes.split(","):
    for fusion in cli.fusions.split(","):
        args = argparse.Namespace(dataset=shape, fusion_method=fusion, modality="full", alpha=4.0, drop=0)
        gdl_b200.setup_seed(0)
        model = gdl_b200.AVClassifier_DGL(args)
        model.apply(gdl_b200.weight_init)
        model.to(dev).eval()
        distinct = []
        for i in range(cli.distinct):
            s, im, lb = make_batch(cli.batch, model.n_classes, shape, seed=10 + i, label_max=LABEL_MAX[shape])
            distinct.append((s.pin_memory(), im.pin_memory(), lb.pin_memory()))
        batches = [distinct[i % cli.distinct] for i in range(cli.batches)]
        times = {"valid": [], "ap": []}
        accs, rep = {}, None
        for r in range(cli.rounds + 1):
            for name in ("valid", "ap"):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                res = valid(args, model, dev, batches) if name == "valid" else \
                    valid_report(args, model, dev, batches, ap=True)
                torch.cuda.synchronize()
                if name == "ap":
                    rep, res = res, (res.acc, res.acc_a, res.acc_v)
                accs[name] = res
                if r:
                    times[name].append(time.perf_counter() - t0)
        med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
        per = {k: 1e3 * v / cli.batches for k, v in med.items()}
        say("%-9s %-6s n = %3d (F, Tt, T, H, W) = %s: valid %.2f ms/batch (%.1f ms)  valid_report(ap=True) %.2f "
            "ms/batch (%.1f ms)  difference %+.3f ms/batch (%+.2f %%); gdl_eval_ap alone over %d rows %.3f ms; "
            "mAP %.4f top-5 %.4f; accuracies valid %s ap %s (%s)"
            % (shape, fusion, model.n_classes, BATCH_SHAPES[shape], per["valid"], 1e3 * med["valid"], per["ap"],
               1e3 * med["ap"], per["ap"] - per["valid"], 100.0 * (med["ap"] / med["valid"] - 1.0),
               cli.batch * cli.batches, ap_ms(cli.batch * cli.batches, model.n_classes), rep.map, rep.top5,
               [round(a, 4) for a in accs["valid"]], [round(a, 4) for a in accs["ap"]],
               "equal" if accs["valid"] == accs["ap"] else "DIFFER"))
        del model, batches, distinct
        torch.cuda.empty_cache()
os.makedirs(os.path.dirname(os.path.abspath(cli.out)), exist_ok=True)
with open(cli.out, "w") as f:
    f.write("\n".join(lines) + "\n")
