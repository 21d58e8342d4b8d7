"""valid() against valid_report() (the same pass plus gdl_eval_confusion per batch) at the CREMA-D and KineticSound
shapes, B = 256, concat and FiLM heads, one GPU.  Both read the same pinned host batches and run alternately
(valid, report, valid, report, ...) in the same process after a warm-up round that captures both graphs; the
accuracies they return are printed side by side.  Also times gdl_eval_confusion alone with CUDA events.  Writes the
report to --out (default profiles/eval_report_bench.txt):
python tools/eval_report_bench.py"""
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
from gdl_b200.train import valid, valid_report  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--batch", type=int, default=256)
ap.add_argument("--batches", type=int, default=6, help="test batches per evaluation")
ap.add_argument("--rounds", type=int, default=5)
ap.add_argument("--shapes", default="CREMAD,KineticSound")
ap.add_argument("--fusions", default="concat,film")
ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "eval_report_bench.txt"))
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


def kernel_us(B, n, reps=200):
    """Mean time of one gdl_eval_confusion over logits [3, B, n] (CUDA events around `reps` launches)."""
    logits = torch.randn(3, B, n, device="cuda")
    labels = torch.randint(0, n, (B,), device="cuda")
    buf = torch.zeros(1 + 3 * n * n, dtype=torch.int64, device="cuda")
    for _ in range(10):
        ops.eval_confusion(logits, labels, buf[1:], buf[:1], B, n)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        ops.eval_confusion(logits, labels, buf[1:], buf[:1], B, n)
    e1.record()
    torch.cuda.synchronize()
    return 1e3 * e0.elapsed_time(e1) / reps


say("# tools/eval_report_bench.py: device %s, power limit %s, max SM clock %s; B = %d, %d test batches per "
    "evaluation, pinned host batches, valid() / valid_report() alternating for %d rounds after one warm-up round "
    "(median reported)" % (torch.cuda.get_device_name(), query("power.limit"), query("clocks.max.sm"), cli.batch,
                           cli.batches, cli.rounds))
dev = torch.device("cuda")
for shape in cli.shapes.split(","):
    for fusion in cli.fusions.split(","):
        args = argparse.Namespace(dataset=shape, fusion_method=fusion, modality="full", alpha=4.0, drop=0)
        gdl_b200.setup_seed(0)
        model = gdl_b200.AVClassifier_DGL(args)
        model.apply(gdl_b200.weight_init)
        model.to(dev).eval()
        batches = []
        for i in range(cli.batches):
            s, im, lb = make_batch(cli.batch, model.n_classes, shape, seed=10 + i, label_max=LABEL_MAX[shape])
            batches.append((s.pin_memory(), im.pin_memory(), lb.pin_memory()))
        times = {"valid": [], "report": []}
        accs = {}
        for r in range(cli.rounds + 1):
            for name, fn in (("valid", lambda: valid(args, model, dev, batches)),
                             ("report", lambda: valid_report(args, model, dev, batches))):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                res = fn()
                torch.cuda.synchronize()
                accs[name] = res if name == "valid" else (res.acc, res.acc_a, res.acc_v)
                if r:
                    times[name].append(time.perf_counter() - t0)
        med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
        per = {k: 1e3 * v / cli.batches for k, v in med.items()}
        say("%-12s %-6s n = %3d (F, Tt, T, H, W) = %s: valid %.2f ms/batch  valid_report %.2f ms/batch  "
            "difference %+.3f ms/batch (%+.2f %%); gdl_eval_confusion alone %.2f us; rounds valid %s report %s ms; "
            "accuracies valid %s report %s (%s)"
            % (shape, fusion, model.n_classes, BATCH_SHAPES[shape], per["valid"], per["report"],
               per["report"] - per["valid"], 100.0 * (med["report"] / med["valid"] - 1.0),
               kernel_us(cli.batch, model.n_classes), [round(1e3 * t, 1) for t in times["valid"]],
               [round(1e3 * t, 1) for t in times["report"]], [round(a, 4) for a in accs["valid"]],
               [round(a, 4) for a in accs["report"]], "equal" if accs["valid"] == accs["report"] else "DIFFER"))
        del model, batches
        torch.cuda.empty_cache()
os.makedirs(os.path.dirname(os.path.abspath(cli.out)), exist_ok=True)
with open(cli.out, "w") as f:
    f.write("\n".join(lines) + "\n")
