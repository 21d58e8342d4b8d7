"""valid() before and after the graph-captured EvalStep, at the CREMA-D and KineticSound shapes, B = 256, concat head,
one GPU.  The old path is the per-batch loop valid() ran before: a blocking `.to(device)` of every batch, the encoders'
training-shadow repack, the eval forward with the BatchNorm fold recomputed per call, torch pooling / bias adds /
arg-max.  The new path is gdl_b200.train.valid.  Both read the same pinned host batches; the two are run alternately
(old, new, old, new, ...) in the same process, and the accuracies they return are printed side by side.  Writes the
report to --out (default profiles/eval_bench.txt):
python tools/eval_bench.py"""
import argparse
import os
import subprocess
import sys
import time

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "iccv2025-gdl_b200"))
import gdl_b200  # noqa: E402
from gdl_b200 import ops  # noqa: E402
from gdl_b200.autograd import to_nhwc8  # noqa: E402
from gdl_b200.shapes import BATCH_SHAPES, LABEL_MAX, make_batch  # noqa: E402
from gdl_b200.train import valid  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--batch", type=int, default=256)
ap.add_argument("--batches", type=int, default=6, help="test batches per evaluation")
ap.add_argument("--rounds", type=int, default=4)
ap.add_argument("--shapes", default="CREMAD,KineticSound")
ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "eval_bench.txt"))
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


def old_valid(model, device, loader):
    """The per-batch loop of valid() before EvalStep (model(...) as it then ran, inlined)."""
    correct = torch.zeros(3, device=device, dtype=torch.float64)
    total = 0
    with torch.no_grad():
        for spec, image, label in loader:
            spec, image, label = spec.to(device), image.to(device), label.to(device)
            feats = []
            for net, x in ((model.audio_net, spec.unsqueeze(1).float()), (model.visual_net, image.float())):
                x8, (N, H, W) = to_nhwc8(net, x)
                eng = net.engine(N, H, W)
                eng.repack()
                eng._eval_key_folded = None  # the per-call version bump always re-folded
                feats.append(eng.forward(x8, training=False).permute(0, 3, 1, 2).float())
            a, v = feats
            B = a.shape[0]
            v = v.view(B, -1, v.shape[1], v.shape[2], v.shape[3]).permute(0, 2, 1, 3, 4)
            a = torch.flatten(F.adaptive_avg_pool2d(a, 1), 1)
            v = torch.flatten(F.adaptive_avg_pool3d(v, 1), 1)
            a_out, v_out, out = model.fusion_module(a, v)
            for i, o in enumerate((out, a_out, v_out)):
                correct[i] += (o.argmax(1) == label).sum()
            total += label.shape[0]
    acc = (correct / max(total, 1)).tolist()
    return acc[0], acc[1], acc[2]


say("# tools/eval_bench.py: device %s, power limit %s, max SM clock %s; concat head, B = %d, %d test batches per "
    "evaluation, pinned host batches, old / new alternating for %d rounds (median reported)"
    % (torch.cuda.get_device_name(), query("power.limit"), query("clocks.max.sm"), cli.batch, cli.batches, cli.rounds))
dev = torch.device("cuda")
for shape in cli.shapes.split(","):
    args = argparse.Namespace(dataset=shape, fusion_method="concat", modality="full", alpha=4.0, drop=0)
    gdl_b200.setup_seed(0)
    model = gdl_b200.AVClassifier_DGL(args)
    model.apply(gdl_b200.weight_init)
    model.to(dev).eval()
    batches = []
    for i in range(cli.batches):
        s, im, lb = make_batch(cli.batch, model.n_classes, shape, seed=10 + i, label_max=LABEL_MAX[shape])
        batches.append((s.pin_memory(), im.pin_memory(), lb.pin_memory()))
    times = {"old": [], "new": []}
    accs = {}
    for r in range(cli.rounds + 1):  # round 0 warms up both paths (engines, folds, graph capture)
        for name, fn in (("old", lambda: old_valid(model, dev, batches)), ("new", lambda: valid(args, model, dev, batches))):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            accs[name] = fn()
            torch.cuda.synchronize()
            if r:
                times[name].append(time.perf_counter() - t0)
    n = cli.batch * cli.batches
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    say("%-12s (F, Tt, T, H, W) = %s: old %.1f ms (%.0f samples/s)  new %.1f ms (%.0f samples/s)  speed-up %.2fx; "
        "rounds old %s new %s ms; accuracies old %s new %s"
        % (shape, BATCH_SHAPES[shape], 1e3 * med["old"], n / med["old"], 1e3 * med["new"], n / med["new"],
           med["old"] / med["new"], [round(1e3 * t, 1) for t in times["old"]], [round(1e3 * t, 1) for t in times["new"]],
           [round(a, 4) for a in accs["old"]], [round(a, 4) for a in accs["new"]]))
    del model, batches
    torch.cuda.empty_cache()
os.makedirs(os.path.dirname(os.path.abspath(cli.out)), exist_ok=True)
with open(cli.out, "w") as f:
    f.write("\n".join(lines) + "\n")
