"""The graph-captured step at a fixed lr against the same step at an lr that changes every iteration (the update reads
it from device memory, so neither re-captures), alternating rounds of CUDA-graph replays in one process, for the
B = 256 CREMA-D concat step and the B = 64 KineticSound concat step; then the host time of one full re-capture of the
step at each shape (graphs cleared, one step, synchronised), which is what every lr change cost while the lr was a
kernel argument baked into the graphs.  Writes the report to --out (default profiles/lr_schedule_bench.txt):
python tools/lr_schedule_bench.py"""
import argparse
import math
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
from gdl_b200.step import DGLStep  # noqa: E402
from gdl_b200.shapes import BATCH_SHAPES, HEAD_WIDTH, LABEL_MAX, make_batch  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=20, help="graph replays per timed round")
ap.add_argument("--rounds", type=int, default=7)
ap.add_argument("--recaptures", type=int, default=5, help="re-captures timed per shape (median reported)")
ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "lr_schedule_bench.txt"))
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


def med(ts):
    return sorted(ts)[len(ts) // 2]


say("# tools/lr_schedule_bench.py: device %s, power limit %s, max SM clock %s"
    % (torch.cuda.get_device_name(), query("power.limit"), query("clocks.max.sm")))
say("# concat head, SGD (momentum 0.9, weight decay 1e-4), CUDA graphs; step times from CUDA events over %d replays "
    "per round, %d rounds, fixed and per-iteration lr alternating" % (cli.steps, cli.rounds))
# a warm-up + cosine sequence: a different lr at every step
varying = [1e-3 * 0.5 * (1 + math.cos(math.pi * k / 97)) + 1e-5 for k in range(97)]
for dataset, B in (("CREMAD", 256), ("KineticSound", 64)):
    Fq, Tt, T, H, W = BATCH_SHAPES[dataset]
    batch = [t.cuda() for t in make_batch(B, HEAD_WIDTH[dataset], dataset, seed=1, label_max=LABEL_MAX[dataset])]
    gdl_b200.setup_seed(0)
    model = gdl_b200.AVClassifier_DGL(argparse.Namespace(dataset=dataset, fusion_method="concat", modality="full"))
    model.apply(gdl_b200.weight_init)
    model.cuda().train()
    st = DGLStep(model, B, (Fq, Tt), (T, H, W), alpha=4.0, lr=1e-3)
    st.load_inputs(*batch)
    for _ in range(3):
        st.step(lr=1e-3)
    torch.cuda.synchronize()
    graphs = {k: id(g) for k, g in st.graphs.items()}
    res = {"fixed": [], "per-iteration": []}
    k = 0
    for r in range(cli.rounds):
        for mode in res:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(cli.steps):
                st.step(lr=1e-3 if mode == "fixed" else varying[k % len(varying)])
                k += 1
            e1.record()
            torch.cuda.synchronize()
            res[mode].append(e0.elapsed_time(e1) / cli.steps)
    assert {k: id(g) for k, g in st.graphs.items()} == graphs, "a graph was re-captured"
    for mode, ts in res.items():
        say("%-12s B=%3d lr %-13s: %s ms per step (median %.3f)" % (dataset, B, mode, " ".join("%.3f" % t for t in ts),
                                                                   med(ts)))
    # host time of one synchronised step: a replay, and a re-capture (graphs cleared) followed by its replay
    plain, recap = [], []
    for _ in range(cli.recaptures):
        for target, clear in ((plain, False), (recap, True)):
            if clear:
                st.graphs.clear()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            st.step(lr=1e-3)
            torch.cuda.synchronize()
            target.append((time.perf_counter() - t0) * 1e3)
    say("%-12s B=%3d host time of one step, synchronised: replay %s ms (median %.2f); re-capture + replay %s ms "
        "(median %.2f); re-capture cost %.2f ms per lr change (%d launches captured)"
        % (dataset, B, " ".join("%.2f" % t for t in plain), med(plain), " ".join("%.2f" % t for t in recap), med(recap),
           med(recap) - med(plain), st.launches_per_step))
    del model, st, batch
    torch.cuda.empty_cache()
os.makedirs(os.path.dirname(os.path.abspath(cli.out)), exist_ok=True)
with open(cli.out, "w") as f:
    f.write("\n".join(lines) + "\n")
