"""Data-parallel replicas run one after another on one GPU (DGLStep replicas): bandwidth of gdl_grad_accumulate over
the concat (22,352,902 floats) and FiLM (156,568,070 floats) gradient arenas, L2 flushed between repetitions, GB/s
from the algorithmic bytes (8 per element for acc <- grad, 12 for acc += grad); then the KineticSound-shape concat step
at a global batch of G = 512 rows three ways, alternating rounds in the same process: one 512-row replica (BatchNorm
over all 512 rows), R = 2 replicas of 256 rows and R = 8 replicas of 64 rows (what nn.DataParallel over 8 GPUs
computes).  Writes the report to --out (default profiles/replica_bench.txt):
python tools/replica_bench.py"""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "iccv2025-gdl_b200"))
import gdl_b200  # noqa: E402
from gdl_b200 import ops  # noqa: E402
from gdl_b200.step import DGLStep  # noqa: E402
from gdl_b200.shapes import BATCH_SHAPES, HEAD_WIDTH, LABEL_MAX, make_batch  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=10, help="global steps per timed round")
ap.add_argument("--rounds", type=int, default=5)
ap.add_argument("--batch", type=int, default=512, help="global batch G")
ap.add_argument("--replicas", default="1,2,8", help="replica counts R to compare (G / R rows each)")
ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "replica_bench.txt"))
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


say("# tools/replica_bench.py: device %s, power limit %s, max SM clock %s"
    % (torch.cuda.get_device_name(), query("power.limit"), query("clocks.max.sm")))

# ---- gdl_grad_accumulate over the gradient arenas ----
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")


def timeit(fn, reps=9):
    fn(); torch.cuda.synchronize(); ts = []  # noqa: E702
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1))  # noqa: E702
    return sorted(ts)[len(ts) // 2]


say("# GB/s = algorithmic bytes / CUDA-event time, L2 flushed (256 MB written) before each call, median of 9")
for name, n in (("concat", 22352902), ("film", 156568070)):
    n += 3  # the loss tail rides along
    acc, grad = torch.randn(n, device="cuda"), torch.randn(n, device="cuda")
    for accumulate, label, nbytes in ((False, "acc <- grad", 8.0), (True, "acc += grad", 12.0)):
        t = timeit(lambda: ops.grad_accumulate(acc, grad, n, accumulate))
        say("%-6s %11d floats  grad_accumulate (%s) %.3f ms  %.0f GB/s" % (name, n, label, t, nbytes * n * 1e-6 / t))
    del acc, grad
    torch.cuda.empty_cache()
del flush

# ---- the KineticSound concat step at G rows: R replicas of G / R rows ----
G = cli.batch
Fq, Tt, T, H, W = BATCH_SHAPES["KineticSound"]
batch = [t.cuda() for t in make_batch(G, HEAD_WIDTH["KineticSound"], "KineticSound", seed=1,
                                      label_max=LABEL_MAX["KineticSound"])]
steps = {}
for R in [int(x) for x in cli.replicas.split(",")]:
    gdl_b200.setup_seed(0)
    model = gdl_b200.AVClassifier_DGL(argparse.Namespace(dataset="KineticSound", fusion_method="concat",
                                                         modality="full"))
    model.apply(gdl_b200.weight_init)
    model.cuda().train()
    st = DGLStep(model, G // R, (Fq, Tt), (T, H, W), alpha=4.0, lr=1e-3, replicas=R)
    st.load_inputs(*batch)
    for _ in range(3):  # eager, capture, replay
        st.step()
    steps[R] = st
torch.cuda.synchronize()
res = {R: [] for R in steps}
for r in range(cli.rounds):
    for R, st in steps.items():
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(cli.steps):
            st.step()
        e1.record()
        torch.cuda.synchronize()
        res[R].append(e0.elapsed_time(e1) / cli.steps)
say("# KineticSound shape, concat, SGD, CUDA graphs; ms per global step of G = %d rows, %d rounds of %d steps, "
    "alternating; samples/s from the median" % (G, cli.rounds, cli.steps))
for R, ts in res.items():
    med = sorted(ts)[len(ts) // 2]
    say("R=%d x %3d rows: %s ms (median %.3f)  %.0f samples/s  %d launches per step"
        % (R, G // R, " ".join("%.3f" % t for t in ts), med, G * 1e3 / med, steps[R].launches_per_step))
os.makedirs(os.path.dirname(os.path.abspath(cli.out)), exist_ok=True)
with open(cli.out, "w") as f:
    f.write("\n".join(lines) + "\n")
