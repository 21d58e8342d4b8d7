"""Update-kernel bandwidth (SGD-momentum, Adam, Adagrad) over the parameter arenas of the concat (22,352,902 floats)
and FiLM (156,568,070 floats) heads, L2 flushed between repetitions, GB/s from the algorithmic bytes (24 / 32 / 24
per element); then the B = 256 CREMA-D concat step with Adam against SGD, alternating, in the same process:
python tools/optim_bench.py"""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "iccv2025-gdl_b200"))
from gdl_b200 import ops  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=20, help="graph replays per timed round of the whole step")
ap.add_argument("--rounds", type=int, default=5)
cli = ap.parse_args()
ops.init()
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")


def timeit(fn, reps=9):
    fn(); torch.cuda.synchronize(); ts = []  # noqa: E702
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1))  # noqa: E702
    return sorted(ts)[len(ts) // 2]


def power_limit():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                               str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    except OSError:
        return "unknown"


print("device: %s, power limit %s" % (torch.cuda.get_device_name(), power_limit()))
GB = 1e-6  # bytes per ms -> GB/s
for name, n in (("concat", 22352902), ("film", 156568070)):
    p, g = torch.randn(n, device="cuda"), torch.randn(n, device="cuda")
    a, b = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    st = torch.zeros(3, device="cuda", dtype=torch.int32)
    stats = torch.tensor([1.0, 1.0, 0.0, 0.0], device="cuda")
    t = timeit(lambda: ops.sgd_momentum(p, g, a, n, 1e-3, 0.9, 1e-4, False, stats))
    print("%-6s %11d floats  sgd_momentum %.3f ms  %.0f GB/s" % (name, n, t, 24.0 * n * GB / t))
    t = timeit(lambda: g.copy_(p))  # the copy bandwidth the update kernels are measured against
    print("%-6s %11d floats  copy         %.3f ms  %.0f GB/s" % (name, n, t, 8.0 * n * GB / t))
    t = timeit(lambda: ops.adam(p, g, a, b, st, n, 1e-3, 0.9, 0.999, 1e-8, 0.0, stats))
    print("%-6s %11d floats  adam         %.3f ms  %.0f GB/s" % (name, n, t, 32.0 * n * GB / t))
    t = timeit(lambda: ops.adagrad(p, g, b, st, n, 1e-3, 0.0, 1e-10, 0.0, stats))
    print("%-6s %11d floats  adagrad      %.3f ms  %.0f GB/s" % (name, n, t, 24.0 * n * GB / t))
    del p, g, a, b
    torch.cuda.empty_cache()

# ---- the whole step: B = 256 CREMA-D concat, SGD vs Adam, CUDA-graph replay, alternating ----
import gdl_b200  # noqa: E402
from gdl_b200.optim import UpdateRule  # noqa: E402
from gdl_b200.step import DGLStep  # noqa: E402
from oracle.synth import SHAPES, make_batch  # noqa: E402

B = 256
Fq, Tt, T, H, W = SHAPES["CREMAD"]
batch = [t.cuda() for t in make_batch(B, 6, "CREMAD", seed=1)]
steps = {}
for kind in ("sgd", "adam"):
    gdl_b200.setup_seed(0)
    model = gdl_b200.AVClassifier_DGL(argparse.Namespace(dataset="CREMAD", fusion_method="concat", modality="full"))
    model.apply(gdl_b200.weight_init)
    model.cuda().train()
    rule = UpdateRule("sgd", 1e-3, 1e-4, momentum=0.9) if kind == "sgd" else UpdateRule("adam", 1e-3)
    st = DGLStep(model, B, (Fq, Tt), (T, H, W), alpha=4.0, rule=rule)
    st.load_inputs(*batch)
    for _ in range(3):
        st.step()
    steps[kind] = st
torch.cuda.synchronize()
res = {k: [] for k in steps}
for r in range(cli.rounds):
    for kind, st in steps.items():
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(cli.steps):
            st.step()
        e1.record()
        torch.cuda.synchronize()
        res[kind].append(e0.elapsed_time(e1) / cli.steps)
for kind, ts in res.items():
    print("B=256 concat step, %-4s: %s ms per step (median %.3f; %d rounds of %d graph replays, alternating)"
          % (kind, " ".join("%.3f" % t for t in ts), sorted(ts)[len(ts) // 2], cli.rounds, cli.steps))
print("launches per step: sgd %d, adam %d" % (steps["sgd"].launches_per_step, steps["adam"].launches_per_step))
