"""Data-parallel replicas run one after another on one GPU (DGLStep replicas, `main_dgl.py --dp_replicas`): the
accumulation kernel, the FP32 check mode against the oracle's R-shard simulation of nn.DataParallel (reference
main_dgl.py:244: torch.chunk order, per-replica BatchNorm, only replica 0's running statistics persist, CE over the
gathered logits == shard sums scaled by 1/G, gradient reduce-add), the bf16 product path (graphs, datapipe), two
GPUs, and the CLI.  GPU only."""
import argparse
import math
import os
import re
import subprocess
import sys

import pytest
import torch

from test_gpu_step import cos

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------------------ kernel
@pytest.mark.parametrize("numel", [1, 3, 4, 1027, 100003, 4 * 1024 * 1024 + 5])
def test_grad_accumulate_is_a_bit_exact_fp32_add(numel):
    from gdl_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(numel)
    src = torch.randn(numel, device="cuda", generator=g)
    dst0 = torch.randn(numel, device="cuda", generator=g) * 7
    dst = dst0.clone()
    ops.grad_accumulate(dst, src, numel, True)
    torch.cuda.synchronize()
    assert torch.equal(dst, dst0 + src)
    ops.grad_accumulate(dst, src, numel, False)
    torch.cuda.synchronize()
    assert torch.equal(dst, src)


def test_grad_accumulate_rejects_bad_arguments():
    import ctypes as C
    from gdl_b200 import ops
    from gdl_b200._lib import GDL_OK, load
    lib = load()
    a, b = torch.zeros(64, device="cuda"), torch.zeros(64, device="cuda")
    s = ops._stream()
    assert lib.gdl_grad_accumulate(None, C.c_void_p(b.data_ptr()), 16, 1, s) != GDL_OK
    assert lib.gdl_grad_accumulate(C.c_void_p(a.data_ptr()), None, 16, 0, s) != GDL_OK
    assert lib.gdl_grad_accumulate(C.c_void_p(a.data_ptr() + 4), C.c_void_p(b.data_ptr()), 16, 1, s) != GDL_OK
    assert lib.gdl_grad_accumulate(C.c_void_p(a.data_ptr()), C.c_void_p(b.data_ptr() + 8), 16, 1, s) != GDL_OK
    assert lib.gdl_grad_accumulate(C.c_void_p(a.data_ptr()), C.c_void_p(b.data_ptr()), 0, 1, s) != GDL_OK


# ------------------------------------------------------------------------------------------------ helpers
def _model(fusion="concat"):
    import gdl_b200
    args = argparse.Namespace(dataset="CREMAD", fusion_method=fusion, modality="full")
    gdl_b200.setup_seed(0)
    model = gdl_b200.AVClassifier_DGL(args)
    model.apply(gdl_b200.weight_init)
    return model.cuda().train()


def _simulate(O, sd, batch, fusion, R):
    """The oracle's R-shard simulation of one step of nn.DataParallel over R devices: per-shard losses and
    (unclipped) gradients summed, and the running statistics of shard 0's BatchNorm."""
    G = batch[0].shape[0]
    b = G // R
    losses, total = [0.0, 0.0, 0.0], None
    for k in range(R):
        res = O.dgl_step(sd, {}, *[t[k * b:(k + 1) * b] for t in batch], fusion=fusion, alpha=4.0, max_norm=1e9,
                         inv_batch=1.0 / G, apply_update=False)
        losses = [x + y for x, y in zip(losses, res["losses"])]
        total = res["grads"] if total is None else {n: res["grads"][n] + total[n] for n in total}
    nb = {}
    with torch.no_grad():
        O.model_forward(sd, batch[0][:b], batch[1][:b], fusion, True, None, True, nb)
    return losses, total, nb


def _sgd(sd, mom, grads, nb, lr, mu=0.9, wd=1e-4, max_norm=40.0):
    """clip_grad_norm_ + torch.optim.SGD on the summed gradients (the oracle's own update block), then the
    running statistics of replica 0; returns the unclipped norm."""
    norm = sum(float(g.double().pow(2).sum()) for g in grads.values()) ** 0.5
    coef = min(1.0, max_norm / (norm + 1e-6))
    with torch.no_grad():
        for k, g in grads.items():
            d = g * coef + wd * sd[k]
            if k not in mom:
                mom[k] = d.clone()
            else:
                mom[k].mul_(mu).add_(d)
            sd[k].add_(mom[k], alpha=-lr)
    for k, v in nb.items():
        sd[k] = v if torch.is_tensor(v) else torch.tensor(v)
    return norm


# ------------------------------------------------------------------------------------------------ check mode
def _run_check(fusion, R, b=4, nsteps=3, lr=0.01):
    """3 SGD steps in check mode, each compared with the oracle's R-shard simulation started from the device's own
    weights, running statistics and momentum (free-running, BatchNorm over b = 4 rows of the tiny shape amplifies
    the two implementations' fp32 rounding within two steps: measured min per-tensor cosine 0.70 at step 2)."""
    from gdl_b200.step import DGLStep
    from oracle import dgl_oracle as O
    from oracle.synth import SHAPES, make_batch
    torch.set_num_threads(os.cpu_count())
    model = _model(fusion)
    Fq, Tt, T, H, W = SHAPES["tiny"]
    step = DGLStep(model, b, (Fq, Tt), (T, H, W), alpha=4.0, lr=lr, check_fp32=True, replicas=R)
    names, bufs = dict(model.named_parameters()), dict(model.named_buffers())
    ar = step.arena
    for s in range(nsteps):
        sd = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}
        mom = {} if s == 0 else {k: ar.momentum[ar.offset_of[id(p)]:ar.offset_of[id(p)] + p.numel()].view(p.shape)
                                 .cpu().clone() for k, p in names.items() if id(p) in ar.offset_of}
        before = {k: v.clone() for k, v in sd.items()}
        batch = make_batch(R * b, 6, "tiny", seed=1 + s)
        step.step(*[t.cuda() for t in batch])
        got = step.read_stats()
        losses, total, nb = _simulate(O, sd, batch, fusion, R)
        norm = _sgd(sd, mom, total, nb, lr)
        rows = sorted((cos(names[k].grad.detach().float().cpu(), g), k) for k, g in total.items())
        upd = sorted((cos(names[k].detach().cpu() - before[k], sd[k] - before[k]), k) for k in total)
        dmax = max((names[k].detach().cpu() - sd[k]).abs().max().item() / (sd[k].abs().max().item() + lr)
                   for k in total)
        untouched = all(torch.equal(names[k].detach().cpu(), before[k]) for k in names if k not in total)
        print("replicas check-mode %s R=%d b=%d step %d: losses %s vs %s; norm %.6g vs %.6g; min grad cos %.7f (%s); "
              "min update cos %.7f (%s); params rel %.2e" % (fusion, R, b, s, got[:3], losses, got[3], norm, rows[0][0],
                                                             rows[0][1], upd[0][0], upd[0][1], dmax))
        for g, r in zip(got[:3], losses):
            assert abs(g - r) <= 1e-4 * abs(r), (s, got[:3], losses)
        assert abs(got[3] - norm) <= 1e-3 * norm, (s, got[3], norm)
        assert rows[0][0] >= 0.999, (s, rows[:3])
        assert upd[0][0] >= 0.999 and dmax < 5e-3 and untouched, (s, upd[:3], dmax)
        for k, v in nb.items():  # replica 0's statistics only: replicas 1 .. R-1 left the buffers untouched
            if k.endswith("num_batches_tracked"):
                assert int(bufs[k]) == s + 1, k
            else:
                assert torch.allclose(bufs[k].detach().cpu(), v, rtol=1e-4, atol=1e-5), \
                    (s, k, (bufs[k].detach().cpu() - v).abs().max().item())
    del model, step
    torch.cuda.empty_cache()


@pytest.mark.parametrize("R", [2, 4])
@pytest.mark.parametrize("fusion", ["concat", "gated"])
def test_check_mode_matches_the_r_shard_simulation(fusion, R):
    _run_check(fusion, R)


def test_adam_counts_global_steps_with_replicas():
    """The update runs once per global step: the device step count advances by one per step, not per replica."""
    from gdl_b200.optim import UpdateRule
    from gdl_b200.step import DGLStep
    from oracle.synth import SHAPES, make_batch
    model = _model()
    Fq, Tt, T, H, W = SHAPES["tiny"]
    step = DGLStep(model, 2, (Fq, Tt), (T, H, W), rule=UpdateRule("adam", 1e-3, eps=1e-8), check_fp32=True,
                   replicas=3)
    for s in range(3):
        step.step(*[t.cuda() for t in make_batch(6, 6, "tiny", seed=1 + s)])
    torch.cuda.synchronize()
    assert all(math.isfinite(x) for x in step.read_stats())
    assert step.arena.steps == 3 and int(step.arena.step_state[0]) == 3


# ------------------------------------------------------------------------------------------------ product path
def _product(R, b, use_graph, shape="CREMAD", fusion="concat"):
    from gdl_b200.step import DGLStep
    from oracle.synth import SHAPES
    model = _model(fusion)
    Fq, Tt, T, H, W = SHAPES[shape]
    return model, DGLStep(model, b, (Fq, Tt), (T, H, W), alpha=4.0, lr=0.01, use_graph=use_graph, replicas=R)


def test_bf16_step_matches_the_simulation_and_graph_replay_is_bit_identical():
    """CREMA-D shape, G = 16 as R = 2 replicas of 8 rows: step 0 against the 2-shard oracle simulation (bf16
    tolerances of tests/dist_step_check.py), then 3 steps through the captured graphs bit-identical to 3 eager steps."""
    from oracle import dgl_oracle as O
    from oracle.synth import make_batch
    torch.set_num_threads(os.cpu_count())
    batches = [make_batch(16, 6, "CREMAD", seed=1 + s) for s in range(3)]
    out = []
    for use_graph in (False, True):
        model, step = _product(2, 8, use_graph)
        names = dict(model.named_parameters())
        for s, batch in enumerate(batches):
            step.step(*[t.cuda() for t in batch])
            torch.cuda.synchronize()
            if s == 0 and not use_graph:
                got = step.read_stats()
                sd = O.init_state("concat", "CREMAD", 0)
                losses, total, _ = _simulate(O, sd, batch, "concat", 2)
                norm = sum(float(v.double().pow(2).sum()) for v in total.values()) ** 0.5
                worst = min(cos(names[k].grad.detach().float().cpu(), total[k])
                            for k in ("fusion_module.fc_out.weight", "fusion_module.fc_out.bias"))
                print("bf16 R=2 step 0: losses %s vs %s, head cos %.5f, norm %.5g vs %.5g" % (got[:3], losses, worst,
                                                                                           got[3], norm))
                for g, r in zip(got[:3], losses):
                    assert abs(g - r) <= 2e-2 * abs(r), (got[:3], losses)
                assert worst >= 0.99, worst
                assert abs(got[3] - norm) <= 6e-2 * norm, (got[3], norm)
        out.append((step.read_stats(), step.arena.param.clone(),
                    {k: v.clone() for k, v in model.named_buffers()}, step.launches_per_step))
        del model, step
    assert out[0][0] == out[1][0]
    assert torch.equal(out[0][1], out[1][1]), "CUDA-graph replay differs from eager execution"
    assert all(torch.equal(v, out[1][2][k]) for k, v in out[0][2].items())


def test_later_replicas_leave_the_running_statistics_bit_identical():
    """After one R = 2 step the running statistics are bit-identical to those of a one-replica step on replica 0's
    rows alone (same weights, same kernels): replica 1 did not touch them.  num_batches_tracked advanced once."""
    from oracle.synth import make_batch
    batch = make_batch(8, 6, "tiny", seed=3)
    bufs = []
    for R in (2, 1):
        model, step = _product(R, 4, False, shape="tiny")
        step.step(*[t[:4 * R].cuda() for t in batch])
        torch.cuda.synchronize()
        bufs.append({k: v.clone() for k, v in model.named_buffers()})
        del model, step
    for k, v in bufs[0].items():
        assert torch.equal(v, bufs[1][k]), k
        if k.endswith("num_batches_tracked"):
            assert int(v) == 1


def test_launches_per_step_count_every_replica_and_one_update():
    """Each further replica adds its input layout, its compute and one accumulation pass; the clip, the update and
    the weight-shadow refresh (7 launches with SGD) run once per global step."""
    from oracle.synth import make_batch
    counts = {}
    for R in (1, 2, 4):
        model, step = _product(R, 2, True, shape="tiny")
        for s in range(2):
            step.step(*[t.cuda() for t in make_batch(2 * R, 6, "tiny", seed=1 + s)])
        torch.cuda.synchronize()
        counts[R] = step.launches_per_step
        del model, step
    print("launches per step by replicas:", counts)
    for R in (2, 4):
        assert counts[R] == R * (counts[1] - 7) + 7 + R, counts


def test_device_datapipe_prefetch_with_replicas():
    """DGLStep.prefetch(..., pipeline=) with R = 2 (the crop-box table covers both replicas' frames) == prefetch of
    the host-transformed frames: same losses, same weights."""
    import numpy as np
    from gdl_b200.datapipe import DeviceFrameStore, VisualPipeline
    from oracle.crop_oracle import crop_resize_flip_normalize
    from oracle.synth import SHAPES, make_batch
    Fq, Tt, T, H, W = SHAPES["tiny"]
    G = 4
    rs = np.random.RandomState(5)
    store = rs.randint(0, 256, size=(G * T, 90, 120, 3), dtype=np.uint8)
    rows = []
    for f in range(G * T):
        h, w = int(rs.randint(20, 91)), int(rs.randint(20, 121))
        rows.append([f, int(rs.randint(0, 90 - h + 1)), int(rs.randint(0, 120 - w + 1)), h, w, int(rs.randint(2))])
    host = torch.zeros(G, 3, T, H, W)
    for f, (src, i, j, h, w, flip) in enumerate(rows):
        host[f // T, :, f % T] = torch.from_numpy(crop_resize_flip_normalize(store[src], i, j, h, w, flip, size=H))
    spec, _, label = make_batch(G, 6, "tiny", seed=2)
    results = []
    for use_pipe in (False, True):
        model, step = _product(2, G // 2, False, shape="tiny")
        if use_pipe:
            pipe = VisualPipeline(DeviceFrameStore(torch.from_numpy(store)), T, size=H)
            step.prefetch(spec.pin_memory(), torch.tensor(rows, dtype=torch.int32).pin_memory(), label.pin_memory(),
                          pipeline=pipe)
        else:
            step.prefetch(spec.pin_memory(), host.pin_memory(), label.pin_memory())
        step.step()
        torch.cuda.synchronize()
        results.append((step.read_stats(), step.arena.param.clone()))
        del model, step
    assert results[0][0] == results[1][0]
    assert torch.equal(results[0][1], results[1][1])


# ------------------------------------------------------------------------------------------------ two GPUs
def test_two_gpus_with_replicas():
    """torchrun, 2 ranks: W = 2, R = 4 against the 4-shard oracle simulation; W = 2, R = 2 bit-identical to one GPU
    running R = 2 (tests/dist_replica_check.py)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = os.path.join(os.path.dirname(__file__), "dist_replica_check.py")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29534", script],
                       capture_output=True, text=True, timeout=600)
    assert "DIST_REPLICA_CHECK_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


# ------------------------------------------------------------------------------------------------ CLI
def test_main_dgl_trains_and_resumes_with_replicas(tmp_path, capsys):
    sys.path.insert(0, ROOT)
    import main_dgl
    ck = tmp_path / "ckpt"
    common = ["--train", "--ckpt_path", str(ck), "--dp_replicas", "2", "--batch_size", "8", "--synthetic_len", "256",
              "--audio_path", "synthetic"]
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        main_dgl.main(common + ["--epochs", "2"])
        out = capsys.readouterr().out
        saved = sorted(p for p in os.listdir(ck) if p.endswith(".pth"))
        assert os.path.isfile(ck / "CREMAD_full.csv") and os.path.isfile(tmp_path / "audio_visual_grad_vanilla.csv")
        assert saved, out[-2000:]
        main_dgl.main(common + ["--epochs", "3", "--resume", str(ck / saved[-1])])
        out += capsys.readouterr().out
    finally:
        os.chdir(cwd)
    assert "Resumed from" in out and "Epoch: 2:" in out, out[-2000:]
    losses = [float(x) for x in re.findall(r"^Loss: ([-+0-9.naif]+)", out, re.M)]
    assert len(losses) == 3 and all(math.isfinite(x) for x in losses), out[-2000:]
