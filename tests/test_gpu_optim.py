"""Adam and Adagrad on the fused step (reference main_dgl.py:251-256 `--optimizer Adam` / `AdaGrad`): the kernels
against torch.optim, CUDA-graph replay of the device step counter, the FP32 check mode free-running against the
oracle driving torch's CPU optimizers, the train_epoch drop-in with a torch.optim.Adam, checkpoint resume, and the
CLI.  GPU only."""
import argparse
import math
import os
import re

import pytest
import torch

from test_gpu_step import cos

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------------------ kernels
def _segments():
    """The arena layout of tests/test_gpu_kernels.py::test_grad_stats_and_sgd; numel ends with the 100003-element
    tensor (no padding), so the numel % 4 tail of the update kernels runs."""
    sizes = [(64, 3, 7, 7), (64,), (64,), (128, 64, 3, 3), (6, 1024), (6,), (100003,)]
    groups = [0, 0, 1, 1, 2, 2, 1]
    pad = lambda n: (n + 63) // 64 * 64
    offs, total = [], 0
    for s in sizes:
        offs.append(total)
        total += pad(math.prod(s))
    numel = offs[-1] + math.prod(sizes[-1])
    g = torch.Generator(device="cuda").manual_seed(8)
    grad = torch.zeros(total, device="cuda")
    param = torch.zeros(total, device="cuda")
    for s, o in zip(sizes, offs):
        n = math.prod(s)
        grad[o:o + n] = torch.randn(n, device="cuda", generator=g) * 3
        param[o:o + n] = torch.randn(n, device="cuda", generator=g)
    seg_end = torch.tensor([min(o + pad(math.prod(s)), numel) for s, o in zip(sizes, offs)], device="cuda",
                           dtype=torch.int64)
    seg = (seg_end, torch.tensor(groups, device="cuda", dtype=torch.int32),
           torch.tensor([1.0 / math.prod(s) for s in sizes], device="cuda"))
    return sizes, offs, numel, param, grad, seg


def _fused(kind, kw, param, grad, numel, stats):
    """State buffers and a closure running one fused update (kw: torch's constructor arguments)."""
    from gdl_b200 import ops
    st = torch.zeros(3, device="cuda", dtype=torch.int32)
    if kind == "adam":
        m, v = torch.zeros_like(param), torch.zeros_like(param)
        b1, b2 = kw.get("betas", (0.9, 0.999))
        run = lambda: ops.adam(param, grad, m, v, st, numel, kw["lr"], b1, b2, kw.get("eps", 1e-8),
                               kw.get("weight_decay", 0.0), stats)
        return {"exp_avg": m, "exp_avg_sq": v}, st, run
    s = torch.full_like(param, kw.get("initial_accumulator_value", 0.0))
    run = lambda: ops.adagrad(param, grad, s, st, numel, kw["lr"], kw.get("lr_decay", 0.0), kw.get("eps", 1e-10),
                              kw.get("weight_decay", 0.0), stats)
    return {"sum": s}, st, run


CASES = [("adam", dict(lr=1e-3)), ("adam", dict(lr=2e-3, betas=(0.8, 0.99), weight_decay=1e-2)),
         ("adagrad", dict(lr=1e-2)), ("adagrad", dict(lr=1e-2, weight_decay=1e-2)),
         ("adagrad", dict(lr=1e-2, lr_decay=0.1)), ("adagrad", dict(lr=1e-2, initial_accumulator_value=0.1))]


@pytest.mark.parametrize("kind,kw", CASES)
def test_update_kernel_matches_torch_optim(kind, kw):
    """3 steps of gdl_adam / gdl_adagrad with the clip coefficient from gdl_grad_stats against clip_grad_norm_ and
    torch.optim.Adam / Adagrad: parameters, clipped gradients (written back) and state to fp32 accuracy."""
    from gdl_b200 import ops
    sizes, offs, numel, param, grad, (seg_end, seg_group, seg_inv) = _segments()
    params = [param[o:o + math.prod(s)].clone().view(s).requires_grad_(True) for s, o in zip(sizes, offs)]
    grads = [grad[o:o + math.prod(s)].clone().view(s) for s, o in zip(sizes, offs)]
    scratch = torch.empty(ops.optim_scratch_floats(numel, len(sizes)), device="cuda")
    stats = torch.empty(4, device="cuda")
    ops.grad_stats(grad, numel, seg_end, seg_group, seg_inv, len(sizes), 40.0, scratch, stats)
    state, st, run = _fused(kind, kw, param, grad, numel, stats)
    for step in range(3):
        run()
        if step == 0:
            stats[1] = 1.0  # later steps: the gradients are already clipped
    torch.cuda.synchronize()

    for p, gr in zip(params, grads):
        p.grad = gr.clone()
    torch.nn.utils.clip_grad_norm_(params, 40.0, 2)
    opt = (torch.optim.Adam if kind == "adam" else torch.optim.Adagrad)(params, **kw)
    for _ in range(3):
        opt.step()
    assert int(st[0]) == 3
    for p, s, o in zip(params, sizes, offs):
        n = p.numel()
        assert torch.allclose(param[o:o + n].view(s), p.detach(), atol=1e-6, rtol=1e-5)
        assert torch.allclose(grad[o:o + n].view(s), p.grad, atol=1e-6, rtol=1e-5)
        for key, buf in state.items():
            assert torch.allclose(buf[o:o + n].view(s), opt.state[p][key], atol=1e-6, rtol=1e-5), key
        assert float(opt.state[p]["step"]) == 3


@pytest.mark.parametrize("kind,kw", [CASES[1], CASES[4]])
def test_update_graph_replay_advances_the_device_step(kind, kw):
    """The update captured once and replayed 3 times is bit-identical to 3 eager calls: the step count (and with it
    the bias corrections / lr decay) advances on the device under replay."""
    from gdl_b200 import ops
    sizes, offs, numel, param, grad, (seg_end, seg_group, seg_inv) = _segments()
    stats = torch.tensor([1.0, 0.5, 0.0, 0.0], device="cuda")
    outs = []
    for graph in (False, True):
        p, g = param.clone(), grad.clone()
        state, st, run = _fused(kind, kw, p, g, numel, stats)
        if graph:
            torch.cuda.synchronize()
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr):
                run()
            for _ in range(3):
                gr.replay()
        else:
            for _ in range(3):
                run()
        torch.cuda.synchronize()
        outs.append([p, g, st] + list(state.values()))
    assert int(outs[1][2][0]) == 3
    for a, b in zip(*outs):
        assert torch.equal(a, b), "CUDA-graph replay differs from eager execution"


# ------------------------------------------------------------------------------------------------ check mode
def _oracle_step(O, sd, batch, update, **kw):
    """The oracle's DGL step with another optimizer: dgl_step runs its own SGD block with lr = 0 (the parameters stay
    as they are, the BatchNorm running statistics advance), then `update` applies the optimizer to the clipped
    gradients it returns."""
    ref = O.dgl_step(sd, {}, *batch, lr=0.0, mu=0.0, wd=0.0, **kw)
    with torch.no_grad():
        update(sd, ref["grads"])
    return ref


def _torch_update(cls, kw):
    """update(sd, grads) for _oracle_step: a CPU torch optimizer over the oracle's parameters (single-tensor path)."""
    box = {}

    def update(sd, grads):
        if "opt" not in box:
            box["params"] = {k: sd[k] for k in grads}
            box["opt"] = cls(list(box["params"].values()), **kw)
        for k, p in box["params"].items():
            p.grad = grads[k].clone()
        box["opt"].step()
    return update


def _run_check(kind, fusion, dataset, B, shape, nsteps, lr=1e-3):
    from gdl_b200 import AVClassifier_DGL, setup_seed, weight_init
    from gdl_b200.optim import UpdateRule
    from gdl_b200.step import DGLStep
    from oracle import dgl_oracle as O
    from oracle.synth import SHAPES, make_batch
    torch.set_num_threads(os.cpu_count())
    args = argparse.Namespace(dataset=dataset, fusion_method=fusion, modality="full")
    setup_seed(0)
    model = AVClassifier_DGL(args)
    model.apply(weight_init)
    model.cuda().train()
    Fq, Tt, T, H, W = SHAPES[shape]
    rule = UpdateRule(kind, lr, eps=1e-8 if kind == "adam" else 1e-10)
    step = DGLStep(model, B, (Fq, Tt), (T, H, W), alpha=4.0, rule=rule, check_fp32=True)
    cls = torch.optim.Adam if kind == "adam" else torch.optim.Adagrad
    update = _torch_update(cls, dict(lr=lr))
    sd = O.init_state(fusion, dataset, 0)
    names = dict(model.named_parameters())
    n_cls = O.N_CLASSES[dataset]
    for s in range(nsteps):
        before = {k: names[k].detach().cpu().clone() for k in sd if k in names}
        ref_before = {k: v.clone() for k, v in sd.items() if k in names}
        batch = make_batch(B, n_cls, shape, seed=1 + s)
        step.step(*[t.cuda() for t in batch])
        got = step.read_stats()
        ref = _oracle_step(O, sd, batch, update, fusion=fusion, alpha=4.0)
        rows = [(cos(names[k].grad.detach().cpu(), g), k) for k, g in ref["grads"].items()]
        # Parameters.  The first Adam / Adagrad update is lr * g / (|g| + eps) per element: +-lr whatever the
        # gradient's size, so an element whose gradient the two fp32 implementations get with opposite signs moves by
        # 2 lr, and one whose gradient is below ~1e-5 on either side (the eps regime: 1e-8 / |g| >= 1e-3) moves by a
        # fraction of lr.  Measured (B200): at step 0, 0.01-0.1 % of the elements move by more than 1e-3 lr, up to
        # 1947 of them with gradients above 1e-3 of their tensor's largest (`loud`: an element whose terms cancel
        # has an fp32 gradient that uncertain), so "only elements with |g| < 1e-3 max|g| may differ" does not hold.
        # Criterion: elements that differ by more than 1e-3 lr for neither reason (`unexplained`) are at most 1e-5
        # of all (measured: none).  Step 1 starts from weights that differ in those elements by 2 lr, and every
        # element's update depends on the ratio of its step-0 and step-1 gradients, so nothing element-wise holds
        # there (measured at the tiny shape: 60-70 % of the elements move by more than 1e-3 lr, update relative L2
        # difference 0.13-0.19, per-tensor gradient cosine median >= 0.9993 and minimum 0.948 (a BN bias), losses
        # within 1.6e-3); step 1 is bounded by those aggregate measures.
        bad = loud = unexplained = total = 0
        du2 = ref2 = 0.0
        for k, g in ref["grads"].items():
            dref = sd[k] - ref_before[k]
            du = (names[k].detach().cpu() - before[k]) - dref
            off = du.abs() > 1e-3 * lr
            gg = names[k].grad.detach().cpu()
            why = (gg * g <= 0) | (torch.minimum(gg.abs(), g.abs()) < 1e-5)
            loud += int((off & (g.abs() >= 1e-3 * g.abs().max())).sum())
            unexplained += int((off & ~why).sum())
            bad += int(off.sum())
            total += g.numel()
            du2 += du.double().pow(2).sum().item()
            ref2 += dref.double().pow(2).sum().item()
        rel = (du2 / ref2) ** 0.5
        untouched = all(torch.equal(names[k].detach().cpu(), before[k]) for k in before if k not in ref["grads"])
        print("check-mode %s %s/%s %s B=%d step %d: losses %s vs %s; grad_norm %.6g vs %.6g; min cos %.7f (%s); "
              "updates off by > 1e-3 lr: %d of %d elements, %d of them with |g| >= 1e-3 max|g|, %d unexplained; "
              "update rel. L2 diff %.2e; diag (%.5g, %.5g) vs (%.5g, %.5g)"
              % (kind, fusion, dataset, shape, B, s, got[:3], ref["losses"], got[3], ref["grad_norm"], min(rows)[0],
                 min(rows)[1], bad, total, loud, unexplained, rel, got[5], got[6], ref["audio_grad_sum"],
                 ref["visual_grad_sum"]))
        assert untouched
        if s == 0:   # identical weights: the check-mode tolerances of tests/test_gpu_check_mode.py
            for g, r in zip(got[:3], ref["losses"]):
                assert abs(g - r) <= 1e-4 * abs(r), (got[:3], ref["losses"])
            assert abs(got[3] - ref["grad_norm"]) <= 1e-3 * ref["grad_norm"]
            assert abs(got[4] - ref["clip_coef"]) <= 5e-3
            assert abs(got[5] - ref["audio_grad_sum"]) <= 2e-3 * ref["audio_grad_sum"]
            assert abs(got[6] - ref["visual_grad_sum"]) <= 2e-3 * ref["visual_grad_sum"]
            assert all(c >= 0.999 for c, _ in rows), min(rows)
            assert unexplained <= 1e-5 * total and bad <= 5e-3 * total, (unexplained, bad, total)
        else:
            for g, r in zip(got[:3], ref["losses"]):
                assert abs(g - r) <= 5e-3 * abs(r), (s, got[:3], ref["losses"])
            cs = sorted(c for c, _ in rows)
            assert cs[len(cs) // 2] >= 0.995 and cs[0] >= 0.9, (s, cs[:3], cs[len(cs) // 2])
            assert rel <= 0.3, (s, rel)
    assert step.arena.steps == nsteps and int(step.arena.step_state[0]) == nsteps
    del model, step
    torch.cuda.empty_cache()


@pytest.mark.parametrize("kind", ["adam", "adagrad"])
@pytest.mark.parametrize("fusion", ["concat", "gated"])
def test_check_mode_tiny_two_steps(kind, fusion):
    _run_check(kind, fusion, "CREMAD", 8, "tiny", nsteps=2)


@pytest.mark.parametrize("kind", ["adam", "adagrad"])
def test_check_mode_cremad_shape(kind):
    _run_check(kind, "concat", "CREMAD", 16, "CREMAD", nsteps=1)


# ------------------------------------------------------------------------------------------------ product path
def _model():
    import gdl_b200
    args = argparse.Namespace(dataset="CREMAD", fusion_method="concat", modality="full", alpha=4.0, epochs=1, drop=0)
    gdl_b200.setup_seed(0)
    m = gdl_b200.AVClassifier_DGL(args)
    m.apply(gdl_b200.weight_init)
    return args, m.cuda()


class _Wrap(torch.nn.Module):
    def __init__(self, m):
        super().__init__()
        self.module = m

    def forward(self, *a):
        return self.module(*a)


def _epochs(tmp_path, args, dp, opt, loader, n):
    from gdl_b200.train import train_epoch
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        return [train_epoch(args, e, dp, torch.device("cuda"), loader, opt, None) for e in range(n)]
    finally:
        os.chdir(cwd)


def test_train_epoch_with_torch_adam(tmp_path):
    """The drop-in with a torch.optim.Adam trains with Adam (the bf16 engine; CUDA graph from the second step)
    and tracks the fp32 oracle driving torch's Adam; the optimizer's state aliases the arena and counts the steps."""
    from oracle import dgl_oracle as O
    from oracle.synth import make_batch
    args, model = _model()
    dp = _Wrap(model)
    opt = torch.optim.Adam(dp.parameters(), lr=1e-3, betas=(0.9, 0.999), eps=1e-8)
    batches = [make_batch(4, 6, "tiny", seed=1 + s) for s in range(3)]
    res = _epochs(tmp_path, args, dp, opt, batches, 1)[0]
    sd, tot = O.init_state("concat", "CREMAD", 0), [0.0, 0.0, 0.0]
    update = _torch_update(torch.optim.Adam, dict(lr=1e-3))
    for b in batches:
        r = _oracle_step(O, sd, b, update, fusion="concat")
        tot = [x + y / 3 for x, y in zip(tot, r["losses"])]
    print("train_epoch with Adam: mean losses %s vs oracle %s" % (list(res[:3]), tot))
    for g, r in zip(res[:3], tot):
        assert abs(g - r) <= 5e-2 * abs(r), (res[:3], tot)
    ar = model._gdl_arena
    assert ar.kind == "adam" and not hasattr(ar, "momentum")
    p = model.audio_net.conv1.weight
    o = ar.offset_of[id(p)]
    assert opt.state[p]["exp_avg"].data_ptr() == ar.exp_avg.data_ptr() + 4 * o
    assert opt.state[p]["exp_avg_sq"].data_ptr() == ar.exp_avg_sq.data_ptr() + 4 * o
    assert float(opt.state[p]["exp_avg_sq"].abs().sum()) > 0
    assert float(opt.state[p]["step"]) == 3 and int(ar.step_state[0]) == 3


def test_adam_short_tail_batch_shares_one_step_count(tmp_path):
    """A loader without drop_last: the full and the short batch get a DGLStep each, on one arena with one step count
    (2 epochs of 4, 4, 2 => 6), tracking the oracle stepping through the same sequence with one torch Adam (the bias
    corrections follow the count).  lr = 1e-4 (every Adam update moves every element by about lr): measured on a B200,
    epoch-2 mean losses within 2 % of the oracle's; Adagrad at lr = 1e-3 memorised the 10 items within the 6 steps,
    and its bf16 unimodal losses of 0.05-0.2 differed from the oracle's by up to 40 %."""
    from torch.utils.data import DataLoader, Dataset
    from oracle import dgl_oracle as O
    from oracle.synth import make_batch
    items = [make_batch(1, 6, "tiny", seed=300 + i) for i in range(10)]

    class DS(Dataset):
        def __len__(self):
            return len(items)

        def __getitem__(self, i):
            return tuple(t[0] for t in items[i])

    args, model = _model()
    dp = _Wrap(model)
    opt = torch.optim.Adam(dp.parameters(), lr=1e-4)
    loader = DataLoader(DS(), batch_size=4, shuffle=False, num_workers=0, pin_memory=True, drop_last=False)
    res = _epochs(tmp_path, args, dp, opt, loader, 2)[-1]
    steps = model._gdl_steps
    assert sorted(k[0] for k in steps) == [2, 4]
    a, b = steps.values()
    assert a.arena is b.arena and a.steps_done + b.steps_done == 6
    assert a.arena.steps == 6 and int(a.arena.step_state[0]) == 6
    assert {float(opt.state[p]["step"]) for p in a.arena.params} == {6.0}
    sd, update = O.init_state("concat", "CREMAD", 0), _torch_update(torch.optim.Adam, dict(lr=1e-4))
    for epoch in range(2):
        tot = [0.0, 0.0, 0.0]
        for lo in (0, 4, 8):
            batch = [torch.cat([c[j] for c in items[lo:lo + 4]]) for j in range(3)]
            r = _oracle_step(O, sd, batch, update, fusion="concat")
            tot = [t + x / 3 for t, x in zip(tot, r["losses"])]
    print("tail-batch run with Adam: epoch-2 mean losses %s vs oracle %s" % (list(res[:3]), tot))
    for g, r in zip(res[:3], tot):
        assert abs(g - r) <= 1e-1 * abs(r), (res[:3], tot)


@pytest.mark.parametrize("kind", ["adam", "adagrad"])
def test_resume_from_a_checkpoint_continues_the_run(tmp_path, kind):
    """Train 3 steps, save model + optimizer the way main_dgl.py does, resume into a new model and optimizer, train 3
    more: the result equals training 6 steps without the interruption (state and step count restored)."""
    from oracle.synth import make_batch
    batches = [make_batch(4, 6, "tiny", seed=1 + s) for s in range(6)]

    def fresh():
        args, model = _model()
        dp = _Wrap(model)
        cls = torch.optim.Adam if kind == "adam" else torch.optim.Adagrad
        return args, model, dp, cls(dp.parameters(), lr=1e-3)
    args, m0, dp0, opt0 = fresh()
    _epochs(tmp_path, args, dp0, opt0, batches[:3], 1)
    path = os.path.join(str(tmp_path), "ckpt.pth")
    torch.save({"model": dp0.state_dict(), "optimizer": opt0.state_dict()}, path)
    _epochs(tmp_path, args, dp0, opt0, batches[3:], 1)

    args, m1, dp1, opt1 = fresh()
    ck = torch.load(path, map_location="cuda")
    dp1.load_state_dict(ck["model"])
    opt1.load_state_dict(ck["optimizer"])
    _epochs(tmp_path, args, dp1, opt1, batches[3:], 1)
    torch.cuda.synchronize()
    assert m1._gdl_arena.steps == 6 and int(m1._gdl_arena.step_state[0]) == 6
    worst = max((p1.detach() - p0.detach()).abs().max().item() for p0, p1 in zip(m0.parameters(), m1.parameters()))
    print("%s resume vs uninterrupted: max |param diff| %.3g" % (kind, worst))
    assert worst <= 1e-6


# ------------------------------------------------------------------------------------------------ CLI
@pytest.mark.parametrize("name", ["Adam", "AdaGrad"])
def test_main_dgl_trains_with_the_optimizer(tmp_path, capsys, name):
    import sys
    sys.path.insert(0, ROOT)
    import main_dgl
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        main_dgl.main(["--train", "--ckpt_path", str(tmp_path / "ckpt"), "--optimizer", name, "--epochs", "1",
                       "--batch_size", "4", "--audio_path", "synthetic", "--synthetic_len", "16"])
    finally:
        os.chdir(cwd)
    out = capsys.readouterr().out
    losses = [float(x) for x in re.findall(r"^Loss: ([-+0-9.naif]+)", out, re.M)]
    assert losses and all(math.isfinite(x) for x in losses), out[-2000:]


def test_main_dgl_rejects_an_unknown_optimizer(tmp_path):
    import sys
    sys.path.insert(0, ROOT)
    import main_dgl
    with pytest.raises(ValueError, match="Incorrect optimizer"):
        main_dgl.main(["--train", "--ckpt_path", str(tmp_path), "--optimizer", "foo", "--audio_path", "synthetic"])
