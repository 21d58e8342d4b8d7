"""The update rule read from the torch optimizer (gdl_b200.optim.update_rule) and the Adam / Adagrad optimizer state
in the parameter arena (train.adopt_momentum): what the fused step trains with, what it refuses, and checkpoints in
both directions.  CPU only (the arena is allocated on the CPU; no kernel runs)."""
import argparse
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "iccv2025-gdl_b200"))


def _model():
    import gdl_b200
    args = argparse.Namespace(dataset="CREMAD", fusion_method="concat", modality="full")
    gdl_b200.setup_seed(0)
    return gdl_b200.AVClassifier_DGL(args)


def _params():
    return [torch.nn.Parameter(torch.zeros(3))]


def test_rule_carries_the_hyper_parameters():
    from gdl_b200.optim import update_rule
    r = update_rule(torch.optim.SGD(_params(), lr=0.002, momentum=0.8, weight_decay=3e-4))
    assert (r.kind, r.lr, r.momentum, r.weight_decay) == ("sgd", 0.002, 0.8, 3e-4)
    r = update_rule(torch.optim.Adam(_params(), lr=0.003, betas=(0.8, 0.99), eps=1e-6, weight_decay=1e-2))
    assert (r.kind, r.lr, r.betas, r.eps, r.weight_decay) == ("adam", 0.003, (0.8, 0.99), 1e-6, 1e-2)
    r = update_rule(torch.optim.Adam(_params(), lr=0.001, betas=(0.9, 0.999), eps=1e-08))  # main_dgl.py --optimizer Adam
    assert (r.kind, r.betas, r.eps, r.weight_decay) == ("adam", (0.9, 0.999), 1e-8, 0.0)
    r = update_rule(torch.optim.Adagrad(_params(), lr=0.004, lr_decay=0.1, weight_decay=2e-4,
                                        initial_accumulator_value=0.5, eps=1e-9))
    assert (r.kind, r.lr, r.lr_decay, r.weight_decay, r.initial_accumulator_value, r.eps) == \
        ("adagrad", 0.004, 0.1, 2e-4, 0.5, 1e-9)
    r = update_rule(torch.optim.Adagrad(_params(), lr=0.001))                              # --optimizer AdaGrad
    assert (r.lr_decay, r.weight_decay, r.initial_accumulator_value, r.eps) == (0.0, 0.0, 0.0, 1e-10)


@pytest.mark.parametrize("make,setting", [
    (lambda p: torch.optim.SGD(p, lr=0.1, momentum=0.9, nesterov=True), "nesterov"),
    (lambda p: torch.optim.SGD(p, lr=0.1, momentum=0.9, dampening=0.1), "dampening"),
    (lambda p: torch.optim.SGD(p, lr=0.1, momentum=0.9, maximize=True), "maximize"),
    (lambda p: torch.optim.Adam(p, amsgrad=True), "amsgrad"),
    (lambda p: torch.optim.Adam(p, maximize=True), "maximize"),
    (lambda p: torch.optim.Adam(p, decoupled_weight_decay=True), "decoupled_weight_decay"),
    (lambda p: torch.optim.Adagrad(p, maximize=True), "maximize"),
    (lambda p: torch.optim.SGD([{"params": p[:1]}, {"params": p[1:]}], lr=0.1), "param group"),
    (lambda p: torch.optim.AdamW(p), "AdamW"),
    (lambda p: torch.optim.RMSprop(p), "RMSprop"),
])
def test_unsupported_settings_raise_naming_the_setting(make, setting):
    from gdl_b200.optim import update_rule
    with pytest.raises(NotImplementedError, match=setting):
        update_rule(make([torch.nn.Parameter(torch.zeros(3)), torch.nn.Parameter(torch.zeros(2))]))


def _views(arena, buf):
    return [buf[o:o + p.numel()] for p, o in zip(arena.params, arena.offsets)]


@pytest.mark.parametrize("kind", ["adam", "adagrad"])
def test_checkpoint_state_is_adopted_by_the_arena(kind):
    """Fresh run: the optimizer's state aliases the arena (Adagrad's construction-time `sum` is copied in); a resumed
    run copies exp_avg / exp_avg_sq / sum and the step count in; the next state_dict() carries the arena's values
    and step; differing per-parameter step counts raise."""
    from gdl_b200.optim import update_rule
    from gdl_b200.step import ParamArena
    from gdl_b200.train import adopt_momentum

    def build():
        m = _model()
        if kind == "adam":
            return m, torch.optim.Adam(m.parameters(), lr=0.001, betas=(0.9, 0.999), eps=1e-08)
        return m, torch.optim.Adagrad(m.parameters(), lr=0.001, initial_accumulator_value=0.25)
    keys = ["exp_avg", "exp_avg_sq"] if kind == "adam" else ["sum"]

    # "previous run"
    m0, opt0 = build()
    a0 = ParamArena(m0, torch.device("cpu"), update_rule(opt0))
    assert not hasattr(a0, "momentum")                   # only the state of the rule in use is allocated
    auxi = m0.fusion_module.fc_auxi.weight               # never trained: outside the arena
    auxi_state = dict(opt0.state[auxi]) if kind == "adagrad" else {}
    assert adopt_momentum(a0, opt0) is (kind == "adagrad")   # Adagrad: torch's initial sums are copied in
    assert a0.steps == 0 and int(a0.step_state[0]) == 0
    for key, (_, buf) in zip(keys, a0.state_buffers):
        assert buf is getattr(a0, key)
        for p, o in zip(a0.params, a0.offsets):      # the optimizer state aliases the arena
            assert opt0.state[p][key].data_ptr() == buf.data_ptr() + 4 * o
        if kind == "adagrad":
            assert all(torch.all(v == 0.25) for v in _views(a0, buf))
    if kind == "adagrad":                            # fc_auxi's construction-time state is left alone
        assert opt0.state[auxi].keys() == auxi_state.keys()
        assert all(opt0.state[auxi][k] is v for k, v in auxi_state.items())
    # the fused kernels update the arena and count 5 steps
    for i, (_, buf) in enumerate(a0.state_buffers):
        buf.copy_(torch.arange(a0.numel, dtype=torch.float32) * 1e-6 + i)
    a0.set_steps(5)
    a0.sync_step_tensors()
    saved = {"model": m0.state_dict(), "optimizer": opt0.state_dict()}
    in_arena = [i for i, q in enumerate(m0.parameters()) if id(q) in a0.offset_of]   # state_dict keys: param index
    assert len(in_arena) == len(a0.params)
    for i in in_arena:
        st = saved["optimizer"]["state"][i]
        assert float(st["step"]) == 5.0 and st["step"].device.type == "cpu"

    # "resumed run"
    m1, opt1 = build()
    m1.load_state_dict(saved["model"])
    opt1.load_state_dict(saved["optimizer"])
    a1 = ParamArena(m1, torch.device("cpu"), update_rule(opt1))

    class _Step:
        momentum_loaded = False
    assert adopt_momentum(a1, opt1, _Step()) is True
    assert a1.steps == 5 and int(a1.step_state[0]) == 5
    for (_, b0), (_, b1) in zip(a0.state_buffers, a1.state_buffers):
        for v0, v1 in zip(_views(a0, b0), _views(a1, b1)):
            assert torch.equal(v0, v1)
    p = a1.params[3]
    for key, (_, buf) in zip(keys, a1.state_buffers):
        assert opt1.state[p][key].data_ptr() == buf[a1.offsets[3]:].data_ptr()
    # a second adoption (the DGLStep of an epoch's short tail batch) changes nothing and keeps the count
    a1.steps += 2
    assert adopt_momentum(a1, opt1) is False and a1.steps == 7
    for _, buf in a1.state_buffers:                  # the fused kernels keep updating the arena ...
        buf.mul_(2.0)
    a1.sync_step_tensors()
    again = opt1.state_dict()["state"]               # ... and the next checkpoint carries those values and the count
    for key, (_, b0) in zip(keys, a0.state_buffers):
        total = sum(again[i][key].double().sum().item() for i in in_arena)
        want = 2.0 * sum(v.double().sum().item() for v in _views(a0, b0))
        assert abs(total - want) <= 1e-9 * max(1.0, abs(want))
    assert {float(again[i]["step"]) for i in in_arena} == {7.0}

    # one parameter restored at another step count: refused
    bad = {"state": dict(saved["optimizer"]["state"]), "param_groups": saved["optimizer"]["param_groups"]}
    i = in_arena[2]
    bad["state"][i] = dict(bad["state"][i], step=torch.tensor(4.0))
    m2, opt2 = build()
    opt2.load_state_dict(bad)
    a2 = ParamArena(m2, torch.device("cpu"), update_rule(opt2))
    with pytest.raises(ValueError, match="step counts"):
        adopt_momentum(a2, opt2)
