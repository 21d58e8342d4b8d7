"""Per-iteration lr schedules without a GPU: the warm-up + cosine factor of main_dgl.py --lr_schedule cosine against its
closed form, the flag validation, the scheduler's state_dict round trip, and gdl_b200.optim.follow_rule (the refusal
of a changed momentum, betas, eps, weight decay or lr_decay) on CPU optimizers."""
import math
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "iccv2025-gdl_b200"))


def _closed_form(k, K, W):
    return (k + 1) / W if k < W else 0.5 * (1 + math.cos(math.pi * (k - W) / (K - W)))


@pytest.mark.parametrize("K,W", [(100, 10), (100, 0), (7, 3), (2, 1), (1, 0)])
def test_warmup_cosine_factor_is_the_closed_form(K, W):
    from gdl_b200.optim import warmup_cosine
    f = warmup_cosine(K, W)
    assert [f(k) for k in range(K + 1)] == [_closed_form(k, K, W) for k in range(K + 1)]
    assert f(0) == (1 / W if W else 1.0)             # first step
    if W:
        assert f(W - 1) == 1.0                       # last warm-up step
    assert f(W) == 1.0                               # first decay step
    assert f(K - 1) == pytest.approx(0.5 * (1 + math.cos(math.pi * (K - 1 - W) / (K - W))))
    assert abs(f(K)) < 1e-15                         # where the schedule ends


@pytest.mark.parametrize("K,W", [(10, 10), (10, 11), (10, -1), (0, 0)])
def test_warmup_cosine_rejects_a_warmup_that_does_not_fit(K, W):
    from gdl_b200.optim import warmup_cosine
    with pytest.raises(ValueError, match="warmup_steps"):
        warmup_cosine(K, W)


def test_lambda_lr_follows_the_factor_per_iteration():
    from gdl_b200.optim import warmup_cosine
    opt = torch.optim.SGD([torch.nn.Parameter(torch.zeros(2))], lr=0.01, momentum=0.9)
    sched = torch.optim.lr_scheduler.LambdaLR(opt, warmup_cosine(20, 4))
    seen = []
    for _ in range(20):
        seen.append(opt.param_groups[0]["lr"])
        opt.step()
        sched.step()
    assert seen == [0.01 * _closed_form(k, 20, 4) for k in range(20)]


def _args(*extra):
    import main_dgl
    return main_dgl.get_arguments(["--ckpt_path", "x"] + list(extra))


def test_flag_defaults_keep_the_reference_schedule():
    import main_dgl
    args = _args()
    assert (args.lr_schedule, args.warmup_steps) == ("multistep", 0)
    main_dgl.check_lr_schedule(args)
    opt = torch.optim.SGD([torch.nn.Parameter(torch.zeros(2))], lr=0.001, momentum=0.9)
    sched, step_sched = main_dgl.make_schedulers(args, opt, 10)
    assert type(sched) is torch.optim.lr_scheduler.MultiStepLR and step_sched is None
    assert list(sched.milestones) == [70] and sched.gamma == 0.1


@pytest.mark.parametrize("extra,match", [(["--warmup_steps", "3"], "cosine only"),
                                         (["--lr_schedule", "multistep", "--warmup_steps", "1"], "cosine only"),
                                         (["--lr_schedule", "cosine", "--warmup_steps", "-1"], ">= 0")])
def test_invalid_flag_combinations_raise_before_any_device_work(extra, match):
    import main_dgl
    with pytest.raises(ValueError, match=match):
        main_dgl.check_lr_schedule(_args(*extra))
    # main() raises it before it touches a device (this machine may have none)
    with pytest.raises(ValueError, match=match):
        main_dgl.main(["--train", "--ckpt_path", "x", "--audio_path", "synthetic"] + extra)


def test_unknown_schedule_is_rejected_by_the_parser():
    with pytest.raises(SystemExit):
        _args("--lr_schedule", "linear")


def test_cosine_scheduler_state_dict_round_trip():
    """The per-iteration scheduler saved after 7 of 30 steps and loaded into a fresh optimizer + scheduler (as
    main_dgl.py --resume does) continues the same lr sequence."""
    import main_dgl
    args = _args("--lr_schedule", "cosine", "--warmup_steps", "4", "--epochs", "3", "--learning_rate", "0.02")
    main_dgl.check_lr_schedule(args)

    def fresh():
        opt = torch.optim.Adam([torch.nn.Parameter(torch.zeros(2))], lr=args.learning_rate)
        sched, step_sched = main_dgl.make_schedulers(args, opt, 10)
        assert sched is None and type(step_sched) is torch.optim.lr_scheduler.LambdaLR
        return opt, step_sched

    def run(opt, sched, n):
        out = []
        for _ in range(n):
            out.append(opt.param_groups[0]["lr"])
            opt.step()
            sched.step()
        return out
    opt, sched = fresh()
    first = run(opt, sched, 7)
    saved = {"optimizer": opt.state_dict(), "scheduler": sched.state_dict()}
    rest = run(opt, sched, 23)
    opt2, sched2 = fresh()
    opt2.load_state_dict(saved["optimizer"])
    sched2.load_state_dict(saved["scheduler"])
    assert sched2.last_epoch == 7
    assert run(opt2, sched2, 23) == rest
    assert first + rest == [0.02 * _closed_form(k, 30, 4) for k in range(30)]


# ------------------------------------------------------------------------------------------------ follow_rule
def _p():
    return [torch.nn.Parameter(torch.zeros(3))]


@pytest.mark.parametrize("make,key,value", [
    (lambda p: torch.optim.SGD(p, lr=0.1, momentum=0.9, weight_decay=1e-4), "momentum", 0.85),
    (lambda p: torch.optim.SGD(p, lr=0.1, momentum=0.9, weight_decay=1e-4), "weight_decay", 1e-3),
    (lambda p: torch.optim.Adam(p, lr=1e-3), "betas", (0.85, 0.999)),
    (lambda p: torch.optim.Adam(p, lr=1e-3), "eps", 1e-6),
    (lambda p: torch.optim.Adam(p, lr=1e-3), "weight_decay", 1e-2),
    (lambda p: torch.optim.Adagrad(p, lr=1e-2), "lr_decay", 0.1),
    (lambda p: torch.optim.Adagrad(p, lr=1e-2), "eps", 1e-8),
])
def test_a_changed_setting_other_than_lr_is_refused_by_name(make, key, value):
    from gdl_b200.optim import follow_rule, update_rule
    opt = make(_p())
    rule = update_rule(opt)
    opt.param_groups[0]["lr"] *= 0.5          # the lr may change
    follow_rule(opt, rule)
    opt.param_groups[0][key] = value
    with pytest.raises(NotImplementedError, match="changing " + key):
        follow_rule(opt, rule)


def test_initial_accumulator_value_is_not_compared():
    """torch's Adagrad reads it only when it creates the state, so changing it later changes nothing."""
    from gdl_b200.optim import follow_rule, update_rule
    opt = torch.optim.Adagrad(_p(), lr=1e-2, initial_accumulator_value=0.1)
    rule = update_rule(opt)
    opt.param_groups[0]["initial_accumulator_value"] = 0.5
    follow_rule(opt, rule)


@pytest.mark.parametrize("make,setting", [(lambda p: torch.optim.SGD(p, lr=0.1, momentum=0.9), "momentum"),
                                          (lambda p: torch.optim.Adam(p, lr=1e-3), "betas")])
def test_one_cycle_with_cycle_momentum_is_refused(make, setting):
    from gdl_b200.optim import follow_rule, update_rule
    opt = make(_p())
    sched = torch.optim.lr_scheduler.OneCycleLR(opt, max_lr=0.1, total_steps=10, cycle_momentum=True)
    rule = update_rule(opt)                   # the step is built after the scheduler set its first momentum
    follow_rule(opt, rule)
    opt.step()
    sched.step()
    with pytest.raises(NotImplementedError, match="changing {}.*cycle_momentum=False".format(setting)):
        follow_rule(opt, rule)


def test_one_cycle_without_cycle_momentum_is_followed():
    from gdl_b200.optim import follow_rule, update_rule
    opt = torch.optim.SGD(_p(), lr=0.1, momentum=0.9)
    sched = torch.optim.lr_scheduler.OneCycleLR(opt, max_lr=0.1, total_steps=10, cycle_momentum=False)
    rule = update_rule(opt)
    lrs = set()
    for _ in range(9):
        follow_rule(opt, rule)
        lrs.add(opt.param_groups[0]["lr"])
        opt.step()
        sched.step()
    assert len(lrs) == 9

