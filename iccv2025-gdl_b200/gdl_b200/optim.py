"""The update rule of the fused step, read from the torch optimizer the caller passes in (reference main_dgl.py:249-256:
`sgd`, `AdaGrad`, `Adam`).  The fused step runs csrc/optim.cu instead of `optimizer.step()`, so every setting of the
optimizer that those kernels do not implement is refused here, by name, rather than silently trained as something
else."""
import math
from dataclasses import dataclass, fields

import torch


@dataclass(frozen=True)
class UpdateRule:
    """kind: "sgd" (torch.optim.SGD with momentum), "adam" or "adagrad".  lr is the value at construction; the step
    re-reads the optimizer's lr every step (the lr schedule).  Every other setting is read once, when the step is
    built (follow_rule refuses a change of one)."""
    kind: str
    lr: float
    weight_decay: float = 0.0
    momentum: float = 0.0                      # sgd
    betas: tuple = (0.9, 0.999)                # adam
    eps: float = 1e-8                          # adam, adagrad
    lr_decay: float = 0.0                      # adagrad
    initial_accumulator_value: float = 0.0     # adagrad


def update_rule(optimizer):
    """UpdateRule of a torch.optim.SGD / Adam / Adagrad with one param group; raises NotImplementedError for any
    other optimizer or setting."""
    name = type(optimizer).__name__
    if type(optimizer) not in (torch.optim.SGD, torch.optim.Adam, torch.optim.Adagrad):
        raise NotImplementedError("the fused DGL step implements torch.optim.SGD, Adam and Adagrad, not {}".format(name))
    if len(optimizer.param_groups) != 1:
        raise NotImplementedError("the fused DGL step takes one param group; this {} has {}"
                                  .format(name, len(optimizer.param_groups)))
    g = optimizer.param_groups[0]

    def refuse(flag, value):
        if value:
            raise NotImplementedError("the fused DGL step does not implement {}({}={!r})".format(name, flag, value))

    refuse("maximize", g.get("maximize", False))
    lr, wd = float(g["lr"]), float(g["weight_decay"])
    if isinstance(optimizer, torch.optim.SGD):
        refuse("nesterov", g["nesterov"])
        refuse("dampening", g["dampening"])
        return UpdateRule("sgd", lr, wd, momentum=float(g["momentum"]))
    if isinstance(optimizer, torch.optim.Adam):
        refuse("amsgrad", g["amsgrad"])
        refuse("decoupled_weight_decay", g.get("decoupled_weight_decay", False))
        return UpdateRule("adam", lr, wd, betas=(float(g["betas"][0]), float(g["betas"][1])), eps=float(g["eps"]))
    return UpdateRule("adagrad", lr, wd, eps=float(g["eps"]), lr_decay=float(g["lr_decay"]),
                      initial_accumulator_value=float(g["initial_accumulator_value"]))


# settings that a scheduler may cycle, and how to keep it from doing so
_CYCLED = {"momentum": " (OneCycleLR / CyclicLR: cycle_momentum=False)", "betas": " (OneCycleLR: cycle_momentum=False)"}


def follow_rule(optimizer, rule):
    """Raise NotImplementedError, naming the setting, when the optimizer's param group now differs from `rule` (the
    update a DGLStep was built with) in anything but the lr: the fused update reads those settings once, so a
    scheduler that changes one of them would otherwise train with the stale value.  Host-side dictionary reads only.
    (Adagrad's initial_accumulator_value is not compared: torch reads it only when it creates the state.)"""
    now = update_rule(optimizer)
    for f in fields(UpdateRule):
        if f.name in ("lr", "initial_accumulator_value"):
            continue
        a, b = getattr(rule, f.name), getattr(now, f.name)
        if a != b:
            raise NotImplementedError("the fused DGL step does not follow a changing {} ({!r} -> {!r}): it reads every "
                                      "setting but the lr once, when the step is built{}"
                                      .format(f.name, a, b, _CYCLED.get(f.name, "")))


def warmup_cosine(total_steps, warmup_steps):
    """The lr factor of step k (k = 0 .. total_steps - 1) for torch.optim.lr_scheduler.LambdaLR stepped once per
    iteration (main_dgl.py --lr_schedule cosine): (k + 1) / W for k < W (linear warm-up, W = warmup_steps), then
    1/2 (1 + cos(pi (k - W) / (K - W))) (cosine decay towards 0 at k = K = total_steps)."""
    K, W = int(total_steps), int(warmup_steps)
    if not 0 <= W < K:
        raise ValueError("a cosine schedule over {} steps needs 0 <= warmup_steps < {}, got {}".format(K, K, W))

    def factor(k):
        if k < W:
            return (k + 1) / W
        return 0.5 * (1.0 + math.cos(math.pi * (k - W) / (K - W)))
    return factor
