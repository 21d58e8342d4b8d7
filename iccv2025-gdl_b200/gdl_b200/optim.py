"""The update rule of the fused step, read from the torch optimizer the caller passes in (reference main_dgl.py:249-256:
`sgd`, `AdaGrad`, `Adam`).  The fused step runs csrc/optim.cu instead of `optimizer.step()`, so every setting of the
optimizer that those kernels do not implement is refused here, by name, rather than silently trained as something
else."""
from dataclasses import dataclass

import torch


@dataclass(frozen=True)
class UpdateRule:
    """kind: "sgd" (torch.optim.SGD with momentum), "adam" or "adagrad".  lr is the value at construction; the step
    re-reads the optimizer's lr every step (the lr schedule)."""
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
