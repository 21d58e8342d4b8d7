"""Drop-in surface on the GPU: the autograd-compatible module mode driven by the reference's own
two-backward loop (restated from main_dgl.py:97-154), eval-mode forward / valid(), and the
train_epoch drop-in.  GPU only."""
import argparse
import csv
import os

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def make_model(fusion="concat", dataset="CREMAD"):
    import gdl_b200
    args = argparse.Namespace(dataset=dataset, fusion_method=fusion, modality="full", alpha=4.0, epochs=1, drop=0)
    gdl_b200.setup_seed(0)
    m = gdl_b200.AVClassifier_DGL(args)
    m.apply(gdl_b200.weight_init)
    return args, m.cuda()


class _Wrap(nn.Module):  # provides the `module.` prefix the reference's wipe loop keys on
    def __init__(self, m):
        super().__init__()
        self.module = m

    def forward(self, *a):
        return self.module(*a)


def cos(a, b):
    return F.cosine_similarity(a.flatten().double(), b.flatten().double(), dim=0).item()


@pytest.mark.parametrize("fusion", ["concat", "sum", "gated", "film"])
def test_reference_two_backward_loop_runs_on_the_modules(fusion):
    """The reference's step, verbatim in structure (main_dgl.py:97-154): zero_grad, forward,
    3x CE, (La+Lv)*alpha backward with retain_graph, wipe `fusion` grads, Lf backward, clip, SGD."""
    from oracle import dgl_oracle as O
    from oracle.synth import make_batch
    args, model = make_model(fusion)
    model.train()
    dp = _Wrap(model)
    opt = torch.optim.SGD(dp.parameters(), lr=0.01, momentum=0.9, weight_decay=1e-4)
    spec, image, label = make_batch(4, 6, "tiny", seed=1)
    spec, image, label = spec.cuda(), image.cuda(), label.cuda()
    crit = nn.CrossEntropyLoss()
    opt.zero_grad()
    out, out_a, out_v = dp(spec.unsqueeze(1).float(), image.float())
    loss_v, loss_a, loss_f = crit(out_v, label), crit(out_a, label), crit(out, label)
    ((loss_a + loss_v) * args.alpha).backward(retain_graph=True)
    for name, parms in dp.named_parameters():
        if 'fusion' in str(name).split('.')[1]:
            parms.grad = None
    loss_f.backward()
    nn.utils.clip_grad_norm_(dp.parameters(), max_norm=40, norm_type=2)
    opt.step()
    torch.cuda.synchronize()
    sd = O.init_state(fusion, "CREMAD", 0)
    ref = O.dgl_step(sd, {}, *make_batch(4, 6, "tiny", seed=1), fusion=fusion, alpha=4.0, lr=0.01)
    for g, r in zip((loss_f.item(), loss_a.item(), loss_v.item()), ref["losses"]):
        assert abs(g - r) <= 2e-2 * abs(r)
    names = dict(model.named_parameters())
    for k, g32 in ref["grads"].items():
        gg = names[k].grad.detach().float().cpu()
        assert cos(gg, g32) > (0.995 if k.startswith("fusion_module") else 0.75), k
    # parameters the reference never trains have no grad after the wipe + Lf backward
    for k, p in names.items():
        if k not in ref["grads"]:
            assert p.grad is None or float(p.grad.abs().sum()) == 0.0, k


def test_eval_forward_and_valid():
    from gdl_b200.train import valid
    from oracle import dgl_oracle as O
    from oracle.synth import make_batch
    args, model = make_model("concat")
    sd = O.init_state("concat", "CREMAD", 0)
    from gdl_b200.step import DGLStep
    from oracle.synth import SHAPES
    Fq, Tt, T, H, W = SHAPES["tiny"]
    step = DGLStep(model, 4, (Fq, Tt), (T, H, W), lr=0.01, use_graph=False)
    mom = {}
    for s in range(2):
        b = make_batch(4, 6, "tiny", seed=1 + s)
        step.step(*[t.cuda() for t in b])
        O.dgl_step(sd, mom, *b, fusion="concat", lr=0.01)
    torch.cuda.synchronize()
    # running statistics follow the reference's update rule
    msd = model.state_dict()
    for k in ("audio_net.bn1.running_mean", "visual_net.layer4.1.bn2.running_var", "audio_net.bn1.num_batches_tracked"):
        assert torch.allclose(msd[k].float().cpu(), sd[k].float(), rtol=5e-2, atol=5e-2), k
    model.eval()
    spec, image, label = make_batch(4, 6, "tiny", seed=9)
    with torch.no_grad():
        out, oa, ov = model(spec.cuda().unsqueeze(1).float(), image.cuda().float())
        # eval-mode forward of the oracle on the SAME weights and running statistics (the drift of the two
        # training trajectories is checked above; here only the eval kernels are under test)
        sd_same = {k: v.detach().float().cpu() if v.is_floating_point() else v.detach().cpu() for k, v in msd.items()}
        ro, ra, rv = O.model_forward(sd_same, spec, image, "concat", training=False)
    for g, r in zip((out, oa, ov), (ro, ra, rv)):
        assert (g.cpu() - r).abs().max().item() < 0.05 * (r.abs().max().item() + 1.0)
    acc = valid(args, _Wrap(model), torch.device("cuda"), [(spec, image, label)])
    assert len(acc) == 3 and all(0.0 <= a <= 1.0 for a in acc)
    assert model.args.drop == 1  # the reference flips this flag back (main_dgl.py:221)


def test_train_epoch_dropin(tmp_path):
    from gdl_b200.train import train_epoch
    from oracle import dgl_oracle as O
    from oracle.synth import make_batch
    args, model = make_model("concat")
    dp = _Wrap(model)
    opt = torch.optim.SGD(dp.parameters(), lr=0.01, momentum=0.9, weight_decay=1e-4)
    batches = [make_batch(4, 6, "tiny", seed=1 + s) for s in range(3)]
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        res = train_epoch(args, 0, dp, torch.device("cuda"), batches, opt, None)
        rows = list(csv.reader(open("audio_visual_grad_vanilla.csv")))
    finally:
        os.chdir(cwd)
    assert len(res) == 7 and res[3:] == (0.0, 0.0, 0.0, 0.0)
    assert len(rows) == 3
    sd, mom, tot = O.init_state("concat", "CREMAD", 0), {}, [0.0, 0.0, 0.0]
    diag0 = None
    for b in batches:
        r = O.dgl_step(sd, mom, *b, fusion="concat", lr=0.01)
        tot = [x + y / 3 for x, y in zip(tot, r["losses"])]
        diag0 = diag0 or (r["audio_grad_sum"], r["visual_grad_sum"])
    for g, r in zip(res[:3], tot):
        assert abs(g - r) <= 5e-2 * abs(r), (res[:3], tot)
    assert abs(float(rows[0][0]) - diag0[0]) <= 5e-2 * diag0[0]
    assert abs(float(rows[0][1]) - diag0[1]) <= 5e-2 * diag0[1]
    # momentum is visible through the torch optimizer for reference-format checkpoints
    p = model.audio_net.conv1.weight
    assert "momentum_buffer" in opt.state[p] and float(opt.state[p]["momentum_buffer"].abs().sum()) > 0


def test_train_epoch_over_a_pinning_dataloader_captures_graphs(tmp_path):
    """The step's CUDA graphs are captured lazily on the SECOND step — while a real DataLoader's pin-memory thread is
    calling cudaHostAlloc / cudaEventQuery (the combination main_dgl.py runs: pin_memory=True, num_workers > 0).
    capture_error_mode="thread_local" keeps those foreign-thread calls legal.  6 steps: eager, capture, 4 replays."""
    from torch.utils.data import DataLoader, Dataset
    from gdl_b200.train import train_epoch
    from oracle.synth import SHAPES, make_batch

    class DS(Dataset):
        def __len__(self):
            return 24

        def __getitem__(self, i):
            spec, image, label = make_batch(1, 6, "tiny", seed=100 + i)
            return spec[0], image[0], label[0]

    args, model = make_model("concat")
    dp = _Wrap(model)
    opt = torch.optim.SGD(dp.parameters(), lr=0.01, momentum=0.9, weight_decay=1e-4)
    loader = DataLoader(DS(), batch_size=4, shuffle=False, num_workers=2, pin_memory=True, drop_last=True)
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        res = train_epoch(args, 0, dp, torch.device("cuda"), loader, opt, None)
        rows = list(csv.reader(open("audio_visual_grad_vanilla.csv")))
    finally:
        os.chdir(cwd)
    torch.cuda.synchronize()
    assert len(rows) == 6 and all(float(r[0]) > 0 and float(r[1]) > 0 for r in rows)
    assert all(x == x and 0 < x < 50 for x in res[:3])  # finite epoch-mean losses
    assert model._gdl_step.graphs                       # the captured path really ran


def test_train_epoch_with_a_short_tail_batch_shares_one_arena(tmp_path):
    """A loader WITHOUT drop_last (the train_epoch drop-in contract allows it): every epoch ends with a short batch.
    The two batch geometries get one cached DGLStep each (graphs, engines), both on ONE parameter / gradient /
    momentum arena — switching refreshes the weight shadows, nothing is re-allocated — and the run tracks the fp32
    oracle stepping through the same 4, 4, 2 | 4, 4, 2 sequence with one momentum state."""
    from torch.utils.data import DataLoader, Dataset
    from gdl_b200.train import train_epoch
    from oracle import dgl_oracle as O
    from oracle.synth import make_batch

    items = [make_batch(1, 6, "tiny", seed=300 + i) for i in range(10)]

    class DS(Dataset):
        def __len__(self):
            return len(items)

        def __getitem__(self, i):
            spec, image, label = items[i]
            return spec[0], image[0], label[0]

    args, model = make_model("concat")
    dp = _Wrap(model)
    opt = torch.optim.SGD(dp.parameters(), lr=0.01, momentum=0.9, weight_decay=1e-4)
    loader = DataLoader(DS(), batch_size=4, shuffle=False, num_workers=0, pin_memory=True, drop_last=False)
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        for epoch in range(2):
            res = train_epoch(args, epoch, dp, torch.device("cuda"), loader, opt, None)
    finally:
        os.chdir(cwd)
    torch.cuda.synchronize()
    steps = model._gdl_steps
    assert sorted(k[0] for k in steps) == [2, 4]
    a, b = steps.values()
    assert a.arena is b.arena and model._gdl_arena is a.arena
    assert a.steps_done + b.steps_done == 6
    for p in dp.parameters():  # the optimizer's momentum buffers alias the shared arena
        if p in opt.state:
            o = a.arena.offset_of[id(p)]
            assert opt.state[p]["momentum_buffer"].data_ptr() == a.arena.momentum.data_ptr() + 4 * o
    # oracle: same sequence, one state dict, one momentum dict
    sd, mom, last = O.init_state("concat", "CREMAD", 0), {}, None
    for epoch in range(2):
        tot, n = [0.0, 0.0, 0.0], 0
        for lo in (0, 4, 8):
            chunk = items[lo:lo + 4]
            batch = [torch.cat([c[j] for c in chunk]) for j in range(3)]
            r = O.dgl_step(sd, mom, *batch, fusion="concat", alpha=args.alpha, lr=0.01)
            tot = [t + float(x) for t, x in zip(tot, r["losses"])]
            n += 1
        last = [t / n for t in tot]
    print("tail-batch run: epoch-2 mean losses %s vs oracle %s" % (list(res[:3]), last))
    # six FREE-RUNNING steps at lr = 0.01 with BatchNorm over 2-4 samples: bf16 storage moves the unimodal losses by a few
    # per cent by then (measured 0.1 % / 2 % / 6 %); a wrong momentum or stale weight shadow after a switch shows up as
    # tens of per cent
    for g, r in zip(res[:3], last):
        assert abs(g - r) <= 1e-1 * abs(r), (res[:3], last)


def test_valid_with_folded_batchnorm_on_a_64_sample_test_set(tmp_path):
    """SURVEY.md §8f rank 1 (reference valid(), main_dgl.py:168-222): eval-mode forward with BatchNorm folded into
    the packed conv weights (one fused conv kernel per unit, no BN pass) on a 64-sample synthetic test set after a
    few training steps: logits within 2e-2 (relative L2) of the fp32 oracle's eval forward on the SAME weights /
    running statistics, (acc, acc_a, acc_v) equal (up to arg-max near-ties, counted), and the fold follows
    load_state_dict."""
    from gdl_b200.step import DGLStep
    from gdl_b200.train import valid
    from oracle import dgl_oracle as O
    from oracle.synth import SHAPES, make_batch
    args, model = make_model("concat")
    Fq, Tt, T, H, W = SHAPES["tiny"]
    step = DGLStep(model, 16, (Fq, Tt), (T, H, W), lr=0.01, use_graph=False)
    for s in range(4):  # non-trivial running statistics and weights
        step.step(*[t.cuda() for t in make_batch(16, 6, "tiny", seed=1 + s)])
    torch.cuda.synchronize()
    model.eval()
    batches = [make_batch(16, 6, "tiny", seed=50 + i) for i in range(4)]  # 64 samples
    msd = model.state_dict()
    sd_same = {k: v.detach().float().cpu() if v.is_floating_point() else v.detach().cpu() for k, v in msd.items()}
    correct = torch.zeros(3)
    worst, num, den, flips, sep_flips = 0.0, 0.0, 0.0, 0, 0
    with torch.no_grad():
        for spec, image, label in batches:
            got = model(spec.cuda().unsqueeze(1).float(), image.cuda().float())
            ref = O.model_forward(sd_same, spec, image, "concat", training=False)
            for i, (g, r) in enumerate(zip(got, ref)):
                d = g.cpu() - r
                worst = max(worst, d.abs().max().item() / r.abs().max().item())
                num, den = num + d.double().pow(2).sum().item(), den + r.double().pow(2).sum().item()
                correct[i] += (r.argmax(1) == label).sum()
                differ = g.cpu().argmax(1) != r.argmax(1)
                flips += int(differ.sum())
                # rows the fp32 reference separates by more than 2.5 % of its logit spread (tests/test_gpu_parity_at_size.py)
                top2 = r.topk(2, dim=1).values
                margin = (top2[:, 0] - top2[:, 1]) / (r.max(1).values - r.min(1).values)
                sep_flips += int((differ & (margin > 2.5e-2)).sum())
    acc = valid(args, _Wrap(model), torch.device("cuda"), batches)
    rel_l2 = (num / den) ** 0.5
    print("eval logits: relative L2 error %.4f, max |diff| / max |logit| %.4f, arg-max flips %d / 192; acc %s vs oracle %s"
          % (rel_l2, worst, flips, acc, (correct / 64).tolist()))
    # 17 layers of bf16 storage WITHOUT the per-batch renormalisation of training-mode BatchNorm: ~0.4 % rounding noise per
    # layer accumulates to 1-2 % of a logit (relative L2), a few % in the worst of the 1152 logits
    assert rel_l2 <= 2e-2 and worst <= 6e-2, (rel_l2, worst)
    assert sep_flips == 0 and flips <= 4, (sep_flips, flips)   # >= 98 % of all rows, every separable row
    if flips == 0:
        assert list(acc) == (correct / 64).tolist()
    else:
        assert all(abs(a - c) <= flips / 64 + 1e-9 for a, c in zip(acc, (correct / 64).tolist()))
    eng = model.audio_net.engine(16, Fq, Tt)
    assert hasattr(eng.stem, "wp_e") and eng._eval_key_folded is not None   # the folded path really ran
    # a changed state dict must re-fold: scaling every BN gamma of the audio encoder changes the audio logits
    sd2 = {k: (v * 1.5 if k.startswith("audio_net") and k.endswith("bn2.weight") else v) for k, v in msd.items()}
    before = model(batches[0][0].cuda().unsqueeze(1).float(), batches[0][1].cuda().float())[1].clone()
    model.load_state_dict(sd2)
    with torch.no_grad():
        after = model(batches[0][0].cuda().unsqueeze(1).float(), batches[0][1].cuda().float())[1]
        sd2c = {k: v.detach().float().cpu() if v.is_floating_point() else v.detach().cpu() for k, v in sd2.items()}
        ref2 = O.model_forward(sd2c, batches[0][0], batches[0][1], "concat", training=False)[1]
    assert (after - before).abs().max().item() > 1e-3
    assert (after.cpu() - ref2).abs().max().item() <= 6e-2 * ref2.abs().max().item()
