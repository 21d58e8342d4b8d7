"""Graph-captured validation (step.EvalStep, train.valid) and its eval head kernel (csrc/eval.cu).  GPU only."""
import argparse
import os

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def make_model(fusion="concat", dataset="CREMAD"):
    import gdl_b200
    args = argparse.Namespace(dataset=dataset, fusion_method=fusion, modality="full", alpha=4.0, epochs=1, drop=0)
    gdl_b200.setup_seed(0)
    m = gdl_b200.AVClassifier_DGL(args)
    m.apply(gdl_b200.weight_init)
    return args, m.cuda()


def trained(fusion, shape, B, steps=3):
    from gdl_b200.step import DGLStep
    from oracle.synth import SHAPES, make_batch
    args, model = make_model(fusion)
    Fq, Tt, T, H, W = SHAPES[shape]
    st = DGLStep(model, B, (Fq, Tt), (T, H, W), lr=0.01, use_graph=False)
    for s in range(steps):
        st.step(*[t.cuda() for t in make_batch(B, 6, shape, seed=1 + s)])
    torch.cuda.synchronize()
    return args, model


# ------------------------------------------------------------------------------------------------ the kernel
def _torch_head(kind, a, v, Wx, bx, Wy, by, Wo, bo, x_gate):
    if kind == 0:
        xa, yv = a @ Wx[:, :512].T, v @ Wx[:, 512:].T
        return (xa + yv) + bx, xa + bx, yv + bx
    if kind == 1:
        xa, yv = a @ Wx.T + bx, v @ Wy.T + by
        return xa + yv, xa, yv
    hx, hy = a @ Wx.T + bx, v @ Wy.T + by
    m = torch.sigmoid(hx) * hy if x_gate else torch.sigmoid(hy) * hx
    return m @ Wo.T + bo, (torch.sigmoid(hx) * hx) @ Wo.T + bo, (torch.sigmoid(hy) * hy) @ Wo.T + bo


@pytest.mark.parametrize("kind,x_gate", [(0, 1), (1, 1), (2, 1), (2, 0)])
def test_eval_head_kernel_against_torch(kind, x_gate):
    from gdl_b200 import ops
    g = torch.Generator().manual_seed(kind * 2 + x_gate)
    B, Ga, Gv, n = 37, 12, 3 * 49, 34
    fa = torch.randn(B, Ga, 512, generator=g).cuda().bfloat16()
    fv = torch.randn(B, Gv, 512, generator=g).cuda().bfloat16()
    r = lambda *s: (torch.randn(*s, generator=g) * 0.05).cuda()
    if kind == 0:
        Wx, bx, Wy, by, Wo, bo, ldw = r(n, 1024), r(n), None, None, None, None, 1024
        Wx[1], bx[1] = Wx[0], bx[0]  # columns 0 and 1 tie in every logit set
    elif kind == 1:
        Wx, bx, Wy, by, Wo, bo, ldw = r(n, 512), r(n), r(n, 512), r(n), None, None, 512
        Wx[1], bx[1], Wy[1], by[1] = Wx[0], bx[0], Wy[0], by[0]
    else:
        Wx, bx, Wy, by, Wo, bo, ldw = r(512, 512), r(512), r(512, 512), r(512), r(n, 512), r(n), 512
        Wo[1], bo[1] = Wo[0], bo[0]
    label = torch.randint(0, 3, (B,), generator=g).cuda()  # many rows land on the tied pair {0, 1}
    logits = torch.empty(3, B, n, device="cuda")
    a_out, v_out = torch.empty(B, 512, device="cuda"), torch.empty(B, 512, device="cuda")
    counts = torch.zeros(3, device="cuda", dtype=torch.int64)
    Wy_ptr = Wx.data_ptr() + 4 * 512 if kind == 0 else Wy.data_ptr()
    ops.eval_head(kind, fa, Ga, fv, Gv, Wx.data_ptr(), Wy_ptr, ldw, bx, by, Wo, bo, x_gate, label, a_out, v_out, logits,
                  counts, B, n)
    a, v = fa.float().mean(1), fv.float().mean(1)
    assert torch.allclose(a_out, a, rtol=1e-5, atol=1e-6) and torch.allclose(v_out, v, rtol=1e-5, atol=1e-6)
    ref = _torch_head(kind, a, v, Wx, bx, Wy, by, Wo, bo, x_gate)
    for h in range(3):
        err = (logits[h] - ref[h]).abs().max().item() / ref[h].abs().max().item()
        assert err <= 1e-5, (h, err)
        pred = logits[h].argmax(1)
        assert int(counts[h]) == int((pred == label).sum()), h
        assert bool((pred != 1).all())  # the lowest index wins the tie
    assert torch.equal(logits[:, :, 0], logits[:, :, 1])
    # the count step of the FiLM head agrees with the fused one on the same logits; labels < 0 never count
    c2 = torch.zeros(3, device="cuda", dtype=torch.int64)
    ops.eval_count(logits, label, c2, B, n)
    ops.eval_count(logits, torch.full_like(label, -1), c2, B, n)
    assert torch.equal(c2, counts)


# ------------------------------------------------------------------------------------------------ valid() vs oracle
@pytest.mark.parametrize("fusion", ["concat", "sum", "gated", "film"])
@pytest.mark.parametrize("shape,B", [("tiny", 16), ("CREMAD", 4)])
def test_valid_against_the_oracle_eval_forward(fusion, shape, B):
    from gdl_b200.step import get_eval_step
    from gdl_b200.train import valid
    from oracle import dgl_oracle as O
    from oracle.synth import SHAPES, make_batch
    args, model = trained(fusion, shape, B)
    batches = [make_batch(B, 6, shape, seed=50 + i) for i in range(2)]
    msd = model.state_dict()
    sd = {k: v.detach().float().cpu() if v.is_floating_point() else v.detach().cpu() for k, v in msd.items()}
    acc = valid(args, model, torch.device("cuda"), batches)
    Fq, Tt, T, H, W = SHAPES[shape]
    last = get_eval_step(model, B, (Fq, Tt), (T, H, W)).logits.clone()
    num = den = 0.0
    worst, flips, sep_flips, correct = 0.0, 0, 0, torch.zeros(3)
    model.eval()
    with torch.no_grad():
        for spec, image, label in batches:
            got = model(spec.cuda().unsqueeze(1).float(), image.cuda().float())
            ref = O.model_forward(sd, spec, image, fusion, training=False)
            for i, (gg, r) in enumerate(zip(got, ref)):
                d = gg.cpu() - r
                worst = max(worst, d.abs().max().item() / r.abs().max().item())
                num, den = num + d.double().pow(2).sum().item(), den + r.double().pow(2).sum().item()
                correct[i] += (gg.argmax(1).cpu() == label).sum()
                differ = gg.cpu().argmax(1) != r.argmax(1)
                flips += int(differ.sum())
                top2 = r.topk(2, dim=1).values
                margin = (top2[:, 0] - top2[:, 1]) / (r.max(1).values - r.min(1).values)
                sep_flips += int((differ & (margin > 2.5e-2)).sum())
    assert torch.equal(torch.stack(got), last)  # valid() and model(...) share one arithmetic
    assert list(acc) == [c / (2 * B) for c in correct.tolist()]
    rel_l2 = (num / den) ** 0.5
    print("%s %s: rel L2 %.4f, worst %.4f, flips %d" % (fusion, shape, rel_l2, worst, flips))
    assert rel_l2 <= 2e-2 and worst <= 6e-2, (rel_l2, worst)
    assert sep_flips == 0 and flips <= 4, (sep_flips, flips)


def test_gated_x_gate_false_follows_the_module():
    from oracle.synth import make_batch
    args, model = trained("gated", "tiny", 8, steps=1)
    model.eval()
    spec, image, _ = make_batch(8, 6, "tiny", seed=5)
    spec, image = spec.cuda().unsqueeze(1), image.cuda()
    with torch.no_grad():
        on = model(spec, image)[0].clone()
        model.fusion_module.x_gate = False
        off = model(spec, image)
        fm = model.fusion_module
        a = F.adaptive_avg_pool2d(model.audio_net(spec), 1).flatten(1)
        v = model.visual_net(image)
        v = v.reshape(8, -1, 512, v.shape[2], v.shape[3]).mean((1, 3, 4))
        hx, hy = F.linear(a, fm.fc_x.weight, fm.fc_x.bias), F.linear(v, fm.fc_y.weight, fm.fc_y.bias)
        ref = F.linear(torch.sigmoid(hy) * hx, fm.fc_out.weight, fm.fc_out.bias)
    assert not torch.equal(on, off[0])
    assert (off[0] - ref).abs().max().item() <= 1e-4 * ref.abs().max().item() + 1e-6


# ------------------------------------------------------------------------------------------------ graphs and caching
@pytest.mark.parametrize("fusion", ["concat", "film"])
def test_eval_graph_replay_is_bit_identical_to_eager(fusion):
    from gdl_b200.step import EvalStep, eval_counts
    from oracle.synth import SHAPES, make_batch
    args, model = trained(fusion, "tiny", 8, steps=1)
    model.eval()
    Fq, Tt, T, H, W = SHAPES["tiny"]
    counts = eval_counts(model, torch.device("cuda"))
    res = {}
    for use_graph in (False, True):
        ev = EvalStep(model, 16, (Fq, Tt), (T, H, W), use_graph=use_graph)
        counts.zero_()
        outs = []
        for i in range(3):
            spec, image, label = make_batch(16, 6, "tiny", seed=70 + i)
            ev.load_inputs(spec, image, label)
            out = torch.empty(3, 16, model.n_classes, device="cuda")
            ev.run(out)
            outs.append(out)
        res[use_graph] = (torch.stack(outs), counts.clone())
        assert bool(ev.graphs) == use_graph
    assert torch.equal(res[False][0], res[True][0]) and torch.equal(res[False][1], res[True][1])


def test_fold_is_cached_and_follows_training_and_load_state_dict():
    from gdl_b200 import ops
    from gdl_b200.step import DGLStep
    from gdl_b200.train import valid
    from oracle.synth import SHAPES, make_batch
    args, model = make_model("concat")
    Fq, Tt, T, H, W = SHAPES["tiny"]
    st = DGLStep(model, 8, (Fq, Tt), (T, H, W), lr=0.01)
    for s in range(2):
        st.step(*[t.cuda() for t in make_batch(8, 6, "tiny", seed=1 + s)])
    batches = [make_batch(8, 6, "tiny", seed=80 + i) for i in range(3)]
    dev = torch.device("cuda")

    def launches():
        n0 = ops.LAUNCHES
        acc = valid(args, model, dev, batches)
        torch.cuda.synchronize()
        return ops.LAUNCHES - n0, acc

    launches()
    n2, acc2 = launches()
    n3, acc3 = launches()
    assert n2 == n3 == 2 * len(batches), (n2, n3)  # the two stem layouts per batch; no fold, no pack, graph replays
    assert acc2 == acc3

    def fresh_logits():
        _, m2 = make_model("concat")
        m2.load_state_dict(model.state_dict())
        m2.eval()
        spec, image, _ = batches[0]
        return m2(spec.cuda().unsqueeze(1), image.cuda())[0]

    def logits():
        model.eval()
        spec, image, _ = batches[0]
        return model(spec.cuda().unsqueeze(1), image.cuda())[0]

    before = logits().clone()
    model.train()
    st.step(*[t.cuda() for t in make_batch(8, 6, "tiny", seed=9)])  # a graph replay: nothing bumps torch's versions
    n4, _ = launches()
    assert n4 > n3  # re-folded
    after = logits()
    assert not torch.equal(before, after)
    assert torch.equal(after, fresh_logits())
    sd = {k: (v * 1.25 if k.endswith("bn1.weight") else v) for k, v in model.state_dict().items()}
    model.load_state_dict(sd)
    assert torch.equal(logits(), fresh_logits())


@pytest.mark.parametrize("dp_replicas", [0, 2])
def test_second_epoch_reuses_every_graph_and_allocates_nothing(tmp_path, dp_replicas):
    from gdl_b200.train import train_epoch, valid
    from oracle.synth import make_batch
    args, model = make_model("concat")
    args.batch_size, args.dp_replicas = 8, dp_replicas
    opt = torch.optim.SGD(model.parameters(), lr=0.01, momentum=0.9, weight_decay=1e-4)
    train = [make_batch(8, 6, "tiny", seed=1 + s) for s in range(3)]
    test = [make_batch(8, 6, "tiny", seed=90 + s) for s in range(3)]
    dev = torch.device("cuda")
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        train_epoch(args, 0, model, dev, train, opt, None)
        valid(args, model, dev, test)
        torch.cuda.synchronize()
        st = model._gdl_step
        evs = dict(model._gdl_evals)
        graphs = [dict(st.graphs)] + [dict(e.graphs) for e in evs.values()]
        mem = torch.cuda.memory_allocated()
        train_epoch(args, 1, model, dev, train, opt, None)
        acc = valid(args, model, dev, test)
        torch.cuda.synchronize()
    finally:
        os.chdir(cwd)
    assert model._gdl_step is st and dict(model._gdl_evals) == evs
    assert [dict(st.graphs)] + [dict(e.graphs) for e in evs.values()] == graphs and all(graphs)
    assert torch.cuda.memory_allocated() == mem
    ev = next(iter(evs.values()))
    assert ev.enc_a is st.enc_a and ev.B == st.B == 8 // max(dp_replicas, 1)  # sub-batches of the training geometry
    assert all(0.0 <= a <= 1.0 for a in acc)


def test_device_pipeline_and_short_tail_batch():
    from torch.utils.data import DataLoader
    from gdl_b200.synthetic import SyntheticCramedDevice
    from gdl_b200.train import valid
    args, model = make_model("concat")
    args.fps, args.use_video_frames = 2, 3
    ds = SyntheticCramedDevice(args, "test", 10)
    ds.attach_pipeline(torch.device("cuda"))
    loader = DataLoader(ds, batch_size=4, shuffle=False, num_workers=0, drop_last=False)  # 4, 4, 2
    acc = valid(args, model, torch.device("cuda"), loader)
    correct, total = torch.zeros(3), 0
    model.eval()
    with torch.no_grad():
        for params, boxes, label in loader:
            spec = ds.device_audio_pipeline(params.cuda())
            image = ds.device_pipeline(boxes.reshape(-1, 6).cuda())
            out = model(spec.unsqueeze(1), image)
            for i, o in enumerate(out):
                correct[i] += (o.argmax(1).cpu() == label).sum()
            total += label.shape[0]
    assert total == 10
    assert list(acc) == [c / total for c in correct.tolist()]


def test_two_gpus_evaluate_shards():
    """torchrun, 2 ranks (tests/dist_eval_check.py)."""
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = os.path.join(os.path.dirname(__file__), "dist_eval_check.py")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29537", script],
                       capture_output=True, text=True, timeout=900)
    assert "DIST_EVAL_CHECK_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
