"""Launched by torchrun (2 ranks, one GPU each) from tests/test_gpu_replicas.py: data-parallel replicas run one after
another on each GPU (DGLStep replicas).
  1. W = 2, R = 4 (two replicas per rank): the FP32 check mode against the oracle's 4-shard simulation of
     nn.DataParallel (losses 1e-4, cosine >= 0.999 for every parameter tensor, grad norm 1e-3, rank 0's running
     statistics == shard 0's), then 3 steps of the bf16 product path (graphs + bucketed all-reduce): ranks agree.
  2. W = 2, R = 2 (one replica per rank) is bit-identical after 3 steps to one GPU running R = 2: a sum of two fp32
     terms does not depend on their order."""
import argparse
import os
import sys

import torch
import torch.distributed as dist
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "iccv2025-gdl_b200"))


def _model(dev):
    import gdl_b200
    args = argparse.Namespace(dataset="CREMAD", fusion_method="concat", modality="full")
    gdl_b200.setup_seed(0)
    model = gdl_b200.AVClassifier_DGL(args)
    model.apply(gdl_b200.weight_init)
    return model.to(dev).train()


def _agree(t, world):
    both = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(both, t)
    return all(torch.equal(b, both[0]) for b in both)


def main():
    from gdl_b200.parallel import replicas_per_rank, shard_range
    from gdl_b200.step import DGLStep
    from oracle import dgl_oracle as O
    from oracle.synth import SHAPES, make_batch
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    Fq, Tt, T, H, W = SHAPES["tiny"]
    b = 2

    # 1. R = 4
    R = 4
    G = R * b
    rl = replicas_per_rank(G, R, world)
    lo, hi = shard_range(rank, world, G)
    for check in (True, False):
        model = _model(dev)
        step = DGLStep(model, b, (Fq, Tt), (T, H, W), alpha=4.0, lr=0.01, world_size=world,
                       process_group=dist.group.WORLD, check_fp32=check, replicas=rl)
        for s in range(1 if check else 3):
            spec, image, label = make_batch(G, 6, "tiny", seed=1 + s)
            step.step(spec[lo:hi].to(dev), image[lo:hi].to(dev), label[lo:hi].to(dev))
            torch.cuda.synchronize()
            got = step.read_stats()
            assert _agree(step.arena.param.double().sum().reshape(1), world), "ranks diverged"
            if check and rank == 0:
                sd = O.init_state("concat", "CREMAD", 0)
                losses, total = [0.0, 0.0, 0.0], None
                for k in range(R):
                    res = O.dgl_step(sd, {}, spec[k * b:(k + 1) * b], image[k * b:(k + 1) * b],
                                     label[k * b:(k + 1) * b], fusion="concat", alpha=4.0, max_norm=1e9,
                                     inv_batch=1.0 / G, apply_update=False)
                    losses = [x + y for x, y in zip(losses, res["losses"])]
                    total = res["grads"] if total is None else {n: res["grads"][n] + total[n] for n in total}
                nb = {}
                with torch.no_grad():
                    O.model_forward(sd, spec[:b], image[:b], "concat", True, None, True, nb)
                for gl, rl_ in zip(got[:3], losses):
                    assert abs(gl - rl_) <= 1e-4 * abs(rl_), (got[:3], losses)
                names, bufs = dict(model.named_parameters()), dict(model.named_buffers())
                worst = min((F.cosine_similarity(names[k].grad.detach().float().cpu().flatten().double(),
                                                 total[k].flatten().double(), dim=0).item(), k) for k in total)
                assert worst[0] >= 0.999, worst
                norm = sum(float(v.double().pow(2).sum()) for v in total.values()) ** 0.5
                assert abs(got[3] - norm) <= 1e-3 * norm, (got[3], norm)
                for k, v in nb.items():
                    if k.endswith("tracked"):
                        assert int(bufs[k]) == 1, k
                    else:
                        assert torch.allclose(bufs[k].detach().cpu(), v, rtol=1e-4, atol=1e-5), k
                print("W=%d R=%d check mode vs the %d-shard oracle simulation: losses %s vs %s, min cos %.6f (%s), "
                      "norm %.6g vs %.6g" % (world, R, R, [round(x, 6) for x in got[:3]],
                                             [round(x, 6) for x in losses], worst[0], worst[1], got[3], norm),
                      flush=True)
        if rank == 0:
            print("W=%d R=%d %s ok: losses %s, launches/step %s" % (world, R, "fp32 check mode" if check else
                                                                    "bf16 product path", [round(x, 4) for x in got[:3]],
                                                                    step.launches_per_step), flush=True)
        del model, step

    # 2. R = 2: two ranks with one replica each == one GPU with two replicas
    R = 2
    G = R * b
    lo, hi = shard_range(rank, world, G)
    batches = [make_batch(G, 6, "tiny", seed=10 + s) for s in range(3)]
    model = _model(dev)
    step = DGLStep(model, b, (Fq, Tt), (T, H, W), alpha=4.0, lr=0.01, world_size=world,
                   process_group=dist.group.WORLD, replicas=replicas_per_rank(G, R, world))
    for spec, image, label in batches:
        step.step(spec[lo:hi].to(dev), image[lo:hi].to(dev), label[lo:hi].to(dev))
    torch.cuda.synchronize()
    if rank == 0:
        one = _model(dev)
        st1 = DGLStep(one, b, (Fq, Tt), (T, H, W), alpha=4.0, lr=0.01, replicas=R)
        for batch in batches:
            st1.step(*[t.to(dev) for t in batch])
        torch.cuda.synchronize()
        assert step.read_stats() == st1.read_stats(), (step.read_stats(), st1.read_stats())
        assert torch.equal(step.arena.param, st1.arena.param), "W=2 R=2 differs from one GPU with R=2"
        b1 = dict(one.named_buffers())
        assert all(torch.equal(v, b1[k]) for k, v in model.named_buffers()), "running statistics differ"
        print("W=%d R=%d bit-identical to one GPU with R=%d after 3 steps" % (world, R, R), flush=True)
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("DIST_REPLICA_CHECK_OK", flush=True)


if __name__ == "__main__":
    main()
