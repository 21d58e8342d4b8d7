"""Launched by torchrun (N ranks, one GPU each; N = 2 under pytest, 8 from tools/r2_dist8.sh): DGLStep data-parallel
vs the CPU oracle's N-shard simulation of nn.DataParallel (reference main_dgl.py:244: contiguous chunk r on replica
r, per-replica BatchNorm, CE over the gathered logits == shard sums scaled by 1/B_global, gradient reduce-add).
Runs the bf16 product path eagerly and through CUDA graphs (which must agree bit for bit), with the bucketed NCCL
all-reduce and with one all-reduce, and then the FP32 check mode, in which the N-rank result must equal the
simulation to fp32 accuracy: losses 1e-4, cosine >= 0.999 for every parameter tensor."""
import argparse
import os
import sys

import torch
import torch.distributed as dist
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "iccv2025-gdl_b200"))


def main():
    import gdl_b200
    from gdl_b200.parallel import shard_range
    from gdl_b200 import step as step_module
    from gdl_b200.step import DGLStep
    from oracle import dgl_oracle as O
    from oracle.synth import SHAPES, make_batch
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    B = 2 * world
    args = argparse.Namespace(dataset="CREMAD", fusion_method="concat", modality="full")
    Fq, Tt, T, H, W = SHAPES["tiny"]
    lo, hi = shard_range(rank, world, B)

    def run(check, use_graph):
        """3 steps; returns the stats, the parameters and the momentum."""
        gdl_b200.setup_seed(0)
        model = gdl_b200.AVClassifier_DGL(args)
        model.apply(gdl_b200.weight_init)
        model.to(dev).train()
        step = DGLStep(model, hi - lo, (Fq, Tt), (T, H, W), alpha=4.0, lr=0.01, world_size=world,
                       process_group=dist.group.WORLD, use_graph=use_graph, check_fp32=check)
        sd = O.init_state("concat", "CREMAD", 0)
        for s in range(3):  # with graphs: step 0 eager, steps 1-2 through the captured graphs + eager NCCL
            spec, image, label = make_batch(B, 6, "tiny", seed=1 + s)
            step.step(spec[lo:hi].to(dev), image[lo:hi].to(dev), label[lo:hi].to(dev))
            torch.cuda.synchronize()
            got = step.read_stats()
            # replicas stay identical
            chk = step.arena.param.double().sum().reshape(1)
            both = [torch.zeros_like(chk) for _ in range(world)]
            dist.all_gather(both, chk)
            if rank == 0:
                assert all(torch.equal(b, both[0]) for b in both), "replicas diverged"
                if s == 0:
                    total, losses = None, [0.0, 0.0, 0.0]
                    for r in range(world):
                        a, b = shard_range(r, world, B)
                        res = O.dgl_step({k: v.clone() for k, v in sd.items()}, {}, spec[a:b], image[a:b], label[a:b],
                                         fusion="concat", alpha=4.0, max_norm=1e9, inv_batch=1.0 / B, apply_update=False)
                        losses = [x + y for x, y in zip(losses, res["losses"])]
                        g = res["grads"]
                        total = g if total is None else {k: total[k] + g[k] for k in g}
                    ltol = 1e-4 if check else 2e-2
                    for gl, rl in zip(got[:3], losses):
                        assert abs(gl - rl) <= ltol * abs(rl), (check, got[:3], losses)
                    names = dict(model.named_parameters())
                    # grads in the arena are clipped: compare directions
                    keys = list(total) if check else ["fusion_module.fc_out.weight", "fusion_module.fc_out.bias"]
                    worst = min((F.cosine_similarity(names[k].grad.detach().float().cpu().flatten().double(),
                                                     total[k].flatten().double(), dim=0).item(), k) for k in keys)
                    assert worst[0] > (0.999 if check else 0.99), worst
                    norm = sum(float(v.double().pow(2).sum()) for v in total.values()) ** 0.5
                    assert abs(got[3] - norm) <= (1e-3 if check else 6e-2) * norm, (got[3], norm)
                    print("   vs the %d-shard oracle simulation: losses %s vs %s, min cos %.6f (%s), norm %.5g vs %.5g"
                          % (world, [round(x, 5) for x in got[:3]], [round(x, 5) for x in losses], worst[0], worst[1],
                             got[3], norm), flush=True)
                print("dist step %d ok (%s, %s, %d ranks, overlap %d): losses %s"
                      % (s, "fp32 check mode" if check else "bf16 product path", "graphs" if use_graph else "eager",
                         world, step.overlap, [round(x, 4) for x in got[:3]]), flush=True)
        return step.stats.clone(), step.arena.param.clone(), step.arena.momentum.clone()

    # the product path eagerly, then through the graphs (2 ranks: every sum of the all-reduce is order-exact), with
    # the two all-reduce buckets and with one all-reduce
    default = step_module.AR_OVERLAP
    for overlap in (True, False):
        step_module.AR_OVERLAP = overlap  # read by the DGLStep constructor
        eager, graphs = run(False, False), run(False, True)
        assert all(torch.equal(a, b) for a, b in zip(eager, graphs)), \
            "overlap %d: CUDA-graph steps differ from eager steps" % overlap
    step_module.AR_OVERLAP = default
    run(True, False)
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("DIST_STEP_CHECK_OK", flush=True)


if __name__ == "__main__":
    main()
