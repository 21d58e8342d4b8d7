"""Launched by torchrun (2 ranks, one GPU each) from tests/test_gpu_lr_schedule.py: a per-step lr on the data-parallel
step with the bucketed gradient all-reduce and the CUDA graphs.  5 steps, a different lr each: every graph is
captured once (the same CUDAGraph objects from step 2 on), the ranks hold bit-identical parameters and momentum after
every step, and the graph replays equal eager steps bit for bit."""
import argparse
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "iccv2025-gdl_b200"))


def _agree(t, world):
    both = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(both, t)
    return all(torch.equal(b, both[0]) for b in both)


def main():
    import gdl_b200
    from gdl_b200.parallel import shard_range
    from gdl_b200.step import DGLStep
    from oracle.synth import SHAPES, make_batch
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    Fq, Tt, T, H, W = SHAPES["tiny"]
    b = 2
    G = b * world
    lo, hi = shard_range(rank, world, G)
    batches = [make_batch(G, 6, "tiny", seed=20 + s) for s in range(5)]
    lrs = [0.004, 0.02, 0.011, 0.003, 0.0005]
    out = []
    for use_graph in (False, True):
        gdl_b200.setup_seed(0)
        model = gdl_b200.AVClassifier_DGL(argparse.Namespace(dataset="CREMAD", fusion_method="concat",
                                                             modality="full"))
        model.apply(gdl_b200.weight_init)
        model.to(dev).train()
        st = DGLStep(model, b, (Fq, Tt), (T, H, W), alpha=4.0, lr=0.5, world_size=world,
                     process_group=dist.group.WORLD, use_graph=use_graph)
        assert st.overlap, "the bucketed all-reduce is the default at N > 1"
        seen = None
        for s, (spec, image, label) in enumerate(batches):
            st.step(spec[lo:hi].to(dev), image[lo:hi].to(dev), label[lo:hi].to(dev), lr=lrs[s])
            torch.cuda.synchronize()
            assert _agree(st.arena.param, world) and _agree(st.arena.momentum, world), "ranks diverged"
            if use_graph and s >= 1:
                ids = {k: id(g) for k, g in st.graphs.items()}
                assert ids and (seen is None or ids == seen), "a graph was captured again at step %d" % (s + 1)
                seen = ids
        out.append((st.read_stats(), st.arena.param.clone(), st.arena.momentum.clone()))
        if rank == 0:
            print("W=%d per-step lr, %s: losses %s, graphs %d" % (world, "graphs" if use_graph else "eager",
                                                                  [round(x, 5) for x in out[-1][0][:3]],
                                                                  len(st.graphs)), flush=True)
        del model, st
    assert out[0][0] == out[1][0], (out[0][0], out[1][0])
    assert torch.equal(out[0][1], out[1][1]) and torch.equal(out[0][2], out[1][2]), "graph replays differ from eager"
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("DIST_LR_CHECK_OK", flush=True)


if __name__ == "__main__":
    main()
