"""Launched by torchrun (2 ranks, one GPU each) from tests/test_gpu_eval.py: data-parallel validation.
  1. main_dgl.py --train for 2 epochs: both ranks see the same accuracies, hence the same best_acc.
  2. valid() over a ChunkShardBatchSampler test loader after training with per-rank BatchNorm statistics: each rank
     evaluates G/2 rows per global batch, both ranks return the same accuracy, and it equals a one-GPU evaluation of
     the same global batches with rank 0's weights and running statistics."""
import argparse
import os
import sys
import tempfile

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "iccv2025-gdl_b200"))


def _gather(obj, world):
    out = [None] * world
    dist.all_gather_object(out, obj)
    return out


def main():
    import main_dgl
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    work = os.path.join(tempfile.gettempdir(), "gdl_dist_eval_%s" % os.environ.get("MASTER_PORT", "0"))
    os.makedirs(work, exist_ok=True)
    os.chdir(work)  # train_epoch appends its gradient CSV to the working directory

    # 1. the CLI (it initialises the process group)
    seen = []
    valid = main_dgl.valid

    def recording_valid(*a):
        seen.append(valid(*a))
        return seen[-1]
    main_dgl.valid = recording_valid
    main_dgl.main(["--train", "--ckpt_path", os.path.join(work, "ckpt"), "--dataset", "CREMAD", "--audio_path",
                   "synthetic", "--batch_size", "8", "--epochs", "2", "--synthetic_len", "128",
                   "--fusion_method", "concat"])
    main_dgl.valid = valid
    both = _gather(seen, world)
    assert len(seen) == 2 and all(s == both[0] for s in both), both
    if rank == 0:
        print("main_dgl --train, 2 epochs: accuracies on both ranks %s" % (seen,), flush=True)

    # 2. valid() on a sharded loader
    import gdl_b200
    from gdl_b200.parallel import ChunkShardBatchSampler, shard_range
    from gdl_b200.step import DGLStep
    from gdl_b200.train import valid as gdl_valid
    from oracle.synth import SHAPES, make_batch
    dev = torch.device("cuda", local)
    Fq, Tt, T, H, W = SHAPES["tiny"]
    G = 8
    args = argparse.Namespace(dataset="CREMAD", fusion_method="concat", modality="full", alpha=4.0, drop=0)
    gdl_b200.setup_seed(0)
    model = gdl_b200.AVClassifier_DGL(args)
    model.apply(gdl_b200.weight_init)
    model.to(dev)
    lo, hi = shard_range(rank, world, G)
    st = DGLStep(model, G // world, (Fq, Tt), (T, H, W), lr=0.01, world_size=world, process_group=dist.group.WORLD)
    for s in range(3):
        spec, image, label = make_batch(G, 6, "tiny", seed=1 + s)
        st.step(spec[lo:hi].to(dev), image[lo:hi].to(dev), label[lo:hi].to(dev))
    torch.cuda.synchronize()
    rm = model.audio_net.layer1[0].bn1.running_mean.clone()
    differ = _gather(rm.cpu(), world)
    assert not torch.equal(differ[0], differ[1])  # each rank's running statistics come from its own shard
    sd0 = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()} if rank == 0 else None

    n = 44  # 5 global batches of 8; the reference drops the last 4 samples
    spec, image, label = make_batch(n, 6, "tiny", seed=123)
    ds = torch.utils.data.TensorDataset(spec, image, label)
    loader = torch.utils.data.DataLoader(
        ds, batch_sampler=ChunkShardBatchSampler(torch.utils.data.SequentialSampler(ds), G, rank, world))
    assert all(b[2].shape[0] == G // world for b in loader)
    acc = gdl_valid(args, model, dev, loader)
    accs = _gather(acc, world)
    assert all(a == accs[0] for a in accs), accs
    rm_after = _gather(model.audio_net.layer1[0].bn1.running_mean.cpu(), world)
    assert torch.equal(rm_after[0], rm_after[1])  # rank 0's statistics everywhere
    if rank == 0:
        gdl_b200.setup_seed(0)
        one = gdl_b200.AVClassifier_DGL(args)
        one.to(dev)
        one.load_state_dict(sd0)
        # the same global batches (floor(n / G) * G samples), in sub-batches of G / world rows like the ranks
        half = G // world
        batches = [(spec[i:i + half], image[i:i + half], label[i:i + half]) for i in range(0, n // G * G, half)]
        ref = gdl_valid(args, one, dev, batches)
        assert tuple(acc) == tuple(ref), (acc, ref)
        print("W=%d sharded valid(): accuracy %s on both ranks == one GPU with rank 0's state %s" % (world, acc, ref),
              flush=True)
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("DIST_EVAL_CHECK_OK", flush=True)


if __name__ == "__main__":
    main()
