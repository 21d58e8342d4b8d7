"""Launched by torchrun (2 ranks, one GPU each) from tests/test_gpu_eval_report.py: data-parallel per-class validation.
valid_report() over a ChunkShardBatchSampler test loader after training with per-rank BatchNorm statistics: each rank
evaluates G/2 rows per global batch, every rank returns the same confusion matrices, and they equal a one-GPU
valid_report() of the same floor(n/G)*G samples with rank 0's weights and running statistics."""
import argparse
import os
import sys

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
    import gdl_b200
    from gdl_b200.parallel import ChunkShardBatchSampler, shard_range
    from gdl_b200.step import DGLStep
    from gdl_b200.train import valid, valid_report
    from oracle.synth import SHAPES, make_batch
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
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
    differ = _gather(model.audio_net.layer1[0].bn1.running_mean.cpu(), world)
    assert not torch.equal(differ[0], differ[1])  # each rank's running statistics come from its own shard
    sd0 = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()} if rank == 0 else None

    n = 44  # 5 global batches of 8; the reference drops the last 4 samples
    spec, image, label = make_batch(n, 6, "tiny", seed=321)
    ds = torch.utils.data.TensorDataset(spec, image, label)
    loader = torch.utils.data.DataLoader(
        ds, batch_sampler=ChunkShardBatchSampler(torch.utils.data.SequentialSampler(ds), G, rank, world))
    rep = valid_report(args, model, dev, loader)
    acc = valid(args, model, dev, loader)
    assert (rep.acc, rep.acc_a, rep.acc_v) == acc, (rep.acc, rep.acc_a, rep.acc_v, acc)
    reps = _gather((rep.confusion, rep.total), world)
    assert all(torch.equal(c, reps[0][0]) and t == reps[0][1] for c, t in reps), reps
    assert rep.total == n // G * G
    assert torch.equal(rep.support, torch.bincount(label[:n // G * G], minlength=model.n_classes))
    if rank == 0:
        gdl_b200.setup_seed(0)
        one = gdl_b200.AVClassifier_DGL(args)
        one.to(dev)
        one.load_state_dict(sd0)
        half = G // world
        batches = [(spec[i:i + half], image[i:i + half], label[i:i + half]) for i in range(0, n // G * G, half)]
        ref = valid_report(args, one, dev, batches)
        assert torch.equal(rep.confusion, ref.confusion) and rep.total == ref.total
        print("W=%d sharded valid_report(): the same %d-sample confusion matrices on both ranks == one GPU with rank "
              "0's state; accuracies %s" % (world, rep.total, acc), flush=True)
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("DIST_REPORT_CHECK_OK", flush=True)


if __name__ == "__main__":
    main()
