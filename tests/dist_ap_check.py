"""Launched by torchrun (2 ranks, one GPU each) from tests/test_gpu_eval_ap.py: data-parallel average precision.
valid_report(ap=True) over a ChunkShardBatchSampler test loader after training with per-rank BatchNorm statistics:
each rank evaluates G/2 rows per global batch, the score stores are gathered, and every rank computes the AP of all
the rows.  Checks: the AP is bit-identical on every rank, it equals sklearn on the gathered scores, and the AP and the
top-5 hits equal a one-GPU valid_report(ap=True) of the same rows with rank 0's weights and running statistics."""
import argparse
import os
import sys
import warnings

import numpy as np
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
    from sklearn.metrics import average_precision_score
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
    sd0 = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()} if rank == 0 else None

    n = 44  # 5 global batches of 8; the reference drops the last 4 samples
    spec, image, label = make_batch(n, 6, "tiny", seed=321)
    ds = torch.utils.data.TensorDataset(spec, image, label)
    loader = torch.utils.data.DataLoader(
        ds, batch_sampler=ChunkShardBatchSampler(torch.utils.data.SequentialSampler(ds), G, rank, world))
    rep = valid_report(args, model, dev, loader, ap=True)
    acc = valid(args, model, dev, loader)
    assert (rep.acc, rep.acc_a, rep.acc_v) == acc, (rep.acc, rep.acc_a, rep.acc_v, acc)
    rows = n // G * G
    assert rep.total == rows
    reps = _gather((rep.ap.view(torch.int64), rep.hits, rep.nonfinite), world)
    assert all(torch.equal(a, reps[0][0]) and torch.equal(h, reps[0][1]) for a, h, _ in reps), reps
    # sklearn on the gathered scores
    g = model._gdl_eval_scores.gathered
    assert int(g.cursor) == rows
    scores, labels = g.store[:, :, :rows].cpu().double().numpy(), g.labels[:rows].cpu().numpy()
    assert sorted(labels.tolist()) == sorted(label[:rows].tolist())
    present = np.unique(labels)
    onehot = (labels[:, None] == present[None, :]).astype(np.int64)
    for h in range(3):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ref = average_precision_score(onehot, scores[h][present].T, average=None)
        got = rep.ap[h].numpy()
        assert np.max(np.abs(got[present] - ref)) <= 1e-12, (h, got, ref)
        assert np.isnan(np.delete(got, present)).all()
    if rank == 0:
        gdl_b200.setup_seed(0)
        one = gdl_b200.AVClassifier_DGL(args)
        one.to(dev)
        one.load_state_dict(sd0)
        half = G // world
        batches = [(spec[i:i + half], image[i:i + half], label[i:i + half]) for i in range(0, rows, half)]
        ref = valid_report(args, one, dev, batches, ap=True)
        assert torch.equal(rep.hits, ref.hits) and rep.total == ref.total, (rep.hits, ref.hits)
        assert torch.equal(rep.ap.view(torch.int64), ref.ap.view(torch.int64)), (rep.ap, ref.ap)
        print("W=%d sharded valid_report(ap=True): the same %d-row AP on both ranks == sklearn on the gathered scores "
              "== one GPU with rank 0's state; mAP %s, top-5 %s" % (world, rep.total, rep.map, rep.top5), flush=True)
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("DIST_AP_CHECK_OK", flush=True)


if __name__ == "__main__":
    main()
