"""Host-side data-parallel logic (replaces the reference's torch.nn.DataParallel wrapper,
main_dgl.py:244): one process per GPU, contiguous batch shards in DataParallel `chunk` order,
per-replica BatchNorm, gradient SUM all-reduce of shards whose losses are scaled by 1/B_global
(== the reference's full-batch mean over gathered logits, main_dgl.py:102-104)."""
import torch
import torch.distributed as dist


def shard_range(rank, world, batch):
    """Rows [lo, hi) of the global batch owned by `rank` (torch.chunk order: rank 0 == reference
    device 0, which owns the persisted BN running statistics)."""
    per = (batch + world - 1) // world
    lo = min(rank * per, batch)
    return lo, min(lo + per, batch)


def replicas_per_rank(global_batch, replicas, world):
    """Data-parallel replicas each of `world` processes runs one after another: `replicas` (R) replicas of
    global_batch / R rows in torch.chunk order, R / world of them per process (rank r runs replicas
    r*R/world .. (r+1)*R/world - 1).  ValueError unless R divides the global batch and world divides R."""
    G, R, W = int(global_batch), int(replicas), int(world)
    if G < 1 or R < 1 or W < 1 or G % R or R % W:
        raise ValueError("batch_size {} must split into {} data-parallel replicas of equal size, and the replicas "
                         "evenly over {} processes".format(G, R, W))
    return R // W


def allreduce_sum_(flat, group=None):
    """In-place SUM all-reduce of a flat gradient arena (NCCL on GPUs, gloo in CPU tests)."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    return flat


def flatten_grads(grads, names):
    return torch.cat([grads[k].reshape(-1) for k in names])


def gradient_buckets(grad, cut_a, end_a, cut_v):
    """Views of the flat gradient arena (order: head | audio_net | visual_net | 3 losses) for the two-bucket
    all-reduce: `late` = layer3 + layer4 of both encoders (their gradients are final first, 94 % of the
    bytes) plus the loss tail, `early` = head + stem / layer1 / layer2.  cut_a / cut_v: arena offsets where
    layer3 of the audio / visual encoder starts; end_a: where the audio group ends."""
    assert 0 < cut_a < end_a < cut_v < grad.numel()
    return dict(late=[grad[cut_a:end_a], grad[cut_v:]], early=[grad[:cut_a], grad[end_a:cut_v]])


def allreduce_async(tensors, group=None):
    """Start SUM all-reduces that run on the backend's own stream beside whatever the caller enqueues next;
    returns the work handles (wait() makes the current stream — not the host — wait on NCCL)."""
    return [dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group, async_op=True) for t in tensors]


def allreduce_finish(works, tensors, group=None):
    """Join the asynchronous bucket, then all-reduce the remaining (small) tensors on the critical path."""
    for w in works:
        w.wait()
    for t in tensors:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)


def broadcast_running_stats(model, group=None):
    """Give every rank rank 0's BatchNorm running statistics (one broadcast of their concatenation).  This is what
    nn.DataParallel evaluates with: its replicas are copies of device 0's module and keep no statistics of their own."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return
    bufs = [b for m in model.modules() if isinstance(m, torch.nn.modules.batchnorm._BatchNorm)
            for b in (m.running_mean, m.running_var)]
    flat = torch.cat([b.reshape(-1) for b in bufs])
    dist.broadcast(flat, src=0, group=group)
    if dist.get_rank(group) != 0:  # rank 0 keeps its buffers untouched (and its BatchNorm fold valid)
        for b, v in zip(bufs, flat.split([b.numel() for b in bufs])):
            b.copy_(v.view_as(b))


class ChunkShardBatchSampler(torch.utils.data.Sampler):
    """Batch sampler for one rank of a data-parallel run that reproduces what nn.DataParallel does to the reference's
    DataLoader (main_dgl.py:244,284-288): ONE global sample order (any sampler — RandomSampler for shuffle=True,
    which draws its permutation seed from the global torch RNG at every epoch exactly like the reference's loader),
    cut into global batches of `global_batch` with drop_last=True, and each global batch split CONTIGUOUSLY in
    torch.chunk order: rank r yields rows [r*B/N, (r+1)*B/N) (shard_range).  So replica r's BatchNorm sees exactly
    the rows reference device r would see, and rank 0 == device 0.

    Every rank must build it over the same order: all ranks run the same script from the same seed, so their global
    RNGs — and hence the RandomSampler permutations — agree; `order_digest` lets the caller verify that with one
    tiny all-reduce per epoch."""

    def __init__(self, sampler, global_batch, rank, world):
        if global_batch % world:
            raise ValueError("batch_size {} is not divisible by the {} ranks".format(global_batch, world))
        self.sampler, self.B, self.rank, self.world = sampler, int(global_batch), int(rank), int(world)
        self.order_digest = None

    def __len__(self):
        return len(self.sampler) // self.B  # drop_last=True like every loader of the reference

    def __iter__(self):
        order = list(self.sampler)
        self.order_digest = sum((i + 1) * (int(v) % 65521) for i, v in enumerate(order[:4096])) % (1 << 31)
        lo, hi = shard_range(self.rank, self.world, self.B)
        for k in range(len(order) // self.B):
            yield order[k * self.B + lo:k * self.B + hi]


def assert_same_order(digest, group=None):
    """All ranks iterate the same global order (see ChunkShardBatchSampler): MIN == MAX of the digests."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1 or digest is None:
        return
    dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend(group) == "nccl" else torch.device("cpu")
    t = torch.tensor([digest, -digest], dtype=torch.int64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN, group=group)
    if int(t[0]) != -int(t[1]):
        raise RuntimeError("data-parallel ranks drew different sample orders (global RNG out of sync)")
