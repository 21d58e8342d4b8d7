"""Data-parallel validation on the host side: the sharded test sampler main_dgl.py builds at W > 1."""
import torch

from gdl_b200.parallel import ChunkShardBatchSampler


def test_sharded_test_sampler_covers_the_reference_samples_in_order():
    """The reference's test loader (batch_size G, drop_last, no shuffle) evaluates floor(n/G)*G samples in order;
    DataParallel splits every batch into contiguous chunks.  Over all ranks the sharded sampler yields exactly those
    samples: global batch k is rank 0's chunk, then rank 1's, ..."""
    for n, G, W in ((64, 16, 2), (70, 16, 2), (100, 24, 4), (23, 8, 8), (7, 8, 2)):
        ds = list(range(n))
        ranks = [list(ChunkShardBatchSampler(torch.utils.data.SequentialSampler(ds), G, r, W)) for r in range(W)]
        assert all(len(b) == n // G for b in ranks)
        assert all(len(chunk) == G // W for b in ranks for chunk in b)
        merged = [i for k in range(n // G) for r in range(W) for i in ranks[r][k]]
        assert merged == list(range(n // G * G)), (n, G, W)
