"""Data-parallel replicas run one after another on one GPU (`main_dgl.py --dp_replicas`, DGLStep replicas): the host-side
validation of the replica count against the batch size and the number of processes, and the flag's default.  No GPU."""
import argparse
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("G,R,W,local", [(512, 8, 1, 8), (512, 2, 1, 2), (512, 8, 8, 1), (8, 4, 2, 2), (6, 3, 3, 1)])
def test_replicas_per_rank(G, R, W, local):
    from gdl_b200.parallel import replicas_per_rank
    assert replicas_per_rank(G, R, W) == local


@pytest.mark.parametrize("G,R,W", [(10, 4, 1), (512, 3, 1), (512, 4, 8), (8, 4, 3), (8, 0, 1), (0, 2, 1)])
def test_indivisible_replicas_raise_naming_the_numbers(G, R, W):
    from gdl_b200.parallel import replicas_per_rank
    with pytest.raises(ValueError) as e:
        replicas_per_rank(G, R, W)
    msg = str(e.value)
    assert all(str(x) in msg for x in (G, R, W)), msg


def test_flag_default_is_one_replica_per_process():
    sys.path.insert(0, ROOT)
    import main_dgl
    assert main_dgl.get_arguments(["--ckpt_path", "x"]).dp_replicas == 0
    assert main_dgl.get_arguments(["--ckpt_path", "x", "--dp_replicas", "8"]).dp_replicas == 8


@pytest.mark.parametrize("G,R,W", [(10, 4, 1), (8, 4, 3)])
def test_main_dgl_rejects_indivisible_replicas(tmp_path, monkeypatch, G, R, W):
    """Raised before any device, dataset or process-group work."""
    sys.path.insert(0, ROOT)
    import main_dgl
    monkeypatch.setenv("WORLD_SIZE", str(W))
    with pytest.raises(ValueError, match="batch_size {} ".format(G)):
        main_dgl.main(["--train", "--ckpt_path", str(tmp_path), "--batch_size", str(G), "--dp_replicas", str(R),
                       "--audio_path", "synthetic"])


def _get_step_args(batch_size, dp_replicas):
    return argparse.Namespace(batch_size=batch_size, dp_replicas=dp_replicas, alpha=4.0)


def test_train_rejects_indivisible_replicas():
    from gdl_b200.train import _get_step
    spec, image = torch.zeros(8, 4, 4), torch.zeros(8, 3, 1, 4, 4)
    with pytest.raises(ValueError, match="batch_size 8 "):
        _get_step(_get_step_args(8, 3), torch.nn.Module(), None, spec, image)


def test_train_rejects_a_batch_that_does_not_split_into_the_replicas():
    """A short last batch (a loader without drop_last) of 6 rows cannot be 4 equal replicas."""
    from gdl_b200.train import _get_step
    spec, image = torch.zeros(6, 4, 4), torch.zeros(6, 3, 1, 4, 4)
    with pytest.raises(ValueError, match="6 rows"):
        _get_step(_get_step_args(8, 4), torch.nn.Module(), None, spec, image)


@pytest.mark.parametrize("R", [1, 2, 3])
@pytest.mark.parametrize("W", [1, 2])
@pytest.mark.parametrize("overlap", [True, False])
def test_step_schedule_and_its_graphs(R, W, overlap):
    """DESIGN.md §5: replica k < R-1 is [layout k] then graph(compute k + accumulate), replicas 1 .. R-2 sharing one
    graph; then the last replica: W = 1 one graph with the update; W > 1 NCCL between graphs, with the two buckets
    graph(forward + late backward) -> bucket 1 -> graph(early backward) -> bucket 2 -> graph(update), without them
    graph(compute) -> all-reduce -> graph(update)."""
    from gdl_b200.step import DEVICE, graph_runs, schedule
    seq = schedule(R, W, overlap)
    runs = graph_runs(seq)
    assert [seg for run in runs for seg in run] == seq
    replicas = [(("inputs", 0),)]
    for k in range(1, R):
        replicas += [(("replica0" if k == 1 else "replica", None),), (("inputs", k),)]
    if W == 1:
        last = [(("last", None), ("update", None))]
    elif overlap:
        last = [(("last", 0),), (("allreduce_late", None),), (("last", 1),), (("allreduce_finish", None),),
                (("update", None),)]
    else:
        last = [(("last", None),), (("allreduce", None),), (("update", None),)]
    assert runs == replicas + last
    graphs = [run for run in runs if run[0][0] in DEVICE]
    assert all(seg[0] in DEVICE for run in graphs for seg in run)
    assert len(set(graphs)) == (R > 1) + (R > 2) + (1 if W == 1 else 3 if overlap else 2)
