"""The order of the EncoderEngine's library calls and the sweep hint (gdl_set_sweep) each one runs under.  CPU only.

A sweep hint changes no result, only which part of a tensor the next pass finds in L2, so no correctness test sees a
wrong one.  Here every launching function of gdl_b200.ops is replaced by a recorder and the engine is built on CPU
tensors (its host-only queries, conv_packed_k, the workspace sizes and stem_geometry, need no GPU).  The recorded
(op, hint) lists of the audio and the visual encoder at two geometries must equal the reviewed table below, for a
training forward, a whole backward, the two-part backward of the overlapped all-reduce and forward_eval.  The training
forward is recorded twice: with the BatchNorm statistics out of the convolution epilogues (what every convolution of
these geometries does) and with none of them (gdl_set_fused_stats_min_k above every K: separate bn_stats passes)."""
import textwrap
import threading

import pytest
import torch

# (dataset, B): the (N, H, W) of the audio and the visual encoder (gdl_b200.shapes.BATCH_SHAPES)
GEOMETRIES = {"CREMAD B=16": {"audio": (16, 257, 188), "visual": (48, 224, 224)},
              "KineticSound B=16": {"audio": (16, 129, 626), "visual": (48, 224, 224)}}
STATS_ROWS = 4  # partial rows a fused-statistics epilogue reports (any count > 0 selects the same schedule)

# op:hint of every library call in order (hint 1: descending pixel order)
EXPECTED = {
    "forward": """
        stem_fwd_stats:0 bn_stats_finalize:0 bn_relu_maxpool_fwd:1 conv_fwd_stats:0 bn_stats_finalize:1 bn_apply:1
        conv_fwd_stats:0 bn_stats_finalize:1 bn_apply:1 conv_fwd_stats:0 bn_stats_finalize:1 bn_apply:1
        conv_fwd_stats:0 bn_stats_finalize:1 bn_apply:1 conv_fwd_stats:0 bn_stats_finalize:1 bn_apply:1
        conv_fwd_stats:0 bn_stats_finalize:1 bn_apply:1 conv_fwd_stats:0 bn_stats_finalize:1 bn_apply:1
        conv_fwd_stats:0 bn_stats_finalize:1 bn_apply:1 conv_fwd_stats:0 bn_stats_finalize:1 bn_apply:1
        conv_fwd_stats:0 bn_stats_finalize:1 bn_apply:1 conv_fwd_stats:0 bn_stats_finalize:1 bn_apply:1
        conv_fwd_stats:0 bn_stats_finalize:1 bn_apply:1 conv_fwd_stats:0 bn_stats_finalize:1 bn_apply:1
        conv_fwd_stats:0 bn_stats_finalize:1 bn_apply:1 conv_fwd_stats:0 bn_stats_finalize:1 bn_apply:1
        conv_fwd_stats:0 bn_stats_finalize:1 bn_apply:1 conv_fwd_stats:0 bn_stats_finalize:1 bn_apply:1
        conv_fwd_stats:0 bn_stats_finalize:1 bn_apply:1 conv_fwd_stats:0 bn_stats_finalize:1 bn_apply:1
    """,
    "backward": """
        bn_bwd:1 conv_wgrad:1 conv_dgrad:0 bn_bwd_nores:1 conv_wgrad:1 conv_dgrad:0 bn_bwd:1 conv_wgrad:1
        conv_dgrad:0 bn_bwd_nores:1 conv_wgrad:1 bn_bwd:1 conv_wgrad:0 conv_dgrad:0 conv_dgrad:0 bn_bwd:1
        conv_wgrad:1 conv_dgrad:0 bn_bwd_nores:1 conv_wgrad:1 conv_dgrad:0 bn_bwd:1 conv_wgrad:1 conv_dgrad:0
        bn_bwd_nores:1 conv_wgrad:1 bn_bwd:1 conv_wgrad:0 conv_dgrad:0 conv_dgrad:0 bn_bwd:1 conv_wgrad:1
        conv_dgrad:0 bn_bwd_nores:1 conv_wgrad:1 conv_dgrad:0 bn_bwd:1 conv_wgrad:1 conv_dgrad:0 bn_bwd_nores:1
        conv_wgrad:1 bn_bwd:1 conv_wgrad:0 conv_dgrad:0 conv_dgrad:0 bn_bwd:1 conv_wgrad:1 conv_dgrad:0
        bn_bwd_nores:1 conv_wgrad:1 conv_dgrad:0 bn_bwd:1 conv_wgrad:1 conv_dgrad:0 bn_bwd_nores:1 conv_wgrad:1
        conv_dgrad:0 bn_relu_maxpool_bwd:1 stem_wgrad:1
    """,
    "backward part=0": """
        bn_bwd:1 conv_wgrad:1 conv_dgrad:0 bn_bwd_nores:1 conv_wgrad:1 conv_dgrad:0 bn_bwd:1 conv_wgrad:1
        conv_dgrad:0 bn_bwd_nores:1 conv_wgrad:1 bn_bwd:1 conv_wgrad:0 conv_dgrad:0 conv_dgrad:0 bn_bwd:1
        conv_wgrad:1 conv_dgrad:0 bn_bwd_nores:1 conv_wgrad:1 conv_dgrad:0 bn_bwd:1 conv_wgrad:1 conv_dgrad:0
        bn_bwd_nores:1 conv_wgrad:1 bn_bwd:1 conv_wgrad:0 conv_dgrad:0 conv_dgrad:0
    """,
    "backward part=1": """
        bn_bwd:1 conv_wgrad:1 conv_dgrad:0 bn_bwd_nores:1 conv_wgrad:1 conv_dgrad:0 bn_bwd:1 conv_wgrad:1
        conv_dgrad:0 bn_bwd_nores:1 conv_wgrad:1 bn_bwd:1 conv_wgrad:0 conv_dgrad:0 conv_dgrad:0 bn_bwd:1
        conv_wgrad:1 conv_dgrad:0 bn_bwd_nores:1 conv_wgrad:1 conv_dgrad:0 bn_bwd:1 conv_wgrad:1 conv_dgrad:0
        bn_bwd_nores:1 conv_wgrad:1 conv_dgrad:0 bn_relu_maxpool_bwd:1 stem_wgrad:1
    """,
    "forward_eval": """
        bn_eval_affine:0 bn_eval_affine:0 bn_eval_affine:0 bn_eval_affine:0 bn_eval_affine:0 bn_eval_affine:0
        bn_eval_affine:0 bn_eval_affine:0 bn_eval_affine:0 bn_eval_affine:0 bn_eval_affine:0 bn_eval_affine:0
        bn_eval_affine:0 bn_eval_affine:0 bn_eval_affine:0 bn_eval_affine:0 bn_eval_affine:0 bn_eval_affine:0
        bn_eval_affine:0 bn_eval_affine:0 stem_pack_weights_scaled:0 conv_pack_weights_multi:0 stem_fwd:0
        bn_relu_maxpool_fwd:0 conv_fwd_bias_act:0 conv_fwd_bias_act:0 conv_fwd_bias_act:0 conv_fwd_bias_act:0
        conv_fwd_bias_act:0 conv_fwd_bias_act:0 conv_fwd_bias_act:0 conv_fwd_bias_act:0 conv_fwd_bias_act:0
        conv_fwd_bias_act:0 conv_fwd_bias_act:0 conv_fwd_bias_act:0 conv_fwd_bias_act:0 conv_fwd_bias_act:0
        conv_fwd_bias_act:0 conv_fwd_bias_act:0 conv_fwd_bias_act:0 conv_fwd_bias_act:0 conv_fwd_bias_act:0
    """,
    "forward without fused statistics": """
        stem_fwd_stats:0 bn_stats_finalize:0 bn_relu_maxpool_fwd:1 conv_fwd_stats:0 bn_stats:1 bn_apply:0
        conv_fwd_stats:0 bn_stats:1 bn_apply:0 conv_fwd_stats:0 bn_stats:1 bn_apply:0 conv_fwd_stats:0 bn_stats:1
        bn_apply:0 conv_fwd_stats:0 bn_stats:1 bn_apply:0 conv_fwd_stats:0 bn_stats:1 bn_apply:0 conv_fwd_stats:0
        bn_stats:1 bn_apply:0 conv_fwd_stats:0 bn_stats:1 bn_apply:0 conv_fwd_stats:0 bn_stats:1 bn_apply:0
        conv_fwd_stats:0 bn_stats:1 bn_apply:0 conv_fwd_stats:0 bn_stats:1 bn_apply:0 conv_fwd_stats:0 bn_stats:1
        bn_apply:0 conv_fwd_stats:0 bn_stats:1 bn_apply:0 conv_fwd_stats:0 bn_stats:1 bn_apply:0 conv_fwd_stats:0
        bn_stats:1 bn_apply:0 conv_fwd_stats:0 bn_stats:1 bn_apply:0 conv_fwd_stats:0 bn_stats:1 bn_apply:0
        conv_fwd_stats:0 bn_stats:1 bn_apply:0 conv_fwd_stats:0 bn_stats:1 bn_apply:0
    """,
}


class Recorder:
    """Replaces ops.init, ops.sweep and every launching function of ops (those carrying the _op decorator)."""

    def __init__(self, ops, mp, conv_rows):
        self.calls = []
        self.hint = {}
        mp.setattr(ops, "init", lambda device=None: None)
        mp.setattr(ops, "sweep", self._sweep)
        for name, fn in list(vars(ops).items()):
            if callable(fn) and hasattr(fn, "__wrapped__"):
                mp.setattr(ops, name, self._wrap(name, conv_rows))

    def _sweep(self, reverse):
        self.hint[threading.get_ident()] = 1 if reverse else 0

    def _wrap(self, name, conv_rows):
        def rec(*a, **k):
            self.calls.append("%s:%d" % (name, self.hint.get(threading.get_ident(), 0)))
            return {"conv_fwd_stats": conv_rows, "stem_fwd_stats": STATS_ROWS}.get(name)
        return rec

    def take(self):
        out, self.calls = self.calls, []
        assert self.hint.get(threading.get_ident(), 0) == 0, "a phase left the sweep hint descending"
        return out


def _record(modality, N, H, W):
    from gdl_b200 import ops
    from gdl_b200.backbone import resnet18
    from gdl_b200.engine import EncoderEngine
    out = {}
    for conv_rows in (STATS_ROWS, 0):
        with pytest.MonkeyPatch.context() as mp:
            rec = Recorder(ops, mp, conv_rows)
            eng = EncoderEngine(resnet18(modality, None), N, H, W, torch.device("cpu"))
            x16 = torch.empty(eng.input_shape, dtype=torch.bfloat16)
            rec.take()
            eng.forward(x16)
            if conv_rows == 0:
                out["forward without fused statistics"] = rec.take()
                continue
            out["forward"] = rec.take()
            eng.backward(x16)
            out["backward"] = rec.take()
            eng.backward(x16, part=0)
            out["backward part=0"] = rec.take()
            eng.backward(x16, part=1)
            out["backward part=1"] = rec.take()
            eng.forward_eval(x16)
            out["forward_eval"] = rec.take()
    return out


def _table(out):
    return "EXPECTED = {\n%s}" % "".join(
        '    "%s": """\n%s\n    """,\n' % (k, textwrap.fill(" ".join(v), 116, initial_indent=" " * 8,
                                                             subsequent_indent=" " * 8, break_on_hyphens=False))
        for k, v in out.items())


@pytest.mark.parametrize("modality", ["audio", "visual"])
@pytest.mark.parametrize("cfg", list(GEOMETRIES))
def test_engine_schedule(cfg, modality):
    got = _record(modality, *GEOMETRIES[cfg][modality])
    assert set(got) == set(EXPECTED), _table(got)
    for phase, calls in got.items():
        assert calls == EXPECTED[phase].split(), "%s %s %s changed:\n%s" % (cfg, modality, phase, _table(got))


if __name__ == "__main__":
    import os
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path[:0] = [root, os.path.join(root, "iccv2025-gdl_b200")]
    print(_table(_record("audio", *GEOMETRIES["CREMAD B=16"]["audio"])))
