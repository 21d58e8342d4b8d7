"""Bit-exact data sampling (BASELINE.json north_star: "data indexing, sampling and crop offsets must be
bit-exact"; SURVEY.md §8d).  The reference's dataset classes (dataset/CramedDataset.py:57-110,
dataset/KSDataset.py:136-201) are run UNMODIFIED with only their file I/O mocked by the seeded stand-ins of
gdl_b200.synthetic (librosa.load -> synth_wave, librosa.stft -> stft, Image.open -> synth_image); under the same
torch / numpy / python seeds the synthetic classes must return bit-identical spectrograms and image tensors
(crop offsets, flips, audio offsets) and leave all three RNGs in the same state.  The outputs are always compared
with the digests of the reference's outputs committed as tests/golden/sampling_golden.json.  With GDL_REFERENCE_DIR
naming a checkout of the reference, its classes are also run live, and GDL_WRITE_GOLDEN=1 rewrites the digests."""
import argparse
import hashlib
import json
import os
import random
import sys
import types

import numpy as np
import pytest
import torch

REF = os.environ.get("GDL_REFERENCE_DIR")
GOLD = os.path.join(os.path.dirname(__file__), "golden", "sampling_golden.json")
IDXS = [0, 3, 7, 12]


def _digest(spec, images, label):
    h = hashlib.sha256()
    h.update(np.ascontiguousarray(np.asarray(spec, dtype=np.float32)).tobytes())
    h.update(images.contiguous().numpy().tobytes())
    h.update(str(int(label)).encode())
    return h.hexdigest()


def _rng_digest():
    h = hashlib.sha256()
    h.update(torch.get_rng_state().numpy().tobytes())
    st = np.random.get_state()
    h.update(st[1].tobytes() + str(st[2]).encode())
    h.update(str(random.getstate()[1][:8]).encode())
    return h.hexdigest()


def _run(ds, seed):
    torch.manual_seed(seed)
    np.random.seed(seed)
    random.seed(seed)
    out = [ds[i] for i in IDXS]
    return out, _rng_digest()


def _synthetic(kind, mode):
    from gdl_b200 import synthetic as S
    args = argparse.Namespace(dataset=kind, fps=3, use_video_frames=3)
    return S.SyntheticCramed(args, mode) if kind == "CREMAD" else S.SyntheticKS(args, mode)


def _reference(kind, mode, tmp_path):
    """The reference class with its constructor bypassed (it walks a dataset directory) and its decoders mocked."""
    from gdl_b200 import synthetic as S
    sys.path.insert(0, REF)
    fake = types.ModuleType("librosa")
    fake.load = lambda path, sr=None, mono=True: S.synth_wave(os.path.basename(os.path.dirname(path)) + "/" +
                                                             os.path.basename(path)[:-4],
                                                             2.5 if sr == 22050 else 4.0, sr)
    fake.stft = lambda x, n_fft, hop_length: S.stft(x, n_fft, hop_length)
    saved = {k: sys.modules.get(k) for k in ("librosa", "skimage")}
    sys.modules["librosa"] = fake
    sys.modules.setdefault("skimage", types.ModuleType("skimage"))
    try:
        for m in ("dataset.CramedDataset", "dataset.KSDataset", "dataset"):
            sys.modules.pop(m, None)
        if kind == "CREMAD":
            import dataset.CramedDataset as M
            ds = object.__new__(M.CramedDataset)
            size = (480, 360)
        else:
            import dataset.KSDataset as M
            ds = object.__new__(M.KSDataset)
            torch.nn.Module.__init__(ds)
            size = (340, 256)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
        sys.path.remove(REF)
    n = max(IDXS) + 1
    args = argparse.Namespace(dataset=kind, fps=3, use_video_frames=3)
    dirs, wavs, labels = [], [], []
    nframes = 3 if kind == "CREMAD" else 10
    for i in range(n):
        d = tmp_path / mode / str(i)
        d.mkdir(parents=True, exist_ok=True)
        for f in range(nframes):
            (d / ("%02d.jpg" % f)).write_bytes(b"")
        dirs.append(str(d))
        wavs.append(str(tmp_path / mode / ("%d.wav" % i)))
        labels.append(S._seed_of(("label", "%s/%d" % (mode, i))) % (6 if kind == "CREMAD" else 31))
    ds.args, ds.mode = args, mode
    if kind == "CREMAD":
        ds.image, ds.audio, ds.label = dirs, wavs, labels
        # directory order is file-system dependent upstream: pin it (the module gets its own `os` shim)
        M.os = types.SimpleNamespace(listdir=lambda p: sorted(os.listdir(p)), path=os.path)
    else:
        ds.video_path_list, ds.audio_path_list, ds.data_label = dirs, wavs, labels
        M.listdir_nohidden = lambda p: sorted(os.path.join(p, f) for f in os.listdir(p))

    class _Img:
        @staticmethod
        def open(path):
            p = str(path)
            key = "%s/%s/%d" % (mode, os.path.basename(os.path.dirname(p)), int(os.path.basename(p)[:2]))
            img = S.synth_image(key, size)
            return types.SimpleNamespace(convert=lambda m: img)
    M.Image = _Img
    return ds


CASES = [("CREMAD", "train"), ("CREMAD", "test"), ("KineticSound", "train"), ("KineticSound", "test")]


@pytest.mark.parametrize("kind,mode", CASES)
def test_sampling_matches_reference_bit_exact(kind, mode, tmp_path):
    syn, syn_rng = _run(_synthetic(kind, mode), seed=1234)
    digests = [_digest(*s) for s in syn]
    key = "%s/%s" % (kind, mode)
    if REF:
        ref, ref_rng = _run(_reference(kind, mode, tmp_path), seed=1234)
        for (s0, i0, l0), (s1, i1, l1) in zip(syn, ref):
            assert np.array_equal(np.asarray(s0), np.asarray(s1)), "spectrogram / audio crop offset differs"
            assert torch.equal(i0, i1), "image tensors differ: crop offsets or flips are not bit-exact"
            assert int(l0) == int(l1)
        assert syn_rng == ref_rng, "the RNG streams were consumed differently"
        if os.environ.get("GDL_WRITE_GOLDEN"):
            gold = json.load(open(GOLD)) if os.path.exists(GOLD) else {}
            gold[key] = {"samples": digests, "rng": syn_rng}
            json.dump(gold, open(GOLD, "w"), indent=1, sort_keys=True)
    gold = json.load(open(GOLD))
    assert gold[key]["samples"] == digests and gold[key]["rng"] == syn_rng


def test_shapes_follow_the_reference_contract():
    for kind, (Fq, Tt) in (("CREMAD", (257, 188)), ("KineticSound", (129, 626))):
        spec, images, label = _synthetic(kind, "train")[0]
        assert tuple(np.asarray(spec).shape) == (Fq, Tt)
        assert tuple(images.shape) == (3, 3, 224, 224) and images.dtype == torch.float32
        assert isinstance(label, int)
