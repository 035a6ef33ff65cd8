"""The oracle (CPU restatement) against the committed golden vectors of the live reference
implementation, and -- when `transformers` is importable -- against the live implementation."""
import hashlib
import os

import numpy as np
import pytest

from oracle import logmel_oracle as O

# HF's own stated tolerance between its two paths is 1e-5 (TF-FE:107-108,137-138); measured
# self-disagreement is <= 5.5e-5 (SURVEY.md 8c).  The restatement is held to 1e-4.
TOL = 1e-4


def _sha(x):
    return hashlib.sha256(np.ascontiguousarray(x).tobytes()).hexdigest()


def test_mel_table_bit_exact(golden):
    z, _ = golden
    for m in (80, 128):
        ours = O.mel_filter_bank(m)
        ref = z[f"mel_filters_m{m}"]
        assert ours.shape == (201, m) and ours.dtype == np.float64
        assert np.array_equal(ours, ref), np.abs(ours - ref).max()


def test_mel_table_structure():
    # each FFT bin feeds at most two, adjacent, filters; bins 0 and 200 feed none (SURVEY 8a2)
    for m, nnz in ((80, 391), (128, 394)):
        fb = O.mel_filter_bank(m)
        nz = fb != 0
        assert nz.sum() == nnz
        assert nz.sum(1).max() == 2
        assert not nz[0].any() and not nz[200].any()
        for k in range(201):
            idx = np.nonzero(nz[k])[0]
            if len(idx) == 2:
                assert idx[1] - idx[0] == 1
        assert nz.sum(0).min() >= 1


def test_hann_matches_torch():
    import torch

    w = torch.hann_window(400).numpy()
    # torch builds the window in fp32 (sin^2 form); it is within 2.4e-7 of the exact value
    assert np.abs(O.hann_window(400, np.float32) - w).max() <= 3e-7
    assert np.allclose(O.hann_window(400), np.hanning(401)[:-1], atol=1e-15)


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_oracle_vs_golden(golden, precision):
    z, meta = golden
    numpy_path = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "logmel_golden_numpy.npz"))
    fs = np.array(meta["frame_subsample"])
    worst = 0.0
    for c in meta["cases"]:
        x = O.synth_clip(c["family"], c["n"], c["seed"])
        assert _sha(x) == c["sha256"], f"synthetic generator drifted for {c['name']}"
        got = O.extract([x], n_mels=c["n_mels"], precision=precision)[0]
        if not c["full"]:
            got = got[:, fs]
        ref = z[c["name"] + "_default"]
        assert got.shape == ref.shape and got.dtype == np.float32
        d = float(np.abs(got - ref).max())
        worst = max(worst, d)
        assert d <= TOL, (c["name"], d)
        if c["name"] in numpy_path:          # stored as its difference from the default path
            d2 = float(np.abs(got - (ref + numpy_path[c["name"]])).max())
            assert d2 <= TOL, (c["name"], "numpy", d2)
    print("worst", precision, worst)


def test_known_answers():
    # all-zero and |x| ~ 1e-6 clips are exactly -1.5 everywhere: (-10 + 4) / 4   (SURVEY 8c)
    for fam in ("zeros",):
        out = O.extract([O.synth_clip(fam, 48000, 1)], 80)
        assert np.all(out == -1.5)
    out = O.extract([O.synth_clip("tiny", 48000, 1)], 80)
    assert np.all(out == -1.5)
    # 35 s == its first 30 s ; short clip == explicitly zero padded clip
    x = O.synth_clip("noise", 560000, 5)
    a = O.extract([x], 80)
    b = O.extract([x[:480000]], 80)
    assert np.array_equal(a, b)
    y = O.synth_clip("noise", 30000, 6)
    ypad = np.concatenate([y, np.zeros(480000 - 30000, np.float32)])
    assert np.array_equal(O.extract([y], 80), O.extract([ypad], 80))
    # dynamic range: everything within [gmax_scaled - 2, gmax_scaled]
    assert a.max() - a.min() <= 2.0 + 1e-6


def test_frame_mask_matches_hf_rule():
    L = np.array([0, 1, 159, 160, 161, 479999, 480000, 600000])
    m = O.frame_mask(L)
    assert m.shape == (8, 3000) and m.dtype == np.int32
    assert m.sum(1).tolist() == [0, 1, 1, 1, 2, 3000, 3000, 3000]


def test_oracle_vs_live_hf():
    pytest.importorskip("transformers")
    from oracle.hf_reference import hf_features

    clips = [O.synth_clip("speech", 50000, 11), O.synth_clip("chirp", 481234, 12)]
    for m in (80, 128):
        ref = hf_features(clips, m, "default")
        got = O.extract(clips, m, "f64")
        assert np.abs(ref - got).max() <= TOL


def test_live_hf_attention_mask_rule():
    pytest.importorskip("transformers")
    from oracle.hf_reference import make_hf_extractor

    fe = make_hf_extractor(80)
    clips = [O.synth_clip("noise", n, 3) for n in (161, 4800, 480000)]
    r = fe(clips, sampling_rate=16000, return_attention_mask=True)
    assert np.array_equal(np.asarray(r["attention_mask"]), O.frame_mask([161, 4800, 480000]))
