"""Long-form call (`truncation=False, padding="longest"`) without a GPU: the long-form restatement
(tests/longform_oracle.py) against the golden vectors of the live reference, the padded-length rule against the
live `pad`, and the restatement at 30 s against the 30-s oracle."""
import hashlib
import importlib.util
import json
import os

import numpy as np
import pytest

from oracle import logmel_oracle as O

_spec = importlib.util.spec_from_file_location("_longform_oracle",
                                               os.path.join(os.path.dirname(os.path.abspath(__file__)), "longform_oracle.py"))
LO = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(LO)

TOL = 1e-4       # as test_oracle.py: the restatement against the live reference
HERE = os.path.dirname(os.path.abspath(__file__))


def _sha(x):
    return hashlib.sha256(np.ascontiguousarray(x).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def longform_golden():
    spec = importlib.util.spec_from_file_location("_make_longform_golden",
                                                  os.path.join(HERE, "golden", "make_longform_golden.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    z = np.load(os.path.join(HERE, "golden", "logmel_longform_golden.npz"))
    meta = json.loads(bytes(z["meta_json"]).decode())
    return z, meta, gen


def test_golden_inputs_are_reproducible(longform_golden):
    z, meta, gen = longform_golden
    assert [c["name"] for c in meta["cases"]] == [c[0] for c in gen.CASES]
    for c, case in zip(meta["cases"], gen.CASES):
        clips = gen.case_clips(case)
        assert [_sha(x) for x in clips] == c["sha256"], c["name"]


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_oracle_vs_longform_golden(longform_golden, precision):
    z, meta, gen = longform_golden
    for c, case in zip(meta["cases"], gen.CASES):
        clips = gen.case_clips(case)
        got, gmax = LO.extract_longform(clips, c["n_mels"], precision, pad_to_multiple_of=c["pad_to_multiple_of"],
                                       return_gmax=True)
        assert got.shape == (len(clips), c["n_mels"], c["n_frames"]), c["name"]
        ref = z[c["name"] + "_features"]
        d = float(np.abs(got[:, :, c["frames"]] - ref).max())
        assert d <= TOL, (c["name"], precision, d)
        assert np.abs(np.maximum(gmax, -10.0) - z[c["name"] + "_gmax"]).max() <= 4 * TOL, c["name"]
        L = LO.padded_length([len(x) for x in clips], c["pad_to_multiple_of"])
        mask = LO.frame_mask([len(x) for x in clips], L)
        assert np.array_equal(mask, z[c["name"] + "_mask"]), c["name"]


def test_burst_case_clamps_early_frames_with_a_later_maximum(longform_golden):
    """The clip's maximum lies at 50 s; its first 30 s alone would be clamped much lower."""
    z, meta, gen = longform_golden
    case = next(c for c in gen.CASES if c[0] == "burst50_m80")
    x = gen.case_clips(case)[0]
    whole = LO.extract_longform([x], 80, "f64")[0][:, :3000]
    first = O.extract([x[:480000]], 80, "f64")[0]
    assert np.abs(whole - first).max() > 0.25


def test_padded_length_rule():
    from whisper_context_biasing_b200.feature_extraction import padded_length

    assert padded_length([45 * 16000 + 37, 160000]) == 720037
    assert padded_length([45 * 16000 + 37, 160000], 480000) == 960000
    assert padded_length([480000], 480000) == 480000
    assert padded_length([201]) == 201
    rng = np.random.default_rng(3)
    for _ in range(200):
        lens = [int(n) for n in rng.integers(0, 3_000_000, size=rng.integers(1, 6))]
        m = [None, 1, 160, 4000, 480000, int(rng.integers(1, 100000))][int(rng.integers(0, 6))]
        assert padded_length(lens, m) == LO.padded_length(lens, m)


def test_padded_length_rule_matches_live_hf_pad():
    pytest.importorskip("transformers")
    from transformers import BatchFeature

    from oracle.hf_reference import make_hf_extractor
    from whisper_context_biasing_b200.feature_extraction import padded_length

    fe = make_hf_extractor(80)
    rng = np.random.default_rng(5)
    sets = [[720037, 160000], [201], [5359, 5000], [480000], [480001, 3], [1, 2, 3]]
    sets += [[int(n) for n in rng.integers(1, 2_000_000, size=rng.integers(1, 5))] for _ in range(25)]
    for lens in sets:
        for m in (None, 160, 480000, 7, 12345):
            speech = [np.zeros((n, 1), np.float32) for n in lens]        # as TF-FE:292-293 shapes the input
            r = fe.pad(BatchFeature({"input_features": speech}), padding="longest", max_length=480000,
                       truncation=False, pad_to_multiple_of=m, return_attention_mask=True)
            assert np.asarray(r["input_features"]).shape[1] == padded_length(lens, m), (lens, m)


def test_restatement_at_480000_is_the_30s_oracle():
    """At L = 480000 the long-form restatement is the 30-s oracle, bit for bit (features, gmax, mask)."""
    clips = [O.synth_clip("speech", 50000, 21), O.synth_clip("noise", 480000, 22)]
    for precision in ("f64", "f32"):
        a, ga = O.log_mel_spectrogram(O.pad_or_trim(clips), 80, precision, return_gmax=True)
        b, gb = LO.extract_longform(clips, 80, precision, return_gmax=True)
        assert a.shape == (2, 80, 3000) and np.array_equal(a, b) and np.array_equal(ga, gb)
    assert LO.frames(O.pad_or_trim(clips)[0], np.float64).shape == (3000, 400)
    lens = [0, 1, 159, 160, 161, 479999, 480000, 600000]
    assert np.array_equal(O.frame_mask(lens), LO.frame_mask(lens, 480000))
    # L % 160 != 0: the last partial frame is dropped, as torch drops the last STFT frame
    assert LO.frame_mask([5361], 5361).shape == (1, 33)
    assert LO.extract_longform([np.zeros(201, np.float32)], 80).shape == (1, 80, 1)
    with pytest.raises(ValueError):
        LO.extract_longform([np.zeros(200, np.float32)], 80)
