"""`do_normalize` and `dither` without a GPU: the numpy Philox against the Random123 known answers, and the conditioned
restatement (tests/conditioning_oracle.py) against the live reference -- for dither with torch.randn replaced by the
restated noise, which pins the order of the steps and the noise on the pad and the reflected samples to HF's own code."""
import importlib.util
import os
import warnings

import numpy as np
import pytest

from oracle import logmel_oracle as O

_spec = importlib.util.spec_from_file_location("_conditioning_oracle",
                                               os.path.join(os.path.dirname(os.path.abspath(__file__)), "conditioning_oracle.py"))
CO = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(CO)

TOL = 1e-4       # as test_oracle.py: the restatement against the live reference
LONG = dict(truncation=False, padding="longest")


def _clips():
    clips = [O.synth_clip(f, 30000 + 7001 * i, 500 + i) for i, f in enumerate(O.FAMILIES)]
    clips.append((40.0 + 0.05 * O.synth_clip("speech", 64000, 520)).astype(np.float32))     # large DC offset
    clips.append(np.zeros(0, np.float32))                                                  # empty
    clips.append(O.synth_clip("chirp", 480000 + 12345, 521))                              # longer than 30 s
    return clips


def _hf(clips, n_mels=80, dither=0.0, **kw):
    pytest.importorskip("transformers")
    from transformers import WhisperFeatureExtractor

    fe = WhisperFeatureExtractor(feature_size=n_mels, dither=dither)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")             # the empty clip's NaN statistics, which HF then overwrites
        return fe([c.astype(np.float32) for c in clips], sampling_rate=16000, return_tensors="np", **kw)


def test_philox_known_answers():
    cases = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
             ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
             ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
              (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for ctr, key, want in cases:
        got = CO.philox4x32_10([np.array([c], np.uint64) for c in ctr], key)
        assert [int(w[0]) for w in got] == list(want)


def test_noise_stream_layout():
    """sample n of clip b takes z_{n & 3} of counter (n >> 2, b): prefixes agree, clips differ, unit variance."""
    a = CO.noise(7, 3, 1001)
    assert np.array_equal(a[:500], CO.noise(7, 3, 500))
    assert not np.allclose(a, CO.noise(7, 4, 1001)) and not np.allclose(a, CO.noise(8, 3, 1001))
    z = CO.noise(2 ** 64 - 1, 0, 400000)
    assert abs(z.mean()) < 0.01 and abs(z.std() - 1.0) < 0.01


@pytest.mark.parametrize("longform", [False, True])
def test_normalize_matches_live_hf(longform):
    clips = _clips()
    kw = dict(LONG, pad_to_multiple_of=160) if longform else {}
    ref = _hf(clips, do_normalize=True, **kw)["input_features"]
    got = CO.extract(clips, 80, do_normalize=True, longform=longform, pad_to_multiple_of=160 if longform else None)
    assert got.shape == ref.shape
    d = float(np.abs(got - ref).max())
    assert d <= TOL, d
    # normalising changes the features (the restatement is not trivially the unconditioned one)
    plain = CO.extract(clips, 80, longform=longform, pad_to_multiple_of=160 if longform else None)
    assert np.abs(plain - got).max() > 0.1


@pytest.mark.parametrize("longform", [False, True])
@pytest.mark.parametrize("do_normalize", [False, True])
def test_dither_matches_live_hf_with_restated_noise(monkeypatch, longform, do_normalize):
    import torch

    clips = _clips()[4:]
    seed, dither = 0x0123456789ABCDEF, 0.5
    N = CO.LO.padded_length([len(c) for c in clips], 480000) if longform else O.N_SAMPLES
    z = torch.from_numpy(CO.noise_batch(seed, len(clips), N))
    calls = []

    def randn(shape, dtype=None, device=None, **kw):
        calls.append(tuple(shape))
        assert tuple(shape) == tuple(z.shape)
        return z.to(dtype=dtype or torch.float32, device=device)

    monkeypatch.setattr(torch, "randn", randn)
    kw = dict(LONG, pad_to_multiple_of=480000) if longform else {}
    ref = _hf(clips, dither=dither, do_normalize=do_normalize, **kw)["input_features"]
    assert calls == [tuple(z.shape)]
    got = CO.extract(clips, 80, do_normalize=do_normalize, dither=dither, seed=seed, longform=longform,
                     pad_to_multiple_of=480000 if longform else None)
    d = float(np.abs(got - ref).max())
    assert d <= TOL, d


def test_hf_mask_quirk_with_do_normalize():
    clips = [O.synth_clip("speech", 20000, 1), O.synth_clip("noise", 5000, 2)]
    r = _hf(clips, do_normalize=True)
    assert r["attention_mask"].shape == (2, 480000)
    r = _hf(clips, do_normalize=True, return_attention_mask=True)
    assert r["attention_mask"].shape == (2, 3000)
    r = _hf(clips, do_normalize=True, **LONG)
    assert r["attention_mask"].shape == (2, 20000)
