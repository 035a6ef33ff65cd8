"""CPU restatement of the conditioned call (`do_normalize=True` and the constructor's `dither`): test infrastructure, built
on the long-form restatement (tests/longform_oracle.py).

HF (TF-FE:189-342 and :141-161, transformers 5.5.0, torch path) runs, on the batch padded to N samples (N = 480000 for the
30-s call, L for the long-form call):
  1. pad / trim;
  2. do_normalize: zero_mean_unit_var_norm with the pad's mask -- (x - mean) / sqrt(var + 1e-7) over the n_b = min(len, N)
     valid samples (float32 numpy arithmetic), 0 on the pad, an empty clip stays 0;
  3. dither: waveform += dither * randn over the whole padded [B, N], before torch.stft reflects it;
  4. the log-mel features.
The noise cannot be torch.randn's, so it is restated as the Philox4x32-10 / Box-Muller stream of include/wlm.h.
"""
from __future__ import annotations

import importlib.util
import os

import numpy as np

from oracle import logmel_oracle as O

_spec = importlib.util.spec_from_file_location("_longform_oracle_c",
                                               os.path.join(os.path.dirname(os.path.abspath(__file__)), "longform_oracle.py"))
LO = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(LO)

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = 0x9E3779B9, 0xBB67AE85
_MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """Philox4x32-10 (Random123).  ctr: 4 uint32 arrays (broadcastable), key: 2 ints -> 4 uint32 arrays."""
    x = [np.asarray(c, dtype=np.uint64) & _MASK for c in ctr]
    k0, k1 = int(key[0]) & 0xFFFFFFFF, int(key[1]) & 0xFFFFFFFF
    for r in range(10):
        if r:
            k0, k1 = (k0 + _W0) & 0xFFFFFFFF, (k1 + _W1) & 0xFFFFFFFF
        p0, p1 = _M0 * x[0], _M1 * x[2]
        x = [(p1 >> np.uint64(32)) ^ x[1] ^ np.uint64(k0), p1 & _MASK, (p0 >> np.uint64(32)) ^ x[3] ^ np.uint64(k1), p0 & _MASK]
    return [v.astype(np.uint32) for v in x]


def noise(seed: int, b: int, n: int) -> np.ndarray:
    """z(seed, b, 0..n-1), float64: counter (i >> 2, b, 0, 0), key (lo32, hi32) of the seed, Box-Muller on (u0, u1) and
    (u2, u3), sample i takes z_{i & 3}."""
    q = np.arange((n + 3) // 4, dtype=np.uint64)
    seed = int(seed) % 2 ** 64
    r = philox4x32_10([q, np.full_like(q, b), np.zeros_like(q), np.zeros_like(q)], (seed & 0xFFFFFFFF, seed >> 32))
    u = [((w >> np.uint32(8)).astype(np.float64) + 0.5) * 2.0 ** -24 for w in r]
    z = np.empty((q.shape[0], 4), np.float64)
    for p in range(2):
        rad = np.sqrt(-2.0 * np.log(u[2 * p]))
        z[:, 2 * p] = rad * np.cos(2.0 * np.pi * u[2 * p + 1])
        z[:, 2 * p + 1] = rad * np.sin(2.0 * np.pi * u[2 * p + 1])
    return z.reshape(-1)[:n]


def noise_batch(seed: int, B: int, n: int) -> np.ndarray:
    return np.stack([noise(seed, b, n) for b in range(B)]).astype(np.float32)


def normalize(padded: np.ndarray, lengths) -> np.ndarray:
    """zero_mean_unit_var_norm of TF-FE (float32 numpy), on [B, N] padded with zeros."""
    out = np.array(padded, dtype=np.float32, copy=True)
    for b, n in enumerate(lengths):
        n = int(min(n, out.shape[1]))
        v = out[b]
        if n == 0:
            v[:] = 0.0
            continue
        v[:] = (v - v[:n].mean()) / np.sqrt(v[:n].var() + 1e-7)
        v[n:] = 0.0
    return out


def condition(clips, N: int, do_normalize=False, dither=0.0, seed=0) -> np.ndarray:
    """pad / trim to N, normalise, + dither z: the waveform [B, N] float32 that HF hands to torch.stft."""
    clips = [np.asarray(c, dtype=np.float32).reshape(-1) for c in clips]
    x = O.pad_or_trim(clips, N)
    if do_normalize:
        x = normalize(x, [len(c) for c in clips])
    if dither:
        x = x + np.float32(dither) * noise_batch(seed, len(clips), N)
    return x.astype(np.float32)


def extract(clips, n_mels=80, do_normalize=False, dither=0.0, seed=0, longform=False, pad_to_multiple_of=None,
            precision="f64"):
    """The conditioned call: 30-s geometry (N = 480000) or long-form (N = the padded length L)."""
    clips = [np.asarray(c, dtype=np.float32).reshape(-1) for c in clips]
    N = LO.padded_length([len(c) for c in clips], pad_to_multiple_of) if longform else O.N_SAMPLES
    return LO.log_mel_spectrogram(condition(clips, N, do_normalize, dither, seed), n_mels, precision)[0]
