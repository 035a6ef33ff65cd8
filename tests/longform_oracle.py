"""CPU restatement of the long-form call (`truncation=False, padding="longest"`): test infrastructure, built on the
unchanged 30-s oracle (`oracle/logmel_oracle.py`: mel bank, window, pad/trim).

What differs from the 30-s path (TF-FE:189-342, TF-SU `pad`/`_pad`, transformers 5.5.0):
  * every clip of the batch is zero-padded to one common length L -- the longest clip, rounded up to a multiple of
    `pad_to_multiple_of` when given; `max_length` plays no part;
  * torch.stft(center=True) reflects 200 samples at sample 0 and at sample L, and the last frame is dropped:
    T = L // 160 frames;
  * each clip is clamped with its own maximum over all M x T values;
  * the attention mask is the sample mask [0, len) subsampled every 160 samples, its last column dropped when
    L % 160 != 0: [B, T].
"""
from __future__ import annotations

import numpy as np

from oracle import logmel_oracle as O


def padded_length(lengths, pad_to_multiple_of=None) -> int:
    L = max((int(n) for n in lengths), default=0)
    if pad_to_multiple_of is not None and L % pad_to_multiple_of != 0:
        L = (L // pad_to_multiple_of + 1) * pad_to_multiple_of
    return L


def frame_mask(lengths, n_samples: int) -> np.ndarray:
    lengths = np.minimum(np.asarray(lengths, dtype=np.int64), n_samples)
    pos = O.HOP_LENGTH * np.arange(n_samples // O.HOP_LENGTH, dtype=np.int64)
    return (pos[None, :] < lengths[:, None]).astype(np.int32)


def frames(padded_clip: np.ndarray, dtype) -> np.ndarray:
    """[T, 400] frames of an already padded clip of L samples, reflected by 200 at both ends."""
    n = padded_clip.shape[0]
    x = np.pad(padded_clip.astype(dtype), (O.N_FFT // 2, O.N_FFT // 2), mode="reflect")
    idx = O.HOP_LENGTH * np.arange(n // O.HOP_LENGTH)[:, None] + np.arange(O.N_FFT)[None, :]
    return x[idx]


def log_mel_spectrogram(padded: np.ndarray, n_mels: int = 80, precision: str = "f64"):
    """[B, L] float32 (already padded) -> ([B, n_mels, L // 160] float32, gmax [B]); the arithmetic of
    O.log_mel_spectrogram, for any L."""
    padded = np.asarray(padded, dtype=np.float32)
    dt = np.float64 if precision == "f64" else np.float32
    fbT = O.mel_filter_bank(n_mels).T.astype(dt)
    win = O.hann_window(O.N_FFT, dt)
    out = np.empty((padded.shape[0], n_mels, padded.shape[1] // O.HOP_LENGTH), dtype=np.float32)
    gmax = np.empty((padded.shape[0],), dtype=np.float32)
    for b in range(padded.shape[0]):
        spec = np.fft.rfft(frames(padded[b], dt) * win[None, :], axis=1)
        if precision == "f32":
            spec = spec.astype(np.complex64)
        power = (np.abs(spec) ** 2).astype(dt)
        log_spec = np.log10(np.maximum(fbT @ power.T, dt(1e-10)))
        g = log_spec.max()
        out[b] = ((np.maximum(log_spec, g - dt(8.0)) + dt(4.0)) / dt(4.0)).astype(np.float32)
        gmax[b] = g
    return out, gmax


def extract_longform(clips, n_mels: int = 80, precision: str = "f64", pad_to_multiple_of=None,
                     return_gmax: bool = False):
    """ragged list of PCM clips -> [B, n_mels, L // 160] float32: `WhisperFeatureExtractor.__call__(...,
    truncation=False, padding="longest", pad_to_multiple_of=...)`."""
    if isinstance(clips, np.ndarray) and clips.ndim == 1:
        clips = [clips]
    clips = list(clips)
    L = padded_length([np.asarray(c).reshape(-1).shape[0] for c in clips], pad_to_multiple_of)
    if L <= O.N_FFT // 2:
        raise ValueError(f"padded length {L}: the reflect padding needs more than {O.N_FFT // 2} samples")
    out, gmax = log_mel_spectrogram(O.pad_or_trim(clips, L), n_mels, precision)
    return (out, gmax) if return_gmax else out
