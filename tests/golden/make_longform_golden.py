"""Generate the committed golden fixtures of the long-form call (`truncation=False, padding="longest"`).

Run in the build container (needs `transformers`):

    python tests/golden/make_longform_golden.py

Writes `tests/golden/logmel_longform_golden.npz`.  Every case is ONE batched call of the live
`transformers.WhisperFeatureExtractor` (installed 5.5.0):

    fe(clips, sampling_rate=16000, truncation=False, padding="longest",
       pad_to_multiple_of=..., return_attention_mask=True)

which pads every clip of the batch to the longest one and clamps each clip with its own maximum over all
its frames.  Inputs are rebuilt from seeds by `case_clips` (oracle.logmel_oracle.synth_clip underneath);
their sha256 is stored.  Outputs are frame-subsampled (`frames` of each case), the masks are stored
whole, and the per-clip maximum `gmax` is recovered from the features (the largest feature is
(gmax + 4) / 4).
"""
from __future__ import annotations

import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle.logmel_oracle import synth_clip  # noqa: E402

S = 16000
# name, n_mels, pad_to_multiple_of, clips: (family, samples, seed[, sample where a loud burst starts])
CASES = [
    ("s45p37_s10_m80", 80, None, [("speech", 45 * S + 37, 5001), ("noise", 10 * S, 5002)]),
    ("s95_c61_m128", 128, None, [("speech", 95 * S, 5003), ("chirp", 61 * S, 5004)]),
    ("s45p37_s10_mult480k_m80", 80, 480000, [("speech", 45 * S + 37, 5001), ("noise", 10 * S, 5002)]),
    ("L201_m80", 80, None, [("speech", 201, 5010), ("noise", 1, 5011)]),
    ("L5359_m80", 80, None, [("speech", 5359, 5012), ("noise", 5359 - 150, 5013)]),
    ("L5360_m128", 128, None, [("noise", 5360, 5014), ("speech", 5000, 5015)]),
    ("L5361_m80", 80, None, [("chirp", 5361, 5016), ("speech", 5361 - 399, 5017)]),
    ("L12345_m128", 128, None, [("speech", 12345, 5018), ("noise", 12345 - 20, 5019)]),
    ("int16_40s_m80", 80, None, [("int16", 40 * S + 123, 5020), ("int16", 7 * S, 5021)]),
    ("zeros_40s_m80", 80, None, [("zeros", 40 * S, 5022)]),
    ("burst50_m80", 80, None, [("speech", 70 * S, 5023, 50 * S), ("noise", 20 * S, 5024)]),
]


def sha(x: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(x).tobytes()).hexdigest()


def make_clip(spec) -> np.ndarray:
    """(family, n, seed[, burst]): synth_clip, and for a burst the clip at 1 % level with a 0.5-s 440-Hz tone of
    amplitude 0.5 from sample `burst` on -- the clip's maximum lies there, after every frame of the first 30 s."""
    fam, n, seed = spec[:3]
    x = synth_clip(fam, n, seed)
    if len(spec) > 3:
        at = spec[3]
        x = (0.01 * x).astype(np.float32)
        x[at:at + S // 2] += synth_clip("sine", S // 2, seed + 1)
        x = np.clip(x, -1.0, 1.0).astype(np.float32)
    return x


def case_clips(case):
    return [make_clip(spec) for spec in case[3]]


def frame_subsample(T: int) -> np.ndarray:
    if T <= 64:
        return np.arange(T)
    return np.unique(np.concatenate([np.arange(0, 6), np.arange(7, T, 37), np.arange(2990, min(3010, T)),
                                     np.arange(T - 6, T)]))


def main():
    import transformers
    from oracle.hf_reference import make_hf_extractor

    store = {}
    meta = {"cases": [], "transformers": transformers.__version__, "torch": __import__("torch").__version__,
            "numpy": np.__version__}
    for case in CASES:
        name, n_mels, mult, specs = case
        clips = case_clips(case)
        fe = make_hf_extractor(n_mels)
        r = fe(clips, sampling_rate=S, truncation=False, padding="longest", pad_to_multiple_of=mult,
               return_attention_mask=True)
        feats = np.asarray(r["input_features"], dtype=np.float32)
        mask = np.asarray(r["attention_mask"])
        T = feats.shape[2]
        fs = frame_subsample(T)
        store[name + "_features"] = feats[:, :, fs]
        store[name + "_mask"] = mask.astype(np.int8)
        store[name + "_gmax"] = (4.0 * feats.reshape(len(clips), -1).max(1) - 4.0).astype(np.float32)
        meta["cases"].append({"name": name, "n_mels": n_mels, "pad_to_multiple_of": mult,
                              "clips": [list(s) for s in specs], "sha256": [sha(x) for x in clips],
                              "n_frames": int(T), "frames": fs.tolist()})
        print(name, feats.shape, mask.shape)
    store["meta_json"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    out = os.path.join(ROOT, "tests", "golden", "logmel_longform_golden.npz")
    np.savez_compressed(out, **store)
    print(out, os.path.getsize(out) / 1e6, "MB", len(meta["cases"]), "cases")


if __name__ == "__main__":
    main()
