"""Generate the committed golden fixtures for the log-mel hot path.

Run in the BUILD CONTAINER only (needs `transformers`; the fixtures travel, this script's
dependencies need not):

    python tests/golden/make_golden.py

Outputs `tests/golden/logmel_golden.npz`.  Every entry is produced by the LIVE third-party
implementation the reference calls (`transformers.WhisperFeatureExtractor`, installed 5.5.0;
reference pins 4.51.3), invoked exactly like REF/data_utils/data_loader.py:171 -- one clip per
call, `.input_features[0]` -- for both dispatch paths (torch fp32 default, numpy fp64 fallback).
Inputs are regenerated from seeds by `oracle.logmel_oracle.synth_clip`; a sha256 of every input
is stored so generator drift is detected rather than silently compared.

The numpy path's outputs go to `tests/golden/logmel_golden_numpy.npz`, each as its difference from
the default path's output of the same case (exact in float32, zero for ~98 % of the elements): that
keeps both files under 1 MB.  `default + difference` gives back the numpy path's output bit for bit.
"""
from __future__ import annotations

import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle.hf_reference import hf_features  # noqa: E402
from oracle.logmel_oracle import FAMILIES, synth_clip  # noqa: E402

SHORT_N = 21923                      # 1.37 s, deliberately not a multiple of 160
FRAME_SUBSAMPLE = np.unique(np.concatenate([np.arange(0, 6), np.arange(7, 3000, 37),
                                             np.arange(2994, 3000)]))
RAGGED_LENGTHS = [1, 159, 160, 161, 399, 400, 401, 4801, 479999, 480000, 480001, 560000]


def sha(x: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(x).tobytes()).hexdigest()


def main():
    store, numpy_path = {}, {}

    def add_numpy_path(name, out):
        numpy_path[name] = out - store[name + "_default"]
        assert np.array_equal(store[name + "_default"] + numpy_path[name], out), name

    meta = {"cases": [], "frame_subsample": FRAME_SUBSAMPLE.tolist(),
            "transformers": __import__("transformers").__version__,
            "torch": __import__("torch").__version__, "numpy": np.__version__}

    # (1) short clips, every family, both mel configs: FULL [M, 3000] outputs (compress well,
    #     everything after frame ~140 is the zero-pad constant)
    for n_mels in (80, 128):
        for fi, fam in enumerate(FAMILIES):
            seed = 1000 + fi
            x = synth_clip(fam, SHORT_N, seed)
            name = f"short_{fam}_m{n_mels}"
            store[name + "_default"] = hf_features([x], n_mels, "default")[0]
            add_numpy_path(name, hf_features([x], n_mels, "numpy")[0])
            meta["cases"].append({"name": name, "kind": "short", "family": fam, "seed": seed,
                                  "n": SHORT_N, "n_mels": n_mels, "sha256": sha(x), "full": True})

    # (2) full 30 s clips: frame-subsampled outputs
    for n_mels, fam, seed in ((80, "noise", 2000), (80, "speech", 2001), (80, "sine", 2002),
                              (128, "noise", 2003), (128, "chirp", 2004), (128, "gap", 2005)):
        x = synth_clip(fam, 480000, seed)
        name = f"full_{fam}_m{n_mels}"
        store[name + "_default"] = hf_features([x], n_mels, "default")[0][:, FRAME_SUBSAMPLE]
        add_numpy_path(name, hf_features([x], n_mels, "numpy")[0][:, FRAME_SUBSAMPLE])
        meta["cases"].append({"name": name, "kind": "full", "family": fam, "seed": seed,
                              "n": 480000, "n_mels": n_mels, "sha256": sha(x), "full": False})

    # (3) ragged edge lengths (pad / trim semantics), speech-like content
    for n_mels in (80, 128):
        for li, L in enumerate(RAGGED_LENGTHS):
            seed = 3000 + li
            x = synth_clip("speech", L, seed)
            name = f"ragged_{L}_m{n_mels}"
            store[name + "_default"] = hf_features([x], n_mels, "default")[0][:, FRAME_SUBSAMPLE]
            meta["cases"].append({"name": name, "kind": "ragged", "family": "speech", "seed": seed,
                                  "n": L, "n_mels": n_mels, "sha256": sha(x), "full": False})

    # (4) the mel tables themselves (fp64, as the ctor builds them)
    from oracle.hf_reference import make_hf_extractor
    for n_mels in (80, 128):
        store[f"mel_filters_m{n_mels}"] = make_hf_extractor(n_mels).mel_filters

    store["meta_json"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    out = os.path.join(ROOT, "tests", "golden", "logmel_golden.npz")
    np.savez_compressed(out, **store)
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "logmel_golden_numpy.npz"), **numpy_path)
    print(out, os.path.getsize(out) / 1e6, "MB", len(meta["cases"]), "cases")


if __name__ == "__main__":
    main()
