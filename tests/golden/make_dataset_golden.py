"""Golden fixture for the PCM dataset row (SURVEY.md section 8f rank 1, second half), generated with the REFERENCE'S OWN
`PromptWhisperDataset` (REF/data_utils/data_loader.py:58-376) imported here with stub modules for its three missing
imports (librosa / av / editdistance; `librosa.load` returns seeded synthetic PCM -- the audio files are absent,
REF/.gitignore:1-4) and the synthetic byte-level tokenizer of make_collator_golden.py.

Rows 0..11 of REF/data/medical-united-syn-med-test-jsonl/test.jsonl, all four prompt strategies (:186-366), phase "test"
(no random perturbation).  Stored: labels and bias_spans of every item, the sha256 of the PCM the reference extractor was
given, and a frame-subsampled copy of the features the reference item carried.

Usage:                  python tests/golden/make_dataset_golden.py REFERENCE_CHECKOUT
Output:                 tests/golden/dataset_golden.npz  (+ dataset_golden_rows.jsonl, the 12 metadata rows)
"""
import hashlib
import importlib.util
import json
import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
STRATEGIES = {"desc": dict(prompt=True, bias_list=False), "bias": dict(prompt=False, bias_list=True, bias_nums=4),
              "desc_bias": dict(prompt=True, bias_list=True, bias_nums=4), "none": dict(prompt=False, bias_list=False)}


def synth_audio_for(path, sr=16000):
    """Deterministic stand-in for `librosa.load(path, sr=16000)`: speech-like noise, 1-9 s, seeded by the file name."""
    from oracle import logmel_oracle as O

    seed = int(hashlib.sha256(os.path.basename(path).encode()).hexdigest()[:8], 16)
    n = 16000 + seed % (8 * 16000)
    return O.synth_clip("speech", n, seed % 100000), sr


def import_reference_dataset(ref):
    """The reference module with stubs for the imports that are missing offline (SURVEY 8c)."""
    import importlib.machinery

    import transformers  # noqa: F401  (before the stubs: its availability probes choke on spec-less modules)

    stubs = {}
    for name in ("librosa", "av", "editdistance"):
        if name not in sys.modules:
            m = types.ModuleType(name)
            m.__spec__ = importlib.machinery.ModuleSpec(name, None)
            stubs[name] = sys.modules[name] = m
    sys.modules["librosa"].load = lambda path, sr=16000: synth_audio_for(path, sr)
    try:
        spec = importlib.util.spec_from_file_location("ref_data_loader", os.path.join(ref, "data_utils", "data_loader.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        for name in stubs:                       # the reference module keeps its own references; nobody else sees them
            sys.modules.pop(name, None)
    return mod


def main(ref):
    import random

    import torch
    from make_collator_golden import synthetic_tokenizer
    from transformers import WhisperFeatureExtractor

    tok = synthetic_tokenizer()
    mod = import_reference_dataset(ref)
    gold_dir = os.path.join(ROOT, "tests", "golden")
    rows = [json.loads(l) for l in open(os.path.join(ref, "data", "medical-united-syn-med-test-jsonl", "test.jsonl"))][:12]
    with open(os.path.join(gold_dir, "dataset_golden_rows.jsonl"), "w") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")
    jsonl_dir = os.path.join(gold_dir, "_dataset_tmp")
    os.makedirs(jsonl_dir, exist_ok=True)
    with open(os.path.join(jsonl_dir, "test.jsonl"), "w") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")
    store, meta = {}, {"strategies": {}, "n": len(rows), "pad": int(tok.pad_token_id),
                       "sot": int(tok.convert_tokens_to_ids("<|startoftranscript|>")),
                       "prev": int(tok.convert_tokens_to_ids("<|startofprev|>"))}
    hf = WhisperFeatureExtractor()
    for name, kw in STRATEGIES.items():
        random.seed(0)
        torch.manual_seed(0)
        ds = mod.PromptWhisperDataset("/nonexistent", jsonl_dir, "test", hf, tok, audio_type=".mp3", **kw)
        items = []
        for i in range(len(ds)):
            random.seed(100 + i)          # bias-list sampling inside __getitem__ uses `random`
            torch.manual_seed(100 + i)
            it = ds[i]
            audio, _ = synth_audio_for(os.path.join("/nonexistent", "test", rows[i]["file"]))
            store[f"{name}_{i}_features_sub"] = it["input_features"].numpy()[:, ::37].copy()
            items.append({"labels": [int(x) for x in it["labels"]], "bias_spans": [[int(t) for t in s] for s in it["bias_spans"]],
                          "pcm_sha256": hashlib.sha256(np.ascontiguousarray(audio).tobytes()).hexdigest(), "n": int(audio.shape[0])})
        meta["strategies"][name] = {"kwargs": kw, "items": items}
    os.remove(os.path.join(jsonl_dir, "test.jsonl"))
    os.rmdir(jsonl_dir)
    store["meta_json"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    out = os.path.join(gold_dir, "dataset_golden.npz")
    np.savez_compressed(out, **store)
    print(out, os.path.getsize(out), "bytes")


if __name__ == "__main__":
    main(sys.argv[1])
