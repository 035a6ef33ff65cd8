"""PCM-returning dataset (SURVEY 8f rank 1, second half) against a golden produced by the reference's OWN
`PromptWhisperDataset` (tests/golden/make_dataset_golden.py).  Token ids are integers: exact.  The reference's source is
not part of this repository, so its class is replaced by a stand-in that makes the same feature-extractor call
(REF/data_utils/data_loader.py:170-172) and hands back the labels and bias spans the reference item carried; everything
the wrapper itself produces is compared with the golden."""
import hashlib
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, GOLD)


def _golden():
    z = np.load(os.path.join(GOLD, "dataset_golden.npz"))
    return z, json.loads(bytes(z["meta_json"]).decode())


def test_passthrough_extractor_contract():
    from whisper_context_biasing_b200 import PcmPassthroughExtractor

    pt = PcmPassthroughExtractor()
    x = np.arange(7, dtype=np.float64)
    out = pt(x, sampling_rate=16000).input_features           # REF/data_utils/data_loader.py:171
    assert len(out) == 1 and out[0].dtype == np.float32 and np.array_equal(out[0], x.astype(np.float32))
    with pytest.raises(ValueError):
        pt(x, sampling_rate=8000)


def test_pcm_dataset_matches_reference_dataset():
    import torch

    pytest.importorskip("transformers")                       # the synthetic tokenizer is a WhisperTokenizer
    from make_collator_golden import synthetic_tokenizer
    from make_dataset_golden import STRATEGIES, synth_audio_for

    from oracle import logmel_oracle as O
    from whisper_context_biasing_b200 import pcm_dataset_class

    z, meta = _golden()
    rows = [json.loads(l) for l in open(os.path.join(GOLD, "dataset_golden_rows.jsonl"))]
    tok = synthetic_tokenizer()
    loads = []

    class ReferenceStandIn:
        """The constructor and `__getitem__` of the reference class as far as the wrapper relies on them: records with
        the bias words at index 4 (what `bias_spans_only` reads), one audio load and one extractor call per item."""

        def __init__(self, base_path, jsonl_data, phase, feature_extractor, tokenizer, audio_type=".mp3",
                     gold_items=(), **kwargs):
            self.base_path, self.phase = base_path, phase
            self.feature_extractor, self.tokenizer = feature_extractor, tokenizer
            self.data = [(r["file"], r["text"], r["description"], r["id"], r["bias_words"]) for r in rows]
            self.gold_items = gold_items

        def __len__(self):
            return len(self.data)

        def __getitem__(self, i):
            path = os.path.join(self.base_path, self.phase, self.data[i][0])
            loads.append(path)
            audio, sr = synth_audio_for(path)                                        # librosa.load stand-in
            processed_audio = self.feature_extractor(audio, sampling_rate=sr).input_features      # :171
            g = self.gold_items[i]
            return {"input_features": torch.tensor(processed_audio[0]),                            # :172
                    "labels": torch.tensor(g["labels"]), "bias_spans": g["bias_spans"]}

    Pcm = pcm_dataset_class(ReferenceStandIn)
    sentinel = object()                                        # the device extractor is only carried along
    for name, kw in STRATEGIES.items():
        gold = meta["strategies"][name]["items"]
        ds = Pcm("/nonexistent", "rows", "test", sentinel, tok, audio_type=".mp3", gold_items=gold, **kw)
        assert ds.device_feature_extractor is sentinel and len(ds) == meta["n"]
        n0 = len(loads)
        spans = ds.all_bias_spans()                            # train.py:163 / evaluation.py:147 without the audio
        assert len(loads) == n0
        for i in range(len(ds)):
            assert spans[i] == gold[i]["bias_spans"], (name, i)   # the restated tokenisation == the reference's spans
            n0 = len(loads)
            it = ds[i]
            assert len(loads) == n0 + 1
            assert set(it) == {"audio", "labels", "bias_spans"}
            assert [int(x) for x in it["labels"]] == gold[i]["labels"], (name, i)
            assert [[int(t) for t in s] for s in it["bias_spans"]] == gold[i]["bias_spans"]
            a = it["audio"]
            assert a.dtype == np.float32 and a.ndim == 1 and a.shape[0] == gold[i]["n"]
            assert hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest() == gold[i]["pcm_sha256"]
            if i < 3:      # the PCM item carries exactly the audio whose features the reference item carried
                ref = z[f"{name}_{i}_features_sub"]
                got = O.extract([a], 80, "f32")[0][:, ::37]
                assert np.abs(got - ref).max() <= 1e-4
