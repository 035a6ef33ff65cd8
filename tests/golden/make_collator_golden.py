"""Golden fixture for the collator row (SURVEY.md section 8f rank 1), generated with the REFERENCE'S OWN
`DataCollatorSpeechSeq2SeqWithPadding` (REF/data_utils/data_collator.py:27-127), imported here through
an offline shim (its module body calls `from_pretrained`, which needs the network).

Usage:                  python tests/golden/make_collator_golden.py REFERENCE_CHECKOUT
Output:                 tests/golden/collator_golden.npz
"""
import importlib.util
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _bytes_to_unicode():
    """GPT-2 byte <-> printable unicode table (the order Whisper's byte-level vocab uses)."""
    bs = list(range(ord("!"), ord("~") + 1)) + list(range(ord("\xa1"), ord("\xac") + 1)) + list(range(ord("\xae"), ord("\xff") + 1))
    cs = bs[:]
    n = 0
    for b in range(256):
        if b not in bs:
            bs.append(b)
            cs.append(256 + n)
            n += 1
    return dict(zip(bs, [chr(c) for c in cs]))


def synthetic_tokenizer():
    """Byte-level Whisper tokenizer with the special tokens in Whisper's order (no real vocab exists offline)."""
    from transformers import WhisperTokenizer
    from transformers.models.whisper.tokenization_whisper import LANGUAGES

    symbols = list(_bytes_to_unicode().values())
    specials = ["<|endoftext|>", "<|startoftranscript|>"] + [f"<|{k}|>" for k in LANGUAGES] + [
        "<|translate|>", "<|transcribe|>", "<|startoflm|>", "<|startofprev|>", "<|nospeech|>", "<|notimestamps|>"]
    vocab = {s: i for i, s in enumerate(symbols + specials)}
    tok = WhisperTokenizer(vocab=vocab, merges=[], pad_token="<|endoftext|>", language="en", task="transcribe")
    return tok


def import_reference_collator(ref, tok):
    from transformers import WhisperFeatureExtractor, WhisperTokenizer

    WhisperFeatureExtractor.from_pretrained = classmethod(lambda cls, *a, **k: cls())
    WhisperTokenizer.from_pretrained = classmethod(lambda cls, *a, **k: tok)
    spec = importlib.util.spec_from_file_location("ref_data_collator", os.path.join(ref, "data_utils", "data_collator.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def main(ref):
    from transformers import WhisperFeatureExtractor, WhisperProcessor

    tok = synthetic_tokenizer()
    mod = import_reference_collator(ref, tok)
    proc = WhisperProcessor(WhisperFeatureExtractor(), tok)
    sot = tok.convert_tokens_to_ids("<|startoftranscript|>")
    prev = tok.convert_tokens_to_ids("<|startofprev|>")
    rng = np.random.default_rng(7)
    store, cases = {}, []
    for ci, (B, with_spans, with_prev) in enumerate([(4, True, True), (3, True, False), (2, False, True), (5, True, True)]):
        feats = []
        for b in range(B):
            n_prompt = int(rng.integers(0, 12))
            n_text = int(rng.integers(1, 20))
            prompt = ([prev] + rng.integers(0, 256, n_prompt).tolist()) if n_prompt else []
            labels = prompt + [sot] + rng.integers(0, 256, n_text).tolist() + [tok.eos_token_id]
            f = {"input_features": np.full((80, 3000), float(b), np.float32), "labels": labels}
            if with_spans:
                n_sp = int(rng.integers(0, 4)) if not (ci == 3 and b == 0) else 0
                f["bias_spans"] = [rng.integers(0, 256, int(rng.integers(1, 6))).tolist() for _ in range(n_sp)]
            feats.append(f)
        coll = mod.DataCollatorSpeechSeq2SeqWithPadding(processor=proc, decoder_start_token_id=sot,
                                                        decoder_prev_token_id=prev if with_prev else None)
        out = coll(feats)
        name = f"case{ci}"
        store[name + "_labels_out"] = out["labels"].numpy()
        store[name + "_decoder_input_ids"] = out["decoder_input_ids"].numpy()
        if "bias_spans" in out:
            store[name + "_bias_spans_out"] = out["bias_spans"].numpy()
        assert tuple(out["input_features"].shape) == (B, 80, 3000) and out["input_features"].dtype == torch.float32
        cases.append({"name": name, "B": B, "with_prev": with_prev, "sot": int(sot), "prev": int(prev),
                      "pad": int(tok.pad_token_id),
                      "labels_in": [f["labels"] for f in feats],
                      "bias_spans_in": [f.get("bias_spans") for f in feats] if with_spans else None})
    store["meta_json"] = np.frombuffer(json.dumps({"cases": cases}).encode(), dtype=np.uint8)
    out_path = os.path.join(ROOT, "tests", "golden", "collator_golden.npz")
    np.savez_compressed(out_path, **store)
    print(out_path, os.path.getsize(out_path), "bytes", len(cases), "cases")


if __name__ == "__main__":
    main(sys.argv[1])
