"""DataLoader throughput with audio decoding in the loop; prints ONE JSON line.

    python tools/loader_bench.py [--workers 4] [--batch 16] [--batches 24] [--warmup 3] [--arms a,b,c]

The dataset stands in for the reference's `__getitem__` (`librosa.load(path, sr=16000)`): each item resamples a seeded
44.1 kHz clip to 16 kHz with `scipy.signal.resample_poly(x, 160, 441)`, the polyphase filter a decoder's resampler runs,
and returns the PCM.  Clip lengths follow the word-rate rule of bench.py's C4, d = clip(0.4 + words / 2.6, 1, 30) s, with
words uniform in [1, 25].  This is a synthetic stand-in: the cost of decoding real mp3 files is not measured here.

  a  the reference's setup: HF's `WhisperFeatureExtractor` featurises each item in `--workers` DataLoader workers, and the
     collator stacks the features there (CPU only; runs without a GPU)
  b  this library with 0 workers: decoding and the collator's in-process featurisation both run in the main process
  c  the deferred collator: decoding and PCM collation in `--workers` fork workers started after the main process made
     its plan, pinned by the loader, then `collator.finish` in the main process (one H2D copy, one ragged launch)

Per arm, after `--warmup` batches: `batches_per_s`, wall time over `--batches` batches (the GPU arms synchronise at the
end), and `main_ms_per_batch`, the main thread's CPU time per batch (`time.thread_time`): what the data path costs the
training loop's thread when nothing waits.  Waiting for workers is not in it.  The line names the GPU and its power
limit, and the host's CPU count.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

SOURCE_RATE = 44100
PAD, SOT = 50257, 50258


class DecodingDataset:
    """Item i: a seeded 44.1 kHz clip resampled to 16 kHz (the decoder's work), plus a label sequence."""

    def __init__(self, n, featurise=None):
        self.n = n
        self.featurise = featurise          # arm a: HF's extractor runs in __getitem__, as in the reference

    def __len__(self):
        return self.n

    def __getitem__(self, i):
        from scipy.signal import resample_poly

        rng = np.random.default_rng(i)
        words = int(rng.integers(1, 26))
        secs = float(np.clip(0.4 + words / 2.6, 1.0, 30.0))
        x = rng.standard_normal(int(secs * SOURCE_RATE)).astype(np.float32) * 0.1
        pcm = resample_poly(x, 160, 441).astype(np.float32)
        labels = [SOT] + rng.integers(0, 50000, 5 * words).tolist() + [PAD]
        if self.featurise is not None:
            return {"input_features": self.featurise(pcm, sampling_rate=16000).input_features[0], "labels": labels}
        return {"audio": pcm, "labels": labels}


class StackCollator:
    """Arm a's collator: the reference's stack of precomputed features plus the label half."""

    def __call__(self, features):
        import torch

        from whisper_context_biasing_b200.collator import collate_labels

        batch = {"input_features": torch.from_numpy(np.stack([f["input_features"] for f in features]))}
        batch.update(collate_labels(features, PAD, SOT, None))
        return batch


def run_arm(loader, finish, warmup, batches, sync):
    it = iter(loader)
    for _ in range(warmup):
        finish(next(it))
    sync()
    t0, c0 = time.perf_counter(), time.thread_time()
    for _ in range(batches):
        finish(next(it))
    sync()
    wall, cpu = time.perf_counter() - t0, time.thread_time() - c0
    return {"batches_per_s": round(batches / wall, 3), "main_ms_per_batch": round(1e3 * cpu / batches, 3)}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--workers", type=int, default=4)
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--batches", type=int, default=24)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--n-mels", type=int, default=80)
    ap.add_argument("--arms", default="a,b,c")
    args = ap.parse_args()
    arms = args.arms.split(",")

    import torch

    n = (args.warmup + args.batches) * args.batch
    out = {"workers": args.workers, "batch": args.batch, "batches": args.batches, "n_mels": args.n_mels,
           "cpus": len(os.sched_getaffinity(0)), "arms": {}}
    if "a" in arms:
        from transformers import WhisperFeatureExtractor

        hf = WhisperFeatureExtractor(feature_size=args.n_mels)
        loader = torch.utils.data.DataLoader(DecodingDataset(n, hf), batch_size=args.batch, num_workers=args.workers,
                                             collate_fn=StackCollator())
        out["arms"]["a_hf_in_workers"] = run_arm(loader, lambda b: b, args.warmup, args.batches, lambda: None)
    if "b" in arms or "c" in arms:
        from longform_bench import gpu_info

        from whisper_context_biasing_b200 import B200DataCollatorSpeechSeq2SeqWithPadding, B200WhisperFeatureExtractor

        fe = B200WhisperFeatureExtractor(feature_size=args.n_mels)
        col = B200DataCollatorSpeechSeq2SeqWithPadding(feature_extractor=fe, pad_token_id=PAD, decoder_start_token_id=SOT)
        sync = torch.cuda.synchronize
        out.update(gpu_info())
        if "b" in arms:
            loader = torch.utils.data.DataLoader(DecodingDataset(n), batch_size=args.batch, num_workers=0, collate_fn=col)
            out["arms"]["b_b200_0_workers"] = run_arm(loader, lambda b: b, args.warmup, args.batches, sync)
        if "c" in arms:
            loader = torch.utils.data.DataLoader(DecodingDataset(n), batch_size=args.batch, num_workers=args.workers,
                                                 collate_fn=col, pin_memory=True)
            out["arms"]["c_deferred_in_workers"] = run_arm(loader, col.finish, args.warmup, args.batches, sync)
        fe.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
