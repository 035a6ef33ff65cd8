"""Cost of `do_normalize` and `dither` (`wlm_logmel_conditioned`) on one GPU; prints ONE JSON line.

    python tools/conditioning_bench.py [--iters 10] [--rounds 3]

Workloads (device-resident float32 PCM larger than the 126 MB L2; CUDA events around `iters` calls after a warm-up; the
entry points alternate `rounds` times and the best round is reported, every round is in the line):
  30s   256 x 30 s, 80 mels: wlm_logmel, wlm_logmel_padded (L = 480000), conditioned with normalise, with dither, with both
  20min 4 x 20 min, 128 mels: wlm_logmel_padded, conditioned with normalise, with dither, with both
and, on the same tensors, HF's device-resident torch operations as the baseline: the normalisation of
zero_mean_unit_var_norm (mean, population variance, (x - mean) / sqrt(var + 1e-7)), `+ dither * torch.randn`, then
TF-FE:141-161 (stft, |.|^2, mel matmul, clamp + log10, per-clip max, affine).
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from longform_bench import gpu_info, time_ms, torch_logmel  # noqa: E402

SR = 16000
DITHER = 1e-4


def torch_conditioned(x, filters_t, window, do_normalize=False, dither=0.0):
    import torch

    if do_normalize:
        mean = x.mean(dim=1, keepdim=True)
        var = x.var(dim=1, keepdim=True, unbiased=False)
        x = (x - mean) / torch.sqrt(var + 1e-7)
    if dither:
        x = x + dither * torch.randn(x.shape, dtype=x.dtype, device=x.device)
    return torch_logmel(x, filters_t, window)


def main():
    import numpy as np
    import torch

    from whisper_context_biasing_b200 import B200WhisperFeatureExtractor, slaney_mel_filters

    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    res = {"metric": "conditioning_audio_s_per_s", **gpu_info(), "iters": args.iters, "rounds": args.rounds,
           "dither": DITHER}
    g = torch.Generator(device=dev).manual_seed(1)
    window = torch.hann_window(400, device=dev)
    conds = {"normalize": dict(do_normalize=True, dither=0.0), "dither": dict(dither=DITHER),
             "both": dict(do_normalize=True, dither=DITHER)}
    for tag, B, N, m in (("30s", 256, 480000, 80), ("20min", 4, 1200 * SR, 128)):
        e = B200WhisperFeatureExtractor(feature_size=m, device=dev)
        filt = torch.from_numpy(slaney_mel_filters(m).astype(np.float32)).to(dev).T.contiguous()
        x = 0.1 * torch.randn(B, N, device=dev, generator=g)
        out = torch.empty(B, m, N // 160, device=dev)
        fns = {}
        if N == 480000:
            fns["wlm_logmel"] = lambda: e.extract_device(x, out=out)
        fns["padded"] = lambda: e.extract_device(x, out=out, padded_len=N)
        for k, c in conds.items():
            fns["cond_" + k] = (lambda c=c: e.extract_device(x, out=out, padded_len=N, seed=5, **c))
        times = {k: [] for k in fns}
        for _ in range(args.rounds):
            for k, fn in fns.items():
                times[k].append(time_ms(fn, args.iters))
        audio = B * N / SR
        for k, ts in times.items():
            res[f"{tag}_{k}_ms"] = [round(t, 3) for t in ts]
            res[f"{tag}_{k}_audio_s_per_s"] = round(audio / (min(ts) / 1e3))
        base = min(times["padded"])
        for k in conds:
            res[f"{tag}_cond_{k}_over_padded"] = round(min(times["cond_" + k]) / base, 3)
        for k, c in {"none": dict(do_normalize=False, dither=0.0), **conds}.items():
            tt = time_ms(lambda: torch_conditioned(x, filt, window, **c), max(2, args.iters // 2), warmup=1)
            res[f"{tag}_torch_{k}_ms"] = round(tt, 3)
            res[f"{tag}_torch_{k}_audio_s_per_s"] = round(audio / (tt / 1e3))
            if k != "none":
                res[f"{tag}_torch_over_cond_{k}"] = round(tt / min(times["cond_" + k]), 2)
        del x, out
        e.close()
        torch.cuda.empty_cache()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
