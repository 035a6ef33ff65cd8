"""Long-form log-mel throughput (`wlm_logmel_padded`) on one GPU; prints ONE JSON line.

    python tools/longform_bench.py [--iters 10] [--rounds 3]

Cases (inputs are larger than the 126 MB L2 and device-resident; CUDA events around `iters` calls after a warm-up):
  a  the 30-s batch of bench.py's C2 config (256 x 30 s, 80 mels, float32 out) through wlm_logmel and through
     wlm_logmel_padded at L = 480000, alternated `rounds` times: what the generality of the long-form kernel costs
  b  32 x 10 min dense, 80 and 128 mels
  c  64 ragged clips of 1 to 20 min (seeded), 80 mels: true audio-s/s (sum of the clip lengths) and padded audio-s/s
     (B x L, what the features cover)
  d  the device-resident torch operations of TF-FE:141-161 (stft, |.|^2, mel matmul, clamp + log10, per-clip max,
     affine) on the same tensors as b and c: the baseline the kernels must beat
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SR = 16000


def gpu_info():
    import torch

    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"], info["sm_clock_idle"] = [s.strip() for s in q.split(",")]
    except Exception as e:         # the numbers stay without their context: say so in the line
        info["nvidia_smi_error"] = str(e)
    return info


def time_ms(fn, iters, warmup=2):
    import torch

    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(iters):
        fn()
    t1.record()
    t1.synchronize()
    return t0.elapsed_time(t1) / iters


def torch_logmel(x, filters_t, window):
    """TF-FE:141-161 on a device-resident [B, L] float32 batch."""
    import torch

    stft = torch.stft(x, 400, 160, window=window, return_complex=True)
    mag = stft[..., :-1].abs() ** 2
    mel = filters_t @ mag
    log_spec = torch.clamp(mel, min=1e-10).log10()
    mx = log_spec.amax(dim=(1, 2), keepdim=True)
    log_spec = torch.maximum(log_spec, mx - 8.0)
    return (log_spec + 4.0) / 4.0


def main():
    import numpy as np
    import torch

    from whisper_context_biasing_b200 import B200WhisperFeatureExtractor, slaney_mel_filters

    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    res = {"metric": "longform_audio_s_per_s", **gpu_info(), "iters": args.iters}
    g = torch.Generator(device=dev).manual_seed(1)
    ex = {m: B200WhisperFeatureExtractor(feature_size=m, device=dev) for m in (80, 128)}
    window = torch.hann_window(400, device=dev)
    filt = {m: torch.from_numpy(slaney_mel_filters(m).astype(np.float32)).to(dev).T.contiguous() for m in (80, 128)}

    # (a) the 30-s batch through both entry points, alternated
    x = 0.1 * torch.randn(256, 480000, device=dev, generator=g)
    out = torch.empty(256, 80, 3000, device=dev)
    a30, apad = [], []
    for _ in range(args.rounds):
        a30.append(time_ms(lambda: ex[80].extract_device(x, out=out), args.iters))
        apad.append(time_ms(lambda: ex[80].extract_device(x, out=out, padded_len=480000), args.iters))
    audio = 256 * 30.0
    res["a_30s_path_audio_s_per_s"] = [round(audio / (t / 1e3)) for t in a30]
    res["a_padded_480000_audio_s_per_s"] = [round(audio / (t / 1e3)) for t in apad]
    res["a_padded_over_30s"] = round(min(a30) / min(apad), 3)
    del x, out

    # (b) 32 x 10 min dense
    N = 600 * SR
    x = 0.1 * torch.randn(32, N, device=dev, generator=g)
    for m in (80, 128):
        out = torch.empty(32, m, N // 160, device=dev)
        t = time_ms(lambda: ex[m].extract_device(x, out=out, padded_len=N), args.iters)
        tt = time_ms(lambda: torch_logmel(x, filt[m], window), max(2, args.iters // 2), warmup=1)
        res[f"b_dense_10min_m{m}_audio_s_per_s"] = round(32 * 600.0 / (t / 1e3))
        res[f"d_torch_dense_10min_m{m}_audio_s_per_s"] = round(32 * 600.0 / (tt / 1e3))
        res[f"b_over_torch_m{m}"] = round(tt / t, 2)
        del out
    del x
    torch.cuda.empty_cache()

    # (c) 64 ragged clips of 1 to 20 min
    rng = np.random.default_rng(7)
    lens = rng.integers(60 * SR, 1200 * SR + 1, size=64)
    L = int(lens.max())
    starts = (lens + 3) // 4 * 4
    offs = np.concatenate([[0], np.cumsum(starts)[:-1]]).astype(np.int64)
    buf = torch.zeros(int(starts.sum()) + 4, device=dev)
    dense = torch.zeros(64, L, device=dev)
    for b in range(64):
        v = 0.1 * torch.randn(int(lens[b]), device=dev, generator=g)
        buf[offs[b]:offs[b] + lens[b]] = v
        dense[b, :lens[b]] = v
    lens_d = torch.from_numpy(lens.astype(np.int32)).to(dev)
    offs_d = torch.from_numpy(offs).to(dev)
    out = torch.empty(64, 80, L // 160, device=dev)
    t = time_ms(lambda: ex[80].extract_device(buf, lengths=lens_d, offsets=offs_d, out=out, padded_len=L), args.iters)
    tt = time_ms(lambda: torch_logmel(dense, filt[80], window), max(2, args.iters // 2), warmup=1)
    res["c_ragged_true_audio_s_per_s"] = round(float(lens.sum()) / SR / (t / 1e3))
    res["c_ragged_padded_audio_s_per_s"] = round(64 * L / SR / (t / 1e3))
    res["d_torch_ragged_padded_audio_s_per_s"] = round(64 * L / SR / (tt / 1e3))
    res["c_over_torch"] = round(tt / t, 2)
    # padded-audio rates over the 30-s path's rate of (a): what the long-form kernel gives up for its generality
    best30 = max(res["a_30s_path_audio_s_per_s"])
    res["b_m80_over_a_30s"] = round(res["b_dense_10min_m80_audio_s_per_s"] / best30, 3)
    res["c_padded_over_a_30s"] = round(res["c_ragged_padded_audio_s_per_s"] / best30, 3)
    for e in ex.values():
        e.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
