#!/usr/bin/env python
"""Benchmark of the log-mel hot path (BASELINE.json metric: log-mel audio-seconds/second).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload c2|c3|c4] [--no-extras]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic PCM.  The headline workload is
BASELINE.json configs[1] (C2: whisper-small 80-mel, batch 256 x 30 s, device-resident PCM, one
B200).  With N > 1 (launched by torchrun, one rank per GPU) every rank processes its own C2 batch
-- the path shards by clip with no data-path collective -- so the headline scaling is WEAK and
`value` is the whole-job audio-seconds/second.  The same line carries, as extra objects measured
in the same run with the same rules:

    c3         BASELINE configs[2]: large-v3 128-mel, 1024 x 30 s sharded by clip over the N ranks (STRONG)
    c4         BASELINE configs[3]: 4096 variable-length clips (word-count histogram of the medical jsonl), ragged
    c1         BASELINE configs[0]: the reference's own call shape -- 16 per-clip calls + the collator's stack
    sustained  >= 2 s of back-to-back C2 launches with clock / power samples
    hf_cuda    Hugging Face's own device="cuda" branch of the extractor on the same batch (N = 1)
    cpu_baseline / cpu_baseline_numpy   the reference's CPU paths on this box's host cores (N = 1)

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for how every field is derived.

--dump-outputs DIR writes what the headline workload's last timed step computed, as the caller of the device path
receives it: DIR/input_features.npy, float32 [K, n_mels, 3000], the features of K clips of rank 0's batch drawn with
numpy's default_rng(0) (every clip while the batch fits in 60 MB, else as many as fit).  The PCM is generated from fixed
seeds, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes
import importlib.util
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark writes nothing into the tree it runs from

N_SAMPLES = 480000
N_FRAMES = 3000
CLIP_SECONDS = 30.0
DUMP_BYTES = 60_000_000

WORKLOADS = {
    "c2": dict(n_mels=80, batch=256, strong=False, profile="c2_80mel",
               label="C2: whisper-small 80-mel, batch 256 x 30 s f32 PCM per GPU (BASELINE configs[1])"),
    "c3": dict(n_mels=128, batch=1024, strong=True, profile="c3_128mel",
               label="C3: whisper-large-v3 128-mel, 1024 x 30 s sharded by clip (BASELINE configs[2])"),
    "c4": dict(n_mels=80, batch=4096, strong=True, variable=True, profile=None,
               label="C4: 4096 variable-length clips (1-30 s, word-count histogram of the medical jsonl) ragged, "
                     "pad/trim in-kernel (BASELINE configs[3])"),
}

# Transcript word-count histogram of REF/data/medical-united-syn-med-75-jsonl/test.jsonl (5114 rows; counts for 1..25
# words: min 1, p5 8, median 11, mean 11.26, p95 15, max 25).  The jsonl carries no durations and the audio is absent
# (REF/.gitignore:1-4), so SURVEY 8d's word-rate proxy d = clip(0.4 + words / 2.6, 1, 30) s stands in for the lengths.
C4_WORD_HIST = [4, 0, 0, 0, 2, 34, 100, 262, 673, 1008, 962, 724, 544, 356, 214, 129, 48, 23, 15, 8, 5, 0, 1, 0, 2]


def c4_lengths(n, seed=3):
    """SURVEY 8d C4: words ~ C4_WORD_HIST, d = clip(0.4 + words/2.6, 1, 30) s, plus a 2 % tail uniform 10-30 s and
    0.5 % at 35 s (exercises the trim).  Returns sample counts (multiples of 8: clips sit back to back in the buffer)."""
    import numpy as np

    rng = np.random.default_rng(seed)
    p = np.asarray(C4_WORD_HIST, dtype=np.float64)
    words = rng.choice(np.arange(1, 26), size=n, p=p / p.sum())
    d = np.clip(0.4 + words / 2.6, 1.0, 30.0)
    tail = rng.random(n)
    d = np.where(tail < 0.02, rng.uniform(10.0, 30.0, n), d)
    d = np.where(tail > 0.995, 35.0, d)
    return (d * 16000).astype(np.int64) // 8 * 8


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            d = json.load(open(path))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def _build_module():
    spec = importlib.util.spec_from_file_location("_wlm_build", os.path.join(ROOT, "whisper_context_biasing_b200", "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def profile_summary(profile):
    """profiles/<latest>_<profile>_summary.json written by tools/ncu_summary.py -- used only when it was taken from a
    build of exactly the kernel sources that are running now."""
    if not profile:
        return None, "no ncu capture for this workload"
    pdir = os.path.join(ROOT, "profiles")
    cands = sorted(f for f in os.listdir(pdir) if f.endswith(f"_{profile}_summary.json")) if os.path.isdir(pdir) else []
    if not cands:
        return None, "no profiles/*_summary.json"
    try:
        doc = json.load(open(os.path.join(pdir, cands[-1])))
        sha = _build_module().kernel_sources_sha()
    except Exception as e:     # noqa: BLE001
        return None, f"unreadable summary: {e}"
    if doc.get("kernel_sources_sha") != sha:
        return None, f"{cands[-1]} was taken from kernel sources {doc.get('kernel_sources_sha')}, running {sha}: not printed"
    return doc, cands[-1]


class ClockSampler(threading.Thread):
    """Samples SM clock, power and throttle reasons of one GPU through NVML while the timed region runs."""

    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index: int, period_s: float = 0.002):
        super().__init__(daemon=True)
        self.index, self.period = index, period_s
        self.samples, self.power, self.reasons, self.max_mhz = [], [], set(), None
        self._stop_ev = threading.Event()
        self.ok = False
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        while not self._stop_ev.is_set():
            try:
                self.samples.append(int(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
                self.power.append(self.nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                mask = int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                for bit, name in self.REASONS.items():
                    if mask & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_ev.set()
        if self.ok:
            self.join(timeout=2)
        s = sorted(self.samples)
        p = sorted(self.power)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s),
                "power_w": (round(p[len(p) // 2], 1) if p else None)}


def visible_nvml_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


def bind_rank_to_cores(local_rank: int, world: int):
    """One process per GPU: give every rank its own slice of the host cores, preferring the cores NVML reports as local
    to its GPU, BEFORE any pinned buffer is allocated (first touch then lands on the near NUMA node)."""
    try:
        avail = sorted(os.sched_getaffinity(0))
    except Exception:
        return None
    if world <= 1 or len(avail) < 2 * world:
        return {"cores": len(avail), "bound": False}
    near = None
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(visible_nvml_index(local_rank))
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (max(avail) // 64) + 1)
        near = [c for c in avail if (words[c // 64] >> (c % 64)) & 1]
    except Exception:
        near = None
    per = len(avail) // world
    mine = avail[local_rank * per:(local_rank + 1) * per]
    if near and len(near) < len(avail):          # the box has more than one NUMA domain: stay inside the GPU's
        inter = [c for c in mine if c in near]
        if not inter:
            k = len(near) // max(1, world // 2)
            inter = near[(local_rank % max(1, world // 2)) * k:][:max(1, k)]
        mine = inter or mine
    try:
        os.sched_setaffinity(0, mine)
        return {"cores": len(mine), "bound": True, "first": mine[0], "numa_local_cores": (len(near) if near else None)}
    except Exception:
        return {"cores": len(avail), "bound": False}


# ------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation (HF WhisperFeatureExtractor through a
# DataLoader shaped like REF/data_utils/data_loader.py:170-172 + data_collator.py:64-76)
# ------------------------------------------------------------------------------------------------
def synth_noise_clips(n, seed):
    import numpy as np

    rng = np.random.default_rng(seed)
    return [(0.1 * rng.standard_normal(N_SAMPLES)).astype(np.float32) for _ in range(n)]


def reference_sample_clips(batch, cores):
    """Bounded sample of the workload for the CPU arm: at least the batch, and at least 4 batches of 16 per worker so
    that every DataLoader worker is busy for the whole epoch."""
    n = max(batch, cores * 64)
    return (n + 15) // 16 * 16


def run_reference(args, wl, rank, world):
    if rank != 0:
        return
    from oracle.hf_reference import time_reference_dataloader

    cores = len(os.sched_getaffinity(0))
    clips_per_step = reference_sample_clips(min(wl["batch"], 1024), cores)
    base = synth_noise_clips(64, seed=1)
    clips = [base[i % len(base)] for i in range(clips_per_step)]
    r = time_reference_dataloader(clips, wl["n_mels"], 16, cores, "default", epochs=args.steps, warmup_epochs=max(1, min(args.warmup, 2)))
    t_total, n_total = sum(r["epoch_seconds"]), r["clips"] * len(r["epoch_seconds"])
    value = CLIP_SECONDS * n_total / t_total
    sample = (f"{clips_per_step} x 30 s white-noise clips per step through a torch DataLoader "
              f"(batch 16, {cores} persistent workers, 1 torch thread each) running the unmodified "
              f"transformers WhisperFeatureExtractor per clip + feature_extractor.pad stack")
    line = {
        "impl": "reference", "metric": "log-mel audio-seconds/second", "value": value, "unit": "audio-s/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t_total / max(1, args.steps), "higher_is_better": True,
        "scaling": "strong" if wl["strong"] else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["label"], "n_mels": wl["n_mels"], "sample_clips_per_step": clips_per_step},
        "cpu_baseline": {"value": value, "unit": "audio-s/s", "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": value, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def cpu_baseline(n_mels, path="default"):
    """The reference's CPU implementation on this box's host cores, bounded sample (~10-30 s of CPU work)."""
    from oracle.hf_reference import time_reference_dataloader

    cores = len(os.sched_getaffinity(0))
    n = reference_sample_clips(256, cores) if path == "default" else max(64, cores * 4) // 16 * 16
    base = synth_noise_clips(32, seed=1)
    clips = [base[i % len(base)] for i in range(n)]
    r = time_reference_dataloader(clips, n_mels, 16 if path == "default" else 4, cores, path, epochs=1, warmup_epochs=1)
    what = ("unmodified transformers WhisperFeatureExtractor (default dispatch: torch fp32 STFT, TF-FE:135-164)" if path == "default"
            else "forced numpy fp64 path of the same class (_np_extract_fbank_features, TF-FE:105-133)")
    return {"value": r["audio_s_per_s"], "unit": "audio-s/s", "cores": cores, "kind": "reference",
            "sample": f"{r['clips']} x 30 s white-noise clips, torch DataLoader, {cores} workers x 1 thread, "
                      f"{what} per clip + pad stack ({r['epoch_seconds'][0]:.1f} s)"}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
class Ctx:
    """Per-process measurement context: device, torch.distributed handle, barrier, extractors."""

    def __init__(self, rank, world, local_rank):
        import torch

        self.torch = torch
        self.rank, self.world, self.local_rank = rank, world, local_rank
        torch.cuda.set_device(local_rank)
        self.dev = torch.device("cuda", local_rank)
        self.dist = None
        self.json_fd = None
        if world > 1:
            import torch.distributed as dist_mod

            # NCCL writes "NCCL version ..." straight to file descriptor 1 (at any NCCL_DEBUG level): point fd 1 at
            # stderr for the duration of the run and keep the real stdout for the ONE JSON line
            sys.stdout.flush()
            self.json_fd = os.dup(1)
            os.dup2(2, 1)
            dist_mod.init_process_group(backend="nccl", device_id=self.dev)
            self.dist = dist_mod
        self.fes = {}

    def fe(self, n_mels):
        import whisper_context_biasing_b200 as W

        if n_mels not in self.fes:
            self.fes[n_mels] = W.B200WhisperFeatureExtractor(feature_size=n_mels, device=self.dev)
        return self.fes[n_mels]

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, vals):
        if self.dist is None:
            return [float(v) for v in vals]
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    def emit(self, line):
        if self.rank != 0:
            return
        if self.json_fd is not None:
            os.write(self.json_fd, (json.dumps(line) + "\n").encode())
        else:
            print(json.dumps(line), flush=True)

    def close(self):
        for f in self.fes.values():
            f.close()
        if self.dist is not None:
            self.dist.barrier()
            self.dist.destroy_process_group()


def make_workload(cx: Ctx, wl):
    """Synthetic PCM of the workload's shape (family F1, white Gaussian sigma 0.1), generated on the host into ONE pinned
    buffer, plus a device-resident copy.  Strong workloads take this rank's contiguous clip shard."""
    import numpy as np

    from whisper_context_biasing_b200.sharding import clip_shard

    torch = cx.torch
    n_mels = wl["n_mels"]
    if wl["strong"]:
        lo, hi = clip_shard(wl["batch"], cx.rank, cx.world)
    else:
        lo, hi = 0, wl["batch"]
    B = hi - lo
    g = torch.Generator(device="cpu").manual_seed(1000 + cx.rank)
    w = dict(B=B, n_mels=n_mels, total_clips=(wl["batch"] if wl["strong"] else B * cx.world), wl=wl)
    if not wl.get("variable"):
        host = torch.empty((B, N_SAMPLES), dtype=torch.float32).pin_memory()
        torch.randn((B, N_SAMPLES), generator=g, out=host)
        host.mul_(0.1)
        w["pcm"] = host.to(cx.dev, non_blocking=True)
        w["clips"] = host.numpy()                      # dense host batch [B, 480000]: no per-clip Python work in the call
        w["true_audio_s"] = CLIP_SECONDS * B
        w["in_bytes"] = B * N_SAMPLES * 4
        w["lengths"] = w["offsets"] = None
    else:
        lens = c4_lengths(wl["batch"])[lo:hi]
        offs = np.zeros(B, dtype=np.int64)
        offs[1:] = np.cumsum((lens[:-1] + 7) // 8 * 8)
        total = int(offs[-1] + (lens[-1] + 7) // 8 * 8)
        host = torch.empty((total,), dtype=torch.float32).pin_memory()
        torch.randn((total,), generator=g, out=host)
        host.mul_(0.1)
        w["pcm"] = host.to(cx.dev, non_blocking=True)
        w["offsets"] = torch.from_numpy(offs).to(cx.dev)
        w["lengths"] = torch.from_numpy(lens.astype(np.int32)).to(cx.dev)
        w["clips"] = (host.numpy(), offs, np.minimum(lens, 2 ** 31 - 1).astype(np.int32))   # (buffer, offsets, lengths)
        w["host_offsets"] = offs
        w["true_audio_s"] = float(np.minimum(lens, N_SAMPLES).sum()) / 16000.0
        w["in_bytes"] = int(np.minimum(lens, N_SAMPLES).sum()) * 4
    w["host"] = host
    w["out"] = torch.empty((B, n_mels, N_FRAMES), dtype=torch.float32, device=cx.dev)
    torch.cuda.synchronize(cx.dev)
    return w


def dump_sample(B, n_mels):
    """Sorted clip indices of the --dump-outputs sample: all B clips, or a seeded draw of as many as fit in DUMP_BYTES."""
    import numpy as np

    k = min(B, DUMP_BYTES // (n_mels * N_FRAMES * 4))
    return np.sort(np.random.default_rng(0).choice(B, size=k, replace=False))


def measure(cx: Ctx, w, steps, warmup, e2e=True, e2e_extra=False, sample=None):
    """Device-resident and end-to-end timing of one workload on this rank; returns the fields of its JSON object
    (max over ranks applied).  With `sample` (clip indices), res["_outputs"] holds those clips' features from the last
    timed step."""
    torch = cx.torch
    fe = cx.fe(w["n_mels"])
    B, n_mels, out = w["B"], w["n_mels"], w["out"]
    pcm, lengths, offsets = w["pcm"], w["lengths"], w["offsets"]

    def run_device():
        fe.extract_device(pcm, lengths=lengths, offsets=offsets, out=out)

    # ---- device-resident: PCM already in HBM -------------------------------------------------
    for _ in range(max(warmup, 3)):
        run_device()
    cx.barrier()
    sampler = ClockSampler(visible_nvml_index(cx.local_rank))
    sampler.start()
    launches0 = fe.launch_count
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for s in range(steps):
        run_device()
    t1.record()
    cx.barrier()
    clocks = sampler.stop()
    launches = fe.launch_count - launches0
    dev_ms = t0.elapsed_time(t1)
    launch_ms = dev_ms / steps        # back-to-back launches between two events on the launch stream: the average step

    res = {}
    if sample is not None:          # copied now: the end-to-end legs below write into `out` again
        res["_outputs"] = {"input_features": out[torch.from_numpy(sample).to(cx.dev)].cpu().numpy()}

    # ---- end to end: pinned host PCM -> H2D -> kernels -> D2H of one float per clip --------------
    e2e_steps = max(2, min(steps, 5))
    gmax_host = torch.empty((max(B, 1),), dtype=torch.float32).pin_memory()
    clips = w["clips"]

    def timed(step_fn, n):
        for _ in range(2):
            step_fn()
        cx.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.perf_counter()
        e0.record()
        for _ in range(n):
            step_fn()
        e1.record()
        cx.barrier()
        return e0.elapsed_time(e1), 1e3 * (time.perf_counter() - w0)

    e2e_ms = e2e_wall = e2e16_ms = e2enp_ms = h2d_ms = float("nan")
    if e2e:
        def e2e_step():
            fe.extract_host(clips, out=out)
            gmax_host[:B].copy_(out[:, 0, 0], non_blocking=True)      # D2H read of the step's result
            torch.cuda.current_stream(cx.dev).synchronize()

        e2e_ms, e2e_wall = timed(e2e_step, e2e_steps)

        # H2D-only probe: the same pinned bytes, the same chunking, no kernel -- the ceiling the host side allows
        stage = torch.empty_like(w["host"], device=cx.dev)

        def h2d_step():
            stage.copy_(w["host"], non_blocking=True)
            torch.cuda.current_stream(cx.dev).synchronize()

        h2d_ms, _ = timed(h2d_step, e2e_steps)
        del stage
    if e2e and e2e_extra:
        import numpy as np

        # int16 ingest (SURVEY 8f rank 2): half the H2D bytes, x/32768 on the GPU
        h16 = torch.empty((w["host"].numel(),), dtype=torch.int16).pin_memory()
        h16.copy_((w["host"].reshape(-1) * 32767.0).round().to(torch.int16))
        a16 = h16.numpy()
        c16 = a16.reshape(B, N_SAMPLES) if w["offsets"] is None else (a16, clips[1], clips[2])

        def e2e16_step():
            fe.extract_host(c16, out=out)
            gmax_host[:B].copy_(out[:, 0, 0], non_blocking=True)
            torch.cuda.current_stream(cx.dev).synchronize()

        e2e16_ms, _ = timed(e2e16_step, e2e_steps)
        del h16, a16, c16
        # the reference's return contract (a host ndarray): features copied back inside the call
        host_out = torch.empty((B, n_mels, N_FRAMES), dtype=torch.float32).pin_memory()
        host_np = host_out.numpy()

        def e2enp_step():
            fe.extract_host(clips, out=out, out_host=host_np)

        e2enp_ms, _ = timed(e2enp_step, e2e_steps)
        del host_out, host_np

    dev_ms, launch_ms, e2e_ms, e2e_wall, e2e16_ms, e2enp_ms, h2d_ms = cx.max_over_ranks(
        [dev_ms, launch_ms, e2e_ms, e2e_wall, e2e16_ms, e2enp_ms, h2d_ms])

    total_clips = w["total_clips"]
    peak, peak_src = measured_peaks()
    in_bytes = w["in_bytes"]
    out_bytes = n_mels * N_FRAMES * 4 * B
    alg_bytes = in_bytes + out_bytes                # SURVEY 8d: valid PCM read + full output written
    achieved = alg_bytes / (launch_ms * 1e-3) / 1e9
    prof, prof_note = profile_summary(w["wl"].get("profile"))
    res["value"] = CLIP_SECONDS * total_clips * steps / (dev_ms * 1e-3)
    res["ms_per_step"] = dev_ms / steps
    res["config"] = {"workload": w["wl"]["label"], "n_mels": n_mels, "clips_per_gpu": B, "clip_seconds": 30,
                     "true_audio_seconds_per_gpu": w["true_audio_s"],
                     "l2_policy": f"inputs larger than L2: {in_bytes / 1e6:.0f} MB PCM + {out_bytes / 1e6:.0f} MB features per step",
                     "timing": "CUDA events on the launch stream, barrier + synchronize both sides, max over ranks"}
    res["gpu_launches"] = int(launches)
    res["roofline"] = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                       "traffic": (int(prof["dram_bytes_per_step"] * B / prof["clips"]) if prof and prof.get("clips") else None),
                       "traffic_source": prof_note, "peak_source": peak_src,
                       "algorithmic_bytes_per_launch": alg_bytes, "launch_ms": launch_ms}
    res["clocks"] = clocks
    res["_prof"] = prof
    res["_launch_ms"] = launch_ms
    if e2e:
        h2d_gbs = in_bytes / (h2d_ms / e2e_steps * 1e-3) / 1e9
        e2e_value = CLIP_SECONDS * total_clips * e2e_steps / (e2e_ms * 1e-3)
        res["e2e"] = {"value": e2e_value, "unit": "audio-s/s", "h2d_bytes_per_step": in_bytes + B * 12,
                      "d2h_bytes_per_step": B * 4, "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps,
                      "wall_ms_per_step": e2e_wall / e2e_steps,
                      "roofline": {"bound": "pcie-h2d", "h2d_gbs_measured": h2d_gbs,
                                   "achieved_gbs": in_bytes / (e2e_ms / e2e_steps * 1e-3) / 1e9,
                                   "frac": (h2d_ms / e2e_ms),
                                   "how": "H2D-only probe: the same pinned bytes copied without any kernel, same ranks "
                                          "at the same time; frac = probe time / end-to-end time (1.0 = the library adds "
                                          "nothing to the copy)"},
                      "what": "wlm_logmel_host: pinned host f32 PCM -> chunked H2D overlapped with the kernels -> "
                              "features stay in HBM; D2H of one float per clip"}
        if e2e_extra:
            res["e2e_int16"] = {"value": CLIP_SECONDS * total_clips * e2e_steps / (e2e16_ms * 1e-3), "unit": "audio-s/s",
                                "h2d_bytes_per_step": in_bytes // 2 + B * 12, "d2h_bytes_per_step": B * 4,
                                "what": "same step with int16 PCM in pinned host memory (an optional ingest path, "
                                        "bit-identical to float(x)/32768; half the H2D bytes)"}
            res["e2e_numpy_contract"] = {"value": CLIP_SECONDS * total_clips * e2e_steps / (e2enp_ms * 1e-3), "unit": "audio-s/s",
                                         "h2d_bytes_per_step": in_bytes + B * 12, "d2h_bytes_per_step": out_bytes,
                                         "what": "same step returning the features to a pinned host array, as the reference's "
                                                 "return contract (output='numpy') requires: + full D2H"}
    return res


ALGORITHMIC_MFLOP_PER_CLIP = {80: 32.49, 128: 33.23}     # SURVEY 8d convention


def fp32_roofline(cx, res, n_mels, B):
    """FP32 CUDA-core side of the roofline: SURVEY 8d's algorithmic flops / launch time against the MEASURED FFMA peak
    (tools/libwlm_ubench.so on this very GPU), with the nominal figure beside it and the ncu pipe counters of the
    committed capture when it belongs to the running kernels."""
    sm_mhz = float((res.get("clocks") or {}).get("sm_max_mhz") or 1965.0)
    nominal = 148 * 128 * 2 * sm_mhz * 1e6 / 1e12
    measured = None
    try:
        lib = ctypes.CDLL(os.path.join(ROOT, "tools", "libwlm_ubench.so"))
        lib.wlm_ubench_ffma_tflops.restype = ctypes.c_double
        lib.wlm_ubench_ffma_tflops.argtypes = [ctypes.c_int, ctypes.c_int]
        v = float(lib.wlm_ubench_ffma_tflops(cx.local_rank, 5))
        measured = v if v > 0 else None
    except OSError:
        measured = None
    ach = ALGORITHMIC_MFLOP_PER_CLIP[n_mels] * 1e6 * B / (res["_launch_ms"] * 1e-3) / 1e12
    peak = measured or nominal
    o = {"bound": "fp32-cuda-core", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
         "peak_source": ("measured: scalar FFMA chains on every SM (tools/ubench_peak.cu), best of 5" if measured
                         else "nominal: 148 SMs x 128 lanes x 2 x max SM clock (tools/libwlm_ubench.so missing)"),
         "peak_nominal": nominal,
         "note": "the FFT is add-heavy (FADD2 = one issue, two lanes, no multiply): the FMA-pipe counter, not the flop "
                 "fraction, says how busy the CUDA cores are"}
    prof = res.get("_prof")
    if prof:
        k = max(prof["kernels"], key=lambda k: k.get("gpu__time_duration.sum", 0))
        o["ncu_pct_of_peak_while_active"] = {
            "fma_pipe": k.get("sm__pipe_fma_cycles_active.avg.pct_of_peak_sustained_active"),
            "shared_memory_wavefronts_elapsed": k.get("l1tex__data_pipe_lsu_wavefronts_mem_shared.sum.pct_of_peak_sustained_elapsed"),
            "issue_slots": k.get("smsp__issue_active.avg.pct_of_peak_sustained_active"),
            "profile": prof.get("tag")}
    return o


def sixteen_bit_store(cx, w, steps, warmup):
    """SURVEY 8f rank 4: the same device-resident batch with the kernel storing float16 features (the dtype the reference
    model's autocast converts them to, REF/scripts/train.py:250).  Its own roofline denominator: 1,920,000 B of PCM +
    n_mels x 3000 x 2 B of features per clip (2.40 MB at 80 mels, 2.69 MB at 128)."""
    import whisper_context_biasing_b200 as W

    torch = cx.torch
    fe = W.B200WhisperFeatureExtractor(feature_size=w["n_mels"], device=cx.dev, feature_dtype=torch.float16)
    out = torch.empty((w["B"], w["n_mels"], N_FRAMES), dtype=torch.float16, device=cx.dev)
    for _ in range(max(warmup, 3)):
        fe.extract_device(w["pcm"], out=out)
    cx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fe.extract_device(w["pcm"], out=out)
    e1.record()
    cx.barrier()
    (ms,) = cx.max_over_ranks([e0.elapsed_time(e1)])
    err = float((out.float() - w["out"]).abs().max())
    fe.close()
    peak, _ = measured_peaks()
    alg = w["in_bytes"] + w["n_mels"] * N_FRAMES * 2 * w["B"]
    ach = alg / (ms / steps * 1e-3) / 1e9
    return {"value": CLIP_SECONDS * w["total_clips"] * steps / (ms * 1e-3), "unit": "audio-s/s", "ms_per_step": ms / steps,
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "algorithmic_bytes_per_launch": alg},
            "max_abs_vs_f32_features": err,
            "what": "float16 feature store (round-to-nearest of the float32 value, bit-exact in tests); the kernel is not "
                    "HBM-bound, so halving the write bytes lowers the fraction, not the time"}


def sustained(cx, w, seconds=2.0):
    """>= `seconds` of back-to-back launches of the workload with clock / power samples every 10 ms."""
    torch = cx.torch
    fe = cx.fe(w["n_mels"])
    pcm, out = w["pcm"], w["out"]
    fe.extract_device(pcm, out=out)
    cx.barrier()
    sampler = ClockSampler(visible_nvml_index(cx.local_rank), period_s=0.01)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 0
    t_start = time.perf_counter()
    e0.record()
    while True:
        for _ in range(100):
            fe.extract_device(pcm, out=out)
        n += 100
        torch.cuda.current_stream(cx.dev).synchronize()
        if time.perf_counter() - t_start >= seconds:
            break
    e1.record()
    torch.cuda.synchronize(cx.dev)
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1)
    (ms,) = cx.max_over_ranks([ms])
    return {"value": CLIP_SECONDS * w["total_clips"] * n / (ms * 1e-3), "unit": "audio-s/s", "launch_batches": n,
            "seconds": ms * 1e-3, "ms_per_step": ms / n, "clocks": clocks}


def c1_call_shape(cx):
    """BASELINE configs[0] / REF/data_utils/data_loader.py:171-172 + data_collator.py:64-76: 16 clips, ONE extractor call
    per clip on a pageable numpy array, then the collator's `.pad` stack -- for this library and, beside it, for the
    unmodified reference extractor in this process (the reference runs it inside its single DataLoader worker)."""
    import numpy as np

    torch = cx.torch
    fe = cx.fe(80)
    clips = synth_noise_clips(16, seed=0)

    def ours():
        feats = [fe(x, sampling_rate=16000).input_features[0] for x in clips]       # :171-172
        batch = fe.pad({"input_features": feats}, padding="longest", return_tensors="pt")   # collator :71-76
        torch.cuda.current_stream(cx.dev).synchronize()
        return batch["input_features"]

    for _ in range(3):
        got = ours()
    reps = 10
    t0 = time.perf_counter()
    for _ in range(reps):
        ours()
    t_ours = (time.perf_counter() - t0) / reps
    from oracle.hf_reference import make_hf_extractor

    hf = make_hf_extractor(80)

    def ref():
        feats = [torch.tensor(hf(x, sampling_rate=16000).input_features[0]) for x in clips]
        return hf.pad({"input_features": feats}, padding="longest", return_tensors="pt")["input_features"]

    want = ref()
    t0 = time.perf_counter()
    for _ in range(2):
        ref()
    t_ref = (time.perf_counter() - t0) / 2
    err = float((got.float().cpu() - want).abs().max())
    return {"clips": 16, "value": CLIP_SECONDS * 16 / t_ours, "unit": "audio-s/s", "us_per_clip": 1e6 * t_ours / 16,
            "reference": {"value": CLIP_SECONDS * 16 / t_ref, "us_per_clip": 1e6 * t_ref / 16,
                          "torch_threads": torch.get_num_threads()},
            "max_abs_vs_reference": err,
            "what": "16 x fe(one pageable 30 s clip, sampling_rate=16000).input_features[0] + .pad stack, host wall clock, "
                    "features left in HBM; beside it the unmodified transformers extractor called the same way in-process"}


def hf_cuda_baseline(cx, w):
    """The existing GPU implementation on the same box: the body of HF's `device="cuda"` branch (cuFFT + cuBLAS + ATen
    elementwise, TF-FE:140-163) on the same device-resident batch.  The reference never uses it."""
    torch = cx.torch
    from oracle.hf_reference import make_hf_extractor

    n_mels = w["n_mels"]
    hf = make_hf_extractor(n_mels)
    wave = w["pcm"]
    window = torch.hann_window(400, device=cx.dev)
    mel = torch.from_numpy(hf.mel_filters).to(cx.dev, torch.float32)

    def step():
        stft = torch.stft(wave, 400, 160, window=window, return_complex=True)
        mag = stft[..., :-1].abs() ** 2
        spec = mel.T @ mag
        log_spec = torch.clamp(spec, min=1e-10).log10()
        mx = log_spec.max(dim=2, keepdim=True)[0].max(dim=1, keepdim=True)[0]
        log_spec = torch.maximum(log_spec, mx - 8.0)
        return (log_spec + 4.0) / 4.0

    for _ in range(3):
        ref = step()
    torch.cuda.synchronize(cx.dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k = 5
    e0.record()
    for _ in range(k):
        ref = step()
    e1.record()
    torch.cuda.synchronize(cx.dev)
    ms = e0.elapsed_time(e1) / k
    err = float((ref - w["out"]).abs().max())
    del ref
    torch.cuda.empty_cache()
    return {"value": CLIP_SECONDS * w["B"] / (ms * 1e-3), "unit": "audio-s/s", "ms_per_step": ms,
            "max_abs_vs_ours": err,
            "what": "torch.stft (cuFFT) + abs()**2 + mel matmul (cuBLAS) + clamp/log10/max/scale on the same device-resident "
                    "batch, CUDA events, 5 steps after 3 warm-ups"}


def run_ours(args, wl_name, rank, world, local_rank):
    affinity = bind_rank_to_cores(local_rank, world)
    cx = Ctx(rank, world, local_rank)
    wl = WORKLOADS[wl_name]
    w = make_workload(cx, wl)
    sample = dump_sample(w["B"], wl["n_mels"]) if args.dump_outputs and rank == 0 else None
    res = measure(cx, w, args.steps, args.warmup, e2e=not args.no_e2e, e2e_extra=not args.no_e2e and not wl.get("variable"),
                  sample=sample)
    if sample is not None:
        import numpy as np

        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in res.pop("_outputs").items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    line = {
        "metric": "log-mel audio-seconds/second", "value": res["value"], "unit": "audio-s/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": res["ms_per_step"], "higher_is_better": True,
        "scaling": "strong" if wl["strong"] else "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": res["config"],
    }
    for k in ("e2e", "e2e_int16", "e2e_numpy_contract", "gpu_launches", "roofline", "clocks"):
        if k in res:
            line[k] = res[k]
    line["config"]["rank_affinity"] = affinity
    if not wl.get("variable"):
        line["roofline_fp32"] = fp32_roofline(cx, res, wl["n_mels"], w["B"])
    extras = not args.no_extras
    if extras and wl_name == "c2":
        line["c2_f16_store"] = sixteen_bit_store(cx, w, args.steps, args.warmup)
        line["sustained"] = sustained(cx, w)
        dv = abs(line["sustained"]["value"] - line["value"]) / line["value"]
        line["sustained"]["differs_from_value_by"] = dv
        line["sustained"]["flag"] = bool(dv > 0.03)
        if world == 1 and rank == 0:
            try:
                line["hf_cuda"] = hf_cuda_baseline(cx, w)
            except Exception as e:     # noqa: BLE001  (e.g. out of memory on a shared box: the baseline is optional)
                line["hf_cuda"] = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
    del w
    cx.torch.cuda.empty_cache()
    if extras and wl_name == "c2":
        for name in ("c3", "c4"):
            wx = make_workload(cx, WORKLOADS[name])
            rx = measure(cx, wx, max(5, min(args.steps, 20)), args.warmup, e2e=not args.no_e2e, e2e_extra=False)
            obj = {"value": rx["value"], "unit": "audio-s/s", "scaling": "strong", "ms_per_step": rx["ms_per_step"],
                   "config": rx["config"], "gpu_launches": rx["gpu_launches"], "roofline": rx["roofline"]}
            if "e2e" in rx:
                obj["e2e"] = rx["e2e"]
            if name == "c3":
                obj["roofline_fp32"] = fp32_roofline(cx, rx, 128, wx["B"])
            if name == "c4":
                # both conventions of SURVEY 8d: nominal 30 s windows per clip (value) and the audio actually present
                true_total = _sum_over_ranks(cx, wx["true_audio_s"])
                obj["true_audio_value"] = true_total / (rx["ms_per_step"] * 1e-3)
                if "e2e" in rx:
                    obj["e2e"]["true_audio_value"] = true_total / (rx["e2e"]["ms_per_step"] * 1e-3)
            line[name] = obj
            del wx
            cx.torch.cuda.empty_cache()
        if rank == 0:
            line["c1"] = c1_call_shape(cx)
    if rank == 0 and not args.no_cpu_baseline and world == 1:
        line["cpu_baseline"] = cpu_baseline(wl["n_mels"], "default")
        if extras:
            line["cpu_baseline_numpy"] = cpu_baseline(wl["n_mels"], "numpy")
    for v in line.values():
        if isinstance(v, dict):
            v.pop("_prof", None)
            v.pop("_launch_ms", None)
    cx.emit(line)
    cx.close()


def _sum_over_ranks(cx, v):
    if cx.dist is None:
        return float(v)
    t = cx.torch.tensor([v], dtype=cx.torch.float64, device=cx.dev)
    cx.dist.all_reduce(t, op=cx.dist.ReduceOp.SUM)
    return float(t.item())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host end-to-end legs (profiling runs)")
    ap.add_argument("--no-extras", action="store_true", help="only the headline workload (no c3/c4/c1/sustained/hf_cuda objects)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the features of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of this project's path (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, WORKLOADS[args.workload], rank, world)
        return
    if world == 1 and args.gpus > 1:
        print(f"bench.py: --gpus {args.gpus} needs torchrun (one rank per GPU); running rank 0 only", file=sys.stderr)
    run_ours(args, args.workload, rank, world, local_rank)


if __name__ == "__main__":
    main()
