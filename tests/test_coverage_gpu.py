"""Coverage on a B200 where the rest of the suite never looks:

  A. poisoned padding and poisoned outputs: large finite garbage past every clip's length (dense rows) and between
     ragged clips, lengths of every residue modulo the 16-byte copy unit, outputs filled with a sentinel before the
     call -- on every kernel path (30-s static, dynamic and flat twin, long-form pass 1 + clamp, conditioned);
  B. every mel bank the plan accepts (the CPU restatement of its acceptance rule in test_coverage_cpu.py says which),
     and the refusal of every other one;
  C. the long-form unit queue under load: 25 units per clip, at least four per group, unit-boundary lengths;
  D. batches past the launch limits: 70,000 clips (grid.y strides) and a 30-s batch whose features cross element 2^31.

Every check is exact (bit identity, no sentinel left, exactly -1.5) or uses the suite's TOL against the float64
oracle."""
import importlib.util
import os

import numpy as np
import pytest

from oracle import logmel_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


LO = _load("_longform_oracle_covg", os.path.join(HERE, "longform_oracle.py"))
CO = _load("_conditioning_oracle_covg", os.path.join(HERE, "conditioning_oracle.py"))
RS = _load("_coverage_restatement", os.path.join(HERE, "test_coverage_cpu.py"))

pytestmark = pytest.mark.gpu

TOL = 5e-4
SENTINEL = 7.0                    # exact in float32, bfloat16 and float16; no feature comes near it
GARBAGE = {np.dtype(np.float32): 1000.0, np.dtype(np.int16): 32767}
CONDS = {"normalize": dict(do_normalize=True), "dither": dict(dither=0.25), "both": dict(do_normalize=True, dither=0.25)}
SEED = 0x5EED_0F_C0FFEE
FAMS = O.FAMILIES


@pytest.fixture(scope="module")
def ex():
    import torch

    from whisper_context_biasing_b200 import B200WhisperFeatureExtractor

    e = {m: B200WhisperFeatureExtractor(feature_size=m) for m in (50, 80, 128)}
    yield e
    for x in e.values():
        x.set_feature_dtype(torch.float32)
        x.set_flat_clips(-1)
        x.close()


# ---- inputs: clips on the int16 grid, so float32 and int16 PCM give the same features ---------------------------------
def _q16(x):
    return np.round(np.clip(x, -1.0, 1.0) * 32767.0).astype(np.int16)


def _grid(x):
    return _q16(x).astype(np.float32) / np.float32(32768.0)


def _to_i16(clips):
    return [np.round(c.astype(np.float64) * 32768.0).astype(np.int16) for c in clips]


def _garbage(n, dt, seed):
    dt = np.dtype(dt)
    g = dt.type(GARBAGE[dt])
    return np.where(np.random.default_rng(seed).integers(0, 2, n, dtype=np.uint8) != 0, g, -g).astype(dt, copy=False)


def _dense(clips, stride, poison, seed=1):
    """[B, stride] rows, clip i in [0, min(len, stride)), the rest zero (clean) or garbage (poisoned)"""
    dt = clips[0].dtype
    buf = _garbage(len(clips) * stride, dt, seed).reshape(len(clips), stride) if poison else np.zeros((len(clips), stride), dt)
    for i, c in enumerate(clips):
        n = min(len(c), stride)
        buf[i, :n] = c[:n]
    return buf


def _ragged(clips, poison, seed=2):
    """one 1-D buffer; clip starts 16-byte aligned with at least one 16-byte unit between clips and after the last;
    everything outside the clips zero (clean) or garbage (poisoned)"""
    dt = clips[0].dtype
    gran = 16 // dt.itemsize
    offs, cur = [], 0
    for c in clips:
        offs.append(cur)
        cur += (len(c) + gran - 1) // gran * gran + gran
    buf = _garbage(cur + gran, dt, seed) if poison else np.zeros(cur + gran, dt)
    for o, c in zip(offs, clips):
        buf[o:o + len(c)] = c
    return buf, np.array(offs, np.int64)


def _inputs(e, clips, layout, poison, stride=None):
    import torch

    dev = e.device
    if layout == "static":
        # no lengths: every row is a whole clip of min(stride, 480000) samples, so [0, 480000) is the zero-padded clip
        # and only the samples past 480000 are padding the kernel must not read (garbage when poisoned)
        rows = _dense([c[:O.N_SAMPLES] for c in clips], O.N_SAMPLES, False)
        if stride > O.N_SAMPLES:
            tail = stride - O.N_SAMPLES
            pad = (_garbage(len(clips) * tail, rows.dtype, 3).reshape(len(clips), tail) if poison
                   else np.zeros((len(clips), tail), rows.dtype))
            rows = np.concatenate([rows, pad], axis=1)
        return dict(pcm=torch.from_numpy(np.ascontiguousarray(rows)).to(dev))
    lens = torch.tensor([len(c) for c in clips], dtype=torch.int32, device=dev)
    if layout == "dense":
        return dict(pcm=torch.from_numpy(_dense(clips, stride, poison)).to(dev), lengths=lens)
    buf, offs = _ragged(clips, poison)
    return dict(pcm=torch.from_numpy(buf).to(dev), lengths=lens, offsets=torch.from_numpy(offs).to(dev))


def _batch(inp):
    return inp["lengths"].shape[0] if "lengths" in inp else inp["pcm"].shape[0]


def _run(e, inp, n_frames, **kw):
    """extract_device into an output filled with the sentinel; no element may keep it"""
    import torch

    out = torch.full((_batch(inp), e.feature_size, n_frames), SENTINEL, dtype=e.feature_dtype, device=e.device)
    got = e.extract_device(**inp, out=out, **kw)
    assert got.data_ptr() == out.data_ptr()
    assert not bool((got == SENTINEL).any()), "an output element was never written"
    return got


def _err(got, ref):
    return float(np.abs(got.float().cpu().numpy() - ref).max())


# =====================================================================================================================
# A. poisoned padding and poisoned outputs
# =====================================================================================================================
# len % 8 takes every value in the first eight; 600006 is trimmed (to 480000 / to L); 0 and 1 leave half-tiles idle
LENS_A = [0, 1, 202, 5123, 77780, 160005, 333334, 479999, 480000, 600006, 250003, 12347]
L_A = 600003


@pytest.mark.parametrize("m", [80, 128, 50])
def test_poisoned_padding_and_outputs(ex, m):
    import torch

    e = ex[m]
    assert e.kernel_variant == (m if m in (80, 128) else 0)
    clips = [_grid(O.synth_clip(FAMS[i % len(FAMS)], n, 1000 + i)) for i, n in enumerate(LENS_A)]
    clips[4] = _grid(0.9 + 0.05 * clips[4])                     # a DC offset: the moments must not cancel it away
    assert sorted({n % 8 for n in LENS_A}) == list(range(8))
    q16 = _to_i16(clips)
    assert all(np.array_equal(q.astype(np.float32) / 32768.0, c) for q, c in zip(q16, clips))

    refs = {"30s": O.extract(clips, m), "long": LO.log_mel_spectrogram(O.pad_or_trim(clips, L_A), m)[0]}
    for geom, N in (("30s", O.N_SAMPLES), ("long", L_A)):
        for name, cond in CONDS.items():
            refs[geom, name] = LO.log_mel_spectrogram(CO.condition(clips, N, seed=SEED, **cond), m)[0]
    # (name, layout, row stride, extract_device arguments, reference, frames)
    paths = [("static", "static", 480008, {}, "30s", 3000),
             ("dynamic_dense", "dense", 600008, {}, "30s", 3000),
             ("dynamic_ragged", "ragged", None, {}, "30s", 3000),
             ("long_dense", "dense", 600008, dict(padded_len=L_A), "long", L_A // 160),
             ("long_ragged", "ragged", None, dict(padded_len=L_A), "long", L_A // 160)]
    for geom in ("30s", "long"):
        for name, cond in CONDS.items():
            kw = dict(seed=SEED, **cond, **(dict(padded_len=L_A) if geom == "long" else {}))
            n_frames = 3000 if geom == "30s" else L_A // 160
            paths += [(f"{geom}_{name}_{lay}", lay, 600008, kw, (geom, name), n_frames) for lay in ("dense", "ragged")]

    worst, clean32 = 0.0, {}
    for pcm_name, cl in (("f32", clips), ("i16", q16)):
        for pname, layout, stride, kw, ref, n_frames in paths:
            e.set_feature_dtype(torch.float32)
            if layout == "static":       # clean: rows of exactly 480000 samples; poisoned: 8 garbage samples after them
                clean = e.extract_device(**_inputs(e, cl, "static", False, 480000), **kw)
            else:
                clean = e.extract_device(**_inputs(e, cl, layout, False, stride), **kw)
            if pcm_name == "f32":
                d = _err(clean, refs[ref])
                worst = max(worst, d)
                assert d <= TOL, (m, pname, d)
                clean32[pname] = clean
            else:
                assert torch.equal(clean, clean32[pname]), (m, pname, "int16 and float32 on the int16 grid")
            poisoned = _inputs(e, cl, layout, True, stride)
            for dt in (torch.float32, torch.bfloat16, torch.float16):
                e.set_feature_dtype(dt)
                got = _run(e, poisoned, n_frames, **kw)
                assert torch.equal(got, clean.to(dt)), (m, pcm_name, pname, dt)
        e.set_feature_dtype(torch.float32)

        # the flat twin of the 30-s kernel: the clusters take the first max_clusters clips (short fillers), the flat CTAs
        # the twelve clips behind them
        assert e.sm_count > 6 * e.max_clusters, "no SM is left for the flat kernel"
        nc = e.max_clusters
        fill = [_grid(O.synth_clip("noise", 3000 + 7 * i, 1100 + i)) for i in range(nc)]
        if pcm_name == "i16":
            fill = _to_i16(fill)
        for layout in ("dense", "ragged"):
            inp = _inputs(e, fill + cl, layout, True, 600008)
            e.set_flat_clips(17)
            for dt in (torch.float32, torch.bfloat16, torch.float16):
                e.set_feature_dtype(dt)
                n0 = e.launch_count
                got = _run(e, inp, 3000)
                assert e.launch_count == n0 + 2                     # cluster kernel + flat kernel
                assert torch.equal(got[nc:], clean32[f"dynamic_{layout}"].to(dt)), (m, pcm_name, layout, dt)
            e.set_flat_clips(-1)
            e.set_feature_dtype(torch.float32)
    print(f"A m={m}: worst vs oracle {worst:.2e}")


# =====================================================================================================================
# B. every mel bank
# =====================================================================================================================
def test_every_mel_bank():
    import torch

    from whisper_context_biasing_b200 import B200WhisperFeatureExtractor

    acc = RS.accepted_banks()
    assert set(acc) == RS.ACCEPTED
    few = {min(acc), 50, 113, 127}
    clips = [_grid(O.synth_clip("speech", 480000, 1200)), _grid(O.synth_clip("noise", 5121, 1201)),
             _grid(O.synth_clip("chirp", 77777, 1202))]
    clips4 = clips + [_grid(O.synth_clip("gap", 600003, 1203))]
    L = 600003
    lib_accepts, worst = set(), 0.0
    for m in range(0, 130):
        if m not in acc:
            with pytest.raises(ValueError):
                B200WhisperFeatureExtractor(feature_size=m)
            continue
        e = B200WhisperFeatureExtractor(feature_size=m)
        lib_accepts.add(m)
        try:
            assert e.kernel_variant == (m if m in (80, 128) else 0), m
            rag3 = _inputs(e, clips, "ragged", True)
            rag4 = _inputs(e, clips4, "ragged", True)
            e.set_flat_clips(0)
            a = _run(e, rag3, 3000)
            d = _err(a, O.extract(clips, m))
            worst = max(worst, d)
            assert d <= TOL, (m, d)
            # the flat twin takes the three clips behind max_clusters fillers
            nc = e.max_clusters
            fill = [_grid(O.synth_clip("noise", 2000 + 8 * i, 1210 + i)) for i in range(nc)]
            e.set_flat_clips(17)
            n0 = e.launch_count
            f = _run(e, _inputs(e, fill + clips, "ragged", True), 3000)
            assert e.launch_count == n0 + 2, m
            assert torch.equal(f[nc:], a), m
            e.set_flat_clips(-1)
            assert torch.equal(_run(e, rag3, 3000, padded_len=480000), a), m
            c = _run(e, rag4, L // 160, padded_len=L)
            d = _err(c, LO.extract_longform(clips4, m))
            worst = max(worst, d)
            assert d <= TOL, (m, "long", d)
            if m in few:
                for dt in (torch.bfloat16, torch.float16):
                    e.set_feature_dtype(dt)
                    e.set_flat_clips(0)
                    assert torch.equal(_run(e, rag3, 3000), a.to(dt)), (m, dt)
                    assert torch.equal(_run(e, rag4, L // 160, padded_len=L), c.to(dt)), (m, dt)
                e.set_feature_dtype(torch.float32)
                for longform in (False, True):
                    got = _run(e, rag4, L // 160 if longform else 3000, padded_len=L if longform else None,
                               do_normalize=True, dither=0.25, seed=SEED)
                    d = _err(got, CO.extract(clips4, m, do_normalize=True, dither=0.25, seed=SEED, longform=longform))
                    worst = max(worst, d)
                    assert d <= TOL, (m, "conditioned", longform, d)
        finally:
            e.close()
    assert lib_accepts == set(acc) == set(range(37, 129))
    print(f"B: accepted banks {min(lib_accepts)}..{max(lib_accepts)} ({len(lib_accepts)}), worst vs oracle {worst:.2e}")


# =====================================================================================================================
# C. the long-form unit queue under load
# =====================================================================================================================
def test_loaded_longform_queue(ex):
    import torch

    e = ex[80]
    L, B = 1_000_003, 64
    T = L // 160
    n_tiles = (T + 31) // 32
    units = (n_tiles + 7) // 8
    assert (T, n_tiles, units) == (6250, 196, 25)
    assert B * units >= 4 * 2 * e.sm_count, "fewer than four units per group"
    boundary = [n for k in (1, 2, 3, 7, 12, 24) for n in (40960 * k - 200, 40960 * k - 199)]   # 8k and 8k + 1 half-tiles
    rng = np.random.default_rng(77)
    lens = [0, 1] + boundary + [L, 1_200_000]
    lens += rng.integers(0, L + 1, B - len(lens)).tolist()
    order = rng.permutation(B)                                    # the families and the edge cases spread over the batch
    lens = [lens[i] for i in order]
    clips = [_grid(O.synth_clip(FAMS[(i * 5) % len(FAMS)], n, 3000 + i)) for i, n in enumerate(lens)]
    q16 = _to_i16(clips)
    trimmed = [c[:L] for c in clips]
    assert LO.padded_length([len(c) for c in trimmed]) == L
    stride = 1_200_000
    lay = {"dense": _inputs(e, clips, "dense", True, stride), "ragged": _inputs(e, clips, "ragged", True),
           "dense_i16": _inputs(e, q16, "dense", True, stride), "ragged_i16": _inputs(e, q16, "ragged", True)}

    a = _run(e, lay["dense"], T, padded_len=L)
    ref = LO.extract_longform(trimmed, 80)
    d = _err(a, ref)
    assert d <= TOL, d
    for name in ("ragged", "dense_i16", "ragged_i16"):
        assert torch.equal(_run(e, lay[name], T, padded_len=L), a), name
    for _ in range(3):                       # the unit-to-group assignment differs from run to run
        assert torch.equal(_run(e, lay["ragged"], T, padded_len=L), a)
    for dt in (torch.bfloat16, torch.float16):
        e.set_feature_dtype(dt)
        assert torch.equal(_run(e, lay["ragged"], T, padded_len=L), a.to(dt)), dt
    e.set_feature_dtype(torch.float32)
    # alone and in the batch: the unit-boundary clips, the empty one, the trimmed one and a few others
    edge = {n for n in boundary} | {0, 1, L, 1_200_000}
    sample = [i for i, n in enumerate(lens) if n in edge] + [int(i) for i in rng.choice(B, 4, replace=False)]
    for i in sorted(set(sample)):
        one = _run(e, _inputs(e, [clips[i]], "ragged", True), T, padded_len=L)
        assert torch.equal(one[0], a[i]), (i, lens[i])
    # conditioned: do_normalize and dither on the same loaded queue
    cond = dict(padded_len=L, do_normalize=True, dither=0.25, seed=SEED)
    c = _run(e, lay["dense"], T, **cond)
    dc = _err(c, CO.extract(trimmed, 80, do_normalize=True, dither=0.25, seed=SEED, longform=True))
    assert dc <= TOL, dc
    for name in ("ragged", "ragged_i16"):
        assert torch.equal(_run(e, lay[name], T, **cond), c), name
    assert torch.equal(_run(e, lay["dense"], T, **cond), c)
    print(f"C: worst vs oracle {d:.2e}, conditioned {dc:.2e}")


# =====================================================================================================================
# D. batches past the launch limits
# =====================================================================================================================
def test_70000_clips(ex):
    """B > 65,535: the clamp and moments kernels stride over clips along grid.y, the merge and mask kernels over warps
    and elements."""
    import torch

    e = ex[80]
    B, L = 70_000, 1603
    T, stride = L // 160, 1608
    rng = np.random.default_rng(70)
    lens = rng.integers(0, L + 1, B).astype(np.int32)
    lens[[0, 65_535, 69_999]] = [L, 0, L]
    silent = np.unique(np.concatenate([rng.choice(B, 300, replace=False), [65_534, 65_536, 69_998]]))
    col = np.arange(stride)[None, :]
    x = _grid(rng.standard_normal((B, stride)).astype(np.float32) * rng.uniform(0.002, 0.3, (B, 1)).astype(np.float32))
    x[silent] = 0.0
    x[col >= lens[:, None]] = 0.0
    padded = x[:, :L]                                             # what the oracle pads each clip to
    pcm = np.where(col < lens[:, None], x, _garbage(B * stride, np.float32, 71).reshape(B, stride))
    dev = e.device
    inp = dict(pcm=torch.from_numpy(pcm).to(dev), lengths=torch.from_numpy(lens).to(dev))
    del pcm
    idx = np.unique(np.concatenate([rng.choice(65_535, 1000, replace=False), np.arange(65_535, B)]))
    runs = {"plain": {}, "normalize": dict(do_normalize=True), "dither": dict(dither=0.25, seed=SEED)}
    worst = {}
    for name, kw in runs.items():
        got = _run(e, inp, T, padded_len=L, **kw)
        y = padded[idx]
        if "do_normalize" in kw:
            y = CO.normalize(y, lens[idx])
        if "dither" in kw:
            y = y + np.float32(0.25) * np.stack([CO.noise(SEED, int(b), L) for b in idx]).astype(np.float32)
        ref = LO.log_mel_spectrogram(y, 80)[0]
        worst[name] = _err(got[torch.from_numpy(idx).to(dev)], ref)
        assert worst[name] <= TOL, (name, worst[name])
        if "dither" not in kw:
            assert bool((got[torch.from_numpy(silent).to(dev)] == -1.5).all()), name
            for k in range(0, B, 1000):               # the same clips in batches of 1000: the same bits
                part = _run(e, dict(pcm=inp["pcm"][k:k + 1000], lengths=inp["lengths"][k:k + 1000]), T, padded_len=L, **kw)
                assert torch.equal(part, got[k:k + 1000]), (name, k)
        del got
    mask = e.frame_mask_device(inp["lengths"], padded_len=L)
    assert np.array_equal(mask.cpu().numpy(), LO.frame_mask(lens, L))
    print(f"D 70000 clips: worst vs oracle {worst}")


def test_30s_features_past_2_pow_31_elements(ex):
    """5,600 clips x 128 mels x 3000 frames: clip 5592 straddles element 2^31 and clips 5588..5599 are full 30-s clips;
    the static split (its flat kernel takes the last clips), the cluster kernel alone and the dynamic queue, in bfloat16,
    and the static split in float32."""
    import torch

    e = ex[128]
    B, M, F = 5600, 128, 3000
    assert 5592 * M * F < 2 ** 31 < 5593 * M * F
    fams = ["noise", "sine", "chirp", "speech", "int16", "gap"] * 2
    full = [_q16(O.synth_clip(f, 480000, 5000 + i)) for i, f in enumerate(fams)]
    oracle = O.extract([q.astype(np.float32) / 32768.0 for q in full], M)
    dev = e.device
    g = torch.Generator(device=dev).manual_seed(56)
    pcm = torch.zeros((B, 480000), dtype=torch.int16, device=dev)
    pcm[:B - 12, :4000] = torch.randint(-3000, 3000, (B - 12, 4000), dtype=torch.int16, device=dev, generator=g)
    pcm[B - 12:] = torch.from_numpy(np.stack(full)).to(dev)
    short_lens = torch.randint(0, 4001, (B - 12,), dtype=torch.int32, device=dev, generator=g)
    lens = torch.cat([short_lens, torch.full((12,), 480000, dtype=torch.int32, device=dev)])
    rag = torch.cat([pcm[:B - 12, :4000].reshape(-1), pcm[B - 12:].reshape(-1)])
    offs = torch.cat([torch.arange(B - 12, dtype=torch.int64, device=dev) * 4000,
                      (B - 12) * 4000 + torch.arange(12, dtype=torch.int64, device=dev) * 480000])
    ragged = dict(pcm=rag, lengths=lens, offsets=offs)
    ragged12 = dict(pcm=pcm[B - 12:].reshape(-1), lengths=lens[B - 12:],
                    offsets=torch.arange(12, dtype=torch.int64, device=dev) * 480000)
    configs = [("dense_split", torch.bfloat16, -1, dict(pcm=pcm), dict(pcm=pcm[B - 12:])),
               ("dense_clusters", torch.bfloat16, 0, dict(pcm=pcm), dict(pcm=pcm[B - 12:])),
               ("ragged", torch.bfloat16, -1, ragged, ragged12),
               ("dense_split_f32", torch.float32, -1, dict(pcm=pcm), dict(pcm=pcm[B - 12:]))]
    worst = {}
    for name, dt, flat, inp, inp12 in configs:
        e.set_feature_dtype(dt)
        e.set_flat_clips(flat)
        n0 = e.launch_count
        out = _run(e, inp, F)
        if name.startswith("dense_split"):
            assert e.launch_count == n0 + 2, name            # the static split hands the last clips to the flat kernel
        tail = out[B - 12:].clone()
        del out
        torch.cuda.synchronize()
        alone = e.extract_device(**inp12)
        assert torch.equal(tail, alone), name
        worst[name] = _err(tail, oracle)
        assert worst[name] <= (TOL if dt == torch.float32 else 8e-3 + TOL), (name, worst[name])
        del tail, alone
    e.set_flat_clips(-1)
    e.set_feature_dtype(torch.float32)
    del pcm, rag, ragged, ragged12, configs
    torch.cuda.empty_cache()
    print(f"D past 2^31: worst vs oracle {worst}")
