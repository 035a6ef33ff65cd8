"""Coverage without a GPU: every mel bank the plan can be asked for (the extractor's table against the oracle's and the
live reference's, and a restatement of the plan's acceptance rule and warp split), and the sensitivity of the checks
tests/test_coverage_gpu.py makes -- a kernel that read its garbage padding, counted it in the moments, left a frame of a
poisoned output unwritten or carried state from one unit of work to the next would fail them by far more than TOL."""
import importlib.util
import os
import re
import warnings

import numpy as np
import pytest

from oracle import logmel_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


LO = _load("_longform_oracle_cov", os.path.join(HERE, "longform_oracle.py"))
CO = _load("_conditioning_oracle_cov", os.path.join(HERE, "conditioning_oracle.py"))

TOL = 5e-4
N_FREQ, GROUP_WARPS, MAX_FILTERS_PER_WARP, MAX_GROUP_BINS = 201, 8, 16, 16
SENTINEL = 7.0

# ---------------------------------------------------------------------------------------------------------------------
# restatement of the plan's acceptance rule: build_sparse (csrc/wlm_api.cu) and build_tables (csrc/logmel_fused.cuh)
# ---------------------------------------------------------------------------------------------------------------------


def sparse_lo(table):
    """build_sparse on the float32 table [201, M] the extractor hands to wlm_plan_create: lo[k] per FFT bin, or None
    when the table is refused.  A bin feeding two filters gets the lower one; a bin feeding one filter m gets m, except
    the rising side of filter 0 before any other filter (lo = -1, the "hi" weight of the pair (-1, 0)); a bin feeding
    none keeps the previous bin's lo."""
    t = np.asarray(table, dtype=np.float32)
    if not np.isfinite(t).all():
        return None
    n_mels = t.shape[1]
    khi = np.full(n_mels, -1)
    lo, prev = np.empty(N_FREQ, np.int64), -1
    for k in range(N_FREQ):
        idx = np.nonzero(t[k] != 0.0)[0]
        if len(idx) > 2:
            return None
        for m in idx:
            if khi[m] >= 0 and khi[m] != k - 1:          # the support of a filter must be contiguous
                return None
            khi[m] = k
        if len(idx) == 2 and idx[1] != idx[0] + 1:
            return None
        if len(idx) == 0:
            v = prev
        elif len(idx) == 2:
            v = int(idx[0])
        elif idx[0] == 0 and prev == -1:
            v = -1
        else:
            v = int(idx[0])
        if v < prev:
            return None
        lo[k] = prev = v
    return lo


def _baked():
    """the group starts and warp split compiled into the unrolled 80- and 128-mel kernels (csrc/mel_structure.inc)"""
    text = open(os.path.join(ROOT, "whisper_context_biasing_b200", "csrc", "mel_structure.inc")).read()

    def arr(name):
        body = re.search(r"static const short " + name + r"\[\d+\] = \{([^}]*)\}", text).group(1)
        return [int(x) for x in body.split(",")]
    return {m: (arr(f"kMelGstartHost{m}"), arr(f"kMelM0Host{m}"), arr(f"kMelNfHost{m}")) for m in (80, 128)}


def plan_tables(table):
    """build_tables: None when refused, else (variant, gstart, [(m0, nf)] per warp of a warp group)."""
    lo = sparse_lo(table)
    if lo is None:
        return None
    n_mels = np.asarray(table).shape[1]
    # gstart[v] = first bin k with lo[k] + 1 >= v, v = 0 .. n_mels + 1; group v = the bins with lo = v - 1
    gstart, k = [], 0
    for v in range(n_mels + 2):
        while k < N_FREQ and lo[k] + 1 < v:
            k += 1
        gstart.append(k)
    if any(gstart[v + 1] - gstart[v] > MAX_GROUP_BINS for v in range(n_mels + 1)):
        return None
    baked = _baked().get(n_mels)
    if baked is not None and gstart == baked[0]:
        return n_mels, gstart, list(zip(baked[1], baked[2]))

    def cost(m):
        return 7.0 + 1.5 * (gstart[m + 2] - gstart[m])
    total = 0.0
    for m in range(n_mels):
        total += cost(m)
    split, m, acc = [], 0, 0.0
    for w in range(GROUP_WARPS):
        target = total * (w + 1) / GROUP_WARPS
        m0, cnt = m, 0
        while m < n_mels and cnt < MAX_FILTERS_PER_WARP:
            must_take = n_mels - m > (GROUP_WARPS - 1 - w) * MAX_FILTERS_PER_WARP   # the other warps could not hold them
            if not must_take and cnt > 0 and acc + 0.5 * cost(m) > target:
                break
            acc += cost(m)
            m += 1
            cnt += 1
        split.append((m0, cnt))
    if m < n_mels:
        return None
    return 0, gstart, split


def accepted_banks():
    """{n_mels: (variant, gstart, split)} for every bank in [1, 128] the plan accepts"""
    from whisper_context_biasing_b200.feature_extraction import slaney_mel_filters

    out = {}
    for m in range(1, 129):
        r = plan_tables(slaney_mel_filters(m).astype(np.float32))
        if r is not None:
            out[m] = r
    return out


ACCEPTED = set(range(37, 129))      # what the restatement gives; test_coverage_gpu.py checks the library agrees


# ---------------------------------------------------------------------------------------------------------------------
# B. every mel bank
# ---------------------------------------------------------------------------------------------------------------------


def test_extractor_table_equals_the_oracle_bank_for_every_n_mels():
    from whisper_context_biasing_b200.feature_extraction import slaney_mel_filters

    for m in range(1, 129):
        a, b = slaney_mel_filters(m), O.mel_filter_bank(m)
        assert a.shape == b.shape == (N_FREQ, m) and a.dtype == b.dtype == np.float64
        assert np.array_equal(a, b), m


def test_oracle_bank_equals_the_live_reference_for_every_n_mels():
    audio_utils = pytest.importorskip("transformers.audio_utils")
    for m in range(1, 129):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")          # the reference warns about all-zero filters of the widest banks
            ref = audio_utils.mel_filter_bank(num_frequency_bins=N_FREQ, num_mel_filters=m, min_frequency=0.0,
                                              max_frequency=8000.0, sampling_rate=16000, norm="slaney",
                                              mel_scale="slaney")
        assert np.array_equal(O.mel_filter_bank(m), ref), m


def test_accepted_banks_and_their_warp_split():
    acc = accepted_banks()
    assert set(acc) == ACCEPTED
    for m, (variant, gstart, split) in acc.items():
        assert variant == (m if m in (80, 128) else 0), m
        assert gstart[0] == 0 and gstart[-1] == N_FREQ
        # the warps own contiguous runs that cover the bank, at most 16 filters each
        assert [s[0] for s in split] == [sum(nf for _, nf in split[:w]) for w in range(GROUP_WARPS)], m
        assert sum(nf for _, nf in split) == m and max(nf for _, nf in split) <= MAX_FILTERS_PER_WARP, m
    # the unrolled banks: the restated structure is the one compiled in
    baked = _baked()
    for m in (80, 128):
        assert acc[m][1] == baked[m][0] and acc[m][2] == list(zip(baked[m][1], baked[m][2]))
    # the edges the GPU test exercises: a 16-bin group at the narrow end, a warp of 16 filters the must_take rule
    # forces near 128 (the cost model alone would not), banks where some warp has no filter at all
    widest = {m: max(g[v + 1] - g[v] for v in range(m + 1)) for m, (_, g, _) in acc.items()}
    assert widest[min(acc)] == MAX_GROUP_BINS
    assert any(max(nf for _, nf in s) == MAX_FILTERS_PER_WARP for m, (v, _, s) in acc.items() if v == 0 and m > 112)
    # below 37 filters some group between two filter centres spans more than 16 bins
    from whisper_context_biasing_b200.feature_extraction import slaney_mel_filters

    assert plan_tables(slaney_mel_filters(36).astype(np.float32)) is None


def test_restatement_refuses_what_build_sparse_refuses():
    from whisper_context_biasing_b200.feature_extraction import slaney_mel_filters

    t = slaney_mel_filters(80).astype(np.float32)
    assert sparse_lo(t) is not None
    bad = t.copy()
    bad[100, 10] = 0.5                   # a third filter on one bin, and a filter with two separate pieces
    assert sparse_lo(bad) is None
    bad = t.copy()
    bad[3, 0] = np.nan
    assert sparse_lo(bad) is None
    lo = sparse_lo(t)
    assert lo[0] == -1 and (np.diff(lo) >= 0).all() and lo[-1] == 79


# ---------------------------------------------------------------------------------------------------------------------
# sensitivity of the poisoned-padding, poisoned-output and loaded-queue checks (shown on the oracle, no kernel runs)
# ---------------------------------------------------------------------------------------------------------------------


def _grid(x):
    return (np.round(np.clip(x, -1, 1) * 32767.0) / 32768.0).astype(np.float32)


def test_garbage_tail_not_zeroed_exceeds_tol():
    """The kernels copy whole 16-byte units: up to 3 float32 or 7 int16 samples past len.  Had the fix-up left them in
    place, the frames around the end of the clip would be off by orders of magnitude more than TOL."""
    for n, extra, garbage in ((5121, 3, 1000.0), (77777, 7, 32767 / 32768)):
        x = _grid(O.synth_clip("speech", n, 3))
        clean = O.pad_or_trim([x])
        dirty = clean.copy()
        dirty[0, n:n + extra] = garbage * np.where(np.arange(extra) % 2, -1.0, 1.0)
        a = O.log_mel_spectrogram(clean, 80)
        b = O.log_mel_spectrogram(dirty, 80)
        assert np.abs(a - b).max() > 100 * TOL, (n, extra)
        # long-form: the same, and the clip's maximum moves, so every frame shifts
        a = LO.log_mel_spectrogram(O.pad_or_trim([x], 100003), 80)[0]
        b = LO.log_mel_spectrogram(np.pad(dirty[:, :100003], ((0, 0), (0, 100003 - min(100003, 480000)))), 80)[0]
        assert np.abs(a - b).max() > 100 * TOL, (n, extra)


def test_moments_that_count_the_tail_exceed_tol():
    """do_normalize: a moments sum that read one quad too far (3 garbage float32 samples of +-1000) scales the clip by
    a different factor; the features move by far more than TOL."""
    n, L = 5121, 480000
    x = _grid(O.synth_clip("noise", n, 4))
    good = CO.condition([x], L, do_normalize=True)
    tail = np.concatenate([x, np.array([1000.0, -1000.0, 1000.0], np.float32)])
    m, s = tail.mean(dtype=np.float32), np.sqrt(tail.var(dtype=np.float32) + 1e-7)
    bad = good.copy()
    bad[0, :n] = (x - m) / s
    a = LO.log_mel_spectrogram(good, 80)[0]
    b = LO.log_mel_spectrogram(bad, 80)[0]
    assert np.abs(a - b).max() > 100 * TOL


def test_poisoned_output_catches_an_unwritten_frame():
    """An output from torch.empty may hold the same features from an earlier call, so a frame the kernel never wrote
    can still match.  A sentinel-filled output cannot: the frame keeps 7.0, which no feature can reach (every feature
    is (max(log10 p, gmax - 8) + 4) / 4 of finite PCM, and 7.0 needs a mel power of 1e24), and the comparison fails."""
    x = _grid(O.synth_clip("chirp", 100003, 5))
    ref = LO.log_mel_spectrogram(O.pad_or_trim([x], 100003), 80)[0]
    assert ref.max() < SENTINEL - 1.0
    stale = ref.copy()                          # the caching allocator handed back a block holding this very result
    poisoned = np.full_like(ref, SENTINEL)
    for out in (stale, poisoned):
        out[:, :, :256] = ref[:, :, :256]       # the kernel wrote every frame but those of half-tile 8 (frames 256..287)
        out[:, :, 288:] = ref[:, :, 288:]
    assert np.array_equal(stale, ref)           # undetectable without poisoning
    assert (poisoned == SENTINEL).any() and np.abs(poisoned - ref).max() > 1000 * TOL


def test_state_carried_between_units_exceeds_tol():
    """The loaded-queue check: a group that ran a unit of clip a and then a unit of clip b.  Had it kept a's PCM for
    the first half-tile of b's unit, or a's running maximum for b's clamp, b would be off by far more than TOL."""
    L = 1_000_003
    a = _grid(O.synth_clip("chirp", L, 6))                         # loud: amplitude 0.5
    b = _grid(0.2 * O.synth_clip("noise", 40960 * 3 - 199, 7))     # 8 * 3 + 1 active half-tiles: three full units + one
    b[:40960] = 0.0                                                # a silent first unit, clamped at b's gmax - 8
    fa, ga = LO.log_mel_spectrogram(O.pad_or_trim([a], L), 80)
    fb, gb = LO.log_mel_spectrogram(O.pad_or_trim([b], L), 80)
    # a's frames in place of the first half-tile of b's second unit (frames 256..287)
    mixed = fb.copy()
    mixed[0, :, 256:288] = fa[0, :, 256:288]
    assert np.abs(mixed - fb).max() > 100 * TOL
    # b clamped with a's maximum (a group whose running maximum was not reset between the units)
    assert float(ga[0]) > float(gb[0]) + 1.0
    carried = np.maximum(fb, np.float32((max(float(ga[0]) - 8.0, -10.0) + 4.0) / 4.0))
    assert np.abs(carried - fb).max() > 100 * TOL
