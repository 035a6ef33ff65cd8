"""`do_normalize` and `dither` on a B200: `wlm_logmel_conditioned` and the extractor's conditioned calls against the
conditioned restatement (tests/conditioning_oracle.py), the noise stream's determinism and independence from the batch,
the layout and the formats, and the ABI's errors."""
import ctypes as C
import importlib.util
import os

import numpy as np
import pytest

from oracle import logmel_oracle as O

_spec = importlib.util.spec_from_file_location("_conditioning_oracle",
                                               os.path.join(os.path.dirname(os.path.abspath(__file__)), "conditioning_oracle.py"))
CO = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(CO)

pytestmark = pytest.mark.gpu

TOL = 5e-4
LONG = dict(sampling_rate=16000, truncation=False, padding="longest")
CONDS = {"normalize": dict(do_normalize=True), "dither": dict(dither=0.25), "both": dict(do_normalize=True, dither=0.25)}
SEED = 0xC0FFEE_0BADF00D


@pytest.fixture(scope="module")
def ex():
    import torch

    from whisper_context_biasing_b200 import B200WhisperFeatureExtractor

    e = {m: B200WhisperFeatureExtractor(feature_size=m) for m in (64, 80, 128)}
    yield e
    for x in e.values():
        x.set_feature_dtype(torch.float32)
        x.close()


def _ragged(clips, gran, dtype):
    offs, cur = [], 0
    for c in clips:
        offs.append(cur)
        cur += (len(c) + gran - 1) // gran * gran
    buf = np.zeros(cur + gran, dtype)
    for o, c in zip(offs, clips):
        buf[o:o + len(c)] = c
    return buf, np.array(offs, np.int64)


def _layouts(e, clips):
    """dense (with lengths) and ragged device inputs of the same clips (float32 or int16 arrays)"""
    import torch

    dev = e.device
    dt = clips[0].dtype
    gran = 16 // dt.itemsize
    n = max(4, (max(len(c) for c in clips) + 7) // 8 * 8)
    lens = torch.tensor([len(c) for c in clips], dtype=torch.int32, device=dev)
    dense = np.zeros((len(clips), n), dt)
    for i, c in enumerate(clips):
        dense[i, :len(c)] = c
    buf, offs = _ragged(clips, gran, dt)
    return {"dense": dict(pcm=torch.from_numpy(dense).to(dev), lengths=lens),
            "ragged": dict(pcm=torch.from_numpy(buf).to(dev), lengths=lens, offsets=torch.from_numpy(offs).to(dev))}


@pytest.mark.parametrize("longform", [False, True])
def test_against_restatement(ex, longform):
    """do_normalize, dither and both; lengths from empty to beyond 30 s; L not a multiple of 160 or 4; dense and ragged,
    float32 and int16 PCM; the 80-, 128- and 64-mel (table-driven) banks; 16-bit outputs against the float32 result."""
    import torch

    lengths = [0, 1, 200, 201, 5359, 77777, 480000, 600000] + ([600003] if longform else [])
    clips = [O.synth_clip(O.FAMILIES[i % len(O.FAMILIES)], n, 700 + i) for i, n in enumerate(lengths)]
    clips[5] = (3.0 + 0.1 * clips[5]).astype(np.float32)           # a DC offset far above the signal
    q16 = [np.round(np.clip(c, -1, 1) * 32767.0).astype(np.int16) for c in clips]
    g16 = [q.astype(np.float32) / 32768.0 for q in q16]
    L = 600003 if longform else 480000
    worst = 0.0
    for m in (80, 128, 64):
        e = ex[m]
        lay = _layouts(e, clips)
        lay16 = _layouts(e, q16)
        for name, cond in CONDS.items():
            ref = CO.extract(clips, m, longform=longform, seed=SEED, **cond)
            ref16 = CO.extract(g16, m, longform=longform, seed=SEED, **cond)
            kw = dict(padded_len=L if longform else None, seed=SEED, **cond)
            a = e.extract_device(**lay["dense"], **kw)
            d = float(np.abs(a.cpu().numpy() - ref).max())
            worst = max(worst, d)
            assert d <= TOL, (m, name, d)
            assert torch.equal(a, e.extract_device(**lay["ragged"], **kw)), (m, name)
            b = e.extract_device(**lay16["dense"], **kw)
            assert float(np.abs(b.cpu().numpy() - ref16).max()) <= TOL, (m, name)
            assert torch.equal(b, e.extract_device(**lay16["ragged"], **kw)), (m, name)
            for dt, atol in ((torch.bfloat16, 2 ** -6), (torch.float16, 2 ** -9)):
                e.set_feature_dtype(dt)
                h = e.extract_device(**lay["dense"], **kw)
                e.set_feature_dtype(torch.float32)
                assert h.dtype == dt
                assert float((h.float() - a.to(dt).float()).abs().max()) <= atol, (m, name, dt)
    print("worst vs conditioned restatement", worst)


def test_no_lengths_layout_and_the_public_call(ex):
    import torch

    e = ex[80]
    rows = np.stack([O.synth_clip("speech", 333336, 60 + i) for i in range(3)])
    for name, cond in CONDS.items():
        got = e.extract_device(torch.from_numpy(rows).to(e.device), padded_len=333336, seed=SEED, **cond)
        ref = CO.extract(list(rows), 80, longform=True, seed=SEED, **cond)
        assert float(np.abs(got.cpu().numpy() - ref).max()) <= TOL, name
    # __call__(do_normalize=True), 30 s and long-form, host and device input, and HF's masks
    clips = [O.synth_clip("speech", 45000, 61), O.synth_clip("noise", 700001, 62), np.zeros(0, np.float32)]
    for longform in (False, True):
        kw = dict(LONG, pad_to_multiple_of=160) if longform else dict(sampling_rate=16000)
        ref = CO.extract(clips, 80, do_normalize=True, longform=longform, pad_to_multiple_of=160 if longform else None)
        r = e(clips, do_normalize=True, return_tensors="np", **kw)
        assert float(np.abs(r["input_features"] - ref).max()) <= TOL, longform
        N = 700160 if longform else 480000
        assert r["attention_mask"].shape == (3, N)                      # the sample-level mask of HF's quirk
        assert r["attention_mask"].sum(1).tolist() == [45000, min(700001, N), 0]
        r = e(clips, do_normalize=True, return_attention_mask=True, return_tensors="np", **kw)
        assert r["attention_mask"].shape == (3, N // 160)
    x = torch.from_numpy(rows[:, :333333].copy()).to(e.device)     # 333333 % 4 != 0: the row is padded on the device
    for longform in (False, True):
        kw = LONG if longform else dict(sampling_rate=16000)
        got = e(x, do_normalize=True, return_tensors="np", **kw)["input_features"]
        ref = CO.extract(list(rows[:, :333333]), 80, do_normalize=True, longform=longform)
        assert float(np.abs(got - ref).max()) <= TOL, longform


def test_zero_pcm_with_unit_dither_is_the_noise_stream(ex):
    """features that are pure noise: they check the mapping (b, n) -> z on its own, pad and reflected samples included"""
    e = ex[80]
    for longform, lens in ((False, [0, 480000, 1000]), (True, [12345, 0, 7])):
        clips = [np.zeros(n, np.float32) for n in lens]
        kw = dict(padded_len=12345) if longform else {}
        import torch
        buf, offs = _ragged(clips, 4, np.float32)
        got = e.extract_device(torch.from_numpy(buf).to(e.device), lengths=torch.tensor(lens, dtype=torch.int32, device=e.device),
                               offsets=torch.from_numpy(offs).to(e.device), dither=1.0, seed=SEED, **kw)
        ref = CO.extract(clips, 80, dither=1.0, seed=SEED, longform=longform)
        assert float(np.abs(got.cpu().numpy() - ref).max()) <= TOL, longform
        assert not np.allclose(ref[0], ref[1])


def test_determinism_and_independence(ex):
    import torch

    e = ex[128]
    dev = e.device
    x = O.synth_clip("speech", 250000, 80)
    y = O.synth_clip("noise", 300000, 81)
    L = 300000
    one = dict(pcm=torch.from_numpy(np.pad(x, (0, 0))).to(dev)[None], lengths=torch.tensor([250000], dtype=torch.int32,
                                                                                         device=dev))
    dense = np.zeros((2, 300000), np.float32)
    dense[0, :250000], dense[1] = x, y
    two = dict(pcm=torch.from_numpy(dense).to(dev), lengths=torch.tensor([250000, 300000], dtype=torch.int32, device=dev))
    for name, cond in CONDS.items():
        a = e.extract_device(**one, padded_len=L, seed=SEED, **cond)
        assert torch.equal(a, e.extract_device(**one, padded_len=L, seed=SEED, **cond)), name        # same seed
        b = e.extract_device(**two, padded_len=L, seed=SEED, **cond)
        assert torch.equal(a[0], b[0]), name                       # alone and at index 0 of a larger batch
        if "dither" in cond:
            c = e.extract_device(**one, padded_len=L, seed=SEED + 1, **cond)
            assert not torch.equal(a, c), name
    # repeated do_normalize calls: the moments are reduced in a fixed order
    big = torch.from_numpy(np.stack([O.synth_clip("chirp", 4_000_000, 82 + i) for i in range(3)])).to(dev)
    first = e.extract_device(big, padded_len=4_000_000, do_normalize=True)
    for _ in range(3):
        assert torch.equal(first, e.extract_device(big, padded_len=4_000_000, do_normalize=True))


def test_int16_and_float32_on_the_int16_grid_and_the_host_forms(ex):
    """A clip on the int16 grid gives bit-identical features as int16 PCM and as its float32 copy q / 32768 (the moments
    and the noise see the same values), and the host input forms of extract_host agree bit for bit."""
    import torch

    e = ex[80]
    dev = e.device
    q = [np.round(O.synth_clip(f, n, 110 + i) * 32767.0).astype(np.int16)
         for i, (f, n) in enumerate((("speech", 250000), ("noise", 480000), ("chirp", 600000), ("sine", 0)))]
    f = [x.astype(np.float32) / 32768.0 for x in q]
    lens = torch.tensor([len(x) for x in q], dtype=torch.int32, device=dev)
    buf16, offs16 = _ragged(q, 8, np.int16)
    buf32, offs32 = _ragged(f, 4, np.float32)
    for longform in (False, True):
        kw = dict(padded_len=600000) if longform else {}
        for name, cond in CONDS.items():
            a = e.extract_device(torch.from_numpy(buf16).to(dev), lengths=lens, offsets=torch.from_numpy(offs16).to(dev),
                                 seed=SEED, **kw, **cond)
            b = e.extract_device(torch.from_numpy(buf32).to(dev), lengths=lens, offsets=torch.from_numpy(offs32).to(dev),
                                 seed=SEED, **kw, **cond)
            assert torch.equal(a, b), (longform, name)
            if not longform:
                assert torch.equal(a, e.extract_host(q, seed=SEED, **cond)), name
                assert torch.equal(a, e.extract_host((buf16, offs16, lens.cpu().numpy()), seed=SEED, **cond)), name
    # dense host input: every row is a full clip
    rows = np.stack([O.synth_clip("speech", 160000, 120 + i) for i in range(3)])
    for name, cond in CONDS.items():
        a = e.extract_host(rows, seed=SEED, **cond)
        assert torch.equal(a, e.extract_host(list(rows), seed=SEED, **cond)), name
        out_host = np.empty((3, 80, 3000), np.float32)
        e.extract_host(rows, out_host=out_host, seed=SEED, **cond)
        assert np.array_equal(out_host, a.cpu().numpy()), name


def test_unconditioned_abi_call_equals_wlm_logmel_padded(ex):
    import torch

    from whisper_context_biasing_b200 import _native as N

    e = ex[80]
    B, L = 3, 123457
    x = torch.from_numpy(np.stack([O.synth_clip("speech", 123460, 90 + i) for i in range(B)])).to(e.device)
    lens = torch.tensor([123457, 5000, 0], dtype=torch.int32, device=e.device)
    a = e.extract_device(x, lengths=lens, padded_len=L)
    out = torch.empty_like(a)
    need = int(N.LIB.wlm_conditioned_workspace_bytes(e._plan, B, L))
    assert need >= int(N.LIB.wlm_padded_workspace_bytes(e._plan, B))
    ws = torch.empty(need, dtype=torch.uint8, device=e.device)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(padded_len=L, do_norm=0, dither=0.0, ws_bytes=need):
        return N.LIB.wlm_logmel_conditioned(e._plan, C.c_void_p(x.data_ptr()), N.WLM_PCM_F32, None,
                                            C.c_void_p(lens.data_ptr()), x.shape[1], padded_len, B, do_norm, dither, 5,
                                            C.c_void_p(out.data_ptr()), None, C.c_void_p(ws.data_ptr()), ws_bytes, st)
    assert call() == N.WLM_OK
    torch.cuda.synchronize()
    assert torch.equal(a, out)
    # errors
    assert call(dither=float("nan")) == N.WLM_ERR_BAD_ARG
    assert call(dither=float("inf")) == N.WLM_ERR_BAD_ARG
    assert call(do_norm=1, ws_bytes=need - 1) == N.WLM_ERR_WORKSPACE
    assert call(padded_len=200) == N.WLM_ERR_BAD_ARG
    assert call(padded_len=2 ** 31) == N.WLM_ERR_BAD_ARG
    assert int(N.LIB.wlm_conditioned_workspace_bytes(e._plan, B, 200)) == 0
    with pytest.raises(ValueError):
        e.extract_device(x, lengths=lens, padded_len=L, dither=float("nan"))


def test_constructor_dither_collator_and_cache():
    import torch

    from whisper_context_biasing_b200 import B200WhisperFeatureExtractor
    from whisper_context_biasing_b200.collator import B200DataCollatorSpeechSeq2SeqWithPadding
    from whisper_context_biasing_b200.feature_cache import FeatureCache

    with pytest.raises(ValueError):
        B200WhisperFeatureExtractor(feature_size=80, dither=float("inf"))
    fe = B200WhisperFeatureExtractor(feature_size=80, dither=1e-4)
    plain = B200WhisperFeatureExtractor(feature_size=80)
    clips = [O.synth_clip("speech", 40000, 95), O.synth_clip("zeros", 16000, 96)]
    torch.manual_seed(1)
    a = fe(clips, sampling_rate=16000).input_features
    b = fe(clips, sampling_rate=16000).input_features
    torch.manual_seed(1)
    c = fe(clips, sampling_rate=16000).input_features
    assert torch.equal(a, c) and not torch.equal(a, b)           # reproducible under torch.manual_seed, fresh per call
    p = plain(clips, sampling_rate=16000).input_features
    assert not torch.equal(a, p)
    # the silent clip: -1.5 without dither, the features of 1e-4 noise with it
    assert bool((p[1] == -1.5).all()) and not bool((a[1] == -1.5).all())
    # extract_device and extract_host dither too
    x = torch.from_numpy(O.pad_or_trim(clips)).to(fe.device)
    assert not torch.equal(fe.extract_device(x), plain.extract_device(x))
    torch.manual_seed(2)
    h = fe.extract_host(clips)
    torch.manual_seed(2)
    assert torch.equal(h, fe.extract_host([np.ascontiguousarray(c) for c in clips]))
    # the collator's batch is dithered
    col = B200DataCollatorSpeechSeq2SeqWithPadding(feature_extractor=fe, pad_token_id=50257, decoder_start_token_id=50258)
    items = [{"audio": c, "labels": [50258, 1, 2, 50257]} for c in clips]
    torch.manual_seed(3)
    batch = col(items)
    torch.manual_seed(3)
    assert torch.equal(batch["input_features"], fe.extract_host(clips))
    assert not torch.equal(batch["input_features"], plain.extract_host(clips))
    with pytest.raises(ValueError):
        FeatureCache(fe)
    FeatureCache(plain, capacity_bytes=1 << 24)
    fe.close()
    plain.close()
