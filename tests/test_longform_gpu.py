"""Long-form features on a B200: `wlm_logmel_padded` (any padded length L) and the `truncation=False,
padding="longest"` call, against the 30-s kernels (bit for bit at L = 480000), the long-form golden
vectors of the live reference and the oracle."""
import ctypes as C
import importlib.util
import json
import os

import numpy as np
import pytest

from oracle import logmel_oracle as O

_spec = importlib.util.spec_from_file_location("_longform_oracle",
                                               os.path.join(os.path.dirname(os.path.abspath(__file__)), "longform_oracle.py"))
LO = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(LO)

pytestmark = pytest.mark.gpu

TOL = 5e-4
HERE = os.path.dirname(os.path.abspath(__file__))
LONG = dict(sampling_rate=16000, truncation=False, padding="longest")


@pytest.fixture(scope="module")
def lf():
    import torch

    from whisper_context_biasing_b200 import B200WhisperFeatureExtractor

    ex = {m: B200WhisperFeatureExtractor(feature_size=m) for m in (64, 80, 128)}
    spec = importlib.util.spec_from_file_location("_make_longform_golden",
                                                  os.path.join(HERE, "golden", "make_longform_golden.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    z = np.load(os.path.join(HERE, "golden", "logmel_longform_golden.npz"))
    meta = json.loads(bytes(z["meta_json"]).decode())
    yield ex, gen, z, meta
    for e in ex.values():
        e.set_feature_dtype(torch.float32)
        e.close()


def _ragged(clips, gran, dtype):
    """one 1-D buffer, clip starts multiples of `gran` elements (16 bytes)"""
    offs, cur = [], 0
    for c in clips:
        offs.append(cur)
        cur += (len(c) + gran - 1) // gran * gran
    buf = np.zeros(cur + gran, dtype)
    for o, c in zip(offs, clips):
        buf[o:o + len(c)] = c
    return buf, np.array(offs, np.int64)


def test_bit_identical_to_30s_path_at_480000(lf):
    """L = 480000 is the 30-s geometry: features and gmax equal wlm_logmel's bit for bit, for every layout, PCM format,
    output format and mel bank (64 mels: the table-driven variant)."""
    import torch

    ex, *_ = lf
    lengths = [480000, 0, 1, 200, 401, 5121, 77777, 479999, 480000, 600000, 250000, 160]
    fams = O.FAMILIES
    clips = [O.synth_clip(fams[i % len(fams)], L, 300 + i) for i, L in enumerate(lengths)]
    q16 = [np.round(c * 32767.0).astype(np.int16) for c in clips]
    assert ex[64].kernel_variant == 0
    for m in (80, 128, 64):
        e = ex[m]
        dev = e.device
        lens = torch.tensor(lengths, dtype=torch.int32, device=dev)
        dense = torch.from_numpy(O.pad_or_trim(clips, 600000)).to(dev)
        dense16 = torch.from_numpy(np.stack([np.pad(c[:600000], (0, 600000 - len(c[:600000]))) for c in q16])).to(dev)
        buf, offs = _ragged(clips, 4, np.float32)
        buf16, offs16 = _ragged(q16, 8, np.int16)
        layouts = {
            "dense": dict(pcm=dense, lengths=lens),
            "dense_nolen": dict(pcm=dense[:, :480000].contiguous()),
            "ragged": dict(pcm=torch.from_numpy(buf).to(dev), lengths=lens, offsets=torch.from_numpy(offs).to(dev)),
            "dense_i16": dict(pcm=dense16, lengths=lens),
            "ragged_i16": dict(pcm=torch.from_numpy(buf16).to(dev), lengths=lens,
                               offsets=torch.from_numpy(offs16).to(dev)),
        }
        for dt in (torch.float32, torch.bfloat16, torch.float16):
            e.set_feature_dtype(dt)
            for name, kw in layouts.items():
                a, ga = e.extract_device(**kw, return_gmax=True)
                n0 = e.launch_count
                b, gb = e.extract_device(**kw, return_gmax=True, padded_len=480000)
                assert e.launch_count == n0 + 2
                assert a.shape == b.shape and a.dtype == b.dtype
                assert torch.equal(a, b), (m, dt, name, (a.float() - b.float()).abs().max().item())
                assert torch.equal(ga, gb), (m, dt, name)
        e.set_feature_dtype(torch.float32)


def test_against_longform_golden_and_oracle(lf):
    ex, gen, z, meta = lf
    worst = 0.0
    for c, case in zip(meta["cases"], gen.CASES):
        clips = gen.case_clips(case)
        e = ex[c["n_mels"]]
        r = e(clips, **LONG, pad_to_multiple_of=c["pad_to_multiple_of"], return_tensors="np", return_attention_mask=True)
        got = r["input_features"]
        assert got.shape == (len(clips), c["n_mels"], c["n_frames"]) and got.dtype == np.float32, c["name"]
        d = float(np.abs(got[:, :, c["frames"]] - z[c["name"] + "_features"]).max())
        worst = max(worst, d)
        assert d <= TOL, (c["name"], d)
        assert np.array_equal(r["attention_mask"], z[c["name"] + "_mask"]), c["name"]
        ref = LO.extract_longform(clips, c["n_mels"], "f64", pad_to_multiple_of=c["pad_to_multiple_of"])
        d2 = float(np.abs(got - ref).max())
        assert d2 <= TOL, (c["name"], "oracle", d2)
    print("worst vs long-form golden", worst)


def test_gmax_and_int16_input(lf):
    import torch

    ex, gen, z, meta = lf
    e = ex[80]
    case = next(c for c in gen.CASES if c[0] == "int16_40s_m80")
    clips = gen.case_clips(case)
    L = LO.padded_length([len(x) for x in clips])
    lens = torch.tensor([len(x) for x in clips], dtype=torch.int32, device=e.device)
    buf, offs = _ragged(clips, 4, np.float32)
    a, ga = e.extract_device(torch.from_numpy(buf).to(e.device), lengths=lens, offsets=torch.from_numpy(offs).to(e.device),
                             padded_len=L, return_gmax=True)
    q = [np.round(x * 32768.0).astype(np.int16) for x in clips]       # the clips lie on the int16 grid
    assert all(np.array_equal(qq.astype(np.float32) / 32768.0, x) for qq, x in zip(q, clips))
    buf16, offs16 = _ragged(q, 8, np.int16)
    b, gb = e.extract_device(torch.from_numpy(buf16).to(e.device), lengths=lens,
                             offsets=torch.from_numpy(offs16).to(e.device), padded_len=L, return_gmax=True)
    assert torch.equal(a, b) and torch.equal(ga, gb)
    assert np.abs(np.maximum(ga.cpu().numpy(), -10) - z["int16_40s_m80_gmax"]).max() <= 4 * TOL


def test_global_maximum_lies_after_the_first_30s(lf):
    """Frames of the first 30 s are clamped by a maximum 50 s into the clip: they match the oracle and differ from what
    the 30-s path (which never sees the burst) gives."""
    ex, gen, z, meta = lf
    case = next(c for c in gen.CASES if c[0] == "burst50_m80")
    clips = gen.case_clips(case)
    got = ex[80](clips, **LONG, return_tensors="np").input_features
    ref = LO.extract_longform(clips, 80, "f64")
    assert np.abs(got[:, :, :3000] - ref[:, :, :3000]).max() <= TOL
    short = ex[80](clips, sampling_rate=16000, return_tensors="np").input_features
    assert np.abs(got[0, :, :3000] - short[0]).max() > 0.25


def test_same_clip_alone_and_in_a_longer_batch(lf):
    import torch

    ex, *_ = lf
    x = O.synth_clip("speech", 733333, 77)
    x[-8000:] = 0.0                          # the clip's maximum is not in its last frames
    y = O.synth_clip("noise", 1_500_001, 78)
    for m in (80, 128):
        e = ex[m]
        buf, offs = _ragged([x], 4, np.float32)
        a, ga = e.extract_device(torch.from_numpy(buf).to(e.device), lengths=torch.tensor([733333], dtype=torch.int32,
                                 device=e.device), offsets=torch.from_numpy(offs).to(e.device), padded_len=733333,
                                 return_gmax=True)
        buf2, offs2 = _ragged([y, x], 4, np.float32)
        b, gb = e.extract_device(torch.from_numpy(buf2).to(e.device),
                                 lengths=torch.tensor([len(y), len(x)], dtype=torch.int32, device=e.device),
                                 offsets=torch.from_numpy(offs2).to(e.device), padded_len=1_920_000, return_gmax=True)
        n = 733333 // 160 - 1                # frames [0, len // 160 - 2]: no reflection at the end in either
        assert torch.equal(a[0, :, :n], b[1, :, :n]), m
        assert torch.equal(ga[0], gb[1]), m
        assert b.shape[2] == 12000


def test_silence_is_exactly_minus_1_5(lf):
    import torch

    ex, *_ = lf
    e = ex[80]
    clips = [np.zeros(n, np.float32) for n in (0, 1000, 700001, 5)]
    for dt in (torch.float32, torch.bfloat16, torch.float16):
        e.set_feature_dtype(dt)
        f = e(clips, **LONG, pad_to_multiple_of=160).input_features
        assert tuple(f.shape) == (4, 80, 700160 // 160)
        assert bool((f.float() == -1.5).all()), dt
    e.set_feature_dtype(torch.float32)


def test_masks(lf):
    import torch

    from whisper_context_biasing_b200 import B200WhisperFeatureExtractor

    ex, *_ = lf
    e = ex[80]
    for L in (201, 5361, 480000, 720037, 12345):
        lens = [0, 1, 159, 160, 161, L - 1, L, max(L - 400, 0)]
        got = e.frame_mask_device(torch.tensor(lens, dtype=torch.int32, device=e.device), padded_len=L)
        assert np.array_equal(got.cpu().numpy(), LO.frame_mask(lens, L)), L
    assert np.array_equal(e.frame_mask_device(torch.tensor([5, 480000], dtype=torch.int32, device=e.device)).cpu().numpy(),
                          O.frame_mask([5, 480000]))
    clips = [O.synth_clip("noise", n, 90 + i) for i, n in enumerate((5361, 3000, 17))]
    r = e(clips, **LONG, return_attention_mask=True, return_tensors="pt")
    assert tuple(r["attention_mask"].shape) == (3, 33)
    assert np.array_equal(r["attention_mask"].cpu().numpy(), LO.frame_mask([5361, 3000, 17], 5361))
    # the constructor's return_attention_mask with the call's None: the sample-level mask [B, L]
    q = B200WhisperFeatureExtractor(feature_size=80, return_attention_mask=True)
    r = q(clips, **LONG, return_tensors="np")
    assert r["attention_mask"].shape == (3, 5361)
    assert r["attention_mask"].sum(1).tolist() == [5361, 3000, 17]
    q.close()


def test_more_than_2_pow_31_output_elements():
    """3 clips x 128 mels x 15.6 h, int16 in, bfloat16 out: 2.16e9 feature elements, 64-bit addressing in both passes.
    The clips are silent but for one tone burst each (the last one beyond element 2^31): the burst frames match the
    oracle on a local window and every other element equals the clip's floor exactly."""
    import torch

    from whisper_context_biasing_b200 import B200WhisperFeatureExtractor

    e = B200WhisperFeatureExtractor(feature_size=128, feature_dtype=torch.bfloat16)
    N = 15 * 3600 * 16000 + 36 * 16000 * 60          # 15.6 h
    T = N // 160
    assert 3 * 128 * T > 2 ** 31
    pcm = torch.zeros((3, N), dtype=torch.int16, device=e.device)
    burst = np.round(O.synth_clip("chirp", 8000, 5) * 32767.0).astype(np.int16)
    at = [160 * 1_000_000, 160 * 3_000_000, N - 160 * 1000]     # sample positions, multiples of 160
    for b, s in enumerate(at):
        pcm[b, s:s + 8000] = torch.from_numpy(burst).to(e.device)
    out, gmax = e.extract_device(pcm, padded_len=N, return_gmax=True)
    assert tuple(out.shape) == (3, 128, T) and out.dtype == torch.bfloat16
    w = burst.astype(np.float32) / 32768.0
    win = np.concatenate([np.zeros(16000, np.float32), w, np.zeros(16000, np.float32)])   # 250 frames around the burst
    ref, gref = LO.extract_longform([win], 128, "f64", return_gmax=True)
    for b, s in enumerate(at):
        f0 = (s - 16000) // 160
        got = out[b, :, f0 + 3:f0 + 247].float().cpu().numpy()
        assert np.abs(got - ref[0, :, 3:247]).max() <= 1e-2, b           # bfloat16: 8 significant bits
        assert abs(float(gmax[b]) - float(gref[0])) <= 4 * TOL
        thr = ((torch.clamp(gmax[b] - 8.0, min=-10.0) + 4.0) * 0.25).to(torch.bfloat16)
        assert out[b, 0, 0] == thr
        v = out[b].clone()
        v[:, f0:f0 + 250] = thr
        assert bool((v == thr).all()), b
        del v
    del out, pcm
    e.close()
    torch.cuda.empty_cache()


def test_stream_order_with_the_30s_path(lf):
    """wlm_logmel and wlm_logmel_padded back to back on the same PCM and output buffers, no synchronisation: each
    call sees the PCM written just before it and the copy behind it sees all of its features."""
    import torch

    ex, *_ = lf
    e = ex[80]
    g = torch.Generator(device="cuda").manual_seed(9)
    B, L = 60, 480000
    versions = [0.1 * torch.randn(B, L, device=e.device, generator=g) for _ in range(6)]
    want = []
    for v in versions:
        want.append(e.extract_device(v).clone())
        torch.cuda.synchronize()
    x = torch.empty(B, L, device=e.device)
    out = torch.empty(B, 80, 3000, device=e.device)
    out_long = torch.empty(B, 80, 720000 // 160, device=e.device)
    got, got_long = [], []
    for i, v in enumerate(versions):             # no synchronisation anywhere in this loop
        x.copy_(v)
        e.extract_device(x, out=out, padded_len=L if i % 2 else None)
        got.append(out.clone())
        e.extract_device(x, out=out_long, padded_len=720000)
        got_long.append(out_long.clone())
    torch.cuda.synchronize()
    for i, (a, b) in enumerate(zip(want, got)):
        assert torch.equal(a, b), i
    for i, v in enumerate(versions):
        one = e.extract_device(v, padded_len=720000)
        assert torch.equal(one, got_long[i]), i


def test_call_forms_and_errors(lf):
    import torch

    from whisper_context_biasing_b200 import B200WhisperFeatureExtractor
    from whisper_context_biasing_b200 import _native as N

    ex, *_ = lf
    e = ex[80]
    q = B200WhisperFeatureExtractor(feature_size=80, return_attention_mask=True)
    n = 333333                                           # n % 4 != 0: the CUDA rows are padded to 16-byte boundaries
    rows = np.stack([O.synth_clip("speech", n, 40 + i) for i in range(3)])
    kinds = {"list": list(rows), "numpy": rows, "cpu": torch.from_numpy(rows), "cuda": torch.from_numpy(rows).to(e.device)}
    # every input kind gives the same features and mask bits, in both geometries, with and without do_normalize, in the
    # three mask modes (none, the call's return_attention_mask=True, the constructor's); a 1-D array gives its row's
    for geometry, L in ((dict(sampling_rate=16000), 480000), (LONG, n)):
        for do_normalize in (False, True):
            for fe, mask_kw in ((e, {}), (e, dict(return_attention_mask=True)), (q, {})):
                kw = dict(**geometry, **mask_kw, do_normalize=do_normalize, return_tensors="np")
                got = {k: fe(x, **kw) for k, x in kinds.items()}
                ref = got["list"]
                case = (L, do_normalize, fe is q, mask_kw)
                assert ref["input_features"].shape == (3, 80, L // 160), case
                if mask_kw:
                    assert ref["attention_mask"].shape == (3, L // 160), case
                elif do_normalize or fe is q:
                    assert ref["attention_mask"].shape == (3, L), case             # HF's sample-level mask
                else:
                    assert "attention_mask" not in ref, case
                got["1-D"] = fe(rows[1], **kw)
                for k, r in got.items():
                    assert sorted(r) == sorted(ref), (case, k)
                    for key in ref:
                        want = ref[key][1:2] if k == "1-D" else ref[key]
                        assert np.array_equal(r[key], want), (case, k, key)
    d = e(kinds["cuda"], **LONG, return_tensors="pt").input_features
    assert d.is_cuda
    one = e(rows[1], **LONG, pad_to_multiple_of=480000, max_length=1000, return_tensors="pt").input_features
    assert tuple(one.shape) == (1, 80, 3000)
    q.close()
    # errors
    for geometry in (dict(sampling_rate=16000), LONG):
        for x in (rows[None], torch.from_numpy(rows)[None], kinds["cuda"][None]):
            with pytest.raises(ValueError):
                e(x, **geometry)
    for x in (kinds["list"], kinds["cuda"]):
        with pytest.raises(ValueError):
            e(x, **LONG, pad_to_multiple_of=2 ** 31)
    with pytest.raises(ValueError):
        e([np.zeros(200, np.float32)], **LONG)
    with pytest.raises(ValueError):
        e.extract_device(torch.zeros(1, 400, device=e.device), padded_len=200)
    with pytest.raises(ValueError):
        e.extract_device(torch.zeros(1, 400, device=e.device), padded_len=2 ** 31)
    x = torch.zeros(2, 1024, device=e.device)
    out = torch.empty(2, 80, 6, device=e.device)
    need = int(N.LIB.wlm_padded_workspace_bytes(e._plan, 2))
    ws = torch.zeros(need + 64, dtype=torch.uint8, device=e.device)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(pcm_ptr, padded_len, ws_bytes, out_ptr=out.data_ptr()):
        return N.LIB.wlm_logmel_padded(e._plan, C.c_void_p(pcm_ptr), N.WLM_PCM_F32, None, None, 1024, padded_len, 2,
                                       C.c_void_p(out_ptr), None, C.c_void_p(ws.data_ptr()), ws_bytes, st)
    assert call(x.data_ptr(), 1000, need) == N.WLM_OK
    assert call(x.data_ptr(), 200, need) == N.WLM_ERR_BAD_ARG
    assert call(x.data_ptr(), 2 ** 31, need) == N.WLM_ERR_BAD_ARG
    assert call(x.data_ptr(), 1000, need - 1) == N.WLM_ERR_WORKSPACE
    assert call(x.data_ptr() + 4, 1000, need) == N.WLM_ERR_BAD_ARG
    assert call(x.data_ptr(), 1000, need, out.data_ptr() + 4) == N.WLM_ERR_BAD_ARG
    assert N.LIB.wlm_logmel(e._plan, None, 0, None, None, 0, 0, None, None, None, 0, st) == N.WLM_OK      # B = 0
    m = torch.empty(2, 6, dtype=torch.int32, device=e.device)
    assert N.LIB.wlm_frame_mask_padded(e._plan, C.c_void_p(torch.zeros(2, dtype=torch.int32, device=e.device).data_ptr()),
                                       2, 200, C.c_void_p(m.data_ptr()), st) == N.WLM_ERR_BAD_ARG
    torch.cuda.synchronize()
    # every combination refused before is still refused
    y = rows[0]
    for kw in (dict(padding="longest"), dict(padding="longest", truncation=True), dict(truncation=False),
               dict(padding="max_length", truncation=False), dict(pad_to_multiple_of=160), dict(max_length=1000),
               dict(padding="do_not_pad", truncation=False), dict(padding=True, truncation=False)):
        with pytest.raises(NotImplementedError):
            e(y, sampling_rate=16000, **kw)
