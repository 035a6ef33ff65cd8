"""DataLoader workers for the device collator on a B200: batches collated in fork and spawn workers and featurised by
`finish` in the main process equal the in-process collator's, bit for bit, for every output format, both PCM formats,
with and without the loader's pinned memory, and with dither.  The workers are started after the main process has
created its plan and run kernels, as under a trainer; they never call CUDA.  The extractor's process guard is tested in
this process, by faking its owner pid and by unpickling it."""
import gc
import pickle

import numpy as np
import pytest

from test_loader_workers_cpu import LENGTHS, Items, check_pending, collator, item

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def fe():
    import torch

    from whisper_context_biasing_b200 import B200WhisperFeatureExtractor

    e = {m: B200WhisperFeatureExtractor(feature_size=m) for m in (80, 128)}
    yield e
    for x in e.values():
        x.set_feature_dtype(torch.float32)
        x.close()


def _loader(ds, col, method, pin):
    import torch

    return torch.utils.data.DataLoader(ds, batch_size=4, num_workers=2, collate_fn=col, pin_memory=pin,
                                       multiprocessing_context=method)


def _run(ex, dtype, method, pin, seed=None):
    """Every batch of a worker loader, finished, against the in-process collator on the same items (computed first)."""
    import torch

    ds = Items(dtype)
    batches = [[ds[i] for i in range(k, min(k + 4, len(ds)))] for k in range(0, len(ds), 4)]
    refs = []
    for items in batches:
        if seed is not None:
            torch.manual_seed(seed)
        refs.append(collator(ex, defer=False)(items))
    col = collator(ex, labels_on_device=True)
    n = 0
    for items, ref, batch in zip(batches, refs, _loader(ds, col, method, pin)):
        p = batch["input_features"]
        check_pending(p, items, ex.feature_size)
        assert p.pcm.is_pinned() == pin
        if seed is not None:
            torch.manual_seed(seed)
        col.finish(batch)
        got = batch["input_features"]
        assert got.is_cuda and got.dtype == ex.feature_dtype and got.shape == ref["input_features"].shape
        assert torch.equal(got, ref["input_features"])
        for k in ("labels", "decoder_input_ids", "bias_spans"):
            assert batch[k].is_cuda and torch.equal(batch[k].cpu(), ref[k])
        n += 1
    assert n == len(batches)


@pytest.mark.parametrize("pcm", [np.float32, np.int16], ids=["f32", "i16"])
@pytest.mark.parametrize("out", ["float32", "bfloat16", "float16"])
@pytest.mark.parametrize("n_mels", [80, 128])
def test_fork_workers_equal_in_process(fe, n_mels, out, pcm):
    import torch

    ex = fe[n_mels]
    ex.set_feature_dtype(getattr(torch, out))
    try:
        for pin in (False, True):
            _run(ex, pcm, "fork", pin)
    finally:
        ex.set_feature_dtype(torch.float32)


@pytest.mark.parametrize("n_mels,out,pcm", [(80, "float32", np.int16), (128, "bfloat16", np.float32)])
def test_spawn_workers_equal_in_process(fe, n_mels, out, pcm):
    import torch

    ex = fe[n_mels]
    ex.set_feature_dtype(getattr(torch, out))
    try:
        _run(ex, pcm, "spawn", True)
    finally:
        ex.set_feature_dtype(torch.float32)


def test_dither_seed_drawn_at_finish():
    import torch

    from whisper_context_biasing_b200 import B200WhisperFeatureExtractor

    ex = B200WhisperFeatureExtractor(feature_size=80, dither=1e-3)
    try:
        _run(ex, np.float32, "fork", True, seed=1234)
        items = [item(i, np.int16) for i in range(len(LENGTHS))]
        col = collator(ex, defer=True)
        torch.manual_seed(5)
        a = col.finish(col(items))["input_features"]
        torch.manual_seed(5)
        b = collator(ex, defer=False)(items)["input_features"]
        c = col.finish(col(items))["input_features"]        # the next draw of the generator: new noise
        assert torch.equal(a, b) and not torch.equal(a, c)
    finally:
        ex.close()


def test_pending_on_the_device_and_ordinary_batches(fe):
    import torch

    ex = fe[80]
    items = [item(i, np.float32) for i in range(len(LENGTHS))]
    ref = collator(ex)(items)                               # defer=None in the main process: featurised in the call
    assert ref["input_features"].is_cuda
    col = collator(ex, defer=True)
    batch = col(items)
    batch["input_features"] = batch["input_features"].to(ex.device, non_blocking=True)
    assert batch["input_features"].pcm.is_cuda
    assert torch.equal(col.finish(batch)["input_features"], ref["input_features"])
    assert col.finish(ref) is ref


def test_process_guard_and_detached_copy(fe):
    import torch

    ex = fe[80]
    clips = [item(i, np.float32)["audio"] for i in range(4)]
    want = ex.extract_host(clips)
    lens = torch.tensor([len(c) for c in clips], dtype=torch.int32, device=ex.device)
    x = torch.zeros((4, 480000), device=ex.device)
    calls = [lambda e: e(clips, sampling_rate=16000), lambda e: e.extract_host(clips), lambda e: e.extract_device(x),
             lambda e: e.frame_mask_device(lens)]
    launches = ex.launch_count
    owner = ex._owner_pid
    ex._owner_pid = owner + 1                               # what a forked child sees
    try:
        for call in calls:
            with pytest.raises(RuntimeError, match="finish"):
                call(ex)
    finally:
        ex._owner_pid = owner
    assert ex.launch_count == launches
    back = pickle.loads(pickle.dumps(ex))
    assert back.feature_size == 80 and back.device == ex.device and back.to_dict() == ex.to_dict()
    for call in calls:
        with pytest.raises(RuntimeError, match="unpickled"):
            call(back)
    back.close()
    del back
    gc.collect()
    assert torch.equal(ex.extract_host(clips), want)      # the owner's plan survived its copy
