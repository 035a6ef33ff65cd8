"""DataLoader workers for the device collator, without a GPU: PCM is collated in fork and spawn workers into
`PendingFeatures`, and `finish` featurises it in the main process.  A stub extractor stands in for the B200 one (its
"features" are each clip's sum and length, so `finish` must hand the kernel the right clips); like the real one it refuses
to featurise outside the process that made it, so a worker that touched it would fail the loader.  The real extractor's
process guard and pickled state are checked here with libwlm's calls replaced by fakes."""
import contextlib
import ctypes as C
import os
import pickle
import types
from collections.abc import Mapping

import numpy as np
import pytest
import torch

from whisper_context_biasing_b200 import (B200DataCollatorSpeechSeq2SeqWithPadding, B200FeaturesTrainerMixin,
                                          LogMelBatch, PendingFeatures, collate_labels, pcm_dataset_class)

LENGTHS = [0, 1, 3, 160, 479999, 480000, 700000]
N_SAMPLES = 480000
PAD, SOT, PREV = 50257, 50258, 50360


class StubExtractor:
    """Duck type of `B200WhisperFeatureExtractor` as the collator uses it, on the CPU."""

    model_input_names = ["input_features"]
    feature_size = 4
    device = torch.device("cpu")

    def __init__(self):
        self.owner = os.getpid()
        self.calls = []

    def __setstate__(self, state):
        self.__dict__.update(state)
        self.owner = None                                  # detached, as the real extractor unpickles

    def _featurise(self, clips):
        if self.owner != os.getpid():
            raise RuntimeError("stub extractor used outside the process that created it")
        out = torch.zeros((len(clips), self.feature_size, 3000))
        for b, c in enumerate(clips):
            c = c[:N_SAMPLES].astype(np.float64)
            out[b, 0] = float(c.sum())
            out[b, 1] = float(len(c))
        return out

    def pad(self, processed_features, padding="longest", return_tensors=None):
        return LogMelBatch({"input_features": torch.stack([torch.as_tensor(x) for x in processed_features["input_features"]])})

    def extract_host(self, clips):
        self.calls.append("extract_host")
        return self._featurise(clips)

    def extract_device(self, pcm, offsets=None, lengths=None):
        self.calls.append(("extract_device", pcm.device, pcm.dtype))
        assert offsets.dtype == torch.int64 and lengths.dtype == torch.int32
        x = pcm.numpy()
        return self._featurise([x[o:o + n] for o, n in zip(offsets.tolist(), lengths.tolist())])


def clip(i, dtype):
    rng = np.random.default_rng(1000 + i)
    n = LENGTHS[i % len(LENGTHS)]
    if dtype == np.int16:
        return rng.integers(-32768, 32768, n).astype(np.int16)
    return rng.standard_normal(n).astype(np.float32)


def item(i, dtype):
    rng = np.random.default_rng(i)
    prompt = [PREV] + rng.integers(0, 1000, int(rng.integers(0, 5))).tolist()
    labels = prompt + [SOT] + rng.integers(0, 1000, int(rng.integers(1, 9))).tolist() + [PAD]
    spans = [rng.integers(0, 1000, int(rng.integers(1, 4))).tolist() for _ in range(int(rng.integers(0, 3)))]
    return {"audio": clip(i, dtype), "labels": labels, "bias_spans": spans}


class Items(torch.utils.data.Dataset):
    def __init__(self, dtype):
        self.dtype = dtype

    def __len__(self):
        return 2 * len(LENGTHS)

    def __getitem__(self, i):
        return item(i, self.dtype)


def collator(fe, **kw):
    return B200DataCollatorSpeechSeq2SeqWithPadding(feature_extractor=fe, pad_token_id=PAD, decoder_start_token_id=SOT,
                                                    decoder_prev_token_id=PREV, **kw)


def check_pending(p, items, n_mels=4):
    """The pending layout holds every clip's samples, trimmed to 30 s, each clip on a 16-byte boundary."""
    assert isinstance(p, PendingFeatures) and len(p) == len(items)
    assert p.shape == (len(items), n_mels, 3000) and p.numel() == len(items) * n_mels * 3000
    assert p.pcm.dim() == 1 and p.offsets.dtype == torch.int64 and p.lengths.dtype == torch.int32
    x = p.pcm.cpu().numpy()
    assert x.dtype == items[0]["audio"].dtype
    for o, n, it in zip(p.offsets.tolist(), p.lengths.tolist(), items):
        want = it["audio"][:N_SAMPLES]
        assert n == len(want) and (o * x.itemsize) % 16 == 0
        assert np.array_equal(x[o:o + n], want)


def check_labels(batch, items):
    want = collate_labels(items, PAD, SOT, PREV)
    assert set(want) == {"labels", "decoder_input_ids", "bias_spans"}
    for k, v in want.items():
        assert batch[k].device.type == "cpu" and torch.equal(batch[k], v), k


@pytest.mark.parametrize("dtype", [np.float32, np.int16], ids=["f32", "i16"])
@pytest.mark.parametrize("method", ["fork", "spawn"])
def test_workers_collate_pcm_and_finish_featurises(method, dtype):
    fe = StubExtractor()
    col = collator(fe)                                      # defer=None: defers inside the workers only
    ds = Items(dtype)
    loader = torch.utils.data.DataLoader(ds, batch_size=3, num_workers=2, collate_fn=col,
                                         multiprocessing_context=method)
    n = 0
    for k, batch in enumerate(loader):
        items = [ds[i] for i in range(3 * k, min(3 * k + 3, len(ds)))]
        assert isinstance(batch, LogMelBatch)
        check_pending(batch["input_features"], items)
        check_labels(batch, items)
        assert fe.calls == []                               # the main process's extractor is untouched until finish
        pcm_dtype = batch["input_features"].pcm.dtype
        out = col.finish(batch)
        assert out is batch and fe.calls == [("extract_device", torch.device("cpu"), pcm_dtype)]
        ref = collator(fe)(items)                           # in the main process: featurised in the call
        assert torch.equal(out["input_features"], ref["input_features"])
        for key in ("labels", "decoder_input_ids", "bias_spans"):
            assert torch.equal(out[key], ref[key])
        fe.calls.clear()
        n += len(items)
    assert n == len(ds)


def test_defer_choice_finish_no_op_and_labels_on_device():
    fe = StubExtractor()
    items = [item(i, np.float32) for i in range(4)]
    eager = collator(fe)(items)                             # defer=None in the main process: as before
    assert isinstance(eager["input_features"], torch.Tensor) and fe.calls == ["extract_host"]
    assert collator(fe).finish(eager) is eager and fe.calls == ["extract_host"]
    fe.calls.clear()
    col = collator(fe, defer=True, labels_on_device=True)
    batch = col(items)
    assert fe.calls == [] and isinstance(batch["input_features"], PendingFeatures)
    check_labels(batch, items)                              # labels stay on the CPU until finish
    col.finish(batch)
    assert torch.equal(batch["input_features"], eager["input_features"])
    with pytest.raises(RuntimeError):                       # defer=False in a process that is not the extractor's
        fe.owner = -1
        collator(fe, defer=False)(items)
    # items that carry features are stacked as before, deferred or not
    pre = [{"input_features": np.full((4, 3000), i, np.float32), "labels": it["labels"]} for i, it in enumerate(items)]
    assert torch.equal(collator(fe, defer=True)(pre)["input_features"], collator(fe)(pre)["input_features"])


def test_collator_pickles_without_the_processor():
    fe = StubExtractor()
    proc = types.SimpleNamespace(feature_extractor=fe, tokenizer=types.SimpleNamespace(pad_token_id=PAD))
    col = B200DataCollatorSpeechSeq2SeqWithPadding(processor=proc, decoder_start_token_id=SOT, decoder_prev_token_id=PREV,
                                                   labels_on_device=True)
    back = pickle.loads(pickle.dumps(col))
    assert back.processor is None and back.feature_extractor.owner is None
    for k in ("pad_token_id", "decoder_start_token_id", "decoder_prev_token_id", "labels_on_device", "defer"):
        assert getattr(back, k) == getattr(col, k), k
    assert col.processor is proc                            # pickling leaves the original alone


class ReferenceStandIn(torch.utils.data.Dataset):
    """The part of the reference's `PromptWhisperDataset` the PCM wrapper relies on: one extractor call per item."""

    def __init__(self, base_path, jsonl_data, phase, feature_extractor, tokenizer, *args, **kwargs):
        self.feature_extractor, self.tokenizer = feature_extractor, tokenizer
        self.data = [("f", "t", "d", i, []) for i in range(2 * len(LENGTHS))]

    def __len__(self):
        return len(self.data)

    def __getitem__(self, i):
        it = item(i, np.float32)
        pcm = self.feature_extractor(it["audio"], sampling_rate=16000).input_features
        return {"input_features": torch.tensor(pcm[0]), "labels": it["labels"], "bias_spans": it["bias_spans"]}


def test_pcm_dataset_reaches_spawn_workers():
    fe = StubExtractor()
    ds = pcm_dataset_class(ReferenceStandIn)("/nonexistent", "rows", "train", fe, None)
    back = pickle.loads(pickle.dumps(ds))
    assert type(back).__name__ == "PcmPromptWhisperDataset" and isinstance(back, ReferenceStandIn)
    assert back.device_feature_extractor.owner is None and len(back) == len(ds)
    assert np.array_equal(back[5]["audio"], ds[5]["audio"])
    col = collator(fe)
    loader = torch.utils.data.DataLoader(ds, batch_size=4, num_workers=2, collate_fn=col, multiprocessing_context="spawn")
    for k, batch in enumerate(loader):
        items = [ds[i] for i in range(4 * k, min(4 * k + 4, len(ds)))]
        check_pending(batch["input_features"], items)
        assert torch.equal(col.finish(batch)["input_features"], collator(fe)(items)["input_features"])


# -- B200FeaturesTrainerMixin ---------------------------------------------------------------------------------------------
class TrainerStandIn:
    """`transformers.Trainer`'s input preparation (trainer.py, 5.5), restated: `_prepare_input` rebuilds mappings with
    `type(data)`, moves tensors, passes anything else through; training and prediction steps call `_prepare_inputs`."""

    def __init__(self, data_collator):
        self.data_collator = data_collator
        self.device = torch.device("cpu")

    def _prepare_input(self, data):
        if isinstance(data, Mapping):
            return type(data)({k: self._prepare_input(v) for k, v in data.items()})
        elif isinstance(data, (tuple, list)):
            return type(data)(self._prepare_input(v) for v in data)
        elif isinstance(data, torch.Tensor):
            return data.to(device=self.device)
        return data

    def _prepare_inputs(self, inputs):
        inputs = self._prepare_input(inputs)
        if len(inputs) == 0:
            raise ValueError("empty batch")
        return inputs

    def floating_point_ops(self, inputs):
        return 6 * inputs["input_features"].numel()       # what Trainer reads on the batch the loader gave

    def training_step(self, model, inputs):
        return model(**self._prepare_inputs(inputs))


def test_mixin_finishes_deferred_batches():
    class Trainer(B200FeaturesTrainerMixin, TrainerStandIn):
        pass

    fe = StubExtractor()
    items = [item(i, np.int16) for i in range(5)]
    t = Trainer(collator(fe, defer=True))
    batch = t.data_collator(items)
    assert t.floating_point_ops(batch) == 6 * 5 * 4 * 3000
    seen = {}
    t.training_step(lambda **kw: seen.update(kw), batch)
    assert set(seen) == {"input_features", "labels", "decoder_input_ids", "bias_spans"}
    assert torch.equal(seen["input_features"], collator(fe)(items)["input_features"])
    ready = t._prepare_inputs(collator(fe)(items))           # an ordinary batch is only prepared
    assert isinstance(ready, LogMelBatch) and torch.equal(ready.input_features, seen["input_features"])


def test_mixin_with_seq2seq_trainer(tmp_path):
    pytest.importorskip("accelerate")
    tr = pytest.importorskip("transformers")

    class Trainer(B200FeaturesTrainerMixin, tr.Seq2SeqTrainer):
        pass

    fe = StubExtractor()
    items = [item(i, np.float32) for i in range(3)]
    args = tr.Seq2SeqTrainingArguments(output_dir=str(tmp_path), use_cpu=True, report_to=[])
    t = Trainer(model=torch.nn.Linear(1, 1), args=args, data_collator=collator(fe, defer=True))
    out = t._prepare_inputs(t.data_collator(items))
    assert isinstance(out, LogMelBatch)
    assert torch.equal(out["input_features"], collator(fe)(items)["input_features"])


# -- the extractor's process guard, with libwlm's calls replaced ----------------------------------------------------------
@pytest.fixture
def fake_lib(monkeypatch):
    """A B200WhisperFeatureExtractor can be made without a GPU: CUDA queries and the wlm_* calls are fakes that log."""
    from whisper_context_biasing_b200 import _native as N

    log = []

    def create(dev, n_mels, table, handle):
        log.append("wlm_plan_create")
        handle._obj.value = 0x1000
        return 0

    def destroy(plan):
        log.append("wlm_plan_destroy")
        return 0

    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(torch.cuda, "current_device", lambda: 0)
    monkeypatch.setattr(torch.cuda, "device", lambda d: contextlib.nullcontext())
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a: types.SimpleNamespace(cuda_stream=0))
    for name in N.SYMBOLS:
        def other(*a, _name=name):
            log.append(_name)
            raise AssertionError(f"{_name} called")
        monkeypatch.setattr(N.LIB, name, other)
    monkeypatch.setattr(N.LIB, "wlm_plan_create", create)
    monkeypatch.setattr(N.LIB, "wlm_plan_destroy", destroy)
    return log


def _featurising_calls(fe):
    pcm = np.zeros(16000, np.float32)
    return [lambda: fe(pcm, sampling_rate=16000), lambda: fe([pcm], sampling_rate=16000, truncation=False, padding="longest"),
            lambda: fe.extract_host([pcm]), lambda: fe.extract_device(torch.zeros(16000)),
            lambda: fe.frame_mask_device(torch.zeros(1, dtype=torch.int32))]


def test_extractor_refuses_other_processes_and_unpickles_detached(fake_lib):
    from whisper_context_biasing_b200 import B200WhisperFeatureExtractor

    fe = B200WhisperFeatureExtractor(feature_size=128, dither=0.5, return_attention_mask=True, output="numpy")
    try:
        _check_guard_and_pickle(fe, fake_lib)
    finally:
        fe._plan = None                                     # never reaches the real wlm_plan_destroy


def _check_guard_and_pickle(fe, fake_lib):
    assert fake_lib == ["wlm_plan_create"] and fe._owner_pid == os.getpid()
    fe._owner_pid = os.getpid() + 1                         # as a forked child sees it
    for call in _featurising_calls(fe):
        with pytest.raises(RuntimeError, match="finish"):
            call()
    fe.close()
    assert fake_lib == ["wlm_plan_create"] and fe._plan is None     # the parent's plan is not freed
    fe._owner_pid = os.getpid()

    fe._plan = C.c_void_p(0x1000)
    back = pickle.loads(pickle.dumps(fe))
    assert back._plan is None and back._ws is None
    assert (back.feature_size, back.dither, back.return_attention_mask, back.output, back.device, back.feature_dtype) == \
        (128, 0.5, True, "numpy", torch.device("cuda", 0), torch.float32)
    assert back.to_dict() == fe.to_dict() and np.array_equal(back.mel_filters, fe.mel_filters)
    assert back.model_input_names == ["input_features"] and back.nb_max_frames == 3000
    for call in _featurising_calls(back):
        with pytest.raises(RuntimeError, match="unpickled"):
            call()
    back.close()
    del back
    assert fake_lib == ["wlm_plan_create"]
    fe.close()                                              # the owner frees its plan, once
    fe.close()
    assert fake_lib == ["wlm_plan_create", "wlm_plan_destroy"]
