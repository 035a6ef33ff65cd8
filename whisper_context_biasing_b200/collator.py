"""Device-side collator: same batch dict as the reference's `DataCollatorSpeechSeq2SeqWithPadding`
(REF/data_utils/data_collator.py:27-127), but the log-mel features are computed for the whole batch
in ONE call of the B200 extractor, in the main process, and stay in HBM.

Differences from the reference, on purpose:
  * items may carry raw PCM under "audio" (1-D float32 / int16 numpy) instead of precomputed
    "input_features" -- the dataset then skips REF/data_utils/data_loader.py:171-172 and the two
    host copies of the features disappear; items that already carry "input_features" are stacked
    exactly like `feature_extractor.pad(..., padding="longest", return_tensors="pt")` (:71-76);
  * label / bias-span logic (:78-125) is restated with plain torch ops and needs only the pad token
    id, not a tokenizer object.  It is bit-identical to the reference on the committed golden batch
    (`tests/golden/collator_golden.npz`, produced by the reference's own class).
"""
from __future__ import annotations

from typing import Any, Dict, List, Optional

import numpy as np


def pad_labels(label_lists: List[List[int]], pad_token_id: int):
    """`tokenizer.pad({"input_ids": ...}, padding="longest", return_tensors="pt")` (REF :78-84):
    right-pad with the pad token, attention_mask 1 on real tokens."""
    import torch

    T = max((len(x) for x in label_lists), default=0)
    ids = torch.full((len(label_lists), T), int(pad_token_id), dtype=torch.long)
    mask = torch.zeros((len(label_lists), T), dtype=torch.long)
    for b, x in enumerate(label_lists):
        n = len(x)
        if n:
            ids[b, :n] = torch.as_tensor(list(x), dtype=torch.long)
            mask[b, :n] = 1
    return ids, mask


def collate_labels(features: List[Dict[str, Any]], pad_token_id: int, decoder_start_token_id: int,
                   decoder_prev_token_id: Optional[int]) -> Dict[str, Any]:
    """REF/data_utils/data_collator.py:78-125 -- shift, -100 on padding and on the prompt before
    `<|startoftranscript|>`, bias spans padded with the literal 50256."""
    import torch

    ids, mask = pad_labels([f["labels"] for f in features], pad_token_id)
    decoder_input_ids = ids[:, :-1]                                    # :90
    labels = ids[:, 1:]                                                # :91
    labels_mask = mask[:, 1:]                                          # :94
    labels = labels.masked_fill(labels_mask.ne(1), -100)               # :96
    if decoder_prev_token_id is not None:                              # :98-102
        bos_index = torch.argmax((labels == decoder_start_token_id).long(), dim=1)
        prompt_mask = torch.arange(labels.shape[1]) < bos_index[:, None]
        labels = torch.where(prompt_mask, -100, labels)
    out: Dict[str, Any] = {"labels": labels, "decoder_input_ids": decoder_input_ids}
    if features and "bias_spans" in features[0]:                       # :107-125
        raw_spans = [f["bias_spans"] for f in features]
        max_span_len = max((len(span) for sample in raw_spans for span in sample), default=0)
        max_n_spans = max((len(sample) for sample in raw_spans), default=0)
        if max_span_len == 0 or max_n_spans == 0:
            out["bias_spans"] = torch.zeros((len(raw_spans), 1, 1), dtype=torch.long)
        else:
            padded = [[list(span) + [50256] * (max_span_len - len(span)) for span in sample]
                      + [[50256] * max_span_len] * (max_n_spans - len(sample)) for sample in raw_spans]
            out["bias_spans"] = torch.tensor(padded, dtype=torch.long)
    return out


class PendingFeatures:
    """One batch of PCM, collated in a DataLoader worker, whose features `collator.finish` computes in the main process.

    pcm       1-D float32 or int16 tensor (as the clips came): every clip trimmed to 480000 samples and starting on a
              16-byte boundary (`feature_extraction.pack_pcm`, the layout the extractor's host packing builds)
    offsets   int64 [B] clip starts in `pcm` (elements)
    lengths   int32 [B] samples of each clip

    It is picklable (a worker sends it to the main process), `pin_memory()` and `to(device)` return copies, so the
    DataLoader's pin thread and a trainer's device placement can handle it like a tensor.  `shape` and `numel()` are those
    of the features it stands for, which is what a trainer reads to count FLOPs.
    """

    def __init__(self, pcm, offsets, lengths, feature_size: int):
        self.pcm, self.offsets, self.lengths = pcm, offsets, lengths
        self.feature_size = int(feature_size)

    def pin_memory(self):
        return PendingFeatures(self.pcm.pin_memory(), self.offsets.pin_memory(), self.lengths.pin_memory(),
                               self.feature_size)

    def to(self, device, non_blocking=False):
        return PendingFeatures(*(t.to(device, non_blocking=non_blocking) for t in (self.pcm, self.offsets, self.lengths)),
                               self.feature_size)

    @property
    def shape(self):
        from .feature_extraction import NB_MAX_FRAMES

        return (len(self), self.feature_size, NB_MAX_FRAMES)

    def numel(self) -> int:
        return int(np.prod(self.shape))

    def __len__(self):
        return int(self.offsets.shape[0])

    def __repr__(self):
        return f"PendingFeatures(B={len(self)}, pcm={self.pcm.dtype}, device={self.pcm.device})"


class B200DataCollatorSpeechSeq2SeqWithPadding:
    """Drop-in for the reference collator with the feature extraction moved onto the B200.

    Args mirror the reference dataclass (`processor`, `decoder_start_token_id`,
    `decoder_prev_token_id`); `processor.feature_extractor` must be a `B200WhisperFeatureExtractor`
    and `processor.tokenizer.pad_token_id` supplies the pad id (or pass `pad_token_id=`).

    defer:  whether a batch of PCM items is featurised later, by `finish` in the main process.  None (default): inside
            a DataLoader worker (`torch.utils.data.get_worker_info() is not None`), where CUDA cannot be used; True /
            False force the choice.  A deferred call touches neither CUDA nor the extractor: the batch carries a
            `PendingFeatures` under the features' key, and labels stay on the CPU until `finish`.
    """

    def __init__(self, processor: Any = None, decoder_start_token_id: int = None, decoder_prev_token_id: Optional[int] = None,
                 feature_extractor: Any = None, pad_token_id: Optional[int] = None, labels_on_device: bool = False,
                 defer: Optional[bool] = None):
        self.processor = processor
        self.feature_extractor = feature_extractor if feature_extractor is not None else processor.feature_extractor
        if pad_token_id is None:
            pad_token_id = processor.tokenizer.pad_token_id
        if decoder_start_token_id is None:
            raise ValueError("decoder_start_token_id is required")
        self.pad_token_id = int(pad_token_id)
        self.decoder_start_token_id = int(decoder_start_token_id)
        self.decoder_prev_token_id = decoder_prev_token_id
        self.labels_on_device = labels_on_device
        self.defer = defer

    def __getstate__(self):
        # a spawned worker needs the extractor (it pickles detached) and the token ids, not the processor
        return {**self.__dict__, "processor": None}

    def __call__(self, features: List[Dict[str, Any]]):
        import torch

        from .feature_extraction import N_SAMPLES, B200WhisperFeatureExtractor, LogMelBatch, pack_pcm

        fe = self.feature_extractor
        name = fe.model_input_names[0]
        defer = self.defer if self.defer is not None else torch.utils.data.get_worker_info() is not None
        if features and "audio" in features[0]:
            clips = [np.ascontiguousarray(np.asarray(f["audio"]).reshape(-1)) for f in features]
            if clips[0].dtype not in (np.float32, np.int16):
                clips = [c.astype(np.float32) for c in clips]
            if defer:
                dt, _, ptr_arr, lens_arr, keep = B200WhisperFeatureExtractor._host_batch(clips)
                pcm, offsets, lengths = pack_pcm(dt, ptr_arr, lens_arr, N_SAMPLES)
                del keep
                batch = LogMelBatch({name: PendingFeatures(pcm, offsets, lengths, fe.feature_size)})
            else:
                feats = fe.extract_host(clips)                   # one batched call; stays in HBM
                batch = LogMelBatch({name: feats})
        else:
            batch = fe.pad({name: [f[name] for f in features]}, padding="longest", return_tensors="pt")
        lab = collate_labels(features, self.pad_token_id, self.decoder_start_token_id, self.decoder_prev_token_id)
        if self.labels_on_device and not defer:
            lab = {k: v.to(fe.device, non_blocking=True) for k, v in lab.items()}
        for k, v in lab.items():
            batch[k] = v
        return batch

    def finish(self, batch):
        """Main-process half of a deferred batch: every `PendingFeatures` in `batch` is replaced, in place, by its features
        in HBM -- one ragged launch of the extractor (`extract_device(pcm, offsets=, lengths=)`), the features the
        collator computes in-process, bit for bit; a dithering extractor draws its seed here, from this process's torch
        generator.  The pending tensors may be on the CPU, pinned, or on the device.  Then `labels_on_device` is applied.
        A batch with nothing pending is returned as it is."""
        fe = self.feature_extractor
        pending = [k for k, v in batch.items() if isinstance(v, PendingFeatures)]
        if not pending:
            return batch
        for k in pending:
            p = batch[k].to(fe.device, non_blocking=True)
            batch[k] = fe.extract_device(p.pcm, offsets=p.offsets, lengths=p.lengths)
        if self.labels_on_device:
            for k in ("labels", "decoder_input_ids", "bias_spans"):
                if k in batch:
                    batch[k] = batch[k].to(fe.device, non_blocking=True)
        return batch


class B200FeaturesTrainerMixin:
    """Featurises deferred batches in a `transformers.Trainer`'s main process:

        class Trainer(B200FeaturesTrainerMixin, Seq2SeqTrainer):
            pass

    with `data_collator=B200DataCollatorSpeechSeq2SeqWithPadding(...)`.  Training and prediction steps both prepare their
    inputs through `_prepare_inputs`; `Trainer._prepare_input` passes the `PendingFeatures` through untouched."""

    def _prepare_inputs(self, inputs):
        return self.data_collator.finish(super()._prepare_inputs(inputs))
