"""PCM-returning variant of the reference's `PromptWhisperDataset` (SURVEY.md section 8f rank 1, second half).

The reference computes the log-mel features INSIDE `Dataset.__getitem__`, one clip per call, in a forked DataLoader
worker (REF/data_utils/data_loader.py:170-172), and its driver scripts sweep the whole test set through that path just
to read `bias_spans` (REF/scripts/train.py:163, REF/scripts/evaluation.py:147).  A CUDA extractor cannot run in a forked
worker, and the sweep throws the features away.  This module keeps the reference's dataset class -- prompt strategies,
label assembly, random-prompt perturbation, everything in `__getitem__` stays the reference's own code -- and replaces
only what lines :170-172 produce:

  * `PcmPassthroughExtractor` stands where the feature extractor stood: called as the reference calls it
    (`feature_extractor(audio, sampling_rate=...).input_features`, :171) it hands the PCM back, so
    `torch.tensor(processed_audio[0])` (:172) becomes the clip itself;
  * `pcm_dataset_class(RefDataset)` subclasses the reference's class: items are
    `{"audio": float32 PCM, "labels": ..., "bias_spans": ...}`, ready for
    `B200DataCollatorSpeechSeq2SeqWithPadding`, which featurises the whole batch in one launch in the main process;
  * `bias_spans_only(i)` answers the train.py:163 / evaluation.py:147 sweeps without touching the audio
    (restates :163-168: tokenise each bias word, lower-cased, no special tokens, drop empties).

The reference class is passed in by the caller (it lives in the user's checkout of the reference and imports librosa /
av / editdistance at module level); nothing here imports it.
"""
from __future__ import annotations

from typing import Any, List

import numpy as np

from .feature_extraction import SAMPLING_RATE, LogMelBatch


class PcmPassthroughExtractor:
    """Duck-types the one call the reference's `__getitem__` makes on its feature extractor (data_loader.py:171) and
    returns the PCM instead of features.  Keeps the sampling-rate check of TF-FE:261-267."""

    model_input_names = ["input_features"]

    def __init__(self, sampling_rate: int = SAMPLING_RATE):
        self.sampling_rate = sampling_rate

    def __call__(self, raw_speech, sampling_rate=None, **kwargs):
        if sampling_rate is not None and sampling_rate != self.sampling_rate:
            raise ValueError(
                f"The model corresponding to this feature extractor: {self.__class__.__name__} was trained using a"
                f" sampling rate of {self.sampling_rate}. Please make sure that the provided `raw_speech` input"
                f" was sampled with {self.sampling_rate} and not {sampling_rate}.")
        pcm = np.ascontiguousarray(np.asarray(raw_speech, dtype=np.float32).reshape(-1))
        return LogMelBatch({"input_features": [pcm]})


def bias_spans_of(bias_words, tokenizer) -> List[List[int]]:
    """REF/data_utils/data_loader.py:163-168."""
    spans = []
    for word in bias_words:
        ids = tokenizer.encode(word.lower(), add_special_tokens=False)
        if ids:
            spans.append(ids)
    return spans


def pcm_dataset_class(ref_dataset_cls):
    """Returns a subclass of the reference's `PromptWhisperDataset` (same constructor, data_loader.py:59-60) whose items
    carry raw PCM under "audio" instead of features under "input_features"."""

    class PcmPromptWhisperDataset(ref_dataset_cls):
        def __init__(self, base_path, jsonl_data, phase, feature_extractor, tokenizer, *args, **kwargs):
            # the real (device) extractor is kept for the collator; the reference's __getitem__ gets the pass-through
            self.device_feature_extractor = feature_extractor
            sr = kwargs.get("sample_rate", args[3] if len(args) > 3 else SAMPLING_RATE)
            super().__init__(base_path, jsonl_data, phase, PcmPassthroughExtractor(sr), tokenizer, *args, **kwargs)

        def __getitem__(self, i) -> dict[str, Any]:
            item = super().__getitem__(i)                    # the reference's own code, prompt logic included
            pcm = item.pop("input_features")
            item["audio"] = pcm.numpy() if hasattr(pcm, "numpy") else np.asarray(pcm, dtype=np.float32)
            return item

        def bias_spans_only(self, i) -> List[List[int]]:
            """What `data_test[i]["bias_spans"]` yields (train.py:163, evaluation.py:147) without loading the audio."""
            return bias_spans_of(self.data[i][4], self.tokenizer)

        def all_bias_spans(self) -> List[List[List[int]]]:
            return [self.bias_spans_only(i) for i in range(len(self))]

        def __reduce__(self):
            # this class is made at run time, so pickle (a spawned DataLoader worker) cannot find it by name: rebuild it
            # from the reference class; `device_feature_extractor` pickles detached
            return _pcm_dataset_instance, (ref_dataset_cls,), self.__getstate__()

    PcmPromptWhisperDataset.__qualname__ = "PcmPromptWhisperDataset"
    return PcmPromptWhisperDataset


def _pcm_dataset_instance(ref_dataset_cls):
    cls = pcm_dataset_class(ref_dataset_cls)
    return cls.__new__(cls)
