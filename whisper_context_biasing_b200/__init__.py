"""B200-native (sm_100a) log-mel front-end: a drop-in for the `WhisperFeatureExtractor` path of
thanh-nt25/Whisper-context-biasing.  Hand-written CUDA behind a C ABI (include/wlm.h, lib/libwlm.so);
Python is the host-side mirror of the reference's interface.  No CPU fallback."""
from .collator import (B200DataCollatorSpeechSeq2SeqWithPadding, B200FeaturesTrainerMixin, PendingFeatures,  # noqa: F401
                       collate_labels)
from .dataset import PcmPassthroughExtractor, bias_spans_of, pcm_dataset_class  # noqa: F401
from .feature_cache import FeatureCache  # noqa: F401
from .feature_extraction import B200WhisperFeatureExtractor, LogMelBatch, slaney_mel_filters  # noqa: F401
from .sharding import clip_shard  # noqa: F401

__all__ = ["B200WhisperFeatureExtractor", "B200DataCollatorSpeechSeq2SeqWithPadding", "B200FeaturesTrainerMixin",
           "FeatureCache", "LogMelBatch", "PcmPassthroughExtractor", "PendingFeatures", "bias_spans_of", "collate_labels",
           "clip_shard", "pcm_dataset_class", "slaney_mel_filters"]
