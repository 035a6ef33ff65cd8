"""In-HBM cache of log-mel features, keyed by clip (SURVEY 8f rank 3).

The reference recomputes the features of a clip every time its dataset row is touched: once per
epoch in training, and for a full sweep of the test set just to read `bias_spans`
(REF/scripts/train.py:163, REF/scripts/evaluation.py:147 iterate the whole dataset, and
`PromptWhisperDataset.__getitem__` decodes and featurises on every access,
REF/data_utils/data_loader.py:170-172).  The features of a clip never change, and at 0.96 MB
(80 mels, float32) a B200's 180 GB of HBM holds the whole medical test set (5k clips: 4.9 GB)
many times over -- so keep them where the model reads them.

    cache = FeatureCache(extractor, capacity_bytes=16 << 30)
    feats = cache.get_many(keys, load_pcm)        # [B, n_mels, 3000] on the device

`load_pcm(key)` is only called for the misses (so the decode/resample cost disappears with the
feature cost), all misses of a call are featurised in ONE batched extractor call, and hits are a
device-side gather.  Storage is a slab `[slots, n_mels, 3000]` allocated once; eviction is LRU.
`dtype=torch.float16` halves the footprint; float32 (default) keeps the features bit-identical.

`extractor` is anything with `.feature_size`, `.device` and `.extract_host(list_of_pcm) ->
Tensor[B, n_mels, 3000]` on that device (`B200WhisperFeatureExtractor`); the cache itself contains
no arithmetic.
"""
from __future__ import annotations

from collections import OrderedDict
from typing import Callable, Hashable, Iterable, List, Sequence

N_FRAMES = 3000


class FeatureCache:
    def __init__(self, extractor, capacity_bytes: int = 8 << 30, dtype=None):
        import torch

        if float(getattr(extractor, "dither", 0.0)) != 0.0:
            raise ValueError("an extractor with dither != 0 draws new noise on every call; caching its features would "
                             "freeze one draw")
        self.extractor = extractor
        self.n_mels = int(extractor.feature_size)
        self.device = extractor.device
        self.dtype = dtype or torch.float32
        if self.dtype not in (torch.float32, torch.float16, torch.bfloat16):
            raise ValueError("dtype must be float32, float16 or bfloat16")
        item_bytes = self.n_mels * N_FRAMES * torch.empty((), dtype=self.dtype).element_size()
        self.slots = int(capacity_bytes // item_bytes)
        if self.slots < 1:
            raise ValueError(f"capacity_bytes={capacity_bytes} holds no clip ({item_bytes} bytes each)")
        self._slab = None                      # allocated on first use: [slots, n_mels, 3000]
        self._slot_of: "OrderedDict[Hashable, int]" = OrderedDict()      # LRU order: oldest first
        self._free: List[int] = list(range(self.slots - 1, -1, -1))
        self.hits = 0
        self.misses = 0
        self.evictions = 0

    # ---- bookkeeping (no device work) -------------------------------------------------------------
    def __len__(self):
        return len(self._slot_of)

    def __contains__(self, key):
        return key in self._slot_of

    @property
    def nbytes(self):
        import torch

        return len(self) * self.n_mels * N_FRAMES * torch.empty((), dtype=self.dtype).element_size()

    def _claim(self, key, pinned: set) -> int:
        """Slot for a new key: a free one, else the least recently used entry that this call does not need."""
        if self._free:
            slot = self._free.pop()
        else:
            victim = next((k for k in self._slot_of if k not in pinned), None)
            if victim is None:
                raise RuntimeError(f"a single call needs more distinct clips than the cache holds ({self.slots})")
            slot = self._slot_of.pop(victim)
            self.evictions += 1
        self._slot_of[key] = slot
        return slot

    def plan(self, keys: Sequence[Hashable]):
        """Resolve a batch of keys -> (slot per key, distinct missing keys in first-seen order, their slots).
        Pure bookkeeping; `get_many` is this plus the device work."""
        pinned = set(keys)
        slots: List[int] = []
        missing: List[Hashable] = []
        missing_slots: List[int] = []
        for k in keys:
            if k in self._slot_of:
                self._slot_of.move_to_end(k)
                if k in missing:               # second occurrence of a key that is being filled by this call
                    pass
                else:
                    self.hits += 1
                slots.append(self._slot_of[k])
            else:
                self.misses += 1
                s = self._claim(k, pinned)
                missing.append(k)
                missing_slots.append(s)
                slots.append(s)
        return slots, missing, missing_slots

    def drop(self, keys: Iterable[Hashable]):
        for k in keys:
            s = self._slot_of.pop(k, None)
            if s is not None:
                self._free.append(s)

    def clear(self):
        self.drop(list(self._slot_of))

    # ---- the call ------------------------------------------------------------------------------------
    def get_many(self, keys: Sequence[Hashable], load_pcm: Callable[[Hashable], "object"]):
        """Features of `keys` as one float32 tensor [len(keys), n_mels, 3000] on the extractor's device."""
        import torch

        if self._slab is None:
            self._slab = torch.empty((self.slots, self.n_mels, N_FRAMES), dtype=self.dtype, device=self.device)
        slots, missing, missing_slots = self.plan(keys)
        if missing:
            try:
                feats = self.extractor.extract_host([load_pcm(k) for k in missing])      # ONE batched launch
            except Exception:
                self.drop(missing)             # nothing was written: forget the claimed slots
                raise
            idx = torch.as_tensor(missing_slots, dtype=torch.long, device=self.device)
            self._slab.index_copy_(0, idx, feats.to(self.dtype))
        idx = torch.as_tensor(slots, dtype=torch.long, device=self.device)
        return self._slab.index_select(0, idx).to(torch.float32)

    def stats(self):
        return {"entries": len(self), "slots": self.slots, "bytes": self.nbytes, "hits": self.hits,
                "misses": self.misses, "evictions": self.evictions}
