"""B200 drop-in for the `WhisperFeatureExtractor` object the reference injects into its dataset
and collator (REF/data_utils/data_loader.py:59,75,171 ; REF/data_utils/data_collator.py:10,19-21,
64-76 ; REF/scripts/train.py:96,121,134,147).

Same call signature, attributes and error behaviour as
`transformers/models/whisper/feature_extraction_whisper.py` ("TF-FE", 5.5.0 line numbers):
`__call__` (TF-FE:189-342), `.pad` (feature_extraction_sequence_utils.py:51-219 as the collator
uses it), `.model_input_names` (TF-FE:67) and the ctor attributes (TF-FE:88-103).

Everything numeric runs in libwlm.so (hand-written sm_100a kernels, include/wlm.h).  PyTorch is
used for device memory and streams only.  There is no CPU fallback: without the library or a
B200 the constructor raises.
"""
from __future__ import annotations

import ctypes as C
import logging
import math
import os
import warnings
from typing import Sequence

import numpy as np

from . import _native as N

logger = logging.getLogger(__name__)

N_FFT = 400
HOP_LENGTH = 160
CHUNK_LENGTH = 30
SAMPLING_RATE = 16000
N_SAMPLES = CHUNK_LENGTH * SAMPLING_RATE
NB_MAX_FRAMES = N_SAMPLES // HOP_LENGTH


# --------------------------------------------------------------------------------------------
# host-side constants: the mel table, built exactly as the reference's constructor builds it
# (TF-FE:95-103 -> audio_utils.mel_filter_bank(201, M, 0, 8000, 16000, "slaney", "slaney"))
# --------------------------------------------------------------------------------------------
def _hz_to_mel(freq):
    freq = np.asarray(freq, dtype=np.float64)
    mels = 3.0 * freq / 200.0
    logstep = 27.0 / np.log(6.4)
    safe = np.maximum(freq, 1000.0)
    return np.where(freq >= 1000.0, 15.0 + np.log(safe / 1000.0) * logstep, mels)


def _mel_to_hz(mels):
    mels = np.asarray(mels, dtype=np.float64)
    freq = 200.0 * mels / 3.0
    logstep = np.log(6.4) / 27.0
    return np.where(mels >= 15.0, 1000.0 * np.exp(logstep * (mels - 15.0)), freq)


def slaney_mel_filters(n_mels: int, n_freq: int = 1 + N_FFT // 2, sampling_rate: int = SAMPLING_RATE,
                       fmin: float = 0.0, fmax: float = 8000.0) -> np.ndarray:
    """[n_freq, n_mels] float64, Slaney scale and area normalisation (audio_utils.py:453-544)."""
    edges = _mel_to_hz(np.linspace(_hz_to_mel(fmin), _hz_to_mel(fmax), n_mels + 2))
    bins = np.linspace(0, sampling_rate // 2, n_freq)
    width = np.diff(edges)
    slopes = edges[None, :] - bins[:, None]
    tri = np.maximum(0.0, np.minimum(-slopes[:, :-2] / width[:-1], slopes[:, 2:] / width[1:]))
    return tri * (2.0 / (edges[2:n_mels + 2] - edges[:n_mels]))[None, :]


def padded_length(lengths, pad_to_multiple_of=None) -> int:
    """Common length L of a `padding="longest", truncation=False` batch, as `SequenceFeatureExtractor.pad` computes
    it (TF-SU:51-219, `_pad`): the longest clip, rounded up to a multiple of `pad_to_multiple_of` when given.
    `max_length` plays no part.  The features then have L // 160 frames."""
    L = max((int(n) for n in lengths), default=0)
    if pad_to_multiple_of is not None and L % pad_to_multiple_of != 0:
        L = (L // pad_to_multiple_of + 1) * pad_to_multiple_of
    return L


def pack_pcm(dt, ptr_arr, lens_arr, max_len=None, pin_memory=False):
    """Host clips (float32 or int16; `ptr_arr` their addresses, `lens_arr` their lengths) -> one 1-D host tensor holding
    every clip, trimmed to `max_len` samples and starting on a 16-byte boundary, plus the int64 offsets and int32 lengths
    of that ragged batch (CPU tensors).  The gaps between clips are not initialised; nothing reads them."""
    import torch

    fmt = _pcm_format(dt)
    esz = np.dtype(dt).itemsize
    gran = 16 // esz
    lens = lens_arr.astype(np.int64)
    if max_len is not None:
        lens = np.minimum(lens, max_len)
    starts = (lens + gran - 1) // gran * gran
    offs = np.concatenate([[0], np.cumsum(starts)[:-1]]).astype(np.int64)
    host = torch.empty(int(starts.sum()) + gran, dtype=torch.float32 if fmt == N.WLM_PCM_F32 else torch.int16,
                       pin_memory=pin_memory)
    base = host.data_ptr()
    for o, n, p in zip(offs.tolist(), lens.tolist(), ptr_arr.tolist()):
        if n:
            C.memmove(base + o * esz, p, n * esz)
    return host, torch.from_numpy(offs), torch.from_numpy(lens.astype(np.int32))


def _pcm_format(dtype) -> int:
    """WLM_PCM_* of a numpy or torch PCM dtype: float32, or int16 (scaled by 1/32768 on the GPU)."""
    import torch

    fmt = {np.dtype(np.float32): N.WLM_PCM_F32, torch.float32: N.WLM_PCM_F32,
           np.dtype(np.int16): N.WLM_PCM_I16, torch.int16: N.WLM_PCM_I16}.get(dtype)
    if fmt is None:
        raise ValueError(f"PCM dtype {dtype} not supported (float32 or int16)")
    return fmt


def _feature_format(dtype):
    """(WLM_OUT_*, numpy dtype of a host copy) of a feature dtype; bfloat16 features are copied as uint16 bit patterns."""
    import torch

    fmt = {torch.float32: (N.WLM_OUT_F32, np.float32), torch.bfloat16: (N.WLM_OUT_BF16, np.uint16),
           torch.float16: (N.WLM_OUT_F16, np.float16)}.get(dtype)
    if fmt is None:
        raise ValueError(f"feature_dtype {dtype} not supported (float32, bfloat16, float16)")
    return fmt


class LogMelBatch(dict):
    """dict with attribute access, like `BatchFeature.__getattr__`
    (feature_extraction_utils.py:95-99): `out.input_features`, `out["input_features"]`, item
    assignment (the collator adds labels etc., data_collator.py:104-125), `.to(device)`."""

    def __getattr__(self, item):
        try:
            return self[item]
        except KeyError:
            raise AttributeError(item) from None

    def to(self, *args, **kwargs):
        import torch

        return LogMelBatch({k: (v.to(*args, **kwargs) if isinstance(v, torch.Tensor) else v)
                            for k, v in self.items()})


class B200WhisperFeatureExtractor:
    """Drop-in for `WhisperFeatureExtractor`; features are computed on a B200 by libwlm.so.

    Extra ctor arguments (not in the reference class):
      device:  CUDA device (int, "cuda", "cuda:N" or torch.device); default current device.
      output:  what `return_tensors=None` yields -- "device" (default): a CUDA `torch.Tensor`
               that stays in HBM for the model (`Trainer._prepare_input(...).to(device)` is then
               a no-op); "numpy": a host `np.ndarray` exactly like the reference returns.
      feature_dtype:  torch.float32 (default, the reference's dtype), torch.bfloat16 or
               torch.float16: element type the kernel STORES (round-to-nearest of the float32
               value; the reference model runs under fp16 autocast, REF/scripts/train.py:250).

    `dither` != 0 adds dither * z to the padded waveform of every featurising call (`__call__`,
    `extract_host`, `extract_device`), as the reference adds dither * torch.randn; z is the
    Philox stream of include/wlm.h, seeded per call from torch's default CPU generator, so
    `torch.manual_seed` makes a run reproducible.

    Deviations from the reference class, on purpose: non-default geometry / padding arguments
    raise NotImplementedError; the object is bound to one CUDA device and (like every stateful
    CUDA plan) is meant to be driven from one host thread and one stream at a time.  It is also
    bound to the process that created it: in a forked child, or as an unpickled copy (a spawned
    DataLoader worker's), its attributes work but featurising raises RuntimeError.
    """

    model_input_names = ["input_features"]          # TF-FE:67

    def __init__(self, feature_size=80, sampling_rate=16000, hop_length=160, chunk_length=30, n_fft=400,
                 padding_value=0.0, dither=0.0, return_attention_mask=False, device=None,
                 output="device", feature_dtype=None, **kwargs):
        import torch

        if (sampling_rate, hop_length, chunk_length, n_fft) != (SAMPLING_RATE, HOP_LENGTH, CHUNK_LENGTH, N_FFT):
            raise NotImplementedError(
                "the sm_100a kernels are specialised for sampling_rate=16000, hop_length=160, "
                "chunk_length=30, n_fft=400 (every Whisper checkpoint); got "
                f"{(sampling_rate, hop_length, chunk_length, n_fft)}")
        if padding_value != 0.0:
            raise NotImplementedError("padding_value != 0.0 is not supported")
        if not math.isfinite(float(dither)):
            raise ValueError(f"dither={dither!r} must be a finite number")
        if output not in ("device", "numpy"):
            raise ValueError("output must be 'device' or 'numpy'")
        if not torch.cuda.is_available():
            raise RuntimeError("B200WhisperFeatureExtractor needs a CUDA device; there is no CPU fallback")
        self.feature_size = int(feature_size)
        self.sampling_rate = sampling_rate
        self.hop_length = hop_length
        self.chunk_length = chunk_length
        self.n_fft = n_fft
        self.padding_value = padding_value
        self.dither = dither
        self.return_attention_mask = return_attention_mask
        self.padding_side = "right"
        self.n_samples = chunk_length * sampling_rate
        self.nb_max_frames = self.n_samples // hop_length
        self.mel_filters = slaney_mel_filters(self.feature_size)       # float64 [201, M]
        self.output = output

        if device is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        else:
            dev = torch.device(device) if not isinstance(device, int) else torch.device("cuda", device)
            if dev.type != "cuda":
                raise RuntimeError(f"device={device!r}: only CUDA devices are supported (no CPU fallback)")
            if dev.index is None:
                dev = torch.device("cuda", torch.cuda.current_device())
        self.device = dev
        with torch.cuda.device(dev):
            torch.cuda.current_stream()         # make sure the primary context exists
        table = np.ascontiguousarray(self.mel_filters.astype(np.float32))
        handle = C.c_void_p()
        N.check(N.LIB.wlm_plan_create(dev.index, self.feature_size, table.ctypes.data, C.byref(handle)))
        self._plan = handle
        self._owner_pid = os.getpid()
        self._ws = None
        self.feature_dtype = torch.float32
        if feature_dtype is not None:
            self.set_feature_dtype(feature_dtype)

    # -- lifecycle ---------------------------------------------------------------------------
    def close(self):
        plan, self._plan = getattr(self, "_plan", None), None
        if plan and getattr(self, "_owner_pid", None) == os.getpid():     # a forked copy never frees the parent's plan
            N.LIB.wlm_plan_destroy(plan)

    def __getstate__(self):
        """The configuration and attributes, without the CUDA plan and workspace: these belong to the creating process."""
        return {k: v for k, v in self.__dict__.items() if k not in ("_plan", "_owner_pid", "_ws")}

    def __setstate__(self, state):
        """An unpickled extractor is detached: its attributes work, featurising raises RuntimeError (see `_check_owner`).
        This is what a spawned DataLoader worker receives with the collator or the PCM dataset."""
        self.__dict__.update(state)
        self._plan, self._owner_pid, self._ws = None, None, None

    def _check_owner(self):
        """Featurising needs the plan's CUDA state, which only the process that created the plan has."""
        if self._owner_pid == os.getpid():
            return
        where = ("this is an unpickled copy, which has no CUDA plan" if self._owner_pid is None else
                 f"this process (pid {os.getpid()}) is not the one that created its CUDA plan (pid {self._owner_pid}), "
                 "e.g. a forked DataLoader worker")
        raise RuntimeError(
            f"B200WhisperFeatureExtractor cannot featurise here: {where}. Compute features in the main process: "
            "collate PCM with B200DataCollatorSpeechSeq2SeqWithPadding (it defers inside DataLoader workers) and call "
            "collator.finish(batch), or B200FeaturesTrainerMixin, in the main process; or use dataloader_num_workers=0.")

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launch_count(self) -> int:
        return int(N.LIB.wlm_plan_launch_count(self._plan))

    @property
    def kernel_variant(self) -> int:
        """80 / 128: unrolled mel stage for that Whisper bank; 0: table-driven mel stage."""
        return int(N.LIB.wlm_plan_kernel_variant(self._plan))

    @property
    def max_clusters(self) -> int:
        return int(N.LIB.wlm_plan_max_clusters(self._plan))

    @property
    def sm_count(self) -> int:
        """SMs of the device; `sm_count - 6 * max_clusters` of them run the cluster-less twin of the kernel."""
        return int(N.LIB.wlm_plan_sm_count(self._plan))

    def set_feature_dtype(self, dtype):
        """Element type of the features the kernel stores: float32, bfloat16 or float16."""
        N.check(N.LIB.wlm_plan_set_output_format(self._plan, _feature_format(dtype)[0]))
        self.feature_dtype = dtype

    def set_flat_clips(self, n: int = -1):
        """Measurement knob: clips of a dense batch handed to the cluster-less twin of the kernel (-1 = the library's split)."""
        N.check(N.LIB.wlm_plan_set_flat_clips(self._plan, int(n)))

    # -- helpers -----------------------------------------------------------------------------
    def _check_out(self, out, B, n_frames=None):
        n_frames = self.nb_max_frames if n_frames is None else n_frames
        if (tuple(out.shape) != (B, self.feature_size, n_frames) or out.dtype != self.feature_dtype
                or not out.is_cuda or out.device != self.device or not out.is_contiguous()):
            raise ValueError(f"out must be a contiguous {self.feature_dtype} tensor [B={B}, {self.feature_size}, "
                             f"{n_frames}] on {self.device}")

    def _stream(self):
        import torch

        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _workspace(self, B, padded_len=None):
        """Workspace of a wlm_logmel call (padded_len None) or of a wlm_logmel_conditioned call."""
        import torch

        if padded_len is None:
            need = int(N.LIB.wlm_workspace_bytes(self._plan, B))
        else:
            need = int(N.LIB.wlm_conditioned_workspace_bytes(self._plan, B, padded_len))
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(max(need, 256), dtype=torch.uint8, device=self.device)
        return self._ws, need

    # -- device-resident entry points (new; the reference has no device path) -------------------
    def _conditioning(self, dither, seed):
        """(dither, seed) of one featurising call: None -> the constructor's dither and a seed drawn from torch's default
        CPU generator (drawn only when the call dithers)."""
        import torch

        dither = self.dither if dither is None else dither
        dither = float(dither)
        if not math.isfinite(dither):
            raise ValueError(f"dither={dither!r} must be a finite number")
        if dither == 0.0:
            return 0.0, 0
        if seed is None:
            seed = int(torch.randint(-2 ** 63, 2 ** 63 - 1, (1,), dtype=torch.int64).item())
        return dither, int(seed) % 2 ** 64

    def extract_device(self, pcm, lengths=None, offsets=None, out=None, return_gmax=False, padded_len=None,
                       do_normalize=False, dither=None, seed=None):
        """PCM already in HBM -> features in HBM.

        pcm      CUDA tensor, float32 or int16 (int16 is scaled by 1/32768 on the GPU).
                 dense: [B, L] (row stride L, L % 4 == 0); ragged: 1-D with `offsets`/`lengths`.
        lengths  optional int32 CUDA tensor [B] of valid samples (required when ragged).
        offsets  optional int64 CUDA tensor [B] of clip starts (elements) in the 1-D buffer.
        padded_len  None: every clip is padded / trimmed to 30 s, features [B, M, 3000].  An int L > 200: every
                 clip is zero-padded to L samples (long-form, `truncation=False`), features [B, M, L // 160].
        do_normalize  HF's `do_normalize=True`: each clip's valid samples are scaled to zero mean, unit variance.
        dither   noise amplitude added to the padded waveform (None: the constructor's `dither`).
        seed     64-bit seed of the noise (None: drawn from torch's default CPU generator when the call dithers).
        """
        import torch

        self._check_owner()
        if not (isinstance(pcm, torch.Tensor) and pcm.is_cuda):
            raise ValueError("extract_device expects a CUDA tensor")
        if pcm.device != self.device:
            raise ValueError(f"pcm is on {pcm.device}, the extractor on {self.device}")
        fmt = _pcm_format(pcm.dtype)
        if not pcm.is_contiguous() or pcm.data_ptr() % 16:
            pcm = pcm.contiguous() if pcm.data_ptr() % 16 == 0 else pcm.clone(memory_format=torch.contiguous_format)
        if offsets is None:
            if pcm.dim() == 1:
                pcm = pcm[None]
            if pcm.dim() != 2:
                raise ValueError(f"Only mono-channel audio is supported for input to {self}")
            B, stride = pcm.shape
        else:
            if pcm.dim() != 1 or lengths is None:
                raise ValueError("ragged input needs a 1-D pcm buffer plus offsets and lengths")
            B, stride = offsets.shape[0], 0
            if offsets.dtype != torch.int64 or not offsets.is_cuda:
                raise ValueError("offsets must be a CUDA int64 tensor")
        if lengths is not None and (lengths.dtype != torch.int32 or not lengths.is_cuda or lengths.shape[0] != B):
            raise ValueError("lengths must be a CUDA int32 tensor of shape [B]")
        if padded_len is not None:
            padded_len = int(padded_len)
            self._check_padded_len(padded_len)
        L = self.n_samples if padded_len is None else padded_len
        dither, seed = self._conditioning(dither, seed)
        plain = padded_len is None and not do_normalize and dither == 0.0
        if out is None:
            out = torch.empty((B, self.feature_size, L // self.hop_length), dtype=self.feature_dtype, device=self.device)
        else:
            self._check_out(out, B, L // self.hop_length)
        gmax = torch.empty((max(B, 1),), dtype=torch.float32, device=self.device) if return_gmax else None
        ws, need = self._workspace(B, None if plain else L)
        if B:
            args = (C.c_void_p(pcm.data_ptr()), fmt,
                    C.c_void_p(offsets.data_ptr()) if offsets is not None else None,
                    C.c_void_p(lengths.data_ptr()) if lengths is not None else None, stride)
            tail = (C.c_void_p(out.data_ptr()), C.c_void_p(gmax.data_ptr()) if gmax is not None else None,
                    C.c_void_p(ws.data_ptr()), need, self._stream())
            with torch.cuda.device(self.device):
                if plain:
                    N.check(N.LIB.wlm_logmel(self._plan, *args, B, *tail))
                else:       # with nothing to condition: the launches of wlm_logmel_padded
                    N.check(N.LIB.wlm_logmel_conditioned(self._plan, *args, L, B, int(bool(do_normalize)), dither, seed,
                                                         *tail))
        return (out, gmax[:B]) if return_gmax else out

    def frame_mask_device(self, lengths, padded_len=None):
        """int32 [B, 3000] attention mask on the device (TF-FE:328-337); with `padded_len` = L the long-form
        mask [B, L // 160]."""
        import torch

        self._check_owner()
        B = lengths.shape[0]
        L = self.n_samples if padded_len is None else int(padded_len)
        mask = torch.empty((B, max(L // self.hop_length, 0)), dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            N.check(N.LIB.wlm_frame_mask_padded(self._plan, C.c_void_p(lengths.data_ptr()), B, L,
                                                C.c_void_p(mask.data_ptr()), self._stream()))
        return mask

    def extract_host(self, clips, out=None, out_host=None, do_normalize=False, dither=None, seed=None):
        """Host PCM -> features in HBM through the plan's pinned H2D pipeline (wlm_logmel_host).

        clips   a list of 1-D float32 / int16 numpy arrays of any lengths (what a dataset yields), or -- without any
                per-clip Python work -- a C-contiguous 2-D array [B, L] (dense batch), or a tuple
                (buffer, offsets, lengths): one 1-D array holding every clip, int64 element offsets and lengths.
        do_normalize, dither, seed  as `extract_device`.  A conditioned call packs the clips into one pinned buffer
                and runs `extract_device` on it (wlm_logmel_host has no conditioning)."""
        import torch

        self._check_owner()
        dither, seed = self._conditioning(dither, seed)
        dt, B, ptr_arr, lens_arr, keep = self._host_batch(clips)
        if B == 0:
            return torch.empty((0, self.feature_size, self.nb_max_frames), dtype=self.feature_dtype, device=self.device)
        fmt = _pcm_format(dt)
        if out is None:
            out = torch.empty((B, self.feature_size, self.nb_max_frames), dtype=self.feature_dtype, device=self.device)
        else:
            self._check_out(out, B)
        if out_host is not None:
            want = _feature_format(self.feature_dtype)[1]
            if (not isinstance(out_host, np.ndarray) or out_host.dtype != want or not out_host.flags["C_CONTIGUOUS"]
                    or out_host.shape != (B, self.feature_size, self.nb_max_frames)):
                raise ValueError(f"out_host must be a C-contiguous {np.dtype(want)} ndarray [B={B}, {self.feature_size}, "
                                 f"{self.nb_max_frames}] (bfloat16 features: uint16 bit patterns)")
        if do_normalize or dither != 0.0:
            pcm, lens_dev, offs_dev = self._pack_host(dt, ptr_arr, lens_arr, self.n_samples)
            del keep, ptr_arr, lens_arr
            self.extract_device(pcm, lengths=lens_dev, offsets=offs_dev, out=out, do_normalize=do_normalize, dither=dither,
                                seed=seed)
            if out_host is not None:
                bits = out.view(torch.int16) if self.feature_dtype == torch.bfloat16 else out
                out_host[...] = bits.cpu().numpy().view(want)
            return out
        ptrs = ptr_arr.ctypes.data_as(C.POINTER(C.c_void_p))
        lens = lens_arr.ctypes.data_as(C.POINTER(C.c_int32))
        with torch.cuda.device(self.device):
            N.check(N.LIB.wlm_logmel_host(
                self._plan, ptrs, lens, fmt, B, C.c_void_p(out.data_ptr()),
                C.c_void_p(out_host.ctypes.data) if out_host is not None else None, self._stream()))
        del keep, ptr_arr, lens_arr
        return out

    @staticmethod
    def _host_batch(clips):
        """The host input forms of `extract_host` -> (dtype, B, uintp clip pointers, int32 lengths, what must stay alive
        while the pointers are used).  dtype and the arrays are None for an empty list."""
        keep = clips
        if isinstance(clips, tuple) and len(clips) == 3 and isinstance(clips[0], np.ndarray):
            buf, offs, lens_np = clips
            if buf.ndim != 1 or not buf.flags["C_CONTIGUOUS"]:
                raise ValueError("ragged host input: the buffer must be a C-contiguous 1-D array")
            dt, B = buf.dtype, int(len(offs))
            offs = np.asarray(offs, dtype=np.int64)
            lens_arr = np.ascontiguousarray(lens_np, dtype=np.int32)
            if B and (offs.min() < 0 or int((offs + lens_arr).max()) > buf.shape[0] or lens_arr.min() < 0):
                raise ValueError("ragged host input: a clip lies outside the buffer")
            ptr_arr = (buf.ctypes.data + offs * buf.itemsize).astype(np.uintp)
        elif isinstance(clips, np.ndarray) and clips.ndim == 2:
            if not clips.flags["C_CONTIGUOUS"]:
                clips = keep = np.ascontiguousarray(clips)
            dt, B = clips.dtype, clips.shape[0]
            ptr_arr = (clips.ctypes.data + np.arange(B, dtype=np.int64) * clips.strides[0]).astype(np.uintp)
            lens_arr = np.full((B,), clips.shape[1], dtype=np.int32)
        else:
            B = len(clips)
            if B == 0:
                return None, 0, None, None, keep
            dt = clips[0].dtype
            if any(x.dtype != dt or x.ndim != 1 for x in clips):
                raise ValueError("all clips must be 1-D arrays of the same dtype")
            if not all(x.flags.c_contiguous for x in clips):
                clips = keep = [np.ascontiguousarray(x) for x in clips]
            ptr_arr = np.fromiter((x.__array_interface__["data"][0] for x in clips), dtype=np.uintp, count=B)
            lens_arr = np.fromiter((x.shape[0] for x in clips), dtype=np.int32, count=B)
        return dt, B, ptr_arr, lens_arr, keep

    def _pack_host(self, dt, ptr_arr, lens_arr, max_len=None):
        """Host clips (`_host_batch`'s pointers and lengths, float32 or int16) -> one pinned buffer on the device, each
        clip trimmed to `max_len` samples and starting on a 16-byte boundary, copied over in one transfer.  Returns the
        device buffer and the int32 lengths and int64 offsets of the ragged batch, on the device."""
        host, offs, lens = pack_pcm(dt, ptr_arr, lens_arr, max_len, pin_memory=True)
        pcm = host.to(self.device, non_blocking=True)     # (the caching host allocator keeps `host` until the copy is done)
        return pcm, lens.to(self.device), offs.to(self.device)

    # -- the reference-facing call (TF-FE:189-342) ---------------------------------------------
    def __call__(self, raw_speech, truncation=True, pad_to_multiple_of=None, return_tensors=None,
                 return_attention_mask=None, padding="max_length", max_length=None, sampling_rate=None,
                 do_normalize=None, device=None, **kwargs):
        import torch

        self._check_owner()
        if sampling_rate is not None:
            if sampling_rate != self.sampling_rate:                         # TF-FE:261-267
                raise ValueError(
                    f"The model corresponding to this feature extractor: {self.__class__.__name__} was trained using a"
                    f" sampling rate of {self.sampling_rate}. Please make sure that the provided `raw_speech` input"
                    f" was sampled with {self.sampling_rate} and not {sampling_rate}.")
        else:                                                               # TF-FE:268-272
            logger.warning(
                f"It is strongly recommended to pass the `sampling_rate` argument to `{self.__class__.__name__}()`. "
                "Failing to do so can result in silent errors that might be hard to debug.")
        longform = padding == "longest" and truncation is False      # max_length is ignored, as TF-SU:51-219 does
        if not longform and (padding != "max_length" or (max_length not in (None, self.n_samples)) or not truncation
                             or pad_to_multiple_of is not None):
            raise NotImplementedError(
                "implemented argument combinations: padding='max_length', max_length=None (30 s), truncation=True, "
                "pad_to_multiple_of=None (the reference's), and padding='longest', truncation=False (long-form)")
        if device not in (None, "cpu") and torch.device(device).type != "cuda":
            raise NotImplementedError(f"device={device!r}: features are always computed on {self.device}")

        do_normalize = bool(do_normalize)
        x = self._speech(raw_speech)
        if isinstance(x, torch.Tensor):
            lengths = np.full((x.shape[0],), x.shape[1], dtype=np.int64)
        else:
            lengths = np.array([c.shape[0] for c in x], dtype=np.int64)
        if longform:                                            # every clip is zero-padded to L samples
            L = padded_length(lengths, pad_to_multiple_of)
            self._check_padded_len(L)
        else:                                                   # every clip is padded or trimmed to 30 s
            L = self.n_samples
        if isinstance(x, torch.Tensor):                         # CUDA rows go to the kernels as they are
            B, n = x.shape
            if n % 4:          # rows must start on 16-byte boundaries; the padding is zeros, as HF pads
                x = torch.nn.functional.pad(x, (0, 4 - n % 4))
            lens = None        # a plain call keeps the dense layout: the static cluster / flat split
            if do_normalize or self.dither != 0.0:
                # the row padding above is not part of the clip: the moments and the noise see n samples
                lens = torch.full((B,), n, dtype=torch.int32, device=self.device)
            feats = self.extract_device(x, lengths=lens, padded_len=L if longform else None, do_normalize=do_normalize)
        elif not longform:
            feats = self.extract_host(x, do_normalize=do_normalize)
        else:
            # one pinned buffer, clip starts 16-byte aligned, copied over in one transfer and run as a ragged batch
            dt, _, ptr_arr, lens_arr, keep = self._host_batch(x)
            pcm, lens_dev, offs_dev = self._pack_host(dt, ptr_arr, lens_arr)
            del keep
            feats = self.extract_device(pcm, lengths=lens_dev, offsets=offs_dev, padded_len=L, do_normalize=do_normalize)

        want = return_tensors
        if want is None:
            want = "pt" if self.output == "device" else "np"
        want = getattr(want, "value", want)
        out = LogMelBatch()
        if want == "np":
            out["input_features"] = (feats.float() if feats.dtype == torch.bfloat16 else feats).cpu().numpy()
        elif want == "pt":
            out["input_features"] = feats
        else:
            raise NotImplementedError(f"return_tensors={return_tensors!r} (use None, 'pt' or 'np')")
        if return_attention_mask or do_normalize or (return_attention_mask is None and self.return_attention_mask):
            lens_dev = torch.from_numpy(np.minimum(lengths, L).astype(np.int32)).to(self.device)
            if return_attention_mask:                                                          # TF-FE:328-337
                mask = self.frame_mask_device(lens_dev, padded_len=L)
            else:
                # The reference's quirk, kept: pad() is asked for the mask (do_normalize needs it; otherwise it falls
                # back to the ctor attribute, TF-SU:135-137) and returns the SAMPLE-level mask [B, L], which TF-FE:328
                # then does not rescale because the call argument is not True.
                mask = (torch.arange(L, device=self.device, dtype=torch.int32)[None, :] < lens_dev[:, None]).to(torch.int32)
            out["attention_mask"] = mask.cpu().numpy() if want == "np" else mask
        return out

    def _speech(self, raw_speech):
        """The input forms of `__call__` -> a CUDA float32 tensor [B, n], or a list of contiguous float32 1-D host clips
        (TF-FE:274-290)."""
        import torch

        if isinstance(raw_speech, torch.Tensor):
            if raw_speech.dim() > 2:
                raise ValueError(f"Only mono-channel audio is supported for input to {self}")
            x = raw_speech if raw_speech.dim() == 2 else raw_speech[None]
            if x.dtype != torch.float32:
                x = x.to(torch.float32)
            return x if x.is_cuda else [np.ascontiguousarray(r.numpy()) for r in x]
        is_batched_numpy = isinstance(raw_speech, np.ndarray) and raw_speech.ndim > 1          # TF-FE:274
        if is_batched_numpy and raw_speech.ndim > 2:
            raise ValueError(f"Only mono-channel audio is supported for input to {self}")      # TF-FE:275-276
        is_batched = is_batched_numpy or (
            isinstance(raw_speech, (list, tuple)) and len(raw_speech) > 0
            and isinstance(raw_speech[0], (np.ndarray, tuple, list)))                           # TF-FE:277-279
        if is_batched:                                                                         # TF-FE:281-282
            return [np.ascontiguousarray(np.asarray(s, dtype=np.float32).reshape(-1)) for s in raw_speech]
        return [np.ascontiguousarray(np.asarray(raw_speech, dtype=np.float32).reshape(-1))]   # TF-FE:283-290

    @staticmethod
    def _check_padded_len(L):
        """A padded length the long-form kernels take: torch.stft's reflect padding needs more than n_fft // 2 samples,
        and the frame positions stay in 32 bits."""
        if L <= N_FFT // 2:
            raise ValueError(f"padded length {L}: the reflect padding of the STFT needs more than {N_FFT // 2} samples "
                             "(torch.stft refuses it too)")
        if L >= 2 ** 31:
            raise ValueError(f"padded length {L} does not fit 32 bits")

    # -- the collator's stack (REF/data_utils/data_collator.py:64-76) --------------------------
    def pad(self, processed_features, padding="longest", max_length=None, truncation=False,
            pad_to_multiple_of=None, return_attention_mask=None, return_tensors=None):
        import torch

        if isinstance(processed_features, (list, tuple)) and processed_features and isinstance(processed_features[0], dict):
            processed_features = {k: [f[k] for f in processed_features] for k in processed_features[0]}
        if self.model_input_names[0] not in processed_features:
            raise ValueError(
                "You should supply an instance of `transformers.BatchFeature` or list of `transformers.BatchFeature`"
                f" to this method that includes {self.model_input_names[0]}, but you provided"
                f" {list(processed_features.keys())}")
        items = processed_features[self.model_input_names[0]]
        if isinstance(items, (torch.Tensor, np.ndarray)) and items.ndim == 3:
            items = list(items)
        if len(items) == 0:
            return LogMelBatch({"input_features": items})
        shapes = {tuple(np.shape(i)) for i in items}
        if len(shapes) != 1:
            raise ValueError(f"all feature arrays must have the same shape to be stacked, got {sorted(shapes)}")
        want = getattr(return_tensors, "value", return_tensors)
        if all(isinstance(i, torch.Tensor) for i in items):
            stacked = torch.stack(list(items), dim=0)
            if want == "np":
                stacked = stacked.cpu().numpy()
        else:
            stacked = np.stack([i.cpu().numpy() if isinstance(i, torch.Tensor) else np.asarray(i, dtype=np.float32)
                                for i in items], axis=0)
            if want == "pt":
                stacked = torch.from_numpy(stacked)
        return LogMelBatch({"input_features": stacked})

    def to_dict(self):
        return {"feature_extractor_type": "WhisperFeatureExtractor", "feature_size": self.feature_size,
                "sampling_rate": self.sampling_rate, "hop_length": self.hop_length,
                "chunk_length": self.chunk_length, "n_fft": self.n_fft, "padding_value": self.padding_value,
                "dither": self.dither, "return_attention_mask": self.return_attention_mask,
                "n_samples": self.n_samples, "nb_max_frames": self.nb_max_frames, "padding_side": "right"}

    def __repr__(self):
        return f"B200WhisperFeatureExtractor(feature_size={self.feature_size}, device={self.device})"
