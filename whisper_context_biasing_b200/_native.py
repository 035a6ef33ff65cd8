"""ctypes binding of include/wlm.h.  No torch types cross this boundary: raw pointers + sizes.

The library is mandatory: importing this module without `lib/libwlm.so` raises, and every
non-zero return code raises -- there is no CPU or PyTorch fallback anywhere in the package.
"""
from __future__ import annotations

import ctypes as C
import os

_LIB_PATH = os.environ.get("WLM_LIBRARY_PATH") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libwlm.so")

WLM_OK = 0
WLM_ERR_BAD_ARG = -1
WLM_ERR_UNSUPPORTED = -2
WLM_ERR_CUDA = -3
WLM_ERR_NO_DEVICE = -4
WLM_ERR_WORKSPACE = -5
WLM_PCM_F32 = 0
WLM_PCM_I16 = 1
WLM_OUT_F32 = 0
WLM_OUT_BF16 = 1
WLM_OUT_F16 = 2

# every symbol include/wlm.h declares: (restype, argtypes)
_vp, _i, _i64, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_size_t
SYMBOLS = {
    "wlm_version": (_i, []),
    "wlm_last_error": (C.c_char_p, []),
    "wlm_plan_create": (_i, [_i, _i, _vp, C.POINTER(_vp)]),
    "wlm_plan_destroy": (_i, [_vp]),
    "wlm_plan_n_mels": (_i, [_vp]),
    "wlm_plan_device": (_i, [_vp]),
    "wlm_plan_sm_count": (_i, [_vp]),
    "wlm_plan_kernel_variant": (_i, [_vp]),
    "wlm_plan_max_clusters": (_i, [_vp]),
    "wlm_workspace_bytes": (_sz, [_vp, _i]),
    "wlm_logmel": (_i, [_vp, _vp, _i, _vp, _vp, _i64, _i, _vp, _vp, _vp, _sz, _vp]),
    "wlm_frame_mask": (_i, [_vp, _vp, _i, _vp, _vp]),
    "wlm_logmel_host": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp]),
    "wlm_plan_launch_count": (_i64, [_vp]),
    "wlm_plan_set_output_format": (_i, [_vp, _i]),
    "wlm_plan_output_format": (_i, [_vp]),
    "wlm_plan_set_flat_clips": (_i, [_vp, _i]),
    "wlm_padded_workspace_bytes": (_sz, [_vp, _i]),
    "wlm_logmel_padded": (_i, [_vp, _vp, _i, _vp, _vp, _i64, _i64, _i, _vp, _vp, _vp, _sz, _vp]),
    "wlm_frame_mask_padded": (_i, [_vp, _vp, _i, _i64, _vp, _vp]),
    "wlm_conditioned_workspace_bytes": (_sz, [_vp, _i, _i64]),
    "wlm_logmel_conditioned": (_i, [_vp, _vp, _i, _vp, _vp, _i64, _i64, _i, _i, C.c_float, C.c_uint64, _vp, _vp, _vp, _sz,
                                    _vp]),
}


class WlmError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libwlm error {code}: {msg}")
        self.code = code


def lib_path() -> str:
    return _LIB_PATH


def _load():
    if not os.path.exists(_LIB_PATH):
        raise ImportError(
            f"{_LIB_PATH} is missing. Build it with `python -m whisper_context_biasing_b200.build` "
            "(needs nvcc); this package has no CPU fallback.")
    lib = C.CDLL(_LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args
    return lib


LIB = _load()


def last_error() -> str:
    return (LIB.wlm_last_error() or b"").decode(errors="replace")


def check(rc: int) -> None:
    if rc != WLM_OK:
        msg = last_error()
        if rc in (WLM_ERR_BAD_ARG, WLM_ERR_UNSUPPORTED):
            raise ValueError(f"libwlm: {msg}")
        raise WlmError(rc, msg)
