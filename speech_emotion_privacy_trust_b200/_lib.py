"""ctypes binding of libsept_b200.so (include/sept.h).  There is no CPU fallback: a missing library is built with
nvcc if the toolchain is present, otherwise importing the compute layer fails loudly."""
from __future__ import annotations

import ctypes as C
from pathlib import Path

from . import build as _build

_LIB = None

c_f32p = C.c_void_p      # device / host pointers travel as integers (tensor.data_ptr())
c_ptr = C.c_void_p

_SIGNATURES = {
    "sept_version": (C.c_int, []),
    "sept_last_error": (C.c_char_p, []),
    "sept_source_hash": (C.c_char_p, []),
    "sept_init": (C.c_int, [C.c_int]),
    "sept_frames_per_item": (C.c_int, [C.c_int]),
    "sept_extract_layout": (C.c_int, [c_ptr, C.c_int, C.c_int, C.c_int, c_ptr, c_ptr]),
    "sept_logmel_f32": (C.c_int, [c_ptr, c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_ptr, c_ptr]),
    "sept_logmel_bwd_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int64]),
    "sept_logmel_bwd_f32": (C.c_int, [c_ptr, c_ptr, c_ptr, c_ptr, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int, c_ptr, c_ptr, c_ptr,
                                      c_ptr]),
    "sept_mfcc_f32": (C.c_int, [c_ptr, c_ptr, c_ptr, c_ptr, C.c_int, C.c_int64, c_ptr, c_ptr, c_ptr, c_ptr]),
    "sept_mfcc_bwd_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int64, C.c_int64]),
    "sept_mfcc_bwd_f32": (C.c_int, [c_ptr, c_ptr, c_ptr, c_ptr, C.c_int, C.c_int64, C.c_int64, c_ptr, c_ptr, c_ptr, c_ptr]),
    "sept_resample_layout": (C.c_int, [c_ptr, C.c_int, C.c_int, C.c_int, c_ptr]),
    "sept_resample_f32": (C.c_int, [c_ptr, c_ptr, c_ptr, C.c_int, C.c_int64, C.c_int, C.c_int, c_ptr, c_ptr]),
    "sept_pcm16_to_f32": (C.c_int, [c_ptr, C.c_int64, c_ptr, c_ptr]),
    "sept_speaker_stats_f32": (C.c_int, [c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, C.c_int, c_ptr, c_ptr, C.c_int, c_ptr, c_ptr, c_ptr]),
    "sept_normalize_f32": (C.c_int, [c_ptr, c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, c_ptr, c_ptr]),
    "sept_normalize_windows_f32": (C.c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, C.c_int, c_ptr, c_ptr]),
    "sept_counter_add_u64": (C.c_int, [c_ptr, C.c_uint64, c_ptr]),
    "sept_cloak_fwd_f32": (C.c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, C.c_uint64, C.c_uint64, c_ptr, C.c_int, C.c_float, C.c_float, C.c_float,
                                     C.c_int, C.c_int, c_ptr, c_ptr, c_ptr, c_ptr]),
    "sept_cloak_bwd_workspace_bytes": (C.c_size_t, [C.c_int]),
    "sept_cloak_grl_bwd_f32": (C.c_int, [c_ptr, c_ptr, C.c_float, c_ptr, c_ptr, c_ptr, C.c_float, C.c_float, C.c_int, C.c_int,
                                         c_ptr, c_ptr, c_ptr, c_ptr, c_ptr]),
    "sept_grl_bwd_f32": (C.c_int, [c_ptr, C.c_float, C.c_int64, c_ptr, c_ptr]),
    "sept_add_noise_rows_f32": (C.c_int, [c_ptr, c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, C.c_uint64, C.c_float, c_ptr, c_ptr]),
}

EXPORTS = tuple(_SIGNATURES)

SEPT_E_BADARG, SEPT_E_UNSUPPORTED, SEPT_E_TOO_SHORT, SEPT_E_CUDA = -1, -2, -3, -4


def library_path() -> Path:
    return _build.LIB


def lib() -> C.CDLL:
    """Load libsept_b200.so.  The library carries the sha256 of the sources it was compiled from; if it is absent or
    that hash differs from the sources in the tree (a stale prebuilt .so), it is rebuilt first (under a file lock:
    several ranks may start together), and if it cannot be rebuilt the call raises -- a stale library is never used
    silently and there is no CPU fallback."""
    global _LIB
    if _LIB is None:
        import os
        override = os.environ.get("SEPT_LIB_PATH")                 # experiments only (A/B of two builds): no hash check
        path = Path(override) if override else _build.LIB
        if not override and _build.stale():
            import fcntl
            with open(str(path) + ".lock", "w") as lock:
                fcntl.flock(lock, fcntl.LOCK_EX)
                if _build.stale():
                    try:
                        _build.build(force=True)
                    except RuntimeError as exc:
                        state = "missing" if not path.exists() else "stale (built from other sources than the tree holds)"
                        raise RuntimeError(f"{path.name} is {state} and cannot be rebuilt: {exc}") from exc
        handle = C.CDLL(str(path))
        for name, (res, args) in _SIGNATURES.items():
            try:
                fn = getattr(handle, name)
            except AttributeError:
                if override:                                       # an older experimental build: A/B timing only
                    continue
                raise
            fn.restype, fn.argtypes = res, args
        if not override:
            got = handle.sept_source_hash().decode().split("=", 1)[1]
            if got != _build.source_hash():
                raise RuntimeError(f"{path.name} was built from other sources than the tree holds ({got[:12]} != "
                                   f"{_build.source_hash()[:12]}); run python -m speech_emotion_privacy_trust_b200.build --force")
        _LIB = handle
    return _LIB


def check(rc: int) -> None:
    """Map a status code to the exception the reference's Python would have raised."""
    if rc == 0:
        return
    msg = lib().sept_last_error().decode()
    if rc in (SEPT_E_BADARG, SEPT_E_UNSUPPORTED):
        raise ValueError(msg)
    raise RuntimeError(msg)       # too-short utterance (torch.stft raises RuntimeError too) and CUDA errors


def require_cuda(t) -> None:
    if not t.is_cuda:
        raise RuntimeError("speech_emotion_privacy_trust_b200 computes on a CUDA device only (no CPU fallback); "
                           f"got a tensor on {t.device}")
