"""ctypes binding of libsept_b200.so (include/sept.h).  There is no CPU fallback: a missing library is built with
nvcc if the toolchain is present, otherwise importing the compute layer fails loudly."""
from __future__ import annotations

import ctypes as C
import re
from pathlib import Path

import torch

from . import build as _build

_LIB = None

SEPT_E_BADARG, SEPT_E_UNSUPPORTED, SEPT_E_TOO_SHORT, SEPT_E_CUDA = -1, -2, -3, -4

_RESTYPES = {"int": C.c_int, "size_t": C.c_size_t, "const char*": C.c_char_p}
_ARGTYPES = {"int": C.c_int, "int64_t": C.c_int64, "uint64_t": C.c_uint64, "float": C.c_float, "size_t": C.c_size_t,
             "sept_stream_t": C.c_void_p}
_PROTO = re.compile(r"^[ \t]*(\w[\w \t]*?[ \t*]+)(sept_\w+)\s*\(([^)]*)\)\s*;", re.M)


def _ctype(table: dict, decl: str, name: str):
    try:
        return table[decl]
    except KeyError:
        raise RuntimeError(f"{_build.HEADER.name}: {name} uses the type {decl!r}, which the binding does not map") from None


def signatures(header: str) -> dict:
    """{name: (restype, argtypes)} of every sept_* prototype of the header text.  Pointers (device and host memory alike
    travel as integers, e.g. tensor.data_ptr()) and the stream are c_void_p; any other type must be one the tables above
    map, or this raises."""
    sigs = {}
    for ret, name, params in _PROTO.findall(re.sub(r"/\*.*?\*/", " ", header, flags=re.S)):
        args = []
        for p in ([] if params.strip() == "void" else params.split(",")):
            args.append(C.c_void_p if "*" in p else _ctype(_ARGTYPES, " ".join(p.split()[:-1]), name))
        sigs[name] = (_ctype(_RESTYPES, " ".join(ret.split()).replace(" *", "*"), name), args)
    return sigs


_SIGS = signatures(_build.HEADER.read_text())     # parsed once, when the binding is imported
EXPORTS = tuple(_SIGS)


def library_path() -> Path:
    return _build.LIB


def lib() -> C.CDLL:
    """Load libsept_b200.so.  The library carries the sha256 of the sources it was compiled from; if it is absent or
    that hash differs from the sources in the tree (a stale prebuilt .so), it is rebuilt first (under a file lock:
    several ranks may start together), and if it cannot be rebuilt the call raises -- a stale library is never used
    silently and there is no CPU fallback.  The ctypes signatures are those of include/sept.h."""
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
        for name, (res, args) in _SIGS.items():
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


def call(name: str, *args) -> None:
    """Call the C entry `name` and check its status.  A tensor passes as its data_ptr(), None as NULL, anything else as
    it is."""
    check(getattr(lib(), name)(*[a.data_ptr() if isinstance(a, torch.Tensor) else a for a in args]))


def launch(name: str, *args, device) -> None:
    """call() with `device` current and its current stream appended as the last argument (the entry's sept_stream_t)."""
    with torch.cuda.device(device):
        call(name, *args, torch.cuda.current_stream(device).cuda_stream)


def workspace(nbytes: int, device, zeroed: bool = False) -> torch.Tensor:
    """A workspace of max(16, nbytes) bytes for an entry that sizes its own (never empty, so never a NULL pointer).
    zeroed: for a kernel that needs it to start at zero."""
    return (torch.zeros if zeroed else torch.empty)(max(16, nbytes), dtype=torch.uint8, device=device)


def require_cuda(t) -> None:
    if not t.is_cuda:
        raise RuntimeError("speech_emotion_privacy_trust_b200 computes on a CUDA device only (no CPU fallback); "
                           f"got a tensor on {t.device}")
