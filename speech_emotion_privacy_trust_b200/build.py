"""Build libsept_b200.so (hand-written sm_100a CUDA + the C ABI of include/sept.h) in-tree with nvcc.

    python -m speech_emotion_privacy_trust_b200.build [--force]

nvcc cross-compiles without a GPU.  The .so lands next to this file (git-ignored, but it travels to the GPU box).
"""
from __future__ import annotations

import hashlib
import os
import re
import shutil
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB = PKG / "libsept_b200.so"
HEADER = PKG.parent / "include" / "sept.h"
SOURCES = ["api.cu", "extract.cu", "extract_bwd.cu", "mfcc_bwd.cu", "mfcc_dct.cu", "cloak.cu", "norm.cu", "norm_bwd.cu", "resample.cu", "augment.cu",
           "wave_cloak.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--expt-relaxed-constexpr",
              "-Xcompiler", "-fPIC,-O2", "-diag-suppress", "20013"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found: libsept_b200.so cannot be built (there is no CPU fallback)")


def source_hash() -> str:
    """sha256 over every source the library is compiled from (+ the compiler flags).  Content, not mtime: the tree is
    copied to the GPU box, where timestamps mean nothing."""
    h = hashlib.sha256()
    deps = sorted(list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + list(CSRC.glob("*.h")) + [HEADER])
    for d in deps:
        h.update(d.name.encode() + b"\0" + d.read_bytes() + b"\0")
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def built_hash(path: Path | None = None) -> str | None:
    """The source hash compiled into an existing library (read from the file, no dlopen), None if there is none."""
    path = LIB if path is None else path
    if not path.exists():
        return None
    m = re.search(rb"SEPT_SRC_HASH=([0-9a-f]{64})", path.read_bytes())
    return m.group(1).decode() if m else None


def stale() -> bool:
    return built_hash() != source_hash()


def build(force: bool = False, verbose: bool = False) -> Path:
    if not force and not stale():
        return LIB
    nvcc = _nvcc()
    digest = source_hash()
    extra = os.environ.get("SEPT_NVCC_EXTRA", "").split()        # experiments only (compiler flag A/B)
    objdir = PKG / "build"
    objdir.mkdir(exist_ok=True)
    headers = sorted(list(CSRC.glob("*.cuh")) + list(CSRC.glob("*.h")) + [HEADER])
    common = hashlib.sha256(b"".join(h.read_bytes() for h in headers) + " ".join(NVCC_FLAGS + extra).encode()).hexdigest()
    procs = []
    for src in SOURCES:
        obj, stamp = objdir / (src + ".o"), objdir / (src + ".o.hash")
        want = hashlib.sha256((CSRC / src).read_bytes() + common.encode() + (digest.encode() if src == "api.cu" else b"")).hexdigest()
        if not verbose and obj.exists() and stamp.exists() and stamp.read_text() == want:
            continue                                             # this object was compiled from exactly these bytes
        cmd = [nvcc, *NVCC_FLAGS, *extra, "-c", str(CSRC / src), "-o", str(obj)]
        if src == "api.cu":
            cmd.insert(1, f'-DSEPT_SRC_HASH="{digest}"')
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, stamp, want, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, stamp, want, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
        stamp.write_text(want)
        if verbose and out:
            print(out)
    tmp = LIB.with_suffix(".so.tmp")
    cmd = [nvcc, "-shared", "-o", str(tmp), *[str(objdir / (s + ".o")) for s in SOURCES], "-lcudart_static", "-lpthread", "-ldl", "-lrt"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    os.replace(tmp, LIB)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
