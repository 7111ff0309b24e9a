"""Launch configurations of the log-mel forward (extract_kernel<R, MODE, FAST>) and of its backward's frame pass, over every
shape the C ABI accepts, computed by the library's own host functions (tests/hostsim/launch_shape.cpp).

A shape's kernel path is decided by n_fft (R = 8 / 16 / 32), by whether its mel program has the step counts of the
compiled-in 128-band filterbank (FAST: tables in tensor memory; otherwise the shared-memory rounds), and by how many warps
per CTA fit in shared memory beside the mel program, which grows with n_mels and not monotonically, and the hop.  The
backward's warp tiles are larger than the forward's; a shape the forward runs and the backward does not fit would fail
with a raw launch error in the middle of training.  The named configurations below are the ones
tests/test_extraction_paths_gpu.py runs, each checked here to still take the path it is meant to reach."""
import subprocess
from pathlib import Path

import numpy as np
import pytest

REPO = Path(__file__).resolve().parents[1]
CSRC = REPO / "speech_emotion_privacy_trust_b200" / "csrc"

# (n_fft, hop, n_mels) -> (mel_fast, forward warps, backward warps)
CLASSES = {
    # the reference's shapes: FAST, 8 forward warps
    (400, 200, 128): (1, 8, 5),
    (800, 160, 128): (1, 8, 6),
    (1600, 160, 128): (1, 8, 7),
    # shared-memory mel rounds: 40 bands (two half rounds), 257..512 bands (9..16 rounds)
    (400, 200, 40): (0, 8, 6),
    (800, 160, 40): (0, 8, 7),
    (1600, 160, 40): (0, 8, 6),
    (400, 200, 300): (0, 8, 4),
    (800, 160, 384): (0, 8, 5),
    (1600, 160, 512): (0, 8, 5),
    # forward with fewer than 8 warps, for every n_fft; 1600 / 128 on the FAST path
    (400, 390, 512): (0, 7, 3),
    (800, 694, 40): (0, 7, 5),
    (1600, 1498, 128): (1, 7, 6),
    (1600, 838, 33): (0, 6, 5),
    # backward with 3, 4 and 8 warps (and 4 at (400, 200, 300) above)
    (400, 200, 512): (0, 8, 3),
    (800, 776, 257): (0, 8, 4),
    (400, 2, 1): (0, 8, 8),
    (800, 2, 1): (0, 8, 8),
    (1600, 2, 1): (0, 8, 8),
    # hop = n_fft, hop 2
    (400, 400, 128): (1, 8, 5),
    (800, 800, 128): (1, 8, 5),
    (1600, 1600, 128): (1, 7, 5),
    (400, 2, 128): (1, 8, 6),
}


def cuda_include() -> Path:
    from speech_emotion_privacy_trust_b200 import build
    return Path(build._nvcc()).resolve().parent.parent / "include"


def build_launch_shape(out_dir: Path) -> Path:
    """Compile the host helper (extract.h includes cuda_runtime.h, hence the CUDA include directory)."""
    exe = out_dir / "launch_shape"
    subprocess.run(["g++", "-O2", "-std=c++17", "-I", str(CSRC), "-I", str(cuda_include()),
                    str(REPO / "tests" / "hostsim" / "launch_shape.cpp"), "-o", str(exe)], check=True)
    return exe


def launch_shape(exe: Path, n_fft: int, hop: int, n_mels: int) -> dict:
    """{"mel_fast", "fwd_warps", "bwd_warps", "n_mel_entries"} of one shape."""
    out = subprocess.run([str(exe), str(n_fft), str(hop), str(n_mels)], check=True, capture_output=True, text=True).stdout
    words = out.split()
    return {k: int(v) for k, v in zip(words[::2], words[1::2])}


def path_of(exe: Path, n_fft: int, hop: int, n_mels: int) -> tuple:
    s = launch_shape(exe, n_fft, hop, n_mels)
    return s["mel_fast"], s["fwd_warps"], s["bwd_warps"]


@pytest.fixture(scope="module")
def sweep(tmp_path_factory):
    d = tmp_path_factory.mktemp("launch_shape")
    exe = build_launch_shape(d)
    subprocess.run([str(exe), "sweep", str(d / "sweep.i32")], check=True)
    rows = np.fromfile(d / "sweep.i32", dtype=np.int32).reshape(-1, 7)
    return exe, {k: rows[:, i] for i, k in enumerate(("n_fft", "hop", "mel_fast", "fwd", "bwd", "entries", "n_mels"))}


def test_sweep_covers_every_accepted_shape(sweep):
    _, s = sweep
    assert len(s["n_fft"]) == 512 * (200 + 400 + 800)
    for n_fft in (400, 800, 1600):
        m = s["n_fft"] == n_fft
        assert set(np.unique(s["hop"][m])) == set(range(2, n_fft + 1, 2))
        assert set(np.unique(s["n_mels"][m])) == set(range(1, 513))


def test_backward_fits_wherever_the_forward_does(sweep):
    _, s = sweep
    runs = s["fwd"] > 0
    refused = runs & (s["bwd"] == 0)
    assert not refused.any(), [tuple(int(s[k][i]) for k in ("n_fft", "hop", "n_mels")) for i in np.flatnonzero(refused)[:10]]
    assert np.all(s["fwd"] <= 8) and np.all(s["bwd"] <= 8)


def test_fast_path_is_exactly_the_128_band_filterbank(sweep):
    _, s = sweep
    assert np.array_equal(s["mel_fast"] == 1, s["n_mels"] == 128)


def test_every_warp_class_is_reached(sweep):
    """The classes the GPU tests run exist: fewer than 8 forward warps at every n_fft (and on the FAST path), every
    backward warp count from 3 to 8."""
    _, s = sweep
    for n_fft in (400, 800, 1600):
        assert np.any((s["n_fft"] == n_fft) & (s["fwd"] < 8)), n_fft
    assert np.any((s["mel_fast"] == 1) & (s["fwd"] < 8))
    assert set(np.unique(s["bwd"])) == set(range(3, 9))
    assert set(np.unique(s["fwd"])) == {6, 7, 8}


@pytest.mark.parametrize("shape", sorted(CLASSES), ids=lambda s: "-".join(map(str, s)))
def test_named_configurations_keep_their_class(sweep, shape):
    exe, s = sweep
    assert path_of(exe, *shape) == CLASSES[shape]
    n_fft, hop, n_mels = shape
    i = np.flatnonzero((s["n_fft"] == n_fft) & (s["hop"] == hop) & (s["n_mels"] == n_mels))
    assert len(i) == 1 and (s["mel_fast"][i[0]], s["fwd"][i[0]], s["bwd"][i[0]]) == CLASSES[shape]
