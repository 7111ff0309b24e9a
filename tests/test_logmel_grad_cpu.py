"""CPU checks of the log-mel waveform gradient: the float64 autograd oracle (oracle/logmel_autograd.py) is pinned against
the numpy restatement and finite differences, and the backward's per-lane phase functions (csrc/extract_bwd.cuh), run
lane by lane on the host (tests/hostsim/logmel_bwd.cpp), match the oracle's gradient for every FFT size."""
import subprocess
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import logmel_autograd, restate

REPO = Path(__file__).resolve().parents[1]
CSRC = REPO / "speech_emotion_privacy_trust_b200" / "csrc"


@pytest.mark.parametrize("n_fft", [800, 1600])
def test_oracle_forward_equals_restatement(golden_extraction, n_fft):
    wav = golden_extraction["wav1"].astype(np.float64)
    got = logmel_autograd.logmel_db(torch.from_numpy(wav), n_fft, 160, 128).numpy()
    ref = restate.mel_spectrogram(wav[None], n_fft, 128, dtype=np.float64)[0].T
    assert got.shape == ref.shape
    assert np.max(np.abs(got - ref)) < 1e-9


def test_oracle_gradient_matches_finite_differences():
    rng = np.random.default_rng(3)
    n, n_fft, hop, n_mels = 1003, 400, 200, 40
    wav = rng.standard_normal(n) * 0.1
    T = 1 + n // hop
    G = rng.standard_normal((T, n_mels))
    g = logmel_autograd.logmel_grad(wav, G, n_fft, hop, n_mels)

    def loss(x):
        return float((logmel_autograd.logmel_db(torch.from_numpy(x), n_fft, hop, n_mels).numpy() * G).sum())

    h = 1e-6
    for s in (0, 1, 57, 199, 200, 201, 500, 801, 1001, 1002):     # reflect region at both ends, interior, last sample
        xp, xm = wav.copy(), wav.copy()
        xp[s] += h
        xm[s] -= h
        fd = (loss(xp) - loss(xm)) / (2 * h)
        assert abs(fd - g[s]) <= 1e-5 * max(1.0, abs(g[s])), (s, fd, g[s])


@pytest.fixture(scope="module")
def hostsim_bwd(tmp_path_factory):
    exe = tmp_path_factory.mktemp("hostsim_bwd") / "logmel_bwd"
    subprocess.run(["g++", "-O2", "-std=c++17", "-I", str(CSRC), str(REPO / "tests" / "hostsim" / "logmel_bwd.cpp"), "-o",
                    str(exe)], check=True)
    return exe


def _host_grad(exe, tmp_path, wav, G, n_fft, hop, n_mels):
    wav.astype(np.float32).tofile(tmp_path / "w.f32")
    G.astype(np.float32).tofile(tmp_path / "g.f32")
    subprocess.run([str(exe), str(n_fft), str(hop), str(n_mels), str(tmp_path / "w.f32"), str(tmp_path / "g.f32"),
                    str(tmp_path / "d.f32")], check=True)
    return np.fromfile(tmp_path / "d.f32", np.float32).astype(np.float64)


@pytest.mark.parametrize("i", [0, 3])
@pytest.mark.parametrize("n_fft,hop,n_mels", [(400, 200, 128), (800, 160, 128), (1600, 160, 128), (800, 80, 40),
                                              (1600, 480, 256)])
def test_backward_phase_functions_on_host(hostsim_bwd, golden_extraction, tmp_path, i, n_fft, hop, n_mels):
    """The per-lane functions of the backward kernel against the float64 autograd gradient, within the GPU tolerance."""
    wav = golden_extraction[f"wav{i}"].astype(np.float32)
    T = 1 + len(wav) // hop
    G = np.random.default_rng(i).standard_normal((T, n_mels)).astype(np.float32)
    got = _host_grad(hostsim_bwd, tmp_path, wav, G, n_fft, hop, n_mels)
    ref = logmel_autograd.logmel_grad(wav.astype(np.float64), G.astype(np.float64), n_fft, hop, n_mels)
    rel = np.linalg.norm(got - ref) / np.linalg.norm(ref)
    assert rel < 1e-5, rel


def test_backward_on_host_short_utterance_and_silence(hostsim_bwd, tmp_path):
    """Lengths just above n_fft/2 (reflection at both ends of the same frames) and digital silence (exactly 0)."""
    rng = np.random.default_rng(7)
    for n_fft, hop in ((400, 200), (800, 160), (1600, 160)):
        wav = (rng.standard_normal(n_fft // 2 + 3) * 0.1).astype(np.float32)
        T = 1 + len(wav) // hop
        G = rng.standard_normal((T, 128))
        got = _host_grad(hostsim_bwd, tmp_path, wav, G, n_fft, hop, 128)
        ref = logmel_autograd.logmel_grad(wav.astype(np.float64), G, n_fft, hop, 128)
        assert np.linalg.norm(got - ref) / np.linalg.norm(ref) < 1e-5
        silent = np.zeros(3000, np.float32)
        got = _host_grad(hostsim_bwd, tmp_path, silent, rng.standard_normal((1 + 3000 // hop, 128)), n_fft, hop, 128)
        assert np.all(got == 0.0)


def test_workspace_size_and_unsupported_shapes():
    from speech_emotion_privacy_trust_b200 import _lib, extraction
    lib = _lib.lib()
    assert lib.sept_logmel_bwd_workspace_bytes(800, 160, 10) == 10 * 4 * (3 * 160 + 800)
    assert lib.sept_logmel_bwd_workspace_bytes(1024, 160, 10) == 0
    rc = lib.sept_logmel_bwd_f32(1, 1, 1, 1, 1, 1, 1024, 160, 128, 1, 16, 1, None)
    assert rc == _lib.SEPT_E_UNSUPPORTED
    with pytest.raises(ValueError, match="n_fft=1024"):
        _lib.check(rc)
    with pytest.raises(ValueError, match="hop=161"):
        _lib.check(lib.sept_logmel_bwd_f32(1, 1, 1, 1, 1, 1, 800, 161, 128, 1, 16, 1, None))
    with pytest.raises(ValueError, match="frame-major"):
        extraction.logmel_grad(None, band_major=True)
    with pytest.raises(ValueError, match="deriv"):
        extraction.logmel_grad(None, deriv=True)
