"""CPU checks of the MFCC waveform gradient: the float64 autograd oracle (oracle/mfcc_autograd.py) is pinned against the
numpy restatement and finite differences, the backward's per-element functions (csrc/mfcc_bwd.cuh) with the frame pass
of both streams and the gather, run on the host (tests/hostsim/mfcc_bwd.cpp), match the oracle's gradient, and the C ABI
checks its arguments."""
import subprocess
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import mfcc_autograd, restate

REPO = Path(__file__).resolve().parents[1]
CSRC = REPO / "speech_emotion_privacy_trust_b200" / "csrc"


def _speechlike(n, seed):
    """noise through a resonance, slowly modulated: every non-empty band well above the top_db floor"""
    rng = np.random.default_rng(seed)
    e = rng.standard_normal(n + 2)
    y = np.zeros(n + 2)
    for i in range(2, n + 2):
        y[i] = e[i] + 1.6 * y[i - 1] - 0.8 * y[i - 2]
    return (0.05 * y[2:] * (1.2 + np.sin(np.arange(n) / 900.0))).astype(np.float32)


def test_oracle_forward_equals_restatement(golden_extraction):
    for i in (0, 3):
        x = golden_extraction[f"wav{i}"].astype(np.float64)
        got = mfcc_autograd.mfcc_blocks(torch.from_numpy(x)).numpy()
        for s, y in enumerate((x, restate.waveform_gradient(x, 1.0), restate.waveform_gradient(x, 2.0))):
            ref = restate.mfcc_one(y, np.float64)
            assert got[40 * s:40 * s + 40].shape == ref.shape
            assert np.max(np.abs(got[40 * s:40 * s + 40] - ref)) < 1e-9, s


def test_oracle_gradient_matches_finite_differences():
    """Normal audio: the empty bands 0, 3, 6, 13 (no FFT bin at n_fft 400) sit at -100 dB under the floor in every frame,
    so their upstream gradient goes to the floor and on to the argmax: the routing is part of what is checked."""
    n = 1603
    wav = _speechlike(n, 3).astype(np.float64)
    T = 1 + n // 200
    L = mfcc_autograd.logmel_db(torch.from_numpy(wav), 400, 200, 128)
    assert bool((L[:, [0, 3, 6, 13]] < L.amax() - 80).all())
    G = np.random.default_rng(4).standard_normal((120, T))
    g = mfcc_autograd.mfcc_grad(wav, G)

    def loss(x):
        return float((mfcc_autograd.mfcc_blocks(torch.from_numpy(x)).numpy() * G).sum())

    h = 1e-6
    for s in (0, 1, 2, 57, 150, 800, n - 150, n - 3, n - 2, n - 1):   # np.gradient edges, reflect regions, interior
        xp, xm = wav.copy(), wav.copy()
        xp[s] += h
        xm[s] -= h
        fd = (loss(xp) - loss(xm)) / (2 * h)
        assert abs(fd - g[s]) <= 1e-5 * max(1.0, abs(g[s])), (s, fd, g[s])


@pytest.fixture(scope="module")
def hostsim_mfcc(tmp_path_factory):
    exe = tmp_path_factory.mktemp("hostsim_mfcc") / "mfcc_bwd"
    subprocess.run(["g++", "-O2", "-std=c++17", "-I", str(CSRC), str(REPO / "tests" / "hostsim" / "mfcc_bwd.cpp"), "-o",
                    str(exe)], check=True)
    return exe


def _host(exe, tmp_path, mode, a, b):
    a.astype(np.float32).tofile(tmp_path / "a.f32")
    b.astype(np.float32).tofile(tmp_path / "b.f32")
    subprocess.run([str(exe), mode, str(tmp_path / "a.f32"), str(tmp_path / "b.f32"), str(tmp_path / "o.f32")], check=True)
    return np.fromfile(tmp_path / "o.f32", np.float32).astype(np.float64)


def _rel(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


@pytest.mark.parametrize("case", ["wav0", "wav3", "short201", "short205", "speech"])
def test_backward_functions_on_host(hostsim_mfcc, golden_extraction, tmp_path, case):
    """Head, route, both frame passes (the second staging np.gradient) and the gather against the float64 gradient."""
    if case.startswith("wav"):
        wav = golden_extraction[case].astype(np.float32)
    elif case == "speech":
        wav = _speechlike(7001, 8)
    else:
        wav = _speechlike(int(case[5:]), 7)        # about 1 draw in 8 of two frames is too ill-conditioned for 1e-5 in fp32
    T = 1 + len(wav) // 200
    G = np.random.default_rng(len(wav)).standard_normal((120, T)).astype(np.float32)
    got = _host(hostsim_mfcc, tmp_path, "grad", wav, G)
    ref = mfcc_autograd.mfcc_grad(wav.astype(np.float64), G.astype(np.float64))
    assert _rel(got, ref) < 1e-5, _rel(got, ref)


def test_backward_on_host_silence_is_exact_zero(hostsim_mfcc, tmp_path):
    G = np.random.default_rng(1).standard_normal((120, 1 + 3000 // 200))
    got = _host(hostsim_mfcc, tmp_path, "grad", np.zeros(3000), G)
    assert np.all(got == 0.0)


def test_np_gradient_adjoint_on_host(hostsim_mfcc, tmp_path):
    """<grad x, v> = <x, grad^T v> for the staged np.gradient and the gather's adjoint, and the staged values are
    np.gradient's."""
    rng = np.random.default_rng(2)
    for n in (4, 5, 201, 1000):
        x, v = rng.standard_normal(n).astype(np.float32), rng.standard_normal(n).astype(np.float32)
        out = _host(hostsim_mfcc, tmp_path, "adjoint", x, v)
        gx, gtv = out[:n], out[n:]
        assert np.allclose(gx, np.gradient(x.astype(np.float64)), rtol=1e-6, atol=1e-6)
        lhs, rhs = float(gx @ v.astype(np.float64)), float(x.astype(np.float64) @ gtv)
        assert abs(lhs - rhs) <= 1e-5 * (abs(lhs) + 1.0), (n, lhs, rhs)


def test_workspace_size_and_arguments():
    from speech_emotion_privacy_trust_b200 import _lib
    lib = _lib.lib()

    def up(x):
        return (x + 255) // 256 * 256

    tf, n_items, n_utts = 1000, 130, 7
    want = (up(2 * tf * 128 * 4) + up(tf * 4) + up(2 * n_utts * 4) + up(tf * 16) + up(tf * 32) + 2 * up(n_items * 1800 * 4))
    assert lib.sept_mfcc_bwd_workspace_bytes(n_utts, tf, n_items) == want
    assert lib.sept_mfcc_bwd_workspace_bytes(0, 0, 0) == 0
    assert lib.sept_mfcc_bwd_f32(None, None, None, None, 0, 0, 0, None, None, None, None) == 0
    assert lib.sept_mfcc_bwd_f32(None, 16, 16, 16, 1, 5, 1, 16, 16, 16, None) == _lib.SEPT_E_BADARG
    assert lib.sept_mfcc_bwd_f32(16, 16, 16, 16, 1, 5, 1, None, 16, 16, None) == _lib.SEPT_E_BADARG
    assert lib.sept_mfcc_bwd_f32(16, 16, 16, 16, 1, 5, 1, 16, 20, 16, None) == _lib.SEPT_E_BADARG   # misaligned
    with pytest.raises(ValueError, match="sept_mfcc_bwd_f32"):
        _lib.check(lib.sept_mfcc_bwd_f32(16, 16, 16, 16, 1, 5, 1, 16, None, 16, None))
