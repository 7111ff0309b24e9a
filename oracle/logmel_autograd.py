"""torch restatement of the log-mel chain for gradients -- TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

D(s) = 10 log10(clamp(|STFT(s)|^2 @ fb, 1e-10)) with torch.stft (center, reflect pad, periodic Hann, onesided) and the
HTK filterbank of restate.melscale_fbanks_htk, on the CPU.  Its autograd is the reference waveform gradient of the
library's log-mel backward: float64 is the ground truth, float32 is what a torch user would get and sets the scale of
the fp32 rounding noise.  Pinned by tests/test_logmel_grad_oracle.py against restate.mel_spectrogram and central finite
differences.
"""
from __future__ import annotations

import numpy as np
import torch

from . import restate


def logmel_db(wav: torch.Tensor, n_fft: int, hop: int, n_mels: int) -> torch.Tensor:
    """(N,) waveform -> (T, n_mels) log-mel dB, differentiable, in wav's dtype."""
    dt = wav.dtype
    win = torch.hann_window(n_fft, periodic=True, dtype=dt)
    X = torch.stft(wav, n_fft, hop, window=win, center=True, pad_mode="reflect", return_complex=True)   # (F, T)
    P = X.real * X.real + X.imag * X.imag
    fb = torch.from_numpy(restate.melscale_fbanks_htk(n_fft // 2 + 1, n_mels)).to(dt)
    M = P.transpose(0, 1) @ fb
    return 10.0 * torch.log10(torch.clamp(M, min=1e-10))


def logmel_grad(wav: np.ndarray, grad: np.ndarray, n_fft: int, hop: int, n_mels: int,
                dtype: torch.dtype = torch.float64) -> np.ndarray:
    """d(sum grad * D(wav)) / d wav, computed by torch autograd in `dtype`; grad is (T, n_mels)."""
    x = torch.tensor(np.asarray(wav), dtype=dtype, requires_grad=True)
    D = logmel_db(x, n_fft, hop, n_mels)
    D.backward(torch.tensor(np.asarray(grad), dtype=dtype))
    return x.grad.numpy()
