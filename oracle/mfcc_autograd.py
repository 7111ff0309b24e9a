"""torch restatement of the MFCC chain for gradients -- TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

The three streams of mfcc(audio) (audio_feature_extraction.py:15-26): y0 = x, y1 = np.gradient(x), y2 =
np.gradient(x, 2), each through torchaudio's MFCC (n_fft 400, hop 200, 128 HTK mels, AmplitudeToDB with top_db 80 below
the stream's maximum, orthonormal DCT-II to 40 coefficients), rows 40 s + c of a (120, T) block.  np.gradient is written
with tensor slicing so that autograd flows through it.  Its autograd in float64 is the reference waveform gradient of
the library's MFCC backward.  Pinned by tests/test_mfcc_grad_cpu.py against restate.mfcc and central finite
differences.
"""
from __future__ import annotations

import numpy as np
import torch

from . import restate
from .logmel_autograd import logmel_db


def np_gradient(x: torch.Tensor, spacing: float = 1.0) -> torch.Tensor:
    """np.gradient(x, spacing), edge_order 1, differentiable."""
    return torch.cat([(x[1:2] - x[0:1]) / spacing, (x[2:] - x[:-2]) / (2.0 * spacing), (x[-1:] - x[-2:-1]) / spacing])


def mfcc_blocks(wav: torch.Tensor) -> torch.Tensor:
    """(N,) waveform -> (120, T) MFCC block, differentiable, in wav's dtype."""
    D = torch.from_numpy(restate.create_dct_ortho(40, 128)).to(wav.dtype)
    out = []
    for y in (wav, np_gradient(wav, 1.0), np_gradient(wav, 2.0)):
        L = logmel_db(y, 400, 200, 128)                                   # (T, 128)
        F = torch.maximum(L, L.amax() - 80.0)
        out.append((F @ D).transpose(0, 1))
    return torch.cat(out, dim=0)


def mfcc_grad(wav: np.ndarray, G: np.ndarray, dtype: torch.dtype = torch.float64) -> np.ndarray:
    """d(sum G * mfcc_blocks(wav)) / d wav, computed by torch autograd in `dtype`; G is (120, T)."""
    x = torch.tensor(np.asarray(wav), dtype=dtype, requires_grad=True)
    B = mfcc_blocks(x)
    B.backward(torch.tensor(np.asarray(G), dtype=dtype))
    return x.grad.numpy()
