"""CPU-only checks of training a waveform cloak with fresh noise per utterance (sept_wave_cloak_bwd_per_utt_f32,
WaveCloak(per_utterance=True)): the ctypes signature the binding derives from the header, the workspace size, the
argument checks of the C entry, its loud failure without a GPU, and the errors the Python layer raises before any launch."""
import ctypes

import numpy as np
import pytest
import torch

import wave_cloak_order as order
from speech_emotion_privacy_trust_b200 import _lib

NAME = "sept_wave_cloak_bwd_per_utt_f32"


def test_derived_signature():
    sigs = _lib.signatures(_lib._build.HEADER.read_text())
    P, I, I64, U64, F = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_uint64, ctypes.c_float
    assert sigs["sept_wave_cloak_bwd_per_utt_workspace_bytes"] == (ctypes.c_size_t, [I])
    assert sigs[NAME] == (I, [P, P, P, I, I64, I, P, P, U64, U64, P, P, F, F, F, P, P, P, P])
    assert getattr(_lib.lib(), NAME).argtypes == sigs[NAME][1]


def test_workspace_bytes():
    lib = _lib.lib()
    assert lib.sept_wave_cloak_bwd_per_utt_workspace_bytes(32000) == 2 * order.SLICES * 32000 * 4   # 151.6 MB
    assert lib.sept_wave_cloak_bwd_per_utt_workspace_bytes(4) == 2 * order.SLICES * 16
    for bad in (0, -4, 6, 30):
        assert lib.sept_wave_cloak_bwd_per_utt_workspace_bytes(bad) == 0


def _bufs():
    """Host buffers of valid shape for 2 utterances of 8 samples at period 4 (16-byte aligned; host memory)."""
    b = {"g": (ctypes.c_float * 24)(), "off": (ctypes.c_int64 * 3)(0, 8, 16), "tiles": (ctypes.c_int64 * 3)(0, 2, 4),
         "rhos": (ctypes.c_float * 8)(), "eps": (ctypes.c_float * 12)(), "draw": (ctypes.c_uint64 * 2)(),
         "ids": (ctypes.c_int64 * 2)(3, 1), "ws": (ctypes.c_float * (2 * order.SLICES * 4 + 4))(),
         "dl": (ctypes.c_float * 8)(), "dr": (ctypes.c_float * 8)()}
    a = {k: (ctypes.addressof(v) + 15) & ~15 for k, v in b.items()}
    return b, a


def _bwd(a, **kw):
    v = dict(a, n_utts=2, n_tiles=4, period=4)
    v.update(kw)
    return getattr(_lib.lib(), NAME)(v["g"], v["off"], v["tiles"], v["n_utts"], v["n_tiles"], v["period"], v["rhos"],
                                     v["eps"], 1, 0, v["draw"], v["ids"], 0.1, 0.001, 0.01, v["ws"], v["dl"], v["dr"], None)


@pytest.mark.parametrize("bad", [dict(g=None), dict(off=None), dict(tiles=None), dict(rhos=None), dict(ws=None),
                                 dict(dl=None), dict(dr=None), dict(n_utts=-1), dict(n_tiles=-1), dict(period=0),
                                 dict(period=-4), dict(period=6), dict(period=30)])
def test_rejects_bad_arguments(bad):
    keep, a = _bufs()
    assert _bwd(a, **bad) == _lib.SEPT_E_BADARG
    assert NAME in _lib.lib().sept_last_error().decode()


@pytest.mark.parametrize("which", ["g", "rhos", "eps", "ws", "dl", "dr"])
def test_rejects_unaligned_pointers(which):
    keep, a = _bufs()
    assert _bwd(a, **{which: a[which] + 4}) == _lib.SEPT_E_BADARG
    assert "16-byte aligned" in _lib.lib().sept_last_error().decode()


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_fails_loudly_without_a_gpu():
    keep, a = _bufs()
    for kw in (dict(), dict(eps=None, draw=None, ids=None)):         # caller's eps / device draw, id table or none
        assert _bwd(a, **kw) == _lib.SEPT_E_CUDA
    from speech_emotion_privacy_trust_b200 import wave_cloak
    layer = wave_cloak.WaveCloak(0.001, 0.01, period=8, per_utterance=True)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        layer(_cpu_batch([8, 8]))


def _cpu_batch(lengths):
    """A RaggedAudio over a host buffer (built around the constructor's device check): enough for the checks that run
    before any launch."""
    from speech_emotion_privacy_trust_b200 import extraction
    b = extraction.RaggedAudio.__new__(extraction.RaggedAudio)
    b.utt_off_host = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    b.wav = torch.zeros(int(b.utt_off_host[-1]))
    return b


def test_python_errors_before_any_launch():
    from speech_emotion_privacy_trust_b200 import wave_cloak
    batch = _cpu_batch([8, 5, 0, 12])
    shared = wave_cloak.WaveCloak(0.001, 0.01, period=8)
    for kw in (dict(utt_ids=[0, 1, 2, 3]), dict(n_draws=4), dict(external_eps=torch.zeros(4, 8))):
        with pytest.raises(ValueError, match="per_utterance=True"):
            shared(batch, **kw)
    layer = wave_cloak.WaveCloak(0.001, 0.01, period=8, per_utterance=True)
    assert layer.per_utterance and not shared.per_utterance
    for ids, n_draws, msg in (([0, 1, 2, -1], None, "lie in"), ([0, 1, 2, 4], None, "lie in"), ([0, 1, 2, 9], 9, "lie in"),
                              ([0, 1, 1, 3], None, "distinct"), ([0, 1, 2], None, "entries"),
                              ([0.0, 1.0, 2.0, 3.0], None, "integers")):
        with pytest.raises(ValueError, match=msg):
            layer(batch, utt_ids=ids, n_draws=n_draws)
    with pytest.raises(ValueError, match="smaller than the batch"):
        layer(batch, n_draws=3)
    for shape in ((4, 4), (3, 8), (32,)):
        with pytest.raises(ValueError, match="external_eps must be"):
            layer(batch, external_eps=torch.zeros(shape))
    layer.external_eps = torch.zeros(8)
    with pytest.raises(ValueError, match="single sample"):
        layer(batch)
    assert layer._draws is None and layer._workspace_per_utt is None      # nothing was allocated or launched
