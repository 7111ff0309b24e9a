"""CPU-only checks of the waveform-domain cloak (csrc/wave_cloak.cu, wave_cloak.py): the tile table of
sept_wave_cloak_layout, the backward's summation order restated on the host (tests/wave_cloak_order.py) against a float64
sum on ragged lengths, the argument checks of the four C entries, their loud failure without a GPU, and the errors the
Python layer raises."""
import ctypes

import numpy as np
import pytest
import torch

import wave_cloak_order as order
from speech_emotion_privacy_trust_b200 import _lib

RAGGED = [0, 3, 7, 0, 8, 31, 32, 33, 95, 1, 64, 130, 5]      # empty, shorter than, equal to and several periods


def _layout(utt_off, period):
    off = np.ascontiguousarray(utt_off, dtype=np.int64)
    tile_off = np.zeros(len(off), dtype=np.int64)
    rc = _lib.lib().sept_wave_cloak_layout(off.ctypes.data, len(off) - 1, period, tile_off.ctypes.data)
    return rc, tile_off


def _offsets(lengths, start=0):
    return np.concatenate([[start], start + np.cumsum(lengths)]).astype(np.int64)


@pytest.mark.parametrize("period", [4, 8, 32, 44])
def test_tiles_cover_every_utterance_sample_once(period):
    off = _offsets(RAGGED, start=5)
    rc, tile_off = _layout(off, period)
    assert rc == 0
    assert np.array_equal(np.diff(tile_off), (np.diff(off) + period - 1) // period)
    base, length = order.tiles_of(off, tile_off, period)
    assert np.all(length >= 1) and np.all(length <= period)
    covered = np.concatenate([np.arange(b, b + n) for b, n in zip(base, length)])
    assert np.array_equal(covered, np.arange(off[0], off[-1]))         # in order, each sample once, gaps excluded
    assert np.all((base - off[np.searchsorted(off, base, side="right") - 1]) % period == 0)   # tiles start at phase 0


@pytest.mark.parametrize("period,lengths", [
    (4, RAGGED * 3),
    (44, RAGGED + [1000, 437, 44, 88, 89]),                             # 44 is not a multiple of 16
    (1000, [999, 1000, 1001, 4003, 17, 2500, 3]),
    (32000, [16000, 32000, 96001, 40003, 7]),
])
def test_host_order_against_float64(period, lengths):
    rng = np.random.default_rng(period)
    off = _offsets(lengths, start=3)
    n = int(off[-1]) + 6                                                 # a gap after the last utterance too
    g = (rng.standard_normal(n) * rng.choice([1e-3, 1.0, 1e3], n)).astype(np.float32)
    _, tile_off = _layout(off, period)
    r = order.phase_sum(g, off, tile_off, period).astype(np.float64)
    r64, tol = order.bound(g, off, period)
    assert np.all(np.abs(r - r64) <= tol), np.max(np.abs(r - r64) - tol)
    g2 = g.copy()
    g2[:3] = g2[-6:] = 1e30                                              # samples outside every utterance do not count
    assert np.array_equal(order.phase_sum(g2, off, tile_off, period), order.phase_sum(g, off, tile_off, period))


def test_host_order_many_slices_and_lanes():
    """More tiles than slices, several chunks per slice, and lanes (period 4: 256 lanes, period 256: 4 lanes)."""
    rng = np.random.default_rng(7)
    lengths = rng.integers(1, 900, 400)
    off = _offsets(lengths)
    g = rng.standard_normal(int(off[-1])).astype(np.float32)
    for period in (4, 256):
        _, tile_off = _layout(off, period)
        assert tile_off[-1] > order.SLICES
        r = order.phase_sum(g, off, tile_off, period).astype(np.float64)
        r64, tol = order.bound(g, off, period)
        assert np.all(np.abs(r - r64) <= tol), period


@pytest.mark.parametrize("off,period", [([0, 4], 6), ([0, 4], 0), ([0, 4], -4), ([-1, 4], 4), ([0, 8, 4], 4),
                                        ([0, 1 << 31], 4)])
def test_layout_rejects_bad_arguments(off, period):
    rc, _ = _layout(off, period)
    assert rc == _lib.SEPT_E_BADARG
    assert "sept_wave_cloak_layout" in _lib.lib().sept_last_error().decode()


def test_layout_rejects_null_and_negative():
    lib = _lib.lib()
    off, tile = np.zeros(2, np.int64), np.zeros(2, np.int64)
    assert lib.sept_wave_cloak_layout(None, 1, 4, tile.ctypes.data) == _lib.SEPT_E_BADARG
    assert lib.sept_wave_cloak_layout(off.ctypes.data, 1, 4, None) == _lib.SEPT_E_BADARG
    assert lib.sept_wave_cloak_layout(off.ctypes.data, -1, 4, tile.ctypes.data) == _lib.SEPT_E_BADARG


def test_workspace_bytes():
    lib = _lib.lib()
    assert lib.sept_wave_cloak_bwd_workspace_bytes(32000) == order.SLICES * 32000 * 4
    assert lib.sept_wave_cloak_bwd_workspace_bytes(4) == order.SLICES * 16
    for bad in (0, -4, 6, 30):
        assert lib.sept_wave_cloak_bwd_workspace_bytes(bad) == 0


def _bufs():
    """Host buffers of valid shape for 2 utterances of 8 samples at period 4 (16-byte aligned; host memory)."""
    b = {"x": (ctypes.c_float * 24)(), "y": (ctypes.c_float * 24)(), "noise": (ctypes.c_float * 8)(),
         "off": (ctypes.c_int64 * 3)(0, 8, 16), "tiles": (ctypes.c_int64 * 3)(0, 2, 4), "r": (ctypes.c_float * 8)(),
         "ws": (ctypes.c_float * (order.SLICES * 4 + 4))()}
    a = {k: (ctypes.addressof(v) + 15) & ~15 for k, v in b.items()}
    return b, a


def _fwd(a, **kw):
    v = dict(a, n_utts=2, n=16, period=4)
    v.update(kw)
    return _lib.lib().sept_wave_cloak_fwd_f32(v["x"], v["off"], v["n_utts"], v["n"], v["noise"], v["period"], v["y"], None)


def _bwd(a, **kw):
    v = dict(a, n_utts=2, n_tiles=4, period=4)
    v.update(kw)
    return _lib.lib().sept_wave_cloak_bwd_f32(v["x"], v["off"], v["tiles"], v["n_utts"], v["n_tiles"], v["period"], v["ws"],
                                              v["r"], None)


@pytest.mark.parametrize("bad", [dict(x=None), dict(off=None), dict(noise=None), dict(y=None), dict(n_utts=-1), dict(n=-1),
                                 dict(period=0), dict(period=-4), dict(period=6), dict(period=30)])
def test_forward_rejects_bad_arguments(bad):
    keep, a = _bufs()
    assert _fwd(a, **bad) == _lib.SEPT_E_BADARG
    assert "sept_wave_cloak_fwd_f32" in _lib.lib().sept_last_error().decode()
    with pytest.raises(ValueError, match="sept_wave_cloak_fwd_f32"):
        _lib.check(_lib.SEPT_E_BADARG)


@pytest.mark.parametrize("bad", [dict(x=None), dict(off=None), dict(tiles=None), dict(ws=None), dict(r=None),
                                 dict(n_utts=-1), dict(n_tiles=-1), dict(period=0), dict(period=6), dict(period=30)])
def test_backward_rejects_bad_arguments(bad):
    keep, a = _bufs()
    assert _bwd(a, **bad) == _lib.SEPT_E_BADARG
    assert "sept_wave_cloak_bwd_f32" in _lib.lib().sept_last_error().decode()


@pytest.mark.parametrize("which", ["x", "noise", "y"])
def test_forward_rejects_unaligned_pointers(which):
    keep, a = _bufs()
    assert _fwd(a, **{which: a[which] + 4}) == _lib.SEPT_E_BADARG
    assert "16-byte aligned" in _lib.lib().sept_last_error().decode()


@pytest.mark.parametrize("which", ["x", "ws", "r"])
def test_backward_rejects_unaligned_pointers(which):
    keep, a = _bufs()
    assert _bwd(a, **{which: a[which] + 4}) == _lib.SEPT_E_BADARG
    assert "16-byte aligned" in _lib.lib().sept_last_error().decode()


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_compute_fails_loudly_without_a_gpu():
    keep, a = _bufs()
    assert _fwd(a) == _lib.SEPT_E_CUDA
    assert _bwd(a) == _lib.SEPT_E_CUDA
    with pytest.raises(RuntimeError):
        _lib.check(_lib.SEPT_E_CUDA)
    from speech_emotion_privacy_trust_b200 import wave_cloak
    layer = wave_cloak.WaveCloak(0.001, 0.01, period=8)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        wave_cloak.WaveCloakFunction.apply(torch.zeros(16), layer.locs, layer.rhos, None, None, 0, 0, 0.1, 0.001, 0.01)


def test_python_layer_errors():
    from speech_emotion_privacy_trust_b200 import wave_cloak
    for period in (0, -4, 6, 30):
        with pytest.raises(ValueError, match="multiple of 4"):
            wave_cloak.WaveCloak(0.001, 0.01, period=period)
    with pytest.raises(ValueError, match="the period is 8"):
        wave_cloak.WaveCloak(0.001, 0.01, period=8, locs=torch.zeros(12))
    layer = wave_cloak.WaveCloak(0.001, 0.01, period=8)
    assert layer.locs.shape == layer.rhos.shape == (8,)
    assert torch.allclose(layer.scales(), (1 + torch.tanh(torch.tensor(-2.0))) / 2 * 0.009 + 0.001)
    layer.external_eps = torch.zeros(7)
    with pytest.raises(ValueError, match="external_eps has 7 elements"):
        layer._eps_source()
    with pytest.raises(ValueError, match="multiple of 4"):
        wave_cloak.new_workspace(torch.device("cpu"), 30)
