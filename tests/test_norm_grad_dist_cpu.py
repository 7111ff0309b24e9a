"""CPU-only checks of the data-parallel statistics gradient: argument checks of the two halves of the statistics backward
(sept_speaker_stats_bwd_ties_i32 / sept_speaker_stats_bwd_frames_f32), their loud failure without a GPU, and the two
exchanges of its backward (parallel.sum_in_rank_order, parallel.allreduce_exact_sum) on a world-size-3 gloo group."""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from speech_emotion_privacy_trust_b200 import _lib, parallel

F = 8


def _bufs():
    """Host buffers for one utterance of 4 frames and one speaker (valid shapes; the pointers are host memory)."""
    b = {
        "feat": (ctypes.c_float * (4 * F))(), "frame_off": (ctypes.c_int64 * 2)(0, 4), "spk": (ctypes.c_int32 * 1)(0),
        "ptr": (ctypes.c_int32 * 2)(0, 1), "utts": (ctypes.c_int32 * 1)(0), "stats": (ctypes.c_float * (5 * F))(),
        "dstats": (ctypes.c_float * (5 * F))(), "ties": (ctypes.c_int32 * (2 * F))(), "dfeat": (ctypes.c_float * (4 * F))(),
        "ws": (ctypes.c_int32 * (2 * F + 8))(),
    }
    a = {k: ctypes.addressof(v) for k, v in b.items()}
    a["ws"] = (a["ws"] + 15) & ~15                         # 16-byte aligned workspace
    return b, a


def _ties(a, **kw):
    v = dict(a, n_utts=1, n_feat=F, win_len=2, shift_len=1, n_spk=1)
    v.update(kw)
    return _lib.lib().sept_speaker_stats_bwd_ties_i32(
        v["feat"], v["frame_off"], None, v["n_utts"], v["n_feat"], v["win_len"], v["shift_len"], v["spk"], v["ptr"],
        v["utts"], v["n_spk"], v["stats"], v["ws"], v["ties"], None)


def _frames(a, **kw):
    v = dict(a, n_utts=1, n_feat=F, win_len=2, shift_len=1)
    v.update(kw)
    return _lib.lib().sept_speaker_stats_bwd_frames_f32(
        v["feat"], v["frame_off"], None, v["n_utts"], v["n_feat"], v["win_len"], v["shift_len"], v["spk"], v["stats"],
        v["dstats"], v["ties"], v["dfeat"], None)


def test_ties_workspace_bytes():
    lib = _lib.lib()
    assert lib.sept_speaker_stats_bwd_ties_workspace_bytes(5, 128) == 5 * 2 * 128 * 4
    assert lib.sept_speaker_stats_bwd_ties_workspace_bytes(3, 3) == 80          # 72 bytes rounded up to 16
    assert lib.sept_speaker_stats_bwd_ties_workspace_bytes(0, 128) == 0
    assert lib.sept_speaker_stats_bwd_ties_workspace_bytes(-1, 128) == 0
    assert lib.sept_speaker_stats_bwd_ties_workspace_bytes(4, 0) == 0


@pytest.mark.parametrize("bad", [dict(feat=None), dict(frame_off=None), dict(spk=None), dict(ptr=None), dict(utts=None),
                                 dict(stats=None), dict(ws=None), dict(ties=None), dict(n_utts=-1), dict(n_spk=-1),
                                 dict(n_feat=0), dict(win_len=0), dict(shift_len=0)])
def test_ties_rejects_bad_arguments(bad):
    keep, a = _bufs()
    assert _ties(a, **bad) == _lib.SEPT_E_BADARG
    with pytest.raises(ValueError, match="sept_speaker_stats_bwd_ties_i32"):
        _lib.check(_lib.SEPT_E_BADARG)


def test_ties_rejects_unaligned_workspace():
    keep, a = _bufs()
    assert _ties(a, ws=a["ws"] + 4) == _lib.SEPT_E_BADARG
    assert "16-byte aligned" in _lib.lib().sept_last_error().decode()


@pytest.mark.parametrize("bad", [dict(feat=None), dict(frame_off=None), dict(spk=None), dict(stats=None), dict(dstats=None),
                                 dict(ties=None), dict(dfeat=None), dict(n_utts=-1), dict(n_feat=0), dict(win_len=0),
                                 dict(shift_len=0)])
def test_frames_rejects_bad_arguments(bad):
    keep, a = _bufs()
    assert _frames(a, **bad) == _lib.SEPT_E_BADARG
    assert "sept_speaker_stats_bwd_frames_f32" in _lib.lib().sept_last_error().decode()


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_both_halves_fail_loudly_without_a_gpu():
    keep, a = _bufs()
    assert _ties(a) == _lib.SEPT_E_CUDA
    with pytest.raises(RuntimeError):
        _lib.check(_lib.SEPT_E_CUDA)
    assert _frames(a) == _lib.SEPT_E_CUDA
    from speech_emotion_privacy_trust_b200 import extraction, normalization
    lay = extraction.Layout(np.array([0, 4]), torch.tensor([0, 4]), torch.zeros(2, dtype=torch.int32))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        normalization.speaker_stats_distributed_grad(torch.zeros(4, F), lay, ["a"], ["a"])


def test_exchanges_without_a_process_group():
    assert not dist.is_initialized()
    t = torch.randn(3, 5, 4)
    assert parallel.sum_in_rank_order(t) is t
    i = torch.arange(6, dtype=torch.int32)
    assert parallel.allreduce_exact_sum(i) is i and torch.equal(i, torch.arange(6, dtype=torch.int32))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        g = torch.Generator().manual_seed(10 + rank)
        x = torch.randn(4, 5, 3, generator=g) * 10 ** rank               # magnitudes 1, 10, 100: the order shows in the bits
        s = parallel.sum_in_rank_order(x.clone())
        ties = torch.full((2, 3), rank + 1, dtype=torch.int32)
        parallel.allreduce_exact_sum(ties)
        torch.save({"x": x, "sum": s, "ties": ties}, os.path.join(out, f"r{rank}.pt"))
    finally:
        dist.destroy_process_group()


def test_exchanges_on_three_gloo_ranks(tmp_path):
    world = 3
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    res = [torch.load(tmp_path / f"r{r}.pt") for r in range(world)]
    want = res[0]["x"].clone()
    for r in range(1, world):
        want += res[r]["x"]                                               # ((x0 + x1) + x2)
    for r in range(world):
        assert torch.equal(res[r]["sum"], want), r                        # the same bits on every rank, in rank order
        assert torch.equal(res[r]["ties"], torch.full((2, 3), 6, dtype=torch.int32))
