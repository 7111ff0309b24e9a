"""Gradient through the data-parallel per-speaker statistics (normalization.speaker_stats_distributed_grad) on the GPU.

Spec: with the ranks' losses summed, each rank's feature gradient equals what speaker_stats_grad -> normalized_windows_grad
(or normalize_grad) gives on ONE GPU over the union of all ranks' utterances, restricted to that rank's frames.  One
device: without a process group, against speaker_stats_grad and the float64 oracle (oracle/norm_autograd.py).  Two and four
ranks started with torch.multiprocessing.spawn, each holding a shard of one seeded corpus, against the one-GPU union and
the oracle: over NCCL with one device per rank (skipped when fewer devices are visible), and over gloo with every rank on
the same device (NCCL refuses two ranks on one device; gloo moves the same CUDA tensors, so the rank-order sum and the
exact int32 sum are the same arithmetic and a one-GPU machine runs the multi-rank path too).
Metric: rel = |g - g_ref| / |g_ref| per utterance."""
import os
from datetime import timedelta
from functools import lru_cache

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import norm_autograd as na

pytestmark = pytest.mark.gpu

N_UTTS, F = 24, 128


def _rel(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def _layout(feats, dev):
    from speech_emotion_privacy_trust_b200.extraction import Layout
    fo = np.concatenate([[0], np.cumsum([len(f) for f in feats])]).astype(np.int64)
    return Layout(fo, torch.from_numpy(fo).to(dev), torch.zeros(len(fo), dtype=torch.int32, device=dev))


def _corpus(kind="normal"):
    """24 utterances (short / padded, T = 249 with frames outside every window, whole-utterance flags), speakers a, b, c
    and one speaker with a single utterance (so only one rank holds it).  kind "ties": values on a few levels (ties of
    the minimum and maximum across ranks); "const": feature 5 is digital silence (std exactly 0)."""
    rng = np.random.default_rng(0)
    frames = rng.integers(120, 700, size=N_UTTS)
    frames[:4] = [37, 200, 249, 250]
    spk = [("a", "b", "c")[u % 3] for u in range(N_UTTS)]
    spk[7] = "solo"
    whole = [u % 5 == 4 for u in range(N_UTTS)]
    feats = [(rng.standard_normal((T, F)) * 9 - 40).astype(np.float32) for T in frames]
    if kind == "ties":
        feats = [np.round((f + 40) / 4.5).astype(np.float32) for f in feats]
    elif kind == "const":
        for f in feats:
            f[:, 5] = -100.0
    return feats, spk, whole


ALL_SPEAKERS = ["a", "b", "c", "solo"]


def _upstream(feats):
    """Per-utterance upstream gradients (window form and frame form), seeded by the utterance, so any shard takes the
    rows of the union."""
    from speech_emotion_privacy_trust_b200 import normalization as nz
    gw = [np.random.default_rng(1000 + u).standard_normal((nz.n_windows(len(f)), 200, F)).astype(np.float32)
          for u, f in enumerate(feats)]
    gf = [np.random.default_rng(2000 + u).standard_normal(f.shape).astype(np.float32) for u, f in enumerate(feats)]
    return gw, gf


def _grads(kind, mine, mode, form, dev, stats_fn):
    """feat.grad per utterance of sum(G * normalized_windows_grad) (form "win") or sum(G * normalize_grad) ("frames")
    over the utterances `mine` of the corpus, `stats_fn(feat, lay, spk, whole)` giving the statistics."""
    from speech_emotion_privacy_trust_b200 import normalization as nz
    feats, spk, whole = _corpus(kind)
    gw, gf = _upstream(feats)
    sf = [feats[u] for u in mine]
    lay = _layout(sf, dev)
    feat = torch.from_numpy(np.concatenate(sf)).to(dev).requires_grad_(True)
    st = stats_fn(feat, lay, [spk[u] for u in mine], [whole[u] for u in mine])
    if form == "win":
        wu, wt = nz.window_table(lay)
        out = nz.normalized_windows_grad(feat, lay, st, wu, wt, mode)
        G = np.concatenate([gw[u] for u in mine])
    else:
        out = nz.normalize_grad(feat, lay, st, mode)
        G = np.concatenate([gf[u] for u in mine])
    out.backward(torch.from_numpy(G).to(dev).view_as(out))
    g = feat.grad.cpu().numpy().astype(np.float64)
    fo = lay.frame_off_host
    return [g[fo[i]:fo[i + 1]] for i in range(len(mine))], st, lay


def _oracle(feats, spk, whole, mode, form):
    from speech_emotion_privacy_trust_b200 import normalization as nz
    gw, gf = _upstream(feats)
    xs = [torch.from_numpy(f).double().requires_grad_(True) for f in feats]
    speakers, stats = na.speaker_stats(xs, spk, whole)
    row = {s: i for i, s in enumerate(speakers)}
    rows = [row[s] for s in spk]
    if form == "win":
        wu = np.concatenate([np.full(nz.n_windows(len(f)), u) for u, f in enumerate(feats)])
        wt = np.concatenate([np.arange(nz.n_windows(len(f))) * nz.SHIFT_LEN for f in feats])
        out = na.normalized_windows(xs, stats, rows, wu, wt, mode)
        (out * torch.from_numpy(np.concatenate(gw)).double()).sum().backward()
    else:
        out = torch.cat(na.normalize_frames(xs, stats, rows, mode))
        (out * torch.from_numpy(np.concatenate(gf)).double()).sum().backward()
    return [x.grad.numpy() for x in xs]


def _dist_stats(group=None):
    from speech_emotion_privacy_trust_b200 import normalization as nz
    return lambda feat, lay, spk, whole: nz.speaker_stats_distributed_grad(feat, lay, spk, ALL_SPEAKERS, whole, group)


def _union_stats(feat, lay, spk, whole):
    from speech_emotion_privacy_trust_b200 import normalization as nz
    return nz.speaker_stats_grad(feat, lay, spk, whole)


CASES = [("normal", "znorm", "win"), ("normal", "min_max", "win"), ("normal", "znorm", "frames"),
         ("ties", "min_max", "win"), ("const", "znorm", "win")]


@lru_cache(maxsize=None)
def _union(kind, mode, form):
    return _grads(kind, list(range(N_UTTS)), mode, form, torch.device("cuda", 0), _union_stats)[0]


@lru_cache(maxsize=None)
def _oracle_of(kind, mode, form):
    feats, spk, whole = _corpus(kind)
    return _oracle(feats, spk, whole, mode, form)


# ---- one device ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,mode,form", CASES)
def test_one_device_matches_speaker_stats_grad(kind, mode, form):
    """No process group: the same gradient as speaker_stats_grad (the std comes from the merge, so it is not bit-equal)
    and the float64 oracle within the DESIGN 3.4d tolerance; the forward is speaker_stats_distributed's, bit for bit."""
    from speech_emotion_privacy_trust_b200 import normalization as nz
    assert not dist.is_initialized()
    feats, spk, whole = _corpus(kind)
    g, st, _ = _grads(kind, list(range(N_UTTS)), mode, form, torch.device("cuda", 0), _dist_stats())
    assert st.stats.grad_fn is not None
    feat = torch.from_numpy(np.concatenate(feats)).cuda()
    ref = nz.speaker_stats_distributed(feat, _layout(feats, "cuda"), spk, ALL_SPEAKERS, whole)
    assert torch.equal(st.stats.detach(), ref.stats)
    union, oracle = _union(kind, mode, form), _oracle_of(kind, mode, form)
    for u in range(N_UTTS):
        assert np.all(np.isfinite(g[u])), u
        assert _rel(g[u], union[u]) < 1e-6, (u, _rel(g[u], union[u]))
        assert _rel(g[u], oracle[u]) < 1e-5, (u, _rel(g[u], oracle[u]))


def test_backward_halves_write_every_element():
    """sept_speaker_stats_bwd_ties_i32 + sept_speaker_stats_bwd_frames_f32 called directly (n_feat 128: the vector
    kernels; 37: the scalar ones) write every element of ties and dfeat, count every speaker's min and max at least once
    on the tie-heavy corpus, and give speaker_stats_grad's feature gradient bit for bit."""
    from speech_emotion_privacy_trust_b200 import _lib
    from speech_emotion_privacy_trust_b200 import normalization as nz
    lib = _lib.lib()
    for n_feat in (128, 37):
        rng = np.random.default_rng(n_feat)
        feats, spk, whole = _corpus("ties")
        feats = [f[:, :n_feat].copy() for f in feats]
        lay = _layout(feats, "cuda")
        feat = torch.from_numpy(np.concatenate(feats)).cuda().requires_grad_(True)
        st = nz.speaker_stats_grad(feat, lay, spk, whole)
        d_ptr, d_order = st.spk_lists
        d_whole = torch.from_numpy(np.asarray(whole, dtype=np.uint8)).cuda()
        stats = st.stats.detach()
        dstats = torch.from_numpy(rng.standard_normal(stats.shape).astype(np.float32)).cuda()
        n_spk, s = len(st.speakers), torch.cuda.current_stream(feat.device).cuda_stream
        ties = torch.full((n_spk, 2, n_feat), -7, dtype=torch.int32, device="cuda")
        ws = torch.empty(lib.sept_speaker_stats_bwd_ties_workspace_bytes(N_UTTS, n_feat), dtype=torch.uint8,
                         device="cuda")
        _lib.check(lib.sept_speaker_stats_bwd_ties_i32(
            feat.data_ptr(), lay.frame_off.data_ptr(), d_whole.data_ptr(), N_UTTS, n_feat, 200, 50,
            st.spk_of_utt.data_ptr(), d_ptr.data_ptr(), d_order.data_ptr(), n_spk, stats.data_ptr(), ws.data_ptr(),
            ties.data_ptr(), s))
        dfeat = torch.full(feat.shape, -7.0, device="cuda")
        _lib.check(lib.sept_speaker_stats_bwd_frames_f32(
            feat.data_ptr(), lay.frame_off.data_ptr(), d_whole.data_ptr(), N_UTTS, n_feat, 200, 50,
            st.spk_of_utt.data_ptr(), stats.data_ptr(), dstats.data_ptr(), ties.data_ptr(), dfeat.data_ptr(), s))
        assert torch.all(ties >= 1), n_feat                  # every speaker's min and max is attained by a weighted frame
        assert not torch.any(dfeat == -7), n_feat
        st.stats.backward(dstats)
        assert torch.equal(feat.grad, dfeat), n_feat


# ---- several devices -------------------------------------------------------------------------------------------------
def _shards(world, sharding, lengths):
    from speech_emotion_privacy_trust_b200 import parallel
    if sharding == "length":
        return [list(p) for p in parallel.shard_by_length(lengths, world, bucket=50)]
    perm = np.random.default_rng(world).permutation(len(lengths))          # an unbalanced random split
    cuts = np.sort(np.random.default_rng(world + 1).choice(np.arange(1, len(lengths)), world - 1, replace=False))
    return [sorted(int(u) for u in p) for p in np.split(perm, cuts)]


def _init(rank, world, init_file, backend):
    dev = torch.device("cuda", rank if backend == "nccl" else 0)
    torch.cuda.set_device(dev)
    kw = {"device_id": dev} if backend == "nccl" else {}
    dist.init_process_group(backend, init_method=f"file://{init_file}", rank=rank, world_size=world,
                            timeout=timedelta(seconds=120), **kw)
    return dev


def _features_worker(rank, world, init_file, out_dir, backend, sharding):
    dev = _init(rank, world, init_file, backend)
    try:
        from speech_emotion_privacy_trust_b200 import normalization as nz
        mine = _shards(world, sharding, [len(f) for f in _corpus()[0]])[rank]
        res = {"mine": np.array(mine)}
        for kind, mode, form in CASES:
            g, st, lay = _grads(kind, mine, mode, form, dev, _dist_stats())
            g2, _, _ = _grads(kind, mine, mode, form, dev, _dist_stats())
            feats, spk, whole = _corpus(kind)
            feat = torch.from_numpy(np.concatenate([feats[u] for u in mine])).to(dev)
            ss, sw = [spk[u] for u in mine], [whole[u] for u in mine]
            ref = nz.speaker_stats_distributed(feat, lay, ss, ALL_SPEAKERS, sw)
            key = f"{kind}|{mode}|{form}"
            res[f"{key}|fwd_equal"] = np.array(torch.equal(st.stats.detach(), ref.stats))
            res[f"{key}|bwd_twice_equal"] = np.array(all(np.array_equal(a, b) for a, b in zip(g, g2)))
            gl, _, _ = _grads(kind, mine, mode, form, dev, _union_stats)     # the local entry, under the process group
            for i, u in enumerate(mine):
                res[f"{key}|{u}"] = g[i]
                res[f"{key}|local|{u}"] = gl[i]
            if kind == "const":                              # the std path alone: exactly nothing for the silent column
                feat.requires_grad_(True)
                st = nz.speaker_stats_distributed_grad(feat, lay, ss, ALL_SPEAKERS, sw)
                res["const|std_is_zero"] = np.array(bool(torch.all(st.stats[:, 2, 5] == 0)))
                st.stats[:, 2].sum().backward()
                res["const|std_only|col5_zero"] = np.array(bool(torch.all(feat.grad[:, 5] == 0)))
                res["const|std_only|finite"] = np.array(bool(torch.isfinite(feat.grad).all()))
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), **res)
    finally:
        dist.destroy_process_group()


def _spawn(worker, world, tmp_path, backend, *args):
    if backend == "nccl" and torch.cuda.device_count() < world:
        pytest.skip(f"NCCL needs {world} GPUs, {torch.cuda.device_count()} visible")
    mp.spawn(worker, args=(world, str(tmp_path / "store"), str(tmp_path), backend, *args), nprocs=world, join=True)
    return [dict(np.load(tmp_path / f"r{r}.npz")) for r in range(world)]


BACKENDS = pytest.mark.parametrize("backend", ["nccl", "gloo"])


@BACKENDS
@pytest.mark.parametrize("world,sharding", [(2, "length"), (2, "random"), (4, "length"), (4, "random")])
def test_ranks_match_the_one_gpu_union(backend, world, sharding, tmp_path):
    res = _spawn(_features_worker, world, tmp_path, backend, sharding)
    held = sorted(int(u) for r in res for u in r["mine"])
    assert held == list(range(N_UTTS))                       # the shards partition the corpus
    assert sum(sum(_corpus()[1][u] == "solo" for u in r["mine"]) for r in res) == 1     # one rank holds speaker "solo"
    for kind, mode, form in CASES:
        key = f"{kind}|{mode}|{form}"
        union, oracle = _union(kind, mode, form), _oracle_of(kind, mode, form)
        for r in res:
            assert r[f"{key}|fwd_equal"], (key, "forward differs from speaker_stats_distributed")
            assert r[f"{key}|bwd_twice_equal"], (key, "two backwards differ")
            # speaker_stats_grad on a rank is that rank's own gradient: it runs no collective, even under a process group
            local = _grads(kind, list(r["mine"]), mode, form, torch.device("cuda", 0), _union_stats)[0]
            for i, u in enumerate(r["mine"]):
                g = r[f"{key}|{u}"]
                assert np.all(np.isfinite(g)), (key, u)
                assert _rel(g, union[u]) < 1e-5, (key, u, _rel(g, union[u]))
                assert _rel(g, oracle[u]) < 1e-5, (key, u, _rel(g, oracle[u]))
                assert torch.equal(torch.from_numpy(r[f"{key}|local|{u}"]), torch.from_numpy(local[i])), (key, u)
    for r in res:
        assert r["const|std_is_zero"] and r["const|std_only|col5_zero"] and r["const|std_only|finite"]


def _ties_worker(rank, world, init_file, out_dir, backend):
    """Every rank holds one 250-frame utterance of speaker t (windows [0, 200) and [50, 250): frames 50..199 count twice)
    whose feature 0 reaches the minimum -50 at frame 60 (multiplicity 2), rank 0 also at frame 10 (multiplicity 1), and
    feature 1 the maximum 50 at frame 120; rank 0 alone holds speaker p (one short utterance, minimum at frame 5)."""
    dev = _init(rank, world, init_file, backend)
    try:
        from speech_emotion_privacy_trust_b200 import normalization as nz
        rng = np.random.default_rng(rank)
        t = rng.uniform(-10, 10, (250, 4)).astype(np.float32)
        t[60, 0] = -50
        t[120, 1] = 50
        feats, spk = [t], ["t"]
        if rank == 0:
            t[10, 0] = -50
            p = rng.uniform(-10, 10, (120, 4)).astype(np.float32)
            p[5, 0] = -60
            feats, spk = [t, p], ["t", "p"]
        lay = _layout(feats, dev)
        feat = torch.from_numpy(np.concatenate(feats)).to(dev).requires_grad_(True)
        st = nz.speaker_stats_distributed_grad(feat, lay, spk, ["t", "p"])
        (st.stats[:, 3, 0].sum() + st.stats[:, 4, 1].sum()).backward()   # feature 0: minima only, feature 1: maxima only
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), g=feat.grad.cpu().numpy(), stats=st.stats.detach().cpu().numpy())
    finally:
        dist.destroy_process_group()


@BACKENDS
@pytest.mark.parametrize("world", [2, 4])
def test_tied_minimum_across_ranks_shares_by_global_multiplicity(backend, world, tmp_path):
    res = _spawn(_ties_worker, world, tmp_path, backend)
    # every rank's loss holds stats[t, min, 0] and stats[t, max, 1]: the summed loss counts each `world` times, and the
    # share of a frame of multiplicity w is world * w / W with W the multiplicity summed over every rank's tied frames
    n = np.float32(world)
    w_min = np.float32(2 * world + 1)                        # frame 60 on every rank (2 each) + frame 10 on rank 0 (1)
    w_max = np.float32(2 * world)                            # frame 120 on every rank (2 each)
    for rank, r in enumerate(res):
        g = r["g"]
        assert np.array_equal(r["stats"], res[0]["stats"])   # every rank holds the same statistics
        assert r["stats"][0, 3, 0] == -50 and r["stats"][0, 4, 1] == 50 and r["stats"][1, 3, 0] == -60
        want = np.zeros(250, np.float32)
        want[60] = np.float32(2) * (n / w_min)
        if rank == 0:
            want[10] = n / w_min
        np.testing.assert_allclose(g[:250, 0], want, rtol=1e-6, atol=0)
        assert g[120, 1] == np.float32(2) * (n / w_max) and np.count_nonzero(g[:250, 1]) == 1
        if rank == 0:                                        # speaker p lives on rank 0 only: its one minimum takes it all
            assert g[250 + 5, 0] == n
            assert np.count_nonzero(g[250:, 0]) == 1


def _e2e_inputs():
    from speech_emotion_privacy_trust_b200 import synth
    rng = np.random.default_rng(15)
    lengths = (16000, 40000, 56000, 24000, 33000, 47000, 20000, 36000)
    spk = ["a", "b", "a", "b", "a", "c", "c", "b"]
    return [synth.speech_shaped(n, rng) for n in lengths], spk


def _e2e(waves, spk, mine, dev, stats_fn):
    """wav -> logmel_grad -> statistics -> normalized_windows_grad -> CloakNoiseFunction (eps supplied) -> sum(y * W)
    over the utterances `mine`; returns the waveform gradient per utterance and the windows' upstream rows."""
    from speech_emotion_privacy_trust_b200 import cloak_ops, extraction
    from speech_emotion_privacy_trust_b200 import normalization as nz
    batch = extraction.RaggedAudio.from_list([waves[u] for u in mine], device=dev)
    wav = batch.wav.requires_grad_(True)
    locs = torch.zeros(200, 128, device=dev, requires_grad=True)
    rhos = torch.full((200, 128), -3.0, device=dev, requires_grad=True)
    eps = torch.randn(200, 128, generator=torch.Generator().manual_seed(14)).to(dev)    # the same sample on every rank
    feats, lay = extraction.logmel_grad(batch)
    st = stats_fn(feats, lay, [spk[u] for u in mine])
    wu, wt = nz.window_table(lay)
    x = nz.normalized_windows_grad(feats, lay, st, wu, wt)
    y = cloak_ops.CloakNoiseFunction.apply(x, locs, rhos, None, eps, 0, 0, 1.0, 0.01, 10.0, False, 0.0)
    W = torch.from_numpy(np.stack([np.random.default_rng((3000 + mine[int(i)]) * 1000 + int(t0)).standard_normal((200, 128))
                                   for i, t0 in zip(wu, wt)]).astype(np.float32)).to(dev)
    (y * W.view_as(y)).sum().backward()
    g = wav.grad.cpu().numpy().astype(np.float64)
    off = batch.utt_off_host
    return [g[off[i]:off[i + 1]] for i in range(len(mine))], W.cpu().numpy(), wu, wt


def _e2e_worker(rank, world, init_file, out_dir, backend):
    dev = _init(rank, world, init_file, backend)
    try:
        from speech_emotion_privacy_trust_b200 import normalization as nz
        from speech_emotion_privacy_trust_b200 import parallel
        waves, spk = _e2e_inputs()
        mine = [int(u) for u in parallel.shard_by_length([len(w) for w in waves], world)[rank]]
        g, _, _, _ = _e2e(waves, spk, mine, dev,
                          lambda f, lay, s: nz.speaker_stats_distributed_grad(f, lay, s, ["a", "b", "c"]))
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), mine=np.array(mine), **{f"g{u}": x for u, x in zip(mine, g)})
    finally:
        dist.destroy_process_group()


@lru_cache(maxsize=None)
def _e2e_reference():
    """The one-GPU run over every utterance, and per utterance torch fp32's error against float64 for the same chain."""
    from oracle import logmel_autograd
    from speech_emotion_privacy_trust_b200 import normalization as nz
    waves, spk = _e2e_inputs()
    allu = list(range(len(waves)))
    g, W, wu, wt = _e2e(waves, spk, allu, torch.device("cuda", 0), lambda f, lay, s: nz.speaker_stats_grad(f, lay, s))

    def oracle(dtype):
        xs = [torch.from_numpy(np.asarray(w, np.float32)).to(dtype).requires_grad_(True) for w in waves]
        fs = [logmel_autograd.logmel_db(w, 800, 160, 128) for w in xs]
        speakers, stats = na.speaker_stats(fs, spk)
        row = {s: i for i, s in enumerate(speakers)}
        win = na.normalized_windows(fs, stats, [row[s] for s in spk], wu, wt)
        (win * torch.from_numpy(W).to(dtype)).sum().backward()        # the cloak passes W through to its input
        return [w.grad.double().numpy() for w in xs]

    ref64, ref32 = oracle(torch.float64), oracle(torch.float32)
    return g, [_rel(a, b) for a, b in zip(ref32, ref64)]


@BACKENDS
@pytest.mark.parametrize("world", [2, 4])
def test_end_to_end_waveform_gradient_data_parallel(backend, world, tmp_path):
    res = _spawn(_e2e_worker, world, tmp_path, backend)
    union, rel32 = _e2e_reference()
    seen = []
    for r in res:
        for u in r["mine"]:
            rel = _rel(r[f"g{u}"], union[u])
            assert rel < max(1e-5, 4 * rel32[u]), (u, rel, rel32[u])
            seen.append(int(u))
    assert sorted(seen) == list(range(len(union)))
