"""Training a waveform cloak with fresh noise per utterance (WaveCloak(per_utterance=True): sept_wave_cloak_eval_f32
forward, sept_wave_cloak_bwd_per_utt_f32 backward) on the GPU.

The forward is held bit for bit to noisy_per_utterance and to per-utterance noise rows drawn by
sept_cloak_fwd_f32(per_sample = 1).  The backward: dlocs bit for bit to sept_wave_cloak_bwd_f32's phase sum; at rho = 0,
min 0.5, max 2.5 (sigma' = 1 exactly) drhos bit for bit to the host restatement of the kernels' order
(tests/wave_cloak_order.py) applied to fl32(g * eps_u); at any rho both within the reordered-sum bound of float64.  Then
batch order and sharding, two forwards before one backward, CUDA-graph replays, the chain to a GRL classifier against
the float64 oracles, and two gloo ranks on one device against one GPU."""
import os
from datetime import timedelta

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import wave_cloak_order as order

pytestmark = pytest.mark.gpu

# shorter than, equal to and several periods; lengths that are not multiples of 4; empty utterances
LENGTHS = [3, 4, 5, 1, 43, 44, 45, 0, 88, 131, 999, 1000, 1001, 2003, 31999, 32000, 32001, 64005, 96003, 7]
LEAD, TRAIL = 5, 3                   # samples before the first (so utterances start at odd offsets) and after the last
PERIODS = [4, 44, 1000, 32000]       # 44 and 1000 are not multiples of 16
MN, MX = 1e-3, 0.05
ULP = 2.0 ** -23


def _batch(lengths=LENGTHS, lead=LEAD, trail=TRAIL, seed=0):
    from speech_emotion_privacy_trust_b200 import extraction
    off = np.concatenate([[lead], lead + np.cumsum(lengths)]).astype(np.int64)
    x = np.random.default_rng(seed).standard_normal(int(off[-1]) + trail).astype(np.float32)
    return extraction.RaggedAudio(torch.from_numpy(x).cuda(), off), x, off


def _layer(period, seed=0, mn=MN, mx=MX, rho=None):
    from speech_emotion_privacy_trust_b200 import wave_cloak
    g = torch.Generator().manual_seed(seed)
    layer = wave_cloak.WaveCloak(mn, mx, period=period, locs=0.01 * torch.randn(period, generator=g),
                                 per_utterance=True).cuda()
    with torch.no_grad():
        if rho is None:
            layer.rhos.add_(torch.randn(period, generator=g).cuda())
        else:
            layer.rhos.fill_(rho)
    return layer


def _counter(layer, value):
    layer._eps_source()
    layer._draws.fill_(value)


def _draw(layer, n_rows, draw0, noise):
    """Rows draw0 .. draw0 + n_rows - 1 of sept_cloak_fwd_f32(per_sample = 1, wf = L) at the layer's seed: the noise
    0 + (mu + sigma * eps) when `noise`, else eps itself."""
    from speech_emotion_privacy_trust_b200 import cloak_ops, wave_cloak
    L = layer.period
    counter = torch.tensor([draw0], dtype=torch.int64, device="cuda")
    out, eps, _ = cloak_ops.cloak_forward_raw(torch.zeros(n_rows * L, device="cuda"), layer.locs.detach(),
                                              layer.rhos.detach(), None, None, torch.initial_seed(), 0, wave_cloak.EPS_STD,
                                              layer.min_scale, layer.max_scale, draw=counter, per_sample=True)
    return (out if noise else eps).view(n_rows, L).cpu().numpy()


def _per_sample(off, n, rows, row_of_utt):
    """(phase of every sample or -1, rows[row_of_utt[u]][phase] per in-utterance sample, 0 elsewhere)."""
    ph = order.phase_of(off, n, rows.shape[1])
    s = np.nonzero(ph >= 0)[0]
    u = np.searchsorted(off, s, side="right") - 1
    v = np.zeros(n, np.float32)
    v[s] = rows[np.asarray(row_of_utt)[u], ph[s]]
    return ph, v


def _grad(n, seed):
    g = np.random.default_rng(seed).standard_normal(n).astype(np.float32)
    return g * np.random.default_rng(seed + 1).choice([1e-3, 1.0, 1e3], n).astype(np.float32)


def _bwd_raw(batch, g, period):
    from speech_emotion_privacy_trust_b200 import _lib
    lib = _lib.lib()
    tiles = batch.tiles(period)
    ws = torch.full((lib.sept_wave_cloak_bwd_workspace_bytes(period) // 4,), float("nan"), device="cuda")
    r = torch.full((period,), float("nan"), device="cuda")
    _lib.check(lib.sept_wave_cloak_bwd_f32(g.data_ptr(), batch.utt_off.data_ptr(), tiles.tile_off.data_ptr(), batch.n_utts,
                                           tiles.n_tiles, period, ws.data_ptr(), r.data_ptr(),
                                           torch.cuda.current_stream().cuda_stream))
    return r


def _run(layer, batch, G, **kw):
    """(noisy audio, dlocs, drhos) of one forward + backward of sum(G * y)."""
    layer.zero_grad(set_to_none=True)
    y = layer(batch, **kw).wav
    y.backward(G)
    return y.detach().cpu().numpy(), layer.locs.grad.cpu().numpy(), layer.rhos.grad.cpu().numpy()


def _float64(G, eps_s, ph, rhos, mn, mx, period):
    """(dlocs, drhos, sigma', q) of sum(G * y) in float64, eps_s the eps of every in-utterance sample."""
    inside = ph >= 0
    g64, e64 = G.astype(np.float64)[inside], eps_s.astype(np.float64)[inside]
    dl64 = np.bincount(ph[inside], weights=g64, minlength=period)
    q64 = np.bincount(ph[inside], weights=g64 * e64, minlength=period)
    t = np.tanh(rhos.astype(np.float64))
    dsig = (1 - t * t) / 2 * (mx - mn)
    return dl64, q64 * dsig, dsig, q64


def _bounds(G, eps_s, off, period, dsig, q64, mn, mx):
    """order.bound of G and of G * eps for the phase sums, carried through drhos = q * sigma' with
    sigma' = (1 - tanh^2) / 2 * (max - min) a few ulps off in fp32."""
    _, tol_l = order.bound(G, off, period)
    _, tol_q = order.bound(G.astype(np.float64) * eps_s, off, period)
    tol_r = tol_q * np.abs(dsig) + np.abs(q64) * (mx - mn) / 2 * 4 * ULP + 4 * ULP * np.abs(q64 * dsig)
    return tol_l, tol_r


@pytest.mark.parametrize("period", PERIODS)
def test_forward_bit_exact(period):
    torch.manual_seed(200 + period)
    batch, x, off = _batch(seed=period)
    n = batch.n_utts
    layer = _layer(period, seed=period)
    noise = _draw(layer, 3 * n + 7, 0, noise=True)
    for draw0, ids, n_draws in ((0, None, None), (7, np.random.default_rng(period).permutation(3 * n)[:n], 3 * n)):
        _counter(layer, draw0)
        y = layer(batch, utt_ids=ids, n_draws=n_draws)
        assert y.utt_off is batch.utt_off and y.wav.grad_fn is not None
        assert int(layer._draws) == draw0 + (n if n_draws is None else n_draws)
        _counter(layer, draw0)
        ev = layer.noisy_per_utterance(batch, utt_ids=ids, n_draws=n_draws).wav
        assert torch.equal(y.wav, ev)
        ph, nz = _per_sample(off, len(x), noise, draw0 + (np.arange(n) if ids is None else ids))
        want = np.where(ph >= 0, x + nz, x)
        assert np.array_equal(y.wav.detach().cpu().numpy(), want)


@pytest.mark.parametrize("period", PERIODS)
def test_backward_bit_exact_at_unit_dsigma(period):
    """rho = 0, min 0.5, max 2.5: sigma' = (1 - 0) * 0.5 * 2 = 1 exactly, so drhos is the eps-weighted phase sum itself."""
    torch.manual_seed(300 + period)
    batch, x, off = _batch(seed=period + 1)
    n = batch.n_utts
    layer = _layer(period, seed=period, mn=0.5, mx=2.5, rho=0.0)
    G = _grad(len(x), 40 + period)
    Gt = torch.from_numpy(G).cuda()
    tile_off = batch.tiles(period).tile_off_host
    r = _bwd_raw(batch, Gt, period).cpu().numpy()
    assert np.array_equal(r, order.phase_sum(G, off, tile_off, period))
    ids = np.random.default_rng(period).permutation(2 * n)[:n]
    _counter(layer, 5)
    _, dl, dr = _run(layer, batch, Gt, utt_ids=ids, n_draws=2 * n)
    _, eps_s = _per_sample(off, len(x), _draw(layer, 2 * n, 5, noise=False), ids)
    assert np.array_equal(dl, r)
    assert np.array_equal(dr, order.phase_sum(G * eps_s, off, tile_off, period))          # G * eps_s: fp32 products
    ext = 0.1 * torch.randn(n, period, device="cuda")                                       # the caller's eps by position
    before = int(layer._draws)
    _, dl, dr = _run(layer, batch, Gt, external_eps=ext)
    _, eps_s = _per_sample(off, len(x), ext.cpu().numpy(), np.arange(n))
    assert np.array_equal(dl, r)
    assert np.array_equal(dr, order.phase_sum(G * eps_s, off, tile_off, period))
    assert int(layer._draws) == before


@pytest.mark.parametrize("period", PERIODS)
def test_gradients_vs_float64(period):
    torch.manual_seed(400 + period)
    batch, x, off = _batch(seed=period + 2)
    n = batch.n_utts
    layer = _layer(period, seed=period + 3)
    G = _grad(len(x), 60 + period)
    _counter(layer, 11)
    batch.wav.requires_grad_(True)
    y, dl, dr = _run(layer, batch, torch.from_numpy(G).cuda())
    assert np.array_equal(batch.wav.grad.cpu().numpy(), G)                                  # dx = g exactly
    ph, eps_s = _per_sample(off, len(x), _draw(layer, n, 11, noise=False), np.arange(n))
    rhos = layer.rhos.detach().cpu().numpy()
    dl64, dr64, dsig, q64 = _float64(G, eps_s, ph, rhos, MN, MX, period)
    tol_l, tol_r = _bounds(G, eps_s, off, period, dsig, q64, MN, MX)
    assert np.all(np.abs(dl - dl64) <= tol_l)
    assert np.all(np.abs(dr - dr64) <= tol_r)
    _counter(layer, 11)
    assert all(np.array_equal(a, b) for a, b in zip(_run(layer, batch, torch.from_numpy(G).cuda()), (y, dl, dr)))


def test_bench_corpus_dlocs_bit_exact():
    """The bench corpus (5531 utterances, 532 M samples) at L = 32 000: dlocs is sept_wave_cloak_bwd_f32's phase sum."""
    import bench
    from speech_emotion_privacy_trust_b200 import extraction
    lengths = bench.corpus_lengths(bench.CORPUS_UTTS, 1234)
    off = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    batch = extraction.RaggedAudio(torch.randn(int(off[-1]), device="cuda"), off)
    layer = _layer(32000, seed=1)
    G = torch.randn(batch.wav.numel(), device="cuda")
    layer(batch).wav.backward(G)
    assert int(layer._draws) == len(lengths)
    assert torch.equal(layer.locs.grad, _bwd_raw(batch, G, 32000))
    assert bool(torch.isfinite(layer.rhos.grad).all()) and bool((layer.rhos.grad != 0).any())


def test_invariance_to_batch_order_and_sharding():
    from speech_emotion_privacy_trust_b200 import extraction
    torch.manual_seed(5)
    batch, x, off = _batch(seed=11)
    n, L = batch.n_utts, 1000
    layer = _layer(L, seed=3)
    gid = np.random.default_rng(4).permutation(50)[:n]                              # global ids of a 50-utterance corpus
    G = _grad(len(x), 7)
    _counter(layer, 2)
    y, dl, dr = _run(layer, batch, torch.from_numpy(G).cuda(), utt_ids=gid, n_draws=50)
    ph, eps_s = _per_sample(off, len(x), _draw(layer, 50, 2, noise=False), gid)
    rhos = layer.rhos.detach().cpu().numpy()
    dl64, dr64, dsig, q64 = _float64(G, eps_s, ph, rhos, MN, MX, L)
    tol_l, tol_r = _bounds(G, eps_s, off, L, dsig, q64, MN, MX)
    for parts in ([np.arange(n)[::-1]], [np.arange(0, n, 2), np.arange(1, n, 2)]):   # reversed; two shards
        sdl, sdr = np.zeros(L, np.float32), np.zeros(L, np.float32)
        for part in parts:
            sb = extraction.RaggedAudio.from_list([x[off[u]:off[u + 1]] for u in part])
            sG = np.concatenate([G[off[u]:off[u + 1]] for u in part])
            _counter(layer, 2)
            sy, pdl, pdr = _run(layer, sb, torch.from_numpy(sG).cuda(), utt_ids=gid[part], n_draws=50)
            assert int(layer._draws) == 52
            so = sb.utt_off_host
            for i, u in enumerate(part):
                assert np.array_equal(sy[so[i]:so[i + 1]], y[off[u]:off[u + 1]]), u
            sdl, sdr = sdl + pdl, sdr + pdr
        assert np.all(np.abs(sdl - dl) <= 2 * tol_l) and np.all(np.abs(sdr - dr) <= 2 * tol_r)
        assert np.all(np.abs(sdl - dl64) <= 2 * tol_l) and np.all(np.abs(sdr - dr64) <= 2 * tol_r)


def test_two_forwards_one_backward():
    torch.manual_seed(6)
    batch, x, off = _batch(seed=12)
    n = batch.n_utts
    layer = _layer(44, seed=6)
    G1, G2 = (torch.from_numpy(_grad(len(x), s)).cuda() for s in (80, 90))
    _counter(layer, 3)
    layer.zero_grad(set_to_none=True)
    y1 = layer(batch).wav
    y2 = layer(batch).wav                                           # counter 3 + n: a different noise
    assert not torch.equal(y1, y2)
    ((y1 * G1).sum() + (y2 * G2).sum()).backward()
    both = layer.locs.grad.clone(), layer.rhos.grad.clone()
    _counter(layer, 3)
    layer.zero_grad(set_to_none=True)
    layer(batch).wav.backward(G1)
    layer(batch).wav.backward(G2)                                   # accumulates onto the first gradient
    assert torch.equal(layer.locs.grad, both[0]) and torch.equal(layer.rhos.grad, both[1])
    assert int(layer._draws) == 3 + 2 * n


def test_cuda_graph_replays():
    torch.manual_seed(7)
    batch, x, off = _batch(seed=13)
    n = batch.n_utts
    layer = _layer(1000, seed=7)
    G = torch.from_numpy(_grad(len(x), 100)).cuda()
    _run(layer, batch, G)                                           # warm-up: workspace, tiles, counter
    layer.zero_grad(set_to_none=True)
    _counter(layer, 9)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static = layer(batch).wav
        static.backward(G)
    assert int(layer._draws) == 9                                   # capture runs nothing
    seen = []
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        seen.append((static.detach().cpu().numpy(), layer.locs.grad.cpu().numpy(), layer.rhos.grad.cpu().numpy()))
    assert int(layer._draws) == 9 + 2 * n
    for k, draw0 in enumerate((9, 9 + n)):
        _counter(layer, draw0)
        want = _run(layer, batch, G)
        assert all(np.array_equal(a, b) for a, b in zip(seen[k], want)), draw0
    assert not np.array_equal(seen[0][0], seen[1][0]) and not np.array_equal(seen[0][2], seen[1][2])


# ---- end to end -------------------------------------------------------------------------------------------------
E2E_LENGTHS = (16000, 40000, 56001, 24003, 33000)
E2E_SPK = ["a", "b", "a", "b", "a"]
E_MN, E_MX, LAM = 1e-4, 2e-2, 0.5


class _Reverse64(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        return x.view_as(x)

    @staticmethod
    def backward(ctx, g):
        return -LAM * g


def _e2e_setup():
    from speech_emotion_privacy_trust_b200 import synth
    rng = np.random.default_rng(21)
    waves = [synth.speech_shaped(n, rng) for n in E2E_LENGTHS]
    g = torch.Generator().manual_seed(22)
    locs0 = 1e-3 * torch.randn(32000, generator=g)
    rhos0 = -2.0 + torch.randn(32000, generator=g)
    eps = 0.1 * torch.randn(len(waves), 32000, generator=g)         # one row per utterance
    We, Wg = torch.randn(4, 128, generator=g) / 8, torch.randn(2, 128, generator=g) / 8
    return waves, locs0, rhos0, eps, We, Wg


def _e2e_gpu(layer, waves, eps, We, Wg, labels=None):
    from speech_emotion_privacy_trust_b200 import cloak_ops, extraction
    from speech_emotion_privacy_trust_b200 import normalization as nz
    batch = extraction.RaggedAudio.from_list(waves, device="cuda")
    feats, lay = extraction.logmel_grad(layer(batch, external_eps=eps))
    st = nz.speaker_stats_grad(feats, lay, E2E_SPK)
    wu, wt = nz.window_table(lay)
    z = nz.normalized_windows_grad(feats, lay, st, wu, wt).view(len(wu), 200, 128).mean(1)
    if labels is None:
        labels = (torch.arange(len(wu)) % 4, torch.arange(len(wu)) % 2, wu, wt)
    ye, yg = labels[0].cuda(), labels[1].cuda()
    le = torch.nn.functional.cross_entropy(z @ We.cuda().T, ye)
    lg = torch.nn.functional.cross_entropy(cloak_ops.GradientReversalFunction.apply(z, LAM) @ Wg.cuda().T, yg)
    return le, lg, labels


def _e2e_oracle(waves, locs0, rhos0, eps, We, Wg, labels, dtype):
    from oracle import logmel_autograd
    from oracle import norm_autograd as na
    locs, rhos = locs0.to(dtype).requires_grad_(True), rhos0.to(dtype).requires_grad_(True)
    sigma = (1.0 + torch.tanh(rhos)) / 2 * (E_MX - E_MN) + E_MN
    xs = [torch.from_numpy(np.asarray(w, np.float32)).to(dtype) + (locs + sigma * eps[u].to(dtype))[torch.arange(len(w)) % 32000]
          for u, w in enumerate(waves)]
    fs = [logmel_autograd.logmel_db(x, 800, 160, 128) for x in xs]
    speakers, stats = na.speaker_stats(fs, E2E_SPK)
    row = {s: i for i, s in enumerate(speakers)}
    ye, yg, wu, wt = labels
    z = na.normalized_windows(fs, stats, [row[s] for s in E2E_SPK], wu, wt).reshape(len(wu), 200, 128).mean(1)
    le = torch.nn.functional.cross_entropy(z @ We.to(dtype).T, ye)
    lg = torch.nn.functional.cross_entropy(_Reverse64.apply(z) @ Wg.to(dtype).T, yg)
    (le + lg).backward()
    return locs.grad.double().numpy(), rhos.grad.double().numpy()


def _rel(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def test_end_to_end_gradient_and_sgd():
    from speech_emotion_privacy_trust_b200 import wave_cloak
    waves, locs0, rhos0, eps, We, Wg = _e2e_setup()
    layer = wave_cloak.WaveCloak(E_MN, E_MX, period=32000, locs=locs0, per_utterance=True).cuda()
    with torch.no_grad():
        layer.rhos.copy_(rhos0)
    le, lg, labels = _e2e_gpu(layer, waves, eps.cuda(), We, Wg)
    (le + lg).backward()
    got = layer.locs.grad.double().cpu().numpy(), layer.rhos.grad.double().cpu().numpy()
    ref64 = _e2e_oracle(waves, locs0, rhos0, eps, We, Wg, labels, torch.float64)
    ref32 = _e2e_oracle(waves, locs0, rhos0, eps, We, Wg, labels, torch.float32)
    for a, b, c in zip(got, ref64, ref32):
        assert _rel(a, b) < max(1e-5, 4 * _rel(c, b)), (_rel(a, b), _rel(c, b))
    opt = torch.optim.SGD(layer.parameters(), lr=1e-3 / float(max(layer.locs.grad.abs().max(), layer.rhos.grad.abs().max())))
    js = []
    for _ in range(4):
        layer.zero_grad()
        le, lg, _ = _e2e_gpu(layer, waves, eps.cuda(), We, Wg, labels)
        js.append(float(le.detach()) - LAM * float(lg.detach()))
        (le + lg).backward()
        opt.step()
    assert js[-1] < js[0], js


# ---- data parallel: two gloo ranks on one device ------------------------------------------------------------------
DP_LENGTHS = (16000, 40000, 56001, 24003, 33000, 47005, 20000, 36002, 52003)


def _dp_run(mine):
    """(noisy audio per utterance, summed dlocs, summed drhos) of sum(G_u * y_u) over the utterances `mine` with their
    global ids, device-drawn eps at counter 0, G_u seeded by the utterance's global id; all-reduced when distributed."""
    from speech_emotion_privacy_trust_b200 import extraction, parallel, synth
    rng = np.random.default_rng(31)
    waves = [synth.speech_shaped(n, rng) for n in DP_LENGTHS]
    torch.manual_seed(0)
    layer = _layer(32000, seed=12)
    flat = parallel.FlatGradients(layer.parameters())
    batch = extraction.RaggedAudio.from_list([waves[u] for u in mine], device="cuda")
    G = np.concatenate([_grad(DP_LENGTHS[u], 500 + u) for u in mine])
    y = layer(batch, utt_ids=mine, n_draws=len(DP_LENGTHS)).wav
    y.backward(torch.from_numpy(G).cuda())
    if dist.is_initialized():
        flat.allreduce(average=False)
    yh, so = y.detach().cpu().numpy(), batch.utt_off_host
    return [yh[so[i]:so[i + 1]] for i in range(len(mine))], layer.locs.grad.cpu().numpy(), layer.rhos.grad.cpu().numpy()


def _dp_worker(rank, world, init_file, out_dir):
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", init_method=f"file://{init_file}", rank=rank, world_size=world,
                            timeout=timedelta(seconds=120))
    try:
        from speech_emotion_privacy_trust_b200 import parallel
        mine = parallel.shard_by_length(DP_LENGTHS, world)[rank]
        audio, dl, dr = _dp_run(mine)
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), mine=mine, dl=dl, dr=dr, **{f"a{u}": a for u, a in zip(mine, audio)})
    finally:
        dist.destroy_process_group()


def test_two_gloo_ranks_match_one_gpu(tmp_path):
    mp.spawn(_dp_worker, args=(2, str(tmp_path / "store"), str(tmp_path)), nprocs=2, join=True)
    allu = list(range(len(DP_LENGTHS)))
    audio, dl, dr = _dp_run(allu)
    res = [np.load(tmp_path / f"r{r}.npz") for r in range(2)]
    seen = set()
    for r in res:
        for u in r["mine"]:
            seen.add(int(u))
            assert np.array_equal(r[f"a{int(u)}"], audio[int(u)]), u                # the same noisy audio, bit for bit
    assert seen == set(allu)
    assert np.array_equal(res[0]["dl"], res[1]["dl"]) and np.array_equal(res[0]["dr"], res[1]["dr"])
    off = np.concatenate([[0], np.cumsum(DP_LENGTHS)]).astype(np.int64)
    G = np.concatenate([_grad(DP_LENGTHS[u], 500 + u) for u in allu])
    torch.manual_seed(0)
    layer = _layer(32000, seed=12)
    ph, eps_s = _per_sample(off, int(off[-1]), _draw(layer, len(allu), 0, noise=False), allu)
    dl64, dr64, dsig, q64 = _float64(G, eps_s, ph, layer.rhos.detach().cpu().numpy(), MN, MX, 32000)
    tol_l, tol_r = _bounds(G, eps_s, off, 32000, dsig, q64, MN, MX)
    assert np.all(np.abs(res[0]["dl"] - dl) <= 2 * tol_l) and np.all(np.abs(res[0]["dr"] - dr) <= 2 * tol_r)
    assert np.all(np.abs(dl - dl64) <= tol_l) and np.all(np.abs(dr - dr64) <= tol_r)
