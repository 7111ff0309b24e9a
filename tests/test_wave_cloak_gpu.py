"""Waveform-domain cloak on the GPU (sept_wave_cloak_fwd_f32 / sept_wave_cloak_bwd_f32, wave_cloak.WaveCloak), against
a float64 torch restatement: noise[phase] gathered per sample and torch autograd.

Forward: bit-exact against x + noise[phase] given the same noise.  Backward: the phase sum equals the host restatement of
the kernels' summation order (tests/wave_cloak_order.py) bit for bit, and float64 within 4 * 2^-23 * sqrt(n_j) * sum|g|
per phase j (a reordered fp32 sum of n_j terms); dx is g.  Then eps (external, device draw, CUDA-graph replays), the
chain wav -> wave cloak -> logmel_grad -> speaker_stats_grad -> normalized_windows_grad -> classifier / GRL against the
float64 oracles, and two gloo ranks on one device against one GPU."""
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


def _batch(lengths=LENGTHS, lead=LEAD, trail=TRAIL, seed=0):
    from speech_emotion_privacy_trust_b200 import extraction
    off = np.concatenate([[lead], lead + np.cumsum(lengths)]).astype(np.int64)
    x = np.random.default_rng(seed).standard_normal(int(off[-1]) + trail).astype(np.float32)
    return extraction.RaggedAudio(torch.from_numpy(x).cuda(), off), x, off


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _fwd_raw(batch, noise):
    from speech_emotion_privacy_trust_b200 import _lib
    y = torch.full_like(batch.wav, float("nan"))
    _lib.check(_lib.lib().sept_wave_cloak_fwd_f32(batch.wav.data_ptr(), batch.utt_off.data_ptr(), batch.n_utts,
                                                  batch.wav.numel(), noise.data_ptr(), noise.numel(), y.data_ptr(),
                                                  _stream()))
    return y


def _bwd_raw(batch, g, period):
    from speech_emotion_privacy_trust_b200 import _lib
    lib = _lib.lib()
    tiles = batch.tiles(period)
    ws = torch.full((lib.sept_wave_cloak_bwd_workspace_bytes(period) // 4,), float("nan"), device="cuda")
    r = torch.full((period,), float("nan"), device="cuda")
    _lib.check(lib.sept_wave_cloak_bwd_f32(g.data_ptr(), batch.utt_off.data_ptr(), tiles.tile_off.data_ptr(), batch.n_utts,
                                           tiles.n_tiles, period, ws.data_ptr(), r.data_ptr(), _stream()))
    return r


def _expected(x, off, noise):
    ph = order.phase_of(off, len(x), len(noise))
    y = x.copy()
    y[ph >= 0] = x[ph >= 0] + noise[ph[ph >= 0]]
    return y


@pytest.mark.parametrize("period", PERIODS)
def test_forward_bit_exact(period):
    batch, x, off = _batch()
    noise = np.random.default_rng(period).standard_normal(period).astype(np.float32)
    y = _fwd_raw(batch, torch.from_numpy(noise).cuda()).cpu().numpy()
    want = _expected(x, off, noise)
    assert np.array_equal(y, want)
    assert np.array_equal(y[:LEAD], x[:LEAD]) and np.array_equal(y[-TRAIL:], x[-TRAIL:])   # outside every utterance


def test_forward_without_utterances_and_aligned_starts():
    from speech_emotion_privacy_trust_b200 import extraction
    noise = torch.randn(64, device="cuda")
    x = torch.randn(1003, device="cuda")
    empty = extraction.RaggedAudio(x, np.array([17], dtype=np.int64))
    assert torch.equal(_fwd_raw(empty, noise), x)
    batch, xh, off = _batch(lengths=[64 * 5, 128, 4 * 33, 64 * 7 + 4], lead=0, trail=0, seed=3)   # every start aligned
    assert np.array_equal(_fwd_raw(batch, noise).cpu().numpy(), _expected(xh, off, noise.cpu().numpy()))


@pytest.mark.parametrize("period", PERIODS)
def test_backward_matches_host_order_and_float64(period):
    batch, x, off = _batch(seed=1)
    g = np.random.default_rng(10 + period).standard_normal(len(x)).astype(np.float32)
    g *= np.random.default_rng(20 + period).choice([1e-3, 1.0, 1e3], len(x)).astype(np.float32)
    gt = torch.from_numpy(g).cuda()
    r = _bwd_raw(batch, gt, period).cpu().numpy()
    tiles = batch.tiles(period)
    assert np.array_equal(r, order.phase_sum(g, off, tiles.tile_off_host, period))
    r64, tol = order.bound(g, off, period)
    assert np.all(np.abs(r - r64) <= tol)
    assert np.array_equal(_bwd_raw(batch, gt, period).cpu().numpy(), r)           # two runs, the same bits


def test_backward_many_tiles_per_slice():
    """More tiles than slices with several 256-tile chunks per slice (period 4: 256 lanes; 256: 4 lanes)."""
    lengths = list(np.random.default_rng(5).integers(1, 2000, 1500))
    batch, x, off = _batch(lengths=lengths, seed=2)
    g = np.random.default_rng(6).standard_normal(len(x)).astype(np.float32)
    for period in (4, 256):
        r = _bwd_raw(batch, torch.from_numpy(g).cuda(), period).cpu().numpy()
        assert batch.tiles(period).n_tiles > order.SLICES
        assert np.array_equal(r, order.phase_sum(g, off, batch.tiles(period).tile_off_host, period)), period


def _restated(x, off, locs, rhos, eps, mn, mx, G):
    """float64 torch autograd of sum(G * (x + (locs + sigma(rhos) * eps)[phase])): (d locs, d rhos, dx)."""
    dev = "cuda"
    period = locs.numel()
    ph = torch.from_numpy(order.phase_of(off, len(x), period)).to(dev)
    l64 = locs.detach().double().requires_grad_(True)
    r64 = rhos.detach().double().requires_grad_(True)
    x64 = torch.from_numpy(x).double().to(dev).requires_grad_(True)
    noise = l64 + ((1.0 + torch.tanh(r64)) / 2 * (mx - mn) + mn) * eps.double()
    inside = ph >= 0
    y = x64 + torch.where(inside, noise[ph.clamp(min=0)], torch.zeros((), dtype=torch.float64, device=dev))
    (y * G.double()).sum().backward()
    return l64.grad, r64.grad, x64.grad


@pytest.mark.parametrize("period", PERIODS)
def test_module_gradients_vs_float64_autograd(period):
    from speech_emotion_privacy_trust_b200 import wave_cloak
    batch, x, off = _batch(seed=4)
    mn, mx = 1e-3, 0.05
    layer = wave_cloak.WaveCloak(mn, mx, period=period, locs=0.01 * torch.randn(period)).cuda()
    with torch.no_grad():
        layer.rhos.add_(torch.randn(period, device="cuda"))
    layer.external_eps = 0.1 * torch.randn(period, device="cuda")
    batch.wav.requires_grad_(True)
    out = layer(batch)
    assert out.wav.grad_fn is not None and out.utt_off is batch.utt_off and out.n_utts == batch.n_utts
    G = torch.randn_like(out.wav)
    out.wav.backward(G)
    assert torch.equal(batch.wav.grad, G)                                       # dx = g exactly
    dl64, dr64, _ = _restated(x, off, layer.locs, layer.rhos, layer.external_eps, mn, mx, G)
    r64, tol = order.bound(G.cpu().numpy(), off, period)
    dl, dr = layer.locs.grad.double(), layer.rhos.grad.double()
    tol = torch.from_numpy(tol).cuda()
    assert torch.all((dl - dl64).abs() <= tol)
    t = layer.rhos.detach().double().tanh()
    lever = (layer.external_eps.double() * (1 - t * t) / 2 * (mx - mn)).abs()     # |d drhos / d r|
    # the phase sum's bound carried through drhos = r * eps * sigma', plus sigma' = (1 - tanh^2) / 2 * (max - min) in
    # fp32: 1 - tanh^2 is a few ulps of 1 off, absolutely, wherever |rho| is large
    sig_err = (dl64 * layer.external_eps.double()).abs() * (mx - mn) / 2 * 4 * 2.0 ** -23
    assert torch.all((dr - dr64).abs() <= tol * lever + sig_err + 4 * 2.0 ** -23 * dr64.abs())
    g1 = (layer.locs.grad.clone(), layer.rhos.grad.clone())
    layer.zero_grad()
    layer(batch).wav.backward(G)
    assert torch.equal(layer.locs.grad, g1[0]) and torch.equal(layer.rhos.grad, g1[1])


def test_bench_corpus_backward():
    """The bench corpus (5531 utterances, 9.24 audio-hours, 13 900 to 19 400 samples per phase at L = 32 000)."""
    import bench
    from speech_emotion_privacy_trust_b200 import extraction, wave_cloak
    dev = torch.device("cuda")
    lengths = bench.corpus_lengths(bench.CORPUS_UTTS, 1234)
    off = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    batch = extraction.RaggedAudio(torch.randn(int(off[-1]), device=dev), off)
    layer = wave_cloak.WaveCloak(1e-3, 0.05, period=32000).cuda()
    layer.external_eps = 0.1 * torch.randn(32000, device=dev)
    G = torch.randn(batch.wav.numel(), device=dev)
    layer(batch).wav.backward(G)
    dl = layer.locs.grad.clone()
    layer.zero_grad()
    layer(batch).wav.backward(G)
    assert torch.equal(layer.locs.grad, dl)
    L = 32000
    starts = torch.from_numpy(off[:-1]).to(dev)
    ph = torch.arange(batch.wav.numel(), device=dev) - torch.repeat_interleave(starts, torch.from_numpy(lengths).to(dev))
    ph %= L
    g64 = G.double()
    r64 = torch.bincount(ph, weights=g64, minlength=L)
    a64 = torch.bincount(ph, weights=g64.abs(), minlength=L)
    n_j = torch.bincount(ph, minlength=L).double()
    del ph, g64
    assert int(n_j.min()) > 13000 and int(n_j.max()) > 19000            # samples per phase: every phase sums ~16 000
    assert torch.all((dl.double() - r64).abs() <= 4 * 2.0 ** -23 * n_j.sqrt() * a64)
    t = layer.rhos.detach().double().tanh()
    dr64 = r64 * layer.external_eps.double() * (1 - t * t) / 2 * (0.05 - 1e-3)
    lever = (layer.external_eps.double() * (1 - t * t) / 2 * (0.05 - 1e-3)).abs()
    sig_err = (r64 * layer.external_eps.double()).abs() * (0.05 - 1e-3) / 2 * 4 * 2.0 ** -23
    tol = 4 * 2.0 ** -23 * n_j.sqrt() * a64 * lever + sig_err + 4 * 2.0 ** -23 * dr64.abs()
    assert torch.all((layer.rhos.grad.double() - dr64).abs() <= tol)


def test_external_eps_equals_torch_restatement():
    from speech_emotion_privacy_trust_b200 import wave_cloak
    batch, x, off = _batch(seed=7)
    layer = wave_cloak.WaveCloak(0.25, 2.0, period=1000, locs=0.01 * torch.randn(1000)).cuda()   # max - min exact in fp32
    with torch.no_grad():
        layer.rhos.add_(torch.randn(1000, device="cuda"))
    layer.external_eps = 0.1 * torch.randn(1000, device="cuda")
    y = layer(batch).wav.detach().cpu().numpy()
    with torch.no_grad():
        noise = (layer.locs + layer.scales() * layer.external_eps).cpu().numpy()
    assert np.array_equal(y, _expected(x, off, noise))


def test_device_draw_and_graph_replays():
    from speech_emotion_privacy_trust_b200 import cloak_ops, wave_cloak
    torch.manual_seed(11)
    batch, x, off = _batch(seed=8)
    layer = wave_cloak.WaveCloak(1e-3, 0.05, period=1000, locs=0.01 * torch.randn(1000)).cuda()

    def noise_at(draw):                                   # the noise-only output of sept_cloak_fwd_f32 at that draw
        counter = torch.tensor([draw], dtype=torch.int64, device="cuda")
        _, _, nz = cloak_ops.cloak_forward_raw(None, layer.locs.detach(), layer.rhos.detach(), None, None,
                                               torch.initial_seed(), 0, wave_cloak.EPS_STD, 1e-3, 0.05, want_noise=True,
                                               draw=counter)
        return nz.cpu().numpy()

    y0 = layer(batch).wav.detach().cpu().numpy()
    y1 = layer(batch).wav.detach().cpu().numpy()
    assert np.array_equal(y0, _expected(x, off, noise_at(0)))
    assert np.array_equal(y1, _expected(x, off, noise_at(1)))
    assert not np.array_equal(y0, y1)
    assert int(layer._draws) == 2
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static = layer(batch).wav
    assert int(layer._draws) == 2                         # capture runs nothing
    seen = []
    for draw in (2, 3):
        graph.replay()
        torch.cuda.synchronize()
        got = static.detach().cpu().numpy()
        assert np.array_equal(got, _expected(x, off, noise_at(draw))), draw
        seen.append(got)
    assert not np.array_equal(seen[0], seen[1])


# ---- end to end -------------------------------------------------------------------------------------------------
E2E_LENGTHS = (16000, 40000, 56001, 24003, 33000)
E2E_SPK = ["a", "b", "a", "b", "a"]
MN, MX, LAM = 1e-4, 2e-2, 0.5


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
    eps = 0.1 * torch.randn(32000, generator=g)
    We, Wg = torch.randn(4, 128, generator=g) / 8, torch.randn(2, 128, generator=g) / 8
    return waves, locs0, rhos0, eps, We, Wg


def _e2e_gpu(layer, waves, We, Wg, labels=None):
    """(emotion loss, gender loss, labels): wave cloak -> log-mel -> statistics -> windows -> mean over time ->
    a linear emotion head and, through gradient reversal, a linear gender head."""
    from speech_emotion_privacy_trust_b200 import cloak_ops, extraction
    from speech_emotion_privacy_trust_b200 import normalization as nz
    batch = extraction.RaggedAudio.from_list(waves, device="cuda")
    feats, lay = extraction.logmel_grad(layer(batch))
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
    noise = locs + ((1.0 + torch.tanh(rhos)) / 2 * (MX - MN) + MN) * eps.to(dtype)
    xs = [torch.from_numpy(np.asarray(w, np.float32)).to(dtype) + noise[torch.arange(len(w)) % 32000] for w in waves]
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
    layer = wave_cloak.WaveCloak(MN, MX, period=32000, locs=locs0).cuda()
    with torch.no_grad():
        layer.rhos.copy_(rhos0)
    layer.external_eps = eps.cuda()
    le, lg, labels = _e2e_gpu(layer, waves, We, Wg)
    (le + lg).backward()
    got = layer.locs.grad.double().cpu().numpy(), layer.rhos.grad.double().cpu().numpy()
    ref64 = _e2e_oracle(waves, locs0, rhos0, eps, We, Wg, labels, torch.float64)
    ref32 = _e2e_oracle(waves, locs0, rhos0, eps, We, Wg, labels, torch.float32)
    for a, b, c in zip(got, ref64, ref32):
        assert _rel(a, b) < max(1e-5, 4 * _rel(c, b)), (_rel(a, b), _rel(c, b))
    # SGD on mu, rho descends J = emotion loss - lambda * gender loss (the gradient reversal's objective)
    opt = torch.optim.SGD(layer.parameters(), lr=1e-3 / float(max(layer.locs.grad.abs().max(), layer.rhos.grad.abs().max())))
    js = []
    for _ in range(4):
        layer.zero_grad()
        le, lg, _ = _e2e_gpu(layer, waves, We, Wg, labels)
        js.append(float(le.detach()) - LAM * float(lg.detach()))
        (le + lg).backward()
        opt.step()
    assert js[-1] < js[0], js


# ---- data parallel: two gloo ranks on one device ------------------------------------------------------------------
DP_LENGTHS = (16000, 40000, 56001, 24003, 33000, 47005, 20000, 36002)
DP_SPK = ["a", "b", "a", "b", "a", "c", "c", "b"]


def _dp_grads(mine, stats_fn):
    """Summed-loss gradient of (locs, rhos) over the utterances `mine`: device-drawn eps (seed 0, first draw),
    wave cloak -> logmel_grad -> statistics -> normalized_windows_grad -> sum(W * windows)."""
    from speech_emotion_privacy_trust_b200 import extraction, parallel, synth, wave_cloak
    from speech_emotion_privacy_trust_b200 import normalization as nz
    rng = np.random.default_rng(31)
    waves = [synth.speech_shaped(n, rng) for n in DP_LENGTHS]
    torch.manual_seed(0)
    layer = wave_cloak.WaveCloak(MN, MX, period=32000, locs=1e-3 * torch.randn(32000)).cuda()
    flat = parallel.FlatGradients(layer.parameters())
    batch = extraction.RaggedAudio.from_list([waves[u] for u in mine], device="cuda")
    feats, lay = extraction.logmel_grad(layer(batch))
    st = stats_fn(feats, lay, [DP_SPK[u] for u in mine])
    wu, wt = nz.window_table(lay)
    win = nz.normalized_windows_grad(feats, lay, st, wu, wt)
    W = torch.from_numpy(np.stack([np.random.default_rng(1000 * mine[int(i)] + int(t0)).standard_normal((200, 128))
                                   for i, t0 in zip(wu, wt)]).astype(np.float32)).cuda()
    (win * W.view_as(win)).sum().backward()
    flat.allreduce(average=False)
    return layer.locs.grad.double().cpu().numpy(), layer.rhos.grad.double().cpu().numpy()


def _dp_worker(rank, world, init_file, out_dir):
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", init_method=f"file://{init_file}", rank=rank, world_size=world,
                            timeout=timedelta(seconds=120))
    try:
        from speech_emotion_privacy_trust_b200 import normalization as nz
        mine = [u for u in range(len(DP_LENGTHS)) if u % world == rank]
        dl, dr = _dp_grads(mine, lambda f, lay, s: nz.speaker_stats_distributed_grad(f, lay, s, ["a", "b", "c"]))
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), dl=dl, dr=dr)
    finally:
        dist.destroy_process_group()


def test_two_gloo_ranks_match_one_gpu(tmp_path):
    from speech_emotion_privacy_trust_b200 import normalization as nz
    mp.spawn(_dp_worker, args=(2, str(tmp_path / "store"), str(tmp_path)), nprocs=2, join=True)
    res = [np.load(tmp_path / f"r{r}.npz") for r in range(2)]
    for k in ("dl", "dr"):
        assert np.array_equal(res[0][k], res[1][k])                 # every rank holds the all-reduced gradient
    dl, dr = _dp_grads(list(range(len(DP_LENGTHS))), lambda f, lay, s: nz.speaker_stats_grad(f, lay, s))
    assert _rel(res[0]["dl"], dl) < 1e-5, _rel(res[0]["dl"], dl)
    assert _rel(res[0]["dr"], dr) < 1e-5, _rel(res[0]["dr"], dr)
