"""Waveform gradient of the MFCC blocks (extraction.mfcc_grad / sept_mfcc_bwd_f32) on the GPU, against the float64 torch
autograd oracle (oracle/mfcc_autograd.py).  Metric: rel = |g - g64| / |g64| per utterance."""
import numpy as np
import pytest
import torch

from oracle import mfcc_autograd

pytestmark = pytest.mark.gpu

STREAMS = {"all": slice(0, 120), "x": slice(0, 40), "grad": slice(40, 80), "grad2": slice(80, 120)}


def _batch(waves):
    from speech_emotion_privacy_trust_b200 import extraction
    return extraction.RaggedAudio.from_list(waves, device="cuda")


def _grad(waves, seed=0, rows=slice(0, 120)):
    """GPU gradient of every utterance for a random normal Gbar on `rows` (zero elsewhere), and the Gbar blocks."""
    from speech_emotion_privacy_trust_b200 import extraction
    batch = _batch(waves)
    batch.wav.requires_grad_(True)
    feats, lay = extraction.mfcc_grad(batch)
    gen = torch.Generator().manual_seed(seed)
    Gs = []
    for u in range(len(waves)):
        G = torch.zeros(120, lay.frames(u))
        G[rows] = torch.randn(G[rows].shape, generator=gen)
        Gs.append(G)
    feats.backward(torch.cat([G.reshape(-1) for G in Gs]).cuda())
    g = batch.wav.grad.cpu().numpy().astype(np.float64)
    off = batch.utt_off_host
    return [g[off[u]:off[u + 1]] for u in range(len(waves))], [G.numpy().astype(np.float64) for G in Gs], batch, feats


def _rel(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def _speech(golden):
    """Golden wav1 is not here: torch's own fp32 autograd is 2-3e-5 from float64 on it (its quiet end, through the
    np.gradient edge), so it is held to the fp32 yardstick in test_floor_heavy_audio_within_torch_fp32 instead."""
    from speech_emotion_privacy_trust_b200 import synth
    rng = np.random.default_rng(11)
    return [golden[f"wav{i}"] for i in (0, 2, 3, 4)] + [synth.speech_shaped(n, rng) for n in (16000, 40001, 7777)]


def _floor_margin(w):
    """smallest |L_s - (m_s - 80)| of the float64 oracle over all streams, bins at exactly -100 dB (empty bands) aside"""
    x = torch.from_numpy(w.astype(np.float64))
    gaps = []
    for y in (x, mfcc_autograd.np_gradient(x, 1.0), mfcc_autograd.np_gradient(x, 2.0)):
        L = mfcc_autograd.logmel_db(y, 400, 200, 128)
        live = L > -100.0
        if live.any():
            gaps.append(float((L[live] - (L.amax() - 80.0)).abs().min()))
    return min(gaps)


@pytest.mark.parametrize("rows", list(STREAMS))
def test_speech_gradient_matches_float64(golden_extraction, rows):
    """Every stream on its own too, so that an error in one cannot hide behind another."""
    waves = _speech(golden_extraction)
    for w in waves:
        assert _floor_margin(w) > 1e-4                           # no bin close enough to its floor to flip sides
    gs, Gs, _, _ = _grad(waves, seed=3, rows=STREAMS[rows])
    for w, g, G in zip(waves, gs, Gs):
        ref = mfcc_autograd.mfcc_grad(w.astype(np.float64), G)
        assert _rel(g, ref) < 1e-5, (rows, len(w), _rel(g, ref))


def test_floor_heavy_audio_within_torch_fp32(golden_extraction):
    """Half an utterance scaled by 1e-4 (most of its frames under the floor), a tone with noise 90 dB down, and golden
    audio with quiet stretches: the yardstick is torch's own fp32 autograd on the same input."""
    from speech_emotion_privacy_trust_b200 import synth
    rng = np.random.default_rng(5)
    half = synth.speech_shaped(24000, rng)
    half[12000:] *= 1e-4
    t = np.arange(32000) / 16000
    tone = (0.3 * np.sin(2 * np.pi * 440 * t) + 0.3 * 10 ** (-90 / 20) * rng.standard_normal(t.size)).astype(np.float32)
    waves = [half, tone, golden_extraction["wav6"], golden_extraction["wav1"]]
    gs, Gs, _, _ = _grad(waves, seed=8)
    for w, g, G in zip(waves, gs, Gs):
        ref = mfcc_autograd.mfcc_grad(w.astype(np.float64), G)
        r32 = mfcc_autograd.mfcc_grad(w, G.astype(np.float32), torch.float32)
        assert _rel(g, ref) < max(1e-5, 4 * _rel(r32, ref)), (len(w), _rel(g, ref), _rel(r32, ref))


def test_exact_zeros():
    """Digital silence, an utterance under the 1e-10 clamp in every band, and a zero Gbar give exactly 0."""
    from speech_emotion_privacy_trust_b200 import extraction, synth
    quiet = synth.speech_shaped(6000, np.random.default_rng(3)) * np.float32(1e-6)
    gs, _, _, _ = _grad([np.zeros(5000, np.float32), np.zeros(1201, np.float32), quiet])
    assert all(np.all(g == 0) for g in gs)
    batch = _batch([synth.speech_shaped(12000, np.random.default_rng(2))])
    batch.wav.requires_grad_(True)
    feats, _ = extraction.mfcc_grad(batch)
    feats.backward(torch.zeros_like(feats))
    assert torch.all(batch.wav.grad == 0)


def test_ragged_batch_covers_edges():
    """Lengths just above n_fft/2 and around frame and item boundaries (frame counts not multiples of 8 frames per
    item) and random lengths; dwav is zero outside the utterances."""
    from speech_emotion_privacy_trust_b200 import extraction, synth
    rng = np.random.default_rng(21)
    lens = [201, 202, 203, 399, 400, 401, 999, 1000, 1001, 1599, 1600, 1601] + list(rng.integers(201, 30000, size=8))
    waves = [synth.speech_shaped(int(n), rng) for n in lens]
    gs, Gs, _, _ = _grad(waves, seed=13)
    for w, g, G in zip(waves, gs, Gs):
        ref = mfcc_autograd.mfcc_grad(w.astype(np.float64), G)
        r32 = mfcc_autograd.mfcc_grad(w, G.astype(np.float32), torch.float32)
        assert _rel(g, ref) < max(1e-5, 4 * _rel(r32, ref)), (len(w), _rel(g, ref), _rel(r32, ref))
    wav = torch.zeros(20000, device="cuda")
    wav[1000:9000] = torch.from_numpy(synth.speech_shaped(8000, rng)).cuda()
    wav[9000:17000] = torch.from_numpy(synth.speech_shaped(8000, rng)).cuda()
    wav.requires_grad_(True)
    batch = extraction.RaggedAudio(wav, np.array([1000, 9000, 17000]))
    feats, _ = extraction.mfcc_grad(batch)
    feats.backward(torch.randn_like(feats))
    assert torch.all(wav.grad[:1000] == 0) and torch.all(wav.grad[17000:] == 0)
    assert torch.count_nonzero(wav.grad[1000:17000]) > 15000


@pytest.mark.parametrize("dct", ["default", "tc"])
def test_forward_bit_identical_and_backward_deterministic(golden_extraction, monkeypatch, dct):
    from speech_emotion_privacy_trust_b200 import extraction
    if dct == "tc":
        monkeypatch.setenv("SEPT_MFCC_DCT", "tc")
    waves = _speech(golden_extraction)
    batch = _batch(waves)
    plain, _ = extraction.mfcc(batch)
    batch.wav.requires_grad_(True)
    feats, lay = extraction.mfcc_grad(batch)
    assert feats.grad_fn is not None
    assert torch.equal(feats.detach(), plain)
    G = torch.randn_like(feats)
    g1 = torch.autograd.grad(feats, batch.wav, G, retain_graph=True)[0]
    g2 = torch.autograd.grad(feats, batch.wav, G)[0]
    assert torch.equal(g1, g2)
    # utterance 2 alone: the same bits as inside the batch
    fo, off = lay.frame_off_host, batch.utt_off_host
    one = _batch([waves[2]])
    one.wav.requires_grad_(True)
    f1, _ = extraction.mfcc_grad(one)
    (ga,) = torch.autograd.grad(f1, one.wav, G[fo[2] * 120:fo[3] * 120].contiguous())
    assert torch.equal(ga, g1[off[2]:off[3]])


def test_cuda_graph_replays_eager():
    """mfcc_grad forward and backward captured in one CUDA graph replay to the eager result."""
    from speech_emotion_privacy_trust_b200 import _lib, extraction, synth
    _lib.lib().sept_init(128)
    rng = np.random.default_rng(9)
    batch = _batch([synth.speech_shaped(n, rng) for n in (16000, 24000, 9000)])
    wav = batch.wav.requires_grad_(True)
    W = torch.randn(batch.layout(400, 200).total_frames * 120, device="cuda")

    def step():
        feats, _ = extraction.mfcc_grad(batch)
        (feats * W).sum().backward()

    step()
    eager = wav.grad.clone()
    assert torch.count_nonzero(eager) > 0
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        wav.grad = None
        step()                                                   # warm-up on the capture stream
    torch.cuda.current_stream().wait_stream(s)
    wav.grad = torch.zeros_like(wav)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    wav.grad.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(wav.grad, eager)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(wav.grad, 2 * eager)                      # accumulated in place: eager + eager
