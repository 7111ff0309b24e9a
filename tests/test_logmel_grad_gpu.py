"""Waveform gradient of the log-mel features (extraction.logmel_grad / sept_logmel_bwd_f32) on the GPU, against the
float64 torch autograd oracle (oracle/logmel_autograd.py).  Metric: rel = |g - g64| / |g64| per utterance, with a
random normal upstream gradient."""
import numpy as np
import pytest
import torch

from oracle import logmel_autograd

pytestmark = pytest.mark.gpu


def _batch(waves):
    from speech_emotion_privacy_trust_b200 import extraction
    return extraction.RaggedAudio.from_list(waves, device="cuda")


def _grad(waves, n_fft, hop, n_mels, seed=0):
    """GPU gradient of every utterance and the G that produced it."""
    from speech_emotion_privacy_trust_b200 import extraction
    batch = _batch(waves)
    batch.wav.requires_grad_(True)
    feats, lay = extraction.logmel_grad(batch, n_fft=n_fft, n_mels=n_mels, hop=hop)
    G = torch.randn(feats.shape, generator=torch.Generator().manual_seed(seed)).cuda()
    feats.backward(G)
    g = batch.wav.grad.cpu().numpy().astype(np.float64)
    G = G.cpu().numpy().astype(np.float64)
    off, fo = batch.utt_off_host, lay.frame_off_host
    return [g[off[u]:off[u + 1]] for u in range(len(waves))], [G[fo[u]:fo[u + 1]] for u in range(len(waves))], batch, feats


def _rel(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def _speech(golden):
    from speech_emotion_privacy_trust_b200 import synth
    rng = np.random.default_rng(11)
    return [golden[f"wav{i}"] for i in range(5)] + [synth.speech_shaped(n, rng) for n in (16000, 40001, 7777)]


@pytest.mark.parametrize("n_fft,hop", [(400, 200), (800, 160), (1600, 160)])
def test_speech_gradient_matches_float64(golden_extraction, n_fft, hop):
    waves = _speech(golden_extraction)
    gs, Gs, _, _ = _grad(waves, n_fft, hop, 128)
    for w, g, G in zip(waves, gs, Gs):
        ref = logmel_autograd.logmel_grad(w.astype(np.float64), G, n_fft, hop, 128)
        assert _rel(g, ref) < 1e-5


@pytest.mark.parametrize("n_fft,hop", [(400, 200), (800, 160), (1600, 160)])
def test_high_dynamic_range_within_torch_fp32(golden_extraction, n_fft, hop):
    """A tone with noise 50 dB down: the gradient is dominated by bins holding fp32 rounding noise (d/dx ~ 1/|X|), so
    the yardstick is torch's own fp32 autograd on the same input."""
    rng = np.random.default_rng(5)
    t = np.arange(32000) / 16000
    tone = (0.3 * np.sin(2 * np.pi * 440 * t) + 0.3 * 10 ** (-50 / 20) * rng.standard_normal(t.size)).astype(np.float32)
    waves = [tone, golden_extraction["wav6"]]
    gs, Gs, _, _ = _grad(waves, n_fft, hop, 128)
    for w, g, G in zip(waves, gs, Gs):
        ref = logmel_autograd.logmel_grad(w.astype(np.float64), G, n_fft, hop, 128)
        r32 = logmel_autograd.logmel_grad(w, G.astype(np.float32), n_fft, hop, 128, torch.float32)
        assert _rel(g, ref) <= 4 * _rel(r32, ref), (_rel(g, ref), _rel(r32, ref))


def test_silence_and_always_zero_bands_give_exact_zero():
    """Digital silence: 0 everywhere.  n_fft 400 with 128 mels: bands 0, 3, 6, 13 hold no bin, so a G that lives only
    on them gives exactly 0."""
    from speech_emotion_privacy_trust_b200 import extraction, synth
    gs, _, _, _ = _grad([np.zeros(5000, np.float32), np.zeros(1201, np.float32)], 400, 200, 128)
    assert all(np.all(g == 0) for g in gs)
    batch = _batch([synth.speech_shaped(12000, np.random.default_rng(2))])
    batch.wav.requires_grad_(True)
    feats, _ = extraction.logmel_grad(batch, n_fft=400, n_mels=128, hop=200)
    G = torch.zeros_like(feats)
    G[:, [0, 3, 6, 13]] = torch.randn(feats.shape[0], 4, device="cuda")
    feats.backward(G)
    assert torch.all(batch.wav.grad == 0)


def test_ragged_batch_covers_edges_and_shapes():
    """About two dozen utterances: lengths just above n_fft/2 (reflection at both ends of the same frames), T not a
    multiple of the frames per item, hops 80 / 200 / 480 and 40 / 256 mels besides 128."""
    from speech_emotion_privacy_trust_b200 import synth
    rng = np.random.default_rng(21)
    for n_fft, hop, n_mels in ((400, 80, 128), (800, 200, 40), (1600, 480, 256), (800, 160, 256), (400, 200, 40)):
        lens = [n_fft // 2 + 1, n_fft // 2 + 7, n_fft + 3] + list(rng.integers(n_fft, 30000, size=5))
        waves = [synth.speech_shaped(int(n), rng) for n in lens]
        gs, Gs, _, _ = _grad(waves, n_fft, hop, n_mels, seed=n_fft + hop)
        for w, g, G in zip(waves, gs, Gs):
            ref = logmel_autograd.logmel_grad(w.astype(np.float64), G, n_fft, hop, n_mels)
            r32 = logmel_autograd.logmel_grad(w, G.astype(np.float32), n_fft, hop, n_mels, torch.float32)
            assert _rel(g, ref) < max(1e-5, 4 * _rel(r32, ref)), (n_fft, hop, n_mels, len(w), _rel(g, ref), _rel(r32, ref))


def test_forward_bit_identical_and_backward_deterministic(golden_extraction):
    from speech_emotion_privacy_trust_b200 import extraction
    waves = _speech(golden_extraction)
    for n_fft, hop in ((400, 200), (800, 160), (1600, 160)):
        batch = _batch(waves)
        plain, _ = extraction.logmel(batch, n_fft=n_fft, hop=hop)
        batch.wav.requires_grad_(True)
        feats, _ = extraction.logmel_grad(batch, n_fft=n_fft, hop=hop)
        assert feats.grad_fn is not None
        assert torch.equal(feats.detach(), plain)
        G = torch.randn_like(feats)
        g1 = torch.autograd.grad(feats, batch.wav, G, retain_graph=True)[0]
        g2 = torch.autograd.grad(feats, batch.wav, G)[0]
        assert torch.equal(g1, g2)
        # utterance 2 alone: the same bits as inside the batch
        lay = batch.layout(n_fft, hop)
        fo, off = lay.frame_off_host, batch.utt_off_host
        one = _batch([waves[2]])
        one.wav.requires_grad_(True)
        f1, _ = extraction.logmel_grad(one, n_fft=n_fft, hop=hop)
        (ga,) = torch.autograd.grad(f1, one.wav, G[fo[2]:fo[3]].contiguous())
        assert torch.equal(ga, g1[off[2]:off[3]])


def test_zero_outside_utterances():
    from speech_emotion_privacy_trust_b200 import extraction, synth
    rng = np.random.default_rng(4)
    wav = torch.zeros(20000, device="cuda")
    wav[1000:9000] = torch.from_numpy(synth.speech_shaped(8000, rng)).cuda()
    wav[9000:17000] = torch.from_numpy(synth.speech_shaped(8000, rng)).cuda()
    wav.requires_grad_(True)
    batch = extraction.RaggedAudio(wav, np.array([1000, 9000, 17000]))
    feats, _ = extraction.logmel_grad(batch)
    feats.backward(torch.randn_like(feats))
    assert torch.all(wav.grad[:1000] == 0) and torch.all(wav.grad[17000:] == 0)
    assert torch.count_nonzero(wav.grad[1000:17000]) > 15000


def test_through_cloak_and_cuda_graph():
    """logmel_grad -> frame-major rows -> CloakNoiseFunction (eps supplied) -> loss: wav.grad accumulates; forward and
    backward captured in one CUDA graph replay to the eager result."""
    from speech_emotion_privacy_trust_b200 import cloak_ops, extraction, synth
    rng = np.random.default_rng(9)
    batch = _batch([synth.speech_shaped(n, rng) for n in (16000, 24000, 9000)])
    wav = batch.wav.requires_grad_(True)
    locs = torch.zeros(200, 128, device="cuda", requires_grad=True)
    rhos = torch.full((200, 128), -3.0, device="cuda", requires_grad=True)
    eps = torch.randn(200, 128, device="cuda")
    W = torch.randn(200, 128, device="cuda")

    def step():
        feats, lay = extraction.logmel_grad(batch)
        x = feats[:200].view(1, 200, 128)
        y = cloak_ops.CloakNoiseFunction.apply(x, locs, rhos, None, eps, 0, 0, 1.0, 0.01, 10.0, False, 0.0)
        (y * W).sum().backward()

    step()
    eager = wav.grad.clone()
    assert torch.count_nonzero(eager) > 0
    wav.grad = None
    step()
    assert torch.equal(wav.grad, eager)
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
