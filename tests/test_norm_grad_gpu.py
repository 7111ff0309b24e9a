"""Gradient through the per-speaker statistics and normalised training windows (normalization.speaker_stats_grad /
normalized_windows_grad / normalize_grad; sept_speaker_stats_bwd_ties_i32 + _frames_f32, sept_normalize_bwd_f32) on the
GPU, against the float64 torch autograd oracle (oracle/norm_autograd.py) on the same fp32 features.  Metric:
rel = |g - g64| / |g64| per utterance, with a random normal upstream gradient."""
import numpy as np
import pytest
import torch

from oracle import norm_autograd as na

pytestmark = pytest.mark.gpu

FRAMES = [37, 199, 200, 249, 250, 251, 1001, 120, 260, 330]
SPK = ["a", "b", "a", "b", "c", "a", "b", "c", "a", "b"]
WHOLE = [False, False, False, False, True, False, False, False, False, True]


def _layout(feats):
    from speech_emotion_privacy_trust_b200.extraction import Layout
    fo = np.concatenate([[0], np.cumsum([len(f) for f in feats])]).astype(np.int64)
    return Layout(fo, torch.from_numpy(fo).cuda(), torch.zeros(len(fo), dtype=torch.int32, device="cuda"))


def _rel(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def _feats(F, seed=0, frames=FRAMES):
    rng = np.random.default_rng(seed)
    return [(rng.standard_normal((T, F)) * 9 - 40).astype(np.float32) for T in frames]


def _gpu(feats, spk, whole, wu, wt, mode, G, stats_grad=True):
    """feat.grad of sum(G * normalized_windows_grad(...)) with statistics from speaker_stats_grad (or detached)."""
    from speech_emotion_privacy_trust_b200 import normalization as nz
    lay = _layout(feats)
    feat = torch.from_numpy(np.concatenate(feats)).cuda().requires_grad_(True)
    st = nz.speaker_stats_grad(feat, lay, spk, whole) if stats_grad else nz.speaker_stats(feat.detach(), lay, spk, whole)
    win = nz.normalized_windows_grad(feat, lay, st, wu, wt, mode)
    win.backward(torch.from_numpy(G).cuda().view_as(win))
    g = feat.grad.cpu().numpy().astype(np.float64)
    fo = lay.frame_off_host
    return [g[fo[u]:fo[u + 1]] for u in range(len(feats))], st


def _oracle(feats, spk, whole, wu, wt, mode, G, dtype=torch.float64, detach_stats=False):
    xs = [torch.from_numpy(f).to(dtype).requires_grad_(True) for f in feats]
    speakers, stats = na.speaker_stats(xs, spk, whole)
    if detach_stats:
        stats = stats.detach().requires_grad_(True)
    row = {s: i for i, s in enumerate(speakers)}
    win = na.normalized_windows(xs, stats, [row[s] for s in spk], wu, wt, mode)
    (win * torch.from_numpy(G).to(dtype)).sum().backward()
    return [x.grad.double().numpy() for x in xs], (stats.grad.double().numpy() if detach_stats else None)


def _table(feats):
    from speech_emotion_privacy_trust_b200 import normalization as nz
    return nz.window_table(_layout(feats))


def test_forward_bit_identical_golden(golden_norm):
    from speech_emotion_privacy_trust_b200 import normalization as nz
    g = golden_norm
    feats = [g[f"feat{u}"] for u in range(int(g["n_utts"]))]
    spk = [str(s) for s in g["speakers"]]
    whole = [s == "s2" for s in spk]
    lay = _layout(feats)
    feat = torch.from_numpy(np.concatenate(feats)).cuda()
    st = nz.speaker_stats(feat, lay, spk, whole)
    stg = nz.speaker_stats_grad(feat.clone().requires_grad_(True), lay, spk, whole)
    assert stg.stats.grad_fn is not None and torch.equal(stg.stats.detach(), st.stats)
    assert stg.as_dict().keys() == st.as_dict().keys()
    wu, wt = nz.window_table(lay)
    for mode in ("znorm", "min_max"):
        a = nz.normalized_windows(feat, lay, st, wu, wt, mode)
        b = nz.normalized_windows_grad(feat, lay, stg, wu, wt, mode)
        assert b.grad_fn is not None and torch.equal(a, b.detach())
        assert torch.equal(nz.normalize(feat, lay, st, mode), nz.normalize_grad(feat, lay, stg, mode).detach())


@pytest.mark.parametrize("mode", ["znorm", "min_max"])
@pytest.mark.parametrize("F", [128, 37])
def test_windows_gradient_vs_oracle(mode, F):
    feats = _feats(F, seed=1)
    wu, wt = _table(feats)
    G = np.random.default_rng(2).standard_normal((len(wu), 200, F)).astype(np.float32)
    g, _ = _gpu(feats, SPK, WHOLE, wu, wt, mode, G)
    ref, _ = _oracle(feats, SPK, WHOLE, wu, wt, mode, G)
    for u in range(len(feats)):
        assert _rel(g[u], ref[u]) < 1e-5, (u, _rel(g[u], ref[u]))
    assert np.all(g[3][200:249] == 0)          # T = 249: frames 200..248 lie in no training window


@pytest.mark.parametrize("mode", ["znorm", "min_max"])
def test_frames_gradient_vs_oracle(mode):
    from speech_emotion_privacy_trust_b200 import normalization as nz
    feats = _feats(128, seed=3)
    lay = _layout(feats)
    feat = torch.from_numpy(np.concatenate(feats)).cuda().requires_grad_(True)
    st = nz.speaker_stats_grad(feat, lay, SPK, WHOLE)
    z = nz.normalize_grad(feat, lay, st, mode)
    G = np.random.default_rng(4).standard_normal(z.shape).astype(np.float32)
    z.backward(torch.from_numpy(G).cuda())
    g = feat.grad.cpu().numpy().astype(np.float64)
    xs = [torch.from_numpy(f).double().requires_grad_(True) for f in feats]
    speakers, stats = na.speaker_stats(xs, SPK, WHOLE)
    row = {s: i for i, s in enumerate(speakers)}
    zr = torch.cat(na.normalize_frames(xs, stats, [row[s] for s in SPK], mode))
    (zr * torch.from_numpy(G).double()).sum().backward()
    fo = lay.frame_off_host
    for u in range(len(feats)):
        assert _rel(g[fo[u]:fo[u + 1]], xs[u].grad.numpy()) < 1e-5, u


@pytest.mark.parametrize("mode", ["znorm", "min_max"])
def test_detached_statistics_and_dstats(mode):
    from speech_emotion_privacy_trust_b200 import normalization as nz
    feats = _feats(128, seed=5)
    wu, wt = _table(feats)
    G = np.random.default_rng(6).standard_normal((len(wu), 200, 128)).astype(np.float32)
    g, st = _gpu(feats, SPK, WHOLE, wu, wt, mode, G, stats_grad=False)
    assert st.stats.grad is None and not st.stats.requires_grad
    ref, _ = _oracle(feats, SPK, WHOLE, wu, wt, mode, G, detach_stats=True)
    for u in range(len(feats)):
        assert _rel(g[u], ref[u]) < 1e-5, u
    # statistics as a leaf: d stats against the oracle's, within 1e-5 or 4x torch fp32's own error (S1, S2 cancel)
    lay = _layout(feats)
    feat = torch.from_numpy(np.concatenate(feats)).cuda()
    st = nz.speaker_stats(feat, lay, SPK, WHOLE)
    st.stats.requires_grad_(True)
    win = nz.normalized_windows_grad(feat, lay, st, wu, wt, mode)
    win.backward(torch.from_numpy(G).cuda().view_as(win))
    ds = st.stats.grad.cpu().numpy().astype(np.float64)
    _, ds64 = _oracle(feats, SPK, WHOLE, wu, wt, mode, G, detach_stats=True)
    _, ds32 = _oracle(feats, SPK, WHOLE, wu, wt, mode, G, dtype=torch.float32, detach_stats=True)
    assert np.all(ds[:, 0] == 0)
    rows = [0, 1] if mode == "znorm" else [2, 3]            # oracle rows: mean, std, min, max
    for s in range(ds.shape[0]):
        got, want, t32 = ds[s, 1:][rows], ds64[s][rows], ds32[s][rows]
        assert _rel(got, want) < max(1e-5, 4 * _rel(t32, want)), (s, _rel(got, want), _rel(t32, want))


def test_arbitrary_window_tables():
    feats = _feats(128, seed=7)
    wu, wt = _table(feats)
    rng = np.random.default_rng(8)
    G = rng.standard_normal((len(wu), 200, 128)).astype(np.float32)
    g, _ = _gpu(feats, SPK, WHOLE, wu, wt, "znorm", G)
    perm = rng.permutation(len(wu))
    gp, _ = _gpu(feats, SPK, WHOLE, wu[perm], wt[perm], "znorm", G[perm])
    for u in range(len(feats)):                      # frames sum their windows by start: a shuffled table is bit-identical
        assert np.array_equal(g[u], gp[u]), u
    sub = np.sort(rng.choice(len(wu), len(wu) // 2, replace=False))[::-1]
    dup = np.concatenate([sub, sub[:3]])             # a subset in reverse order, three windows twice
    wu2 = np.concatenate([wu[dup], [6, 8]]).astype(np.int32)
    wt2 = np.concatenate([wt[dup], [975, 70]]).astype(np.int32)   # a window past the end of utterance 6, one off the grid
    G2 = rng.standard_normal((len(wu2), 200, 128)).astype(np.float32)
    for mode in ("znorm", "min_max"):
        g2, _ = _gpu(feats, SPK, WHOLE, wu2, wt2, mode, G2)
        ref, _ = _oracle(feats, SPK, WHOLE, wu2, wt2, mode, G2)
        for u in range(len(feats)):
            assert _rel(g2[u], ref[u]) < 1e-5, (mode, u)


def test_tied_minima_and_maxima():
    rng = np.random.default_rng(9)
    feats = [np.round(rng.standard_normal((T, 128)) * 2).astype(np.float32) for T in FRAMES]   # values in a few levels
    wu, wt = _table(feats)
    G = rng.standard_normal((len(wu), 200, 128)).astype(np.float32)
    g, _ = _gpu(feats, SPK, WHOLE, wu, wt, "min_max", G)
    ref, _ = _oracle(feats, SPK, WHOLE, wu, wt, "min_max", G)
    for u in range(len(feats)):
        assert _rel(g[u], ref[u]) < 1e-5, u


def test_constant_feature_column():
    from speech_emotion_privacy_trust_b200 import normalization as nz
    feats = _feats(128, seed=10)
    for f in feats:
        f[:, 5] = -100.0                                     # digital silence in one band
    lay = _layout(feats)
    feat = torch.from_numpy(np.concatenate(feats)).cuda().requires_grad_(True)
    st = nz.speaker_stats_grad(feat, lay, SPK, WHOLE)
    assert torch.all(st.stats[:, 2, 5] == 0)
    W = torch.randn(st.stats.shape, device="cuda")
    W[:, 0] = 0
    (st.stats * W).sum().backward()
    g = feat.grad
    assert torch.isfinite(g).all()
    xs = [torch.from_numpy(f).double().requires_grad_(True) for f in feats]
    speakers, stats = na.speaker_stats(xs, SPK, WHOLE)
    (stats * W[:, 1:].double().cpu()).sum().backward()
    ref = torch.cat([x.grad for x in xs]).numpy()
    assert _rel(g.cpu().numpy().astype(np.float64), ref) < 1e-5
    # the std path alone gives exactly nothing to the constant column
    feat.grad = None
    st = nz.speaker_stats_grad(feat, lay, SPK, WHOLE)
    st.stats[:, 2].sum().backward()
    assert torch.all(feat.grad[:, 5] == 0) and torch.isfinite(feat.grad).all()
    wu, wt = _table(feats)
    G = np.random.default_rng(11).standard_normal((len(wu), 200, 128)).astype(np.float32)
    g, _ = _gpu(feats, SPK, WHOLE, wu, wt, "znorm", G)
    assert all(np.isfinite(x).all() for x in g)


def test_deterministic_and_speaker_invariant():
    feats = _feats(128, seed=12)
    wu, wt = _table(feats)
    G = np.random.default_rng(13).standard_normal((len(wu), 200, 128)).astype(np.float32)
    a, _ = _gpu(feats, SPK, WHOLE, wu, wt, "znorm", G)
    b, _ = _gpu(feats, SPK, WHOLE, wu, wt, "znorm", G)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    # speaker "a" alone against "a" among the others: its utterances' gradients are bit-identical
    keep = [u for u, s in enumerate(SPK) if s == "a"]
    sel = np.isin(wu, keep)
    remap = {u: i for i, u in enumerate(keep)}
    wua = np.array([remap[u] for u in wu[sel]], dtype=np.int32)
    alone, _ = _gpu([feats[u] for u in keep], ["a"] * len(keep), [WHOLE[u] for u in keep], wua, wt[sel], "znorm", G[sel])
    Gz = G.copy()
    Gz[~sel] = 0                                      # the others' windows carry no gradient into speaker "a"
    mixed, _ = _gpu(feats, SPK, WHOLE, wu, wt, "znorm", Gz)
    for i, u in enumerate(keep):
        assert np.array_equal(alone[i], mixed[u]), u


def test_bad_window_table_raises():
    from speech_emotion_privacy_trust_b200 import normalization as nz
    feats = _feats(16, seed=14, frames=[220, 90])
    lay = _layout(feats)
    feat = torch.from_numpy(np.concatenate(feats)).cuda()
    st = nz.speaker_stats(feat, lay, ["a", "a"])
    with pytest.raises(ValueError):
        nz.normalized_windows_grad(feat, lay, st, np.array([0]), np.array([-1]))
    with pytest.raises(ValueError):
        nz.normalized_windows_grad(feat, lay, st, np.array([2]), np.array([0]))
    with pytest.raises(ValueError):
        nz.normalized_windows_grad(feat, lay, st, np.array([-1]), np.array([0]))


def test_end_to_end_waveform_gradient_through_cloak():
    """wav -> logmel_grad -> speaker_stats_grad -> normalized_windows_grad -> CloakNoiseFunction (eps supplied) -> loss,
    against the composed float64 oracle (and torch fp32 autograd of the same chain for scale)."""
    from oracle import logmel_autograd
    from speech_emotion_privacy_trust_b200 import cloak_ops, extraction, synth
    from speech_emotion_privacy_trust_b200 import normalization as nz
    rng = np.random.default_rng(15)
    lengths = (16000, 40000, 56000, 24000, 33000)
    spk = ["a", "b", "a", "b", "a"]
    waves = [synth.speech_shaped(n, rng) for n in lengths]
    batch = extraction.RaggedAudio.from_list(waves, device="cuda")
    wav = batch.wav.requires_grad_(True)
    locs = torch.zeros(200, 128, device="cuda", requires_grad=True)
    rhos = torch.full((200, 128), -3.0, device="cuda", requires_grad=True)
    eps = torch.randn(200, 128, device="cuda")
    feats, lay = extraction.logmel_grad(batch)
    st = nz.speaker_stats_grad(feats, lay, spk)
    wu, wt = nz.window_table(lay)
    x = nz.normalized_windows_grad(feats, lay, st, wu, wt)
    y = cloak_ops.CloakNoiseFunction.apply(x, locs, rhos, None, eps, 0, 0, 1.0, 0.01, 10.0, False, 0.0)
    W = torch.randn(y.shape, generator=torch.Generator().manual_seed(16)).cuda()
    (y * W).sum().backward()
    g = wav.grad.cpu().numpy().astype(np.float64)
    Wh = W.cpu().reshape(len(wu), 200, 128)

    def oracle(dtype):
        xs = [torch.from_numpy(np.asarray(w, np.float32)).to(dtype).requires_grad_(True) for w in waves]
        fs = [logmel_autograd.logmel_db(w, 800, 160, 128) for w in xs]
        speakers, stats = na.speaker_stats(fs, spk)
        row = {s: i for i, s in enumerate(speakers)}
        win = na.normalized_windows(fs, stats, [row[s] for s in spk], wu, wt)
        (win * Wh.to(dtype)).sum().backward()         # the cloak passes W through to its input (mask None)
        return [w.grad.double().numpy() for w in xs]

    ref, ref32 = oracle(torch.float64), oracle(torch.float32)
    off = batch.utt_off_host
    for u in range(len(waves)):
        rel, rel32 = _rel(g[off[u]:off[u + 1]], ref[u]), _rel(ref32[u], ref[u])
        assert rel < max(1e-5, 4 * rel32), (u, rel, rel32)
