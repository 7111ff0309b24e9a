"""The float64 autograd oracle of the per-speaker statistics and normalisation (oracle/norm_autograd.py): its forward
against the numpy restatement and the golden fixture, its gradient against finite differences, the multiplicity-weighted
split of tied minima / maxima, and the std = 0 rule."""
import numpy as np
import torch

from oracle import norm as onorm
from oracle import norm_autograd as na


def _t(feats):
    return [torch.from_numpy(np.asarray(f, np.float64)) for f in feats]


def test_forward_matches_numpy_restatement_and_golden(golden_norm):
    g = golden_norm
    n = int(g["n_utts"])
    feats = [g[f"feat{u}"] for u in range(n)]
    spk = [str(s) for s in g["speakers"]]
    whole = [s == "s2" for s in spk]
    speakers, stats = na.speaker_stats(_t(feats), spk, whole)
    ref = onorm.speaker_stats_f64(feats, spk, whole)
    for i, s in enumerate(speakers):
        for j, k in enumerate(("mean", "std", "min", "max")):
            np.testing.assert_allclose(stats[i, j].numpy(), ref[s][k], rtol=1e-9, atol=1e-9)
            assert np.max(np.abs(stats[i, j].numpy() - g[f"{s}_{k}"])) < 2e-4, (s, k)
    row = {s: i for i, s in enumerate(speakers)}
    spk_row = [row[s] for s in spk]
    wu, wt = [0, 2, 2, 5], [0, 0, 50, 0]
    win = na.normalized_windows(_t(feats), stats, spk_row, wu, wt).numpy()
    for j, (u, t0) in enumerate(zip(wu, wt)):
        want = onorm.normalize(onorm.windows_of(feats[u].astype(np.float64))[t0 // 50], ref[spk[u]])
        np.testing.assert_allclose(win[j], want, rtol=1e-9, atol=1e-9)
        gold = np.asarray(g[f"z|utt{u}_{t0 // 50}"]).reshape(-1, feats[0].shape[1])
        assert np.max(np.abs(win[j] - gold)) < 1e-4, (u, t0)
    z = na.normalize_frames(_t(feats), stats, spk_row)
    for u in (3, 6):
        gold = np.asarray(g[f"z|utt{u}_0"]).reshape(-1, feats[0].shape[1])
        assert np.max(np.abs(z[u].numpy() - gold[:len(feats[u])])) < 1e-4


def _small(seed=0):
    rng = np.random.default_rng(seed)
    frames = [7, 12, 17, 10]                                   # win_len 10, shift 4: short, 1 window, 2 windows, exact
    spk = ["a", "b", "a", "b"]
    feats = [torch.from_numpy(rng.standard_normal((T, 3))).requires_grad_(True) for T in frames]
    return feats, spk


def test_gradcheck_windows_and_frames():
    feats, spk = _small()
    whole = [False, False, False, True]
    wu, wt = [0, 1, 2, 2, 3, 2], [0, 0, 4, 0, 0, 9]         # padded rows, unsorted, a window past frame 7 of utterance 2

    for mode in ("znorm", "min_max"):
        def f_win(*xs):
            speakers, stats = na.speaker_stats(list(xs), spk, whole, 10, 4)
            row = {s: i for i, s in enumerate(speakers)}
            return na.normalized_windows(list(xs), stats, [row[s] for s in spk], wu, wt, mode, 10)

        def f_frames(*xs):
            speakers, stats = na.speaker_stats(list(xs), spk, whole, 10, 4)
            row = {s: i for i, s in enumerate(speakers)}
            return torch.cat(na.normalize_frames(list(xs), stats, [row[s] for s in spk], mode))

        assert torch.autograd.gradcheck(f_win, tuple(feats))
        assert torch.autograd.gradcheck(f_frames, tuple(feats))


def test_tied_minimum_split_by_multiplicity():
    # win_len 4, shift 2, T = 6: windows [0, 4) and [2, 6), multiplicities 1 1 2 2 1 1.  The minimum sits at frames 0
    # (one stacked row) and 2 (two stacked rows): torch.amin gives each row one third, so frame 2 gets two thirds.
    x = torch.tensor([[-3.0], [1.0], [-3.0], [2.0], [0.5], [5.0]], dtype=torch.float64, requires_grad=True)
    assert list(onorm.frame_multiplicity(6, False, 4, 2)) == [1, 1, 2, 2, 1, 1]
    _, stats = na.speaker_stats([x], ["s"], None, 4, 2)
    stats[0, 2].sum().backward()
    np.testing.assert_allclose(x.grad[:, 0].numpy(), [1 / 3, 0, 2 / 3, 0, 0, 0], rtol=0, atol=1e-15)
    x.grad = None
    _, stats = na.speaker_stats([x], ["s"], None, 4, 2)
    stats[0, 3].sum().backward()                               # the maximum sits once, at frame 5 (multiplicity 1)
    np.testing.assert_allclose(x.grad[:, 0].numpy(), [0, 0, 0, 0, 0, 1], rtol=0, atol=1e-15)


def test_zero_std_rule_gives_finite_gradient():
    rng = np.random.default_rng(3)
    x = rng.standard_normal((250, 4))
    x[:, 1] = -100.0                                           # digital silence: a constant column
    xt = torch.from_numpy(x).requires_grad_(True)
    _, stats = na.speaker_stats([xt], ["s"])
    assert stats[0, 1, 1].item() == 0.0
    stats[0, 1].sum().backward()                               # d(sum of std)/dx: column 1 takes no std path
    assert torch.isfinite(xt.grad).all()
    assert torch.all(xt.grad[:, 1] == 0)
    xt.grad = None
    _, stats = na.speaker_stats([xt], ["s"])
    win = na.normalized_windows([xt], stats, [0], [0, 0], [0, 50])
    (win * torch.from_numpy(rng.standard_normal(win.shape))).sum().backward()
    assert torch.isfinite(xt.grad).all()
