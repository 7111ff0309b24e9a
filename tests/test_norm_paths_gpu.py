"""Per-speaker statistics, normalisation and their gradients (csrc/norm.cu, csrc/norm_bwd.cu) on every kernel path, against
float64 references: oracle/norm.py (statistics, frame multiplicity, windows, normalisation) and oracle/norm_autograd.py
(torch autograd).

The kernel a call takes depends on the feature width F, the utterances per speaker and pointer alignment:
  F = 128                      utt_partial128_kernel, normalize4_kernel, backward V = 4 with 8 row groups
  F = 120                      utt_partial_kernel, normalize4_kernel with 30 columns (16 threads idle)
  F = 12                       normalize4_kernel with 85 rows per pass
  F = 37, 1                    normalize_kernel, backward V = 1 with 6 and 256 row groups
  F = 129                      normalize_kernel; two passes of the feature loops (fbase) of the three per-speaker merge
                               kernels; backward V = 1 with one row group of 129 threads
  F = 302                      normalize_kernel; three fbase passes; backward V = 1 with one row group over 302 columns,
                               so threads 0..45 also take columns 256..301
  F = 1024                    normalize4_kernel with one row per pass, backward V = 4 with one row group
  F = 1028                     F / 4 > 256: normalize_kernel; backward V = 4 with one row group and 257 columns, so
                               thread 0 also takes column 256
  F = 128, 120 at storage      the same features 4 bytes off 16-byte alignment: utt_partial_kernel and normalize_kernel
  offset 1 float
Speakers hold 1, 7, 8, 9, 16, 17 and 40 utterances (the merge kernels' 8 slices take list entries s, s + 8, ...),
interleaved in utterance order.  Utterance lengths sit on the edges of the window rule, test-split (whole) utterances are
mixed in, and four window configurations run: the reference's 200 / 50, a shift that does not divide the window, a tiny
window, and a shift longer than the window (frames between two windows weigh 0 and must not reach min / max)."""
import numpy as np
import pytest
import torch

from oracle import norm as onorm
from oracle import norm_autograd as na

pytestmark = pytest.mark.gpu

FEATS = [128, 120, 12, 37, 1, 129, 302, 1024, 1028]
WINDOWS = [(200, 50), (100, 30), (7, 3), (50, 80)]
SPK_UTTS = (1, 7, 8, 9, 16, 17, 40)
MODES = ("znorm", "min_max")


def _nz():
    from speech_emotion_privacy_trust_b200 import normalization
    return normalization


def _layout(lengths):
    from speech_emotion_privacy_trust_b200.extraction import Layout
    fo = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    return Layout(fo, torch.from_numpy(fo).cuda(), torch.zeros(len(fo), dtype=torch.int32, device="cuda"))


def _edge_lengths(win, shift):
    return [1, 2, win - 1, win, win + 1, win + shift - 1, win + shift, 2 * win + 3]


def _corpus(F, win, shift, seed, counts=SPK_UTTS, n_long=2, quantise=False):
    """Utterances of speakers s0, s1, ... holding counts[i] utterances each, in shuffled utterance order; lengths cycle
    through the window rule's edges, n_long utterances have ~3000 frames; features ~ N(-40, 9^2) plus a per-utterance
    offset (rounded to multiples of 4 with `quantise`, so min / max are tied over many frames)."""
    rng = np.random.default_rng(seed)
    n = sum(counts)
    spk = [str(s) for s in np.repeat([f"s{i}" for i in range(len(counts))], counts)[rng.permutation(n)]]
    edge = _edge_lengths(win, shift)
    lengths = np.array([edge[i % len(edge)] for i in rng.permutation(n)])
    lengths[rng.choice(n, n_long, replace=False)] = 2990 + rng.integers(0, 20, n_long)
    for i, c in enumerate(counts):
        if c == 1:                                           # a lone utterance of one frame would have min == max
            lengths[spk.index(f"s{i}")] = 2 * win + 3
    whole = list(rng.random(n) < 0.25)
    feats = []
    for T in lengths:
        x = rng.standard_normal((int(T), F)) * 9 - 40 + rng.standard_normal() * 5
        feats.append((np.round(x / 4) * 4 if quantise else x).astype(np.float32))
    return feats, spk, whole


def _offset_view(feat):
    """The same values as a contiguous tensor at storage offset 1 float (4 bytes off 16-byte alignment)."""
    buf = torch.empty(feat.numel() + 1, dtype=feat.dtype, device=feat.device)
    buf[1:].copy_(feat.reshape(-1))
    view = buf[1:].view(feat.shape)
    assert view.is_contiguous() and view.data_ptr() % 16 == 4
    return view


def _bits(t):
    return t.detach().contiguous().view(torch.int32)


def _check_stats(st, feats, spk, whole, win, shift, tol, per_chain=False):
    """count exact; min / max bit-equal to the float32 extremes of the frames of nonzero weight; mean / std within tol
    of float64.  Returns the largest mean and std errors.

    per_chain: utt_partial_kernel walks each utterance's frames in one sequential float32 Welford chain per feature, and
    the rounding of the running mean (half an ulp a frame) random-walks along it: ~1e-4 at |mean| ~ 45 for a 3000-frame
    utterance, as a float32 emulation of the kernel's arithmetic gives too (numpy's own float32 reduction of the stacked
    rows, the reference's, is up to 3e-4 off on the same speakers).  So a speaker's bound grows with its longest
    utterance L: max(tol, 2^-23 |mean| sqrt(3 L)), about twice the largest error that emulation gives on this grid."""
    d = st.as_dict()
    ref = onorm.speaker_stats_f64(feats, spk, whole, win, shift)
    err_mean = err_std = 0.0
    for s in ref:
        n_ref, mn, mx, longest = 0, None, None, 0
        for u, f in enumerate(feats):
            if spk[u] != s:
                continue
            w = onorm.frame_multiplicity(len(f), whole is not None and bool(whole[u]), win, shift)
            n_ref += int(w.sum())
            longest = max(longest, len(f))
            used = f[w > 0]
            if len(used):
                mn = used.min(0) if mn is None else np.minimum(mn, used.min(0))
                mx = used.max(0) if mx is None else np.maximum(mx, used.max(0))
        assert np.all(d[s]["count"] == n_ref), (s, d[s]["count"][0], n_ref)
        assert np.array_equal(d[s]["min"], mn), s
        assert np.array_equal(d[s]["max"], mx), s
        e_mean = float(np.max(np.abs(d[s]["mean"] - ref[s]["mean"])))
        e_std = float(np.max(np.abs(d[s]["std"] - ref[s]["std"])))
        bound = max(tol, 2.0 ** -23 * float(np.max(np.abs(ref[s]["mean"]))) * np.sqrt(3 * longest)) if per_chain else tol
        assert e_mean < bound and e_std < bound, (s, longest, e_mean, e_std, bound)
        err_mean, err_std = max(err_mean, e_mean), max(err_std, e_std)
    return err_mean, err_std


def _close(z, z64):
    return np.all(np.abs(z - z64) <= 1e-5 * np.maximum(1.0, np.abs(z64)))


@pytest.mark.parametrize("win,shift", WINDOWS)
@pytest.mark.parametrize("F", FEATS)
def test_statistics_and_normalisation(F, win, shift):
    nz = _nz()
    wide = F >= 1024                                       # fewer utterances: the float64 windows stay small
    feats, spk, whole = _corpus(F, win, shift, seed=F * 1000 + win, counts=(1, 9, 17) if wide else SPK_UTTS,
                                n_long=1 if wide else 2)
    lengths = [len(f) for f in feats]
    lay = _layout(lengths)
    fo = lay.frame_off_host
    feat = torch.from_numpy(np.concatenate(feats)).cuda()
    st = nz.speaker_stats(feat, lay, spk, whole, win, shift)
    _check_stats(st, feats, spk, whole, win, shift, 2e-5, per_chain=True)

    # normalisation with the kernel's own statistics against float64 on the same statistics
    h = st.stats.cpu().numpy().astype(np.float64)
    row = {s: i for i, s in enumerate(st.speakers)}
    st64 = [{"mean": h[row[s], 1], "std": h[row[s], 2], "min": h[row[s], 3], "max": h[row[s], 4]} for s in spk]
    wu, wt = nz.window_table(lay, win_len=win, shift_len=shift)
    assert len(wu) == sum(onorm.n_windows(T, win, shift) for T in lengths)
    u_long = int(np.argmax(lengths))
    # beyond the table: a window running past the end of the longest utterance, one off the grid, one wholly past the
    # end of a short utterance (all padding), and a repeat
    extra_u = np.array([u_long, u_long, int(np.argmin(lengths)), 0], np.int32)
    extra_t = np.array([lengths[u_long] - win // 2, 1, lengths[int(np.argmin(lengths))] + 3, 0], np.int32)
    wu_all, wt_all = np.concatenate([wu, extra_u]), np.concatenate([wt, extra_t])
    views = {"aligned": feat}
    if F in (128, 120):
        views["offset"] = _offset_view(feat)
        st_off = nz.speaker_stats(views["offset"], lay, spk, whole, win, shift)
        _check_stats(st_off, feats, spk, whole, win, shift, 2e-5, per_chain=True)
        if F == 120:                                       # the same kernel on both: the same bits
            assert torch.equal(_bits(st_off.stats), _bits(st.stats))
    for mode in MODES:
        out = {k: (nz.normalize(v, lay, st, mode), nz.normalized_windows(v, lay, st, wu_all, wt_all, mode, win))
               for k, v in views.items()}
        z, zw = (t.cpu().numpy() for t in out["aligned"])
        for u, f in enumerate(feats):
            z64 = onorm.normalize(f.astype(np.float64), st64[u], mode)
            assert _close(z[fo[u]:fo[u + 1]], z64), (mode, u)
        j = 0
        for u, f in enumerate(feats):                       # the table's windows: oracle.norm.windows_of, padded first
            for w64 in onorm.windows_of(f.astype(np.float64), win, shift):
                assert wu_all[j] == u
                assert _close(zw[j, 0], onorm.normalize(w64, st64[u], mode)), (mode, u, j)
                j += 1
        for k in range(len(extra_u)):
            u, t0 = int(extra_u[k]), int(extra_t[k])
            w64 = np.zeros((win, F))
            rows = feats[u][t0:t0 + win]
            w64[:len(rows)] = rows
            assert _close(zw[j + k, 0], onorm.normalize(w64, st64[u], mode)), (mode, u, t0)
        if "offset" in out:                                 # same statistics, other kernel: identical bits
            for a, b in zip(out["aligned"], out["offset"]):
                assert torch.equal(_bits(a), _bits(b)), mode


def _rel(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def _grad_case(F, win, shift, mode, seed, quantise=False):
    """feat.grad through speaker_stats_grad -> normalized_windows_grad and -> normalize_grad against float64 autograd:
    per utterance rel < max(1e-5, 4 x the rel of the same autograd in float32)."""
    nz = _nz()
    feats, spk, whole = _corpus(F, win, shift, seed, counts=(1, 9, 3), n_long=0, quantise=quantise)
    lay = _layout([len(f) for f in feats])
    fo = lay.frame_off_host
    wu, wt = nz.window_table(lay, win_len=win, shift_len=shift)
    wu = np.concatenate([wu, [0]]).astype(np.int32)
    wt = np.concatenate([wt, [len(feats[0]) - 1]]).astype(np.int32)   # a window of one frame and win - 1 padded rows
    rng = np.random.default_rng(seed + 1)
    Gw = rng.standard_normal((len(wu), win, F)).astype(np.float32)
    Gf = rng.standard_normal((int(fo[-1]), F)).astype(np.float32)

    def gpu(frames):
        feat = torch.from_numpy(np.concatenate(feats)).cuda().requires_grad_(True)
        st = nz.speaker_stats_grad(feat, lay, spk, whole, win, shift)
        if frames:
            nz.normalize_grad(feat, lay, st, mode).backward(torch.from_numpy(Gf).cuda())
        else:
            y = nz.normalized_windows_grad(feat, lay, st, wu, wt, mode, win)
            y.backward(torch.from_numpy(Gw).cuda().view_as(y))
        g = feat.grad.cpu().numpy().astype(np.float64)
        return [g[fo[u]:fo[u + 1]] for u in range(len(feats))]

    def oracle(frames, dtype):
        xs = [torch.from_numpy(f).to(dtype).requires_grad_(True) for f in feats]
        speakers, stats = na.speaker_stats(xs, spk, whole, win, shift)
        rows = [speakers.index(s) for s in spk]
        if frames:
            y = torch.cat(na.normalize_frames(xs, stats, rows, mode))
            (y * torch.from_numpy(Gf).to(dtype)).sum().backward()
        else:
            y = na.normalized_windows(xs, stats, rows, wu, wt, mode, win)
            (y * torch.from_numpy(Gw).to(dtype)).sum().backward()
        return [x.grad.double().numpy() for x in xs]

    for frames in (False, True):
        g, ref, ref32 = gpu(frames), oracle(frames, torch.float64), oracle(frames, torch.float32)
        for u in range(len(feats)):
            rel, rel32 = _rel(g[u], ref[u]), _rel(ref32[u], ref[u])
            assert rel < max(1e-5, 4 * rel32), (frames, u, rel, rel32)


GRAD_CASES = [(F, 200, 50) for F in FEATS] + [(F, w, s) for F in (128, 37) for w, s in WINDOWS[1:]]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("F,win,shift", GRAD_CASES)
def test_gradients(F, win, shift, mode):
    _grad_case(F, win, shift, mode, seed=7 * F + win)


@pytest.mark.parametrize("F", [1028, 37])
def test_gradients_tied_extremes(F):
    _grad_case(F, 200, 50, "min_max", seed=F, quantise=True)


def test_normalisation_rejects_bad_input():
    """Every check runs before a launch."""
    nz = _nz()
    lay = _layout([5, 7])
    st = nz.SpeakerStats(["a"], torch.ones((1, 5, 8), device="cuda"), torch.zeros(2, dtype=torch.int32, device="cuda"))
    feat = torch.zeros((12, 8), device="cuda")
    calls = (lambda f: nz.normalize(f, lay, st), lambda f: nz.normalized_windows(f, lay, st, [0], [0]),
             lambda f: nz.normalize_grad(f, lay, st), lambda f: nz.normalized_windows_grad(f, lay, st, [0], [0]))
    for call in calls:
        with pytest.raises(ValueError):
            call(feat.double())
        with pytest.raises(ValueError):
            call(torch.zeros((8, 12), device="cuda").t())        # not contiguous
        with pytest.raises(ValueError):
            call(torch.zeros((12, 9), device="cuda"))            # F differs from the statistics'
        with pytest.raises(RuntimeError):
            call(feat.cpu())
    # a start whose last row t0 + 199 passes 2^31 - 1 would wrap to a negative frame index in int32, and one past 2^32
    # would wrap to a small start in the int32 cast
    bad = (([0], [-1]), ([2], [0]), ([-1], [0]), ([0, 1], [0]), ([0], [2 ** 31 - 200]), ([0], [2 ** 32 + 5]))
    for call in (nz.normalized_windows, nz.normalized_windows_grad):
        for win_utt, win_t0 in bad:
            with pytest.raises(ValueError):
                call(feat, lay, st, win_utt, win_t0)
        with pytest.raises(ValueError):
            call(feat, lay, st, [0], [0], win_len=0)
    wu, wt = nz._check_window_table([1], [2 ** 31 - 201], 2, 200)      # the last start whose rows all fit in int32
    assert wu.dtype == wt.dtype == np.int32 and wt[0] == 2 ** 31 - 201


def _device_feats(lengths, F, seed):
    """~N(-40, 9^2) features plus a per-utterance offset, made on the device."""
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    n = int(lengths.sum())
    off = torch.randn(len(lengths), generator=g, device="cuda") * 5
    feat = torch.randn((n, F), generator=g, device="cuda") * 9 - 40
    feat += off.repeat_interleave(torch.from_numpy(lengths).cuda(), output_size=n)[:, None]
    return feat


def _split(feat, lengths):
    h = feat.cpu().numpy()
    fo = np.concatenate([[0], np.cumsum(lengths)])
    return [h[fo[u]:fo[u + 1]] for u in range(len(lengths))]


def test_corpus_scale_statistics():
    """10 speakers x 500 utterances of 2-10 s (bench.py's length distribution), F = 128, interleaved speakers."""
    import bench
    nz = _nz()
    lengths = bench.corpus_lengths(5000, seed=21) // 160 + 1                  # frames at hop 160
    spk = [f"s{u % 10}" for u in range(len(lengths))]
    whole = list(np.random.default_rng(22).random(len(lengths)) < 0.1)
    feat = _device_feats(lengths, 128, 23)
    st = nz.speaker_stats(feat, _layout(lengths), spk, whole)
    err = _check_stats(st, _split(feat, lengths), spk, whole, 200, 50, 3e-5)
    print(f"\ncorpus F=128 (max {int(st.stats[:, 0, 0].max())} weighted frames a speaker): "
          f"max |mean err| {err[0]:.2e}, max |std err| {err[1]:.2e}")


def test_one_speaker_many_weighted_frames():
    """One speaker with 3000 utterances of 200-1500 frames: ~8 M weighted frames, below the 2^24 up to which the float
    count is exact."""
    nz = _nz()
    lengths = np.random.default_rng(31).integers(200, 1501, 3000).astype(np.int64)
    n_w = sum(int(onorm.frame_multiplicity(int(T)).sum()) for T in lengths)
    assert 7_000_000 < n_w < 1 << 24
    feat = _device_feats(lengths, 16, 32)
    spk = ["a"] * len(lengths)
    st = nz.speaker_stats(feat, _layout(lengths), spk)
    err = _check_stats(st, _split(feat, lengths), spk, None, 200, 50, 3e-5)
    print(f"\none speaker, {n_w} weighted frames: max |mean err| {err[0]:.2e}, max |std err| {err[1]:.2e}")
