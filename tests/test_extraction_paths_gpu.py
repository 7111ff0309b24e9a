"""Log-mel extraction (sept_logmel_f32, csrc/extract.cu) and its waveform gradient (sept_logmel_bwd_f32,
csrc/extract_bwd.cu) on every kernel path the C ABI accepts, against float64: restate.power_spectrogram and
melscale_fbanks_htk for the forward (logmel_error: TOL_DB on bins within 50 dB of their frame's peak, TOL_DB_FLOOR on all
bins), oracle/logmel_autograd.py for the gradient (rel < max(1e-5, 4 rel(torch fp32)); 8 for the thousands of
utterances of a few frames, see test_many_short_utterances).

Which path a shape takes -- n_fft (R = 8 / 16 / 32), the FAST 128-band tensor-memory mel path or the shared-memory mel
rounds, the warps per CTA of the forward and of the backward's frame pass -- is asked of the library's own launch
arithmetic (tests/hostsim/launch_shape.cpp) and asserted, so a tiling change cannot move a case off the path it is meant
to reach without failing here.
  path matrix  n_fft x {128, 40, 300..512 bands} x {frame, band major} x {waveform, np.gradient stream}, ragged batches of
               interior and edge items; band-major blocks must be the frame-major rows transposed, bit for bit
  edges        n_mels 1 .. 512 around the 32-band rounds, hop 2 and hop = n_fft, forwards with 6 and 7 warps, backwards
               with 3, 4 and 8 warps; bands whose filterbank column holds no bin sit exactly at the 1e-10 clamp
  batch        NaN at every sample outside the utterances, a waveform 4 bytes off 16-byte alignment, 12000 short
               utterances, batches with fewer items than the grid has warps
  overflow     one 47-minute utterance at hop 2, band major: bands 96-127 lie more than 2^31 floats into the output
The largest errors of every class are printed at the end of the module (pytest -s)."""
import functools

import numpy as np
import pytest
import torch

from oracle import logmel_autograd, restate
from test_extraction_gpu import TOL_DB, TOL_DB_FLOOR, logmel_error
from test_extraction_paths_cpu import CLASSES, build_launch_shape, path_of

pytestmark = pytest.mark.gpu

N_FFTS = (400, 800, 1600)
HOP = {400: 200, 800: 160, 1600: 160}          # the reference's hops
WIDE = {400: 300, 800: 384, 1600: 512}         # more than 256 bands: 10, 12 and 16 shared-memory mel rounds
FPW = {400: 8, 800: 4, 1600: 2}                # frames per work item
WORST = {}                                     # class -> largest strong-bin / all-bin dB error and gradient rel


def _worst(cls, **errs):
    w = WORST.setdefault(cls, {})
    for k, v in errs.items():
        w[k] = max(w.get(k, 0.0), float(v))


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for cls, w in sorted(WORST.items()):
        print(f"\n{cls}: " + ", ".join(f"{k} {v:.3g}" for k, v in sorted(w.items())))


@pytest.fixture(scope="module")
def tool(tmp_path_factory):
    return build_launch_shape(tmp_path_factory.mktemp("launch_shape"))


def _ex():
    from speech_emotion_privacy_trust_b200 import extraction
    return extraction


def _speech(lengths, seed):
    from speech_emotion_privacy_trust_b200 import synth
    rng = np.random.default_rng(seed)
    return [synth.speech_shaped(int(n), rng) for n in lengths]


def _edge_lengths(n_fft, hop, seed, n_random=6):
    """Reflection at both ends of the same frames (n_fft/2 + 1, + 7, n_fft + 3), T just below, at and above a multiple of
    the frames per item, random lengths up to 3 s."""
    f = FPW[n_fft]
    rng = np.random.default_rng(seed)
    lens = [n_fft // 2 + 1, n_fft // 2 + 7, n_fft + 3, (5 * f - 1) * hop - 1, (5 * f - 1) * hop, 5 * f * hop]
    lens += [int(n) for n in rng.integers(n_fft, 48000, n_random)]
    return [max(n, n_fft // 2 + 1) for n in lens]


@functools.lru_cache(maxsize=None)
def _floor_db():
    """What the kernel stores for a band at the 1e-10 power clamp (digital silence): exactly -100 dB."""
    ex = _ex()
    got, _ = ex.logmel(ex.RaggedAudio.from_list([np.zeros(3000, np.float32)]), n_fft=800, n_mels=40)
    got = got.cpu().numpy()
    assert np.all(got == -100.0), got[got != -100.0][:4]
    return -100.0


def _oracle_db(w, n_fft, hop, n_mels, deriv=False):
    """(n_mels, T) float64 log-mel dB of the waveform, or of its np.gradient."""
    x = restate.waveform_gradient(w, 1.0).astype(np.float64) if deriv else np.asarray(w, np.float64)
    p = restate.power_spectrogram(x, n_fft, hop, np.float64)
    return restate.amplitude_to_db_power((p.T @ restate.melscale_fbanks_htk(n_fft // 2 + 1, n_mels)).T)


def _check_db(cls, rows, w, n_fft, hop, n_mels, deriv=False):
    """rows: the (T, n_mels) frame-major output of one utterance."""
    got = np.asarray(rows).T
    ref = _oracle_db(w, n_fft, hop, n_mels, deriv)
    assert got.shape == ref.shape, (cls, got.shape, ref.shape)
    assert np.all(np.isfinite(got)), (cls, n_fft, hop, n_mels, deriv, len(w))
    e_strong, e_all = logmel_error(got, ref)
    assert e_strong < TOL_DB and e_all < TOL_DB_FLOOR, (cls, n_fft, hop, n_mels, deriv, len(w), e_strong, e_all)
    empty = ~restate.melscale_fbanks_htk(n_fft // 2 + 1, n_mels).any(axis=0)    # bands whose triangle holds no bin
    assert np.all(got[empty] == _floor_db()), (cls, n_fft, hop, n_mels)
    _worst(cls, db_strong=e_strong, db_all=e_all)


def _rel(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def _check_grad(cls, g, w, G, n_fft, hop, n_mels, factor=4):
    ref = logmel_autograd.logmel_grad(np.asarray(w, np.float64), G, n_fft, hop, n_mels)
    r32 = logmel_autograd.logmel_grad(w, G.astype(np.float32), n_fft, hop, n_mels, torch.float32)
    rel, rel32 = _rel(g, ref), _rel(r32, ref)
    assert np.all(np.isfinite(g)) and rel < max(1e-5, factor * rel32), (cls, n_fft, hop, n_mels, len(w), rel, rel32)
    _worst(cls, grad_rel=rel)


def _grad(batch, n_fft, hop, n_mels, seed=0):
    """(dwav of the whole buffer, G, layout, features) of logmel_grad with a normal upstream gradient G."""
    batch.wav.grad = None
    batch.wav.requires_grad_(True)
    feats, lay = _ex().logmel_grad(batch, n_fft=n_fft, n_mels=n_mels, hop=hop)
    G = torch.randn(feats.shape, generator=torch.Generator().manual_seed(seed)).cuda()
    feats.backward(G)
    return batch.wav.grad.cpu().numpy().astype(np.float64), G.cpu().numpy().astype(np.float64), lay, feats.detach()


def _forward_all(cls, batch, waves, n_fft, hop, n_mels, utts=None, derivs=(False, True)):
    """Frame- and band-major launches of each stream: band-major blocks == frame-major rows transposed, bit for bit, and
    the frame-major rows of utterances `utts` (default all) against float64."""
    ex = _ex()
    utts = range(batch.n_utts) if utts is None else utts
    for deriv in derivs:
        fm, lay = ex.logmel(batch, n_fft=n_fft, n_mels=n_mels, hop=hop, deriv=deriv)
        bm, _ = ex.logmel(batch, n_fft=n_fft, n_mels=n_mels, hop=hop, deriv=deriv, band_major=True)
        fm, bm, fo = fm.cpu().numpy(), bm.cpu().numpy(), lay.frame_off_host
        for u, w in zip(utts, waves):
            rows = fm[fo[u]:fo[u + 1]]
            assert np.array_equal(bm[fo[u] * n_mels:fo[u + 1] * n_mels].reshape(n_mels, -1), rows.T), (cls, n_mels, deriv, u)
            _check_db(cls, rows, w, n_fft, hop, n_mels, deriv)


def _backward_all(cls, batch, waves, n_fft, hop, n_mels, utts=None, seed=0):
    utts = range(batch.n_utts) if utts is None else utts
    g, G, lay, _ = _grad(batch, n_fft, hop, n_mels, seed)
    off, fo = batch.utt_off_host, lay.frame_off_host
    for u, w in zip(utts, waves):
        _check_grad(cls, g[off[u]:off[u + 1]], w, G[fo[u]:fo[u + 1]], n_fft, hop, n_mels)
    return g


# ---- the path matrix ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_fft", N_FFTS)
def test_path_matrix(tool, n_fft):
    """Both mel paths (FAST 128 bands; the shared-memory rounds at 40 bands and at 300..512 bands, which no other test
    reaches) x both layouts x both streams, and the backward of each band count."""
    hop = HOP[n_fft]
    waves = _speech(_edge_lengths(n_fft, hop, seed=n_fft), seed=n_fft + 1)
    batch = _ex().RaggedAudio.from_list(waves)
    for n_mels, fast in ((128, 1), (40, 0), (WIDE[n_fft], 0)):
        assert path_of(tool, n_fft, hop, n_mels) == CLASSES[(n_fft, hop, n_mels)] and CLASSES[(n_fft, hop, n_mels)][0] == fast
        _forward_all(f"path matrix, n_fft {n_fft}", batch, waves, n_fft, hop, n_mels)
        _backward_all(f"path matrix, n_fft {n_fft}", batch, waves, n_fft, hop, n_mels, seed=n_mels)


# ---- edges of the accepted space ---------------------------------------------------------------------------------
@pytest.mark.parametrize("n_fft", N_FFTS)
def test_mel_count_edges(tool, n_fft):
    """1 band (a round of width 1), 31 / 32 / 33 (one round, two rounds), 255 .. 257, 511 / 512 (16 rounds); at 300 and
    more bands many filterbank columns hold no bin (190 of 512 at n_fft 400) and must sit at the clamp."""
    hop = HOP[n_fft]
    waves = _speech([n_fft // 2 + 1, n_fft + 3, 9 * FPW[n_fft] * hop + 1, 16000], seed=3 * n_fft)
    batch = _ex().RaggedAudio.from_list(waves)
    for n_mels in (1, 31, 32, 33, 255, 256, 257, 511, 512):
        fast, fwd, bwd = path_of(tool, n_fft, hop, n_mels)
        assert fast == 0 and fwd > 0 and bwd > 0
        _forward_all("n_mels 1..512", batch, waves, n_fft, hop, n_mels, derivs=(False,))
    if n_fft == 400:                                              # the clamp check above is not vacuous
        assert (~restate.melscale_fbanks_htk(201, 512).any(axis=0)).sum() == 190


@pytest.mark.parametrize("n_fft", N_FFTS)
def test_hop_edges(tool, n_fft):
    """hop 2 (the smallest accepted: every item's frames overlap almost entirely) and hop = n_fft (no overlap)."""
    for hop in (2, n_fft):
        lens = [n_fft // 2 + 1, n_fft // 2 + 7, n_fft + 3, 2345] if hop == 2 else _edge_lengths(n_fft, hop, seed=hop)
        waves = _speech(lens, seed=n_fft + hop)
        batch = _ex().RaggedAudio.from_list(waves)
        for n_mels in (128, 40):
            assert path_of(tool, n_fft, hop, n_mels)[0] == (n_mels == 128)
            _forward_all("hop 2 / hop n_fft", batch, waves, n_fft, hop, n_mels)


@pytest.mark.parametrize("shape", [(400, 390, 512), (800, 694, 40), (1600, 1498, 128), (1600, 838, 33)])
def test_forward_with_fewer_than_8_warps(tool, shape):
    """Forwards whose warp tiles leave room for only 7 (6) warps per CTA, at every n_fft and on the FAST path."""
    n_fft, hop, n_mels = shape
    assert path_of(tool, *shape) == CLASSES[shape] and CLASSES[shape][1] < 8
    waves = _speech(_edge_lengths(n_fft, hop, seed=hop), seed=hop + 1)
    batch = _ex().RaggedAudio.from_list(waves)
    _forward_all("forward < 8 warps", batch, waves, n_fft, hop, n_mels)
    _backward_all("forward < 8 warps", batch, waves, n_fft, hop, n_mels)


@pytest.mark.parametrize("shape", [(400, 200, 512), (400, 390, 512), (800, 776, 257), (400, 2, 1), (800, 2, 1), (1600, 2, 1),
                                   (400, 400, 128), (800, 800, 128), (1600, 1600, 128)])
def test_backward_edges(tool, shape):
    """Backward frame passes with 3 warps (512 bands at n_fft 400), 4 (257 bands at hop 776), 8 (one band at hop 2, short
    utterances) and at hop = n_fft."""
    n_fft, hop, n_mels = shape
    assert path_of(tool, *shape) == CLASSES[shape]
    lens = [n_fft // 2 + 1, n_fft // 2 + 7, n_fft + 3, 3001] if hop == 2 else _edge_lengths(n_fft, hop, seed=hop + 5)
    waves = _speech(lens, seed=n_fft * hop + n_mels)
    batch = _ex().RaggedAudio.from_list(waves)
    _backward_all("backward edges", batch, waves, n_fft, hop, n_mels, seed=hop)
    _forward_all("backward edges", batch, waves, n_fft, hop, n_mels, derivs=(False,))


# ---- batch structure ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_fft", N_FFTS)
def test_nan_outside_utterances(n_fft):
    """NaN at every sample outside the utterances: 3 in front (utt_off[0] = 3), 1-5 behind, and between neighbours NaN
    utterances of the shortest legal lengths (the offsets put utterances back to back, so a gap inside the batch is an
    utterance of its own).  A read outside an utterance -- staging, reflection, the np.gradient stream's halo -- would
    poison an output or a gradient.  dwav stays exactly 0 outside the utterances."""
    ex = _ex()
    hop = HOP[n_fft]
    rng = np.random.default_rng(n_fft + 7)
    waves = _speech(_edge_lengths(n_fft, hop, seed=n_fft + 8, n_random=4), seed=n_fft + 9)
    parts, off, real = [np.full(3, np.nan, np.float32)], [3], []
    for i, w in enumerate(waves):
        if i:
            gap = np.full(n_fft // 2 + int(rng.integers(1, 6)), np.nan, np.float32)
            parts.append(gap)
            off.append(off[-1] + len(gap))
        real.append(len(off) - 1)
        parts.append(w)
        off.append(off[-1] + len(w))
    parts.append(np.full(int(rng.integers(1, 6)), np.nan, np.float32))
    wav = torch.from_numpy(np.concatenate(parts)).cuda()
    batch = ex.RaggedAudio(wav, np.array(off))
    for n_mels in (128, 40):
        _forward_all("NaN outside utterances", batch, waves, n_fft, hop, n_mels, utts=real)
    g = _backward_all("NaN outside utterances", batch, waves, n_fft, hop, 128, utts=real)
    assert np.all(g[:3] == 0) and np.all(g[off[-1]:] == 0)


def _offset_copy(t):
    """The same values as a contiguous tensor at storage offset 1 float (4 bytes off 16-byte alignment)."""
    buf = torch.zeros(t.numel() + 1, dtype=t.dtype, device=t.device)
    buf[1:].copy_(t)
    view = buf[1:]
    assert view.is_contiguous() and view.data_ptr() % 16 == 4
    return view


def _bwd_raw(batch, n_fft, hop, n_mels, G, dwav):
    """sept_logmel_bwd_f32 straight from the C ABI, so that dwav can be any buffer."""
    from speech_emotion_privacy_trust_b200 import _lib
    lay = batch.layout(n_fft, hop)
    ws = _lib.workspace(_lib.lib().sept_logmel_bwd_workspace_bytes(n_fft, hop, lay.n_items), batch.wav.device)
    _lib.launch("sept_logmel_bwd_f32", batch.wav, batch.utt_off, lay.frame_off, lay.item_off, batch.n_utts, lay.n_items,
                n_fft, hop, n_mels, G, ws, dwav, device=batch.wav.device)


@pytest.mark.parametrize("n_fft", N_FFTS)
def test_misaligned_waveform(n_fft):
    """wav (and dwav) 4 bytes off 16-byte alignment: the asynchronous staging copies, reflection and the gather give the
    aligned copy's bits."""
    ex = _ex()
    hop = HOP[n_fft]
    waves = _speech(_edge_lengths(n_fft, hop, seed=n_fft + 11), seed=n_fft + 12)
    aligned = ex.RaggedAudio.from_list(waves)
    shifted = ex.RaggedAudio(_offset_copy(aligned.wav), aligned.utt_off_host)
    for n_mels in (128, 40):
        for deriv in (False, True):
            for band_major in (False, True):
                a, _ = ex.logmel(aligned, n_fft=n_fft, n_mels=n_mels, hop=hop, deriv=deriv, band_major=band_major)
                b, lay = ex.logmel(shifted, n_fft=n_fft, n_mels=n_mels, hop=hop, deriv=deriv, band_major=band_major)
                assert torch.equal(a, b), (n_fft, n_mels, deriv, band_major)
        fo = lay.frame_off_host
        fm, _ = ex.logmel(shifted, n_fft=n_fft, n_mels=n_mels, hop=hop)
        fm = fm.cpu().numpy()
        for u, w in enumerate(waves):
            _check_db("misaligned waveform", fm[fo[u]:fo[u + 1]], w, n_fft, hop, n_mels)
        G = torch.randn((lay.total_frames, n_mels), generator=torch.Generator().manual_seed(n_mels)).cuda()
        da = torch.zeros_like(aligned.wav)
        db = _offset_copy(torch.zeros_like(aligned.wav))
        _bwd_raw(aligned, n_fft, hop, n_mels, G, da)
        _bwd_raw(shifted, n_fft, hop, n_mels, G, db)
        assert torch.equal(da, db), (n_fft, n_mels)
        g, Gh, off = db.cpu().numpy().astype(np.float64), G.cpu().numpy().astype(np.float64), aligned.utt_off_host
        for u, w in enumerate(waves):
            _check_grad("misaligned waveform", g[off[u]:off[u + 1]], w, Gh[fo[u]:fo[u + 1]], n_fft, hop, n_mels)


@pytest.mark.parametrize("n_fft", N_FFTS)
def test_many_short_utterances(n_fft):
    """12000 utterances of n_fft/2 + 1 .. 2 n_fft samples and three long ones: a CTA's item range (the grid has one CTA
    per SM) spans about 80 utterances, and a warp walks from one utterance into the next many times.  Every 97th
    utterance, the first, the last and the long ones against float64; four alone against their bits inside the batch."""
    ex = _ex()
    hop = HOP[n_fft]
    rng = np.random.default_rng(n_fft + 13)
    lens = rng.integers(n_fft // 2 + 1, 2 * n_fft + 1, 12000)
    lens[[700, 5100, 9000]] = (160000, 96001, 48123)
    waves = _speech(lens, seed=n_fft + 14)
    batch = ex.RaggedAudio.from_list(waves)
    check = sorted({0, len(waves) - 1, 700, 5100, 9000} | set(range(0, len(waves), 97)))
    fm, lay = ex.logmel(batch, n_fft=n_fft, hop=hop)
    fo = lay.frame_off_host
    fmh = fm.cpu().numpy()
    for u in check:
        _check_db("12000 short utterances", fmh[fo[u]:fo[u + 1]], waves[u], n_fft, hop, 128)
    g, G, _, feats = _grad(batch, n_fft, hop, 128, seed=n_fft)
    assert torch.equal(feats, fm)
    off = batch.utt_off_host
    # Over hundreds of utterances of a few frames, every one reflected, the ratio of two correct fp32 errors has a tail
    # past 4: the same log-mel with its DFT as a dense fp32 matrix product is 5.3 times torch.stft's error on 1 of 300
    # such utterances at n_fft 400 (median 0.47), and this kernel reached 4.2.  A gradient taken from the wrong
    # utterance or the wrong rows is off by O(1).
    for u in check:
        _check_grad("12000 short utterances", g[off[u]:off[u + 1]], waves[u], G[fo[u]:fo[u + 1]], n_fft, hop, 128,
                    factor=8)
    for u in (0, 700, 4321, len(waves) - 1):                      # alone == inside the batch, forward and backward
        solo = ex.RaggedAudio.from_list([waves[u]])
        s, _ = ex.logmel(solo, n_fft=n_fft, hop=hop)
        assert torch.equal(s, fm[fo[u]:fo[u + 1]]), u
        solo.wav.requires_grad_(True)
        f1, _ = ex.logmel_grad(solo, n_fft=n_fft, hop=hop)
        (gs,) = torch.autograd.grad(f1, solo.wav, torch.from_numpy(G[fo[u]:fo[u + 1]]).float().cuda())
        assert np.array_equal(gs.cpu().numpy().astype(np.float64), g[off[u]:off[u + 1]]), u


@pytest.mark.parametrize("n_fft", N_FFTS)
def test_fewer_items_than_warps(n_fft):
    """One utterance of the shortest legal length (one item at n_fft 400 / 800), and five: most warps of the grid get
    nothing to do and must still reach the CTA's barriers."""
    ex = _ex()
    hop = HOP[n_fft]
    for lens in ([n_fft // 2 + 1], [n_fft // 2 + 1, n_fft // 2 + 2, n_fft // 2 + 5, n_fft // 2 + 9, n_fft]):
        waves = _speech(lens, seed=n_fft + len(lens))
        batch = ex.RaggedAudio.from_list(waves)
        assert batch.layout(n_fft, hop).n_items < torch.cuda.get_device_properties(0).multi_processor_count
        for n_mels in (128, 40):
            _forward_all("fewer items than warps", batch, waves, n_fft, hop, n_mels)
            _backward_all("fewer items than warps", batch, waves, n_fft, hop, n_mels)


# ---- band-major offsets past 2^31 floats -------------------------------------------------------------------------
def test_band_major_offsets_past_2_31_floats(tool):
    """One utterance of 44,739,300 samples (47 minutes) at n_fft 400, hop 2, 128 bands, band major: 22,369,651 frames, so
    band 96 starts 96 T > 2^31 floats into the output (11.5 GB).  Every value is written (the output starts as NaN), and
    all 128 bands of the first and the last 200 frames -- bands 96-127 are the ones whose offsets overflowed int --
    match float64 computed on a prefix and on a suffix that starts on a hop boundary, keeping only frames that do not
    see the cut."""
    ex = _ex()
    n_fft, hop, n_mels, n = 400, 2, 128, 44_739_300
    assert path_of(tool, n_fft, hop, n_mels)[0] == 1
    T = 1 + n // hop
    assert 96 * T >= 2 ** 31
    ex.logmel(ex.RaggedAudio.from_list([np.zeros(1000, np.float32)]), n_fft=n_fft, hop=hop, band_major=True)   # module load
    wav = 0.1 * torch.randn(n, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    batch = ex.RaggedAudio(wav, np.array([0, n]))
    batch.layout(n_fft, hop)
    out = torch.full((T * n_mels,), float("nan"), device="cuda")
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    ex.logmel(batch, n_fft=n_fft, n_mels=n_mels, hop=hop, band_major=True, out=out)
    stop.record()
    torch.cuda.synchronize()
    blk = out.view(n_mels, T)
    try:
        assert not bool(torch.isnan(blk).any())
        head, tail = blk[:, :200].cpu().numpy(), blk[:, T - 200:].cpu().numpy()
    finally:
        del blk, out
        torch.cuda.empty_cache()
    s0 = 2 * (T - 200) - n_fft                                    # the suffix's frame 200 is frame T - 200
    ref_head = _oracle_db(wav[:2000].cpu().numpy(), n_fft, hop, n_mels)[:, :200]
    ref_tail = _oracle_db(wav[s0:].cpu().numpy(), n_fft, hop, n_mels)[:, -200:]
    for got, ref in ((head, ref_head), (tail, ref_tail)):
        for bands in (slice(96, 128), slice(0, 32)):
            e_strong, e_all = logmel_error(got[bands], ref[bands])
            assert e_strong < TOL_DB and e_all < TOL_DB_FLOOR, (bands, e_strong, e_all)
            _worst("22.4 M frames band major", db_strong=e_strong, db_all=e_all)
        assert np.all(np.isfinite(got))
        e_strong, e_all = logmel_error(got, ref)
        assert e_strong < TOL_DB and e_all < TOL_DB_FLOOR, (e_strong, e_all)
    print(f"\n{T} frames x {n_mels} bands, band major, in {start.elapsed_time(stop):.1f} ms on {torch.cuda.get_device_name()}")
