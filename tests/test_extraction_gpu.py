"""GPU parity of the extraction path, through the C ABI, against the golden vectors of the real reference and the
numpy oracle.  Tolerances are north_star's: log-mel 1e-3 dB max abs, MFCC 1e-4 of the utterance's max |coefficient|."""
import numpy as np
import pytest
import torch

from oracle import restate

pytestmark = pytest.mark.gpu

TOL_DB = 1e-3
TOL_MFCC_REL = 1e-4
TOL_DB_FLOOR = 0.05        # bins > 50 dB below their frame's peak hold fp32 rounding noise of whichever FFT made them
N_GOLD = 7
SPEECH = range(5)          # golden utterances 0-4 are speech shaped, 5 is silence, 6 a pure tone


def logmel_error(got, exact):
    """(max |dB error| over bins within 50 dB of their frame's strongest band, max over all bins) against fp64-exact
    arithmetic.  The tolerance of north_star (1e-3 dB) is meaningful where the signal is: a bin 60-90 dB below the
    frame's peak is the difference of numbers 1e6-1e9 times larger, and the reference's own fp32 FFT is up to 2e-2 dB
    from exact there (measured with torchaudio on the same inputs), so those bins get the looser TOL_DB_FLOOR."""
    d = np.abs(got - exact)
    strong = exact > exact.max(axis=0, keepdims=True) - 50.0
    return float(d[strong].max()), float(d.max())


@pytest.fixture(scope="module")
def ex():
    from speech_emotion_privacy_trust_b200 import extraction
    return extraction


@pytest.fixture(scope="module")
def gold_batch(ex, golden_extraction):
    waves = [golden_extraction[f"wav{i}"] for i in range(N_GOLD)]
    return ex.RaggedAudio.from_list(waves), waves


def _ok_for(n_fft, waves):
    return [i for i, w in enumerate(waves) if len(w) > n_fft // 2]


@pytest.mark.parametrize("key,n_fft", [("mel1", 800), ("mel2", 1600)])
def test_logmel_golden_both_layouts(ex, golden_extraction, key, n_fft):
    idx = _ok_for(n_fft, [golden_extraction[f"wav{i}"] for i in range(N_GOLD)])
    batch = ex.RaggedAudio.from_list([golden_extraction[f"wav{i}"] for i in idx])
    fm, lay = ex.logmel(batch, n_fft=n_fft)
    bm, _ = ex.logmel(batch, n_fft=n_fft, band_major=True)
    blocks = ex.split_band_major(bm, lay, 128)
    fo = lay.frame_off_host
    for j, i in enumerate(idx):
        ref = golden_extraction[f"{key}_{i}"][0]
        got_bm = blocks[j].cpu().numpy()
        got_fm = fm[fo[j]:fo[j + 1]].cpu().numpy().T
        assert got_bm.shape == ref.shape
        assert np.array_equal(got_bm, got_fm)                     # the two layouts hold the same bits
        if i in SPEECH:
            assert np.max(np.abs(got_bm - ref)) < TOL_DB, (i, np.max(np.abs(got_bm - ref)))
        elif i == 5:                                               # silence: the 1e-10 floor, exactly -100 dB
            assert np.max(np.abs(got_bm + 100.0)) < 1e-4
        else:
            # pure tone: bins 60 dB below the peak hold only the fp32 rounding noise of whichever FFT computed them
            # (the reference itself is 1.4e-2 dB from exact arithmetic there); compare where the signal is
            exact = restate.mel_spectrogram(golden_extraction[f"wav{i}"][None], n_fft, 128, dtype=np.float64)[0]
            strong = exact > exact.max() - 40.0
            assert np.max(np.abs(got_bm - exact)[strong]) < TOL_DB
            assert np.max(np.abs(got_bm - exact)) < 0.05


def test_mfcc_golden(ex, gold_batch, golden_extraction):
    batch, waves = gold_batch
    flat, lay = ex.mfcc(batch)
    blocks = ex.split_band_major(flat, lay, 120)
    for i in range(N_GOLD):
        ref = golden_extraction[f"mfcc_{i}"][0]
        got = blocks[i].cpu().numpy()
        assert got.shape == ref.shape
        # every golden utterance, including the pure tone (6): its mel bins 60-90 dB below the peak are rounding noise, but
        # top_db clamps everything under max - 80 dB and the DCT averages the rest -- the reference itself is 1.2e-6 from
        # fp64-exact arithmetic there, so the north_star tolerance applies unchanged
        rel = np.max(np.abs(got - ref)) / max(np.max(np.abs(ref)), 1e-12)
        assert rel < TOL_MFCC_REL, (i, rel)
        exact = restate.mfcc(waves[i][None], dtype=np.float64)[0]
        assert np.max(np.abs(got - exact)) / max(np.max(np.abs(exact)), 1e-12) < TOL_MFCC_REL, i


def test_logmel_random_ragged_batch_vs_oracle(ex):
    from speech_emotion_privacy_trust_b200 import synth
    rng = np.random.default_rng(77)
    lens = rng.integers(900, 48000, size=24)
    lens[:4] = [801, 960, 1599, 16001]                            # edges: just above pad, frame-count boundaries
    waves = [synth.speech_shaped(int(n), rng) for n in lens]
    batch = ex.RaggedAudio.from_list(waves)
    for n_fft in (800, 1600, 400):
        hop = 200 if n_fft == 400 else 160
        fm, lay = ex.logmel(batch, n_fft=n_fft, hop=hop)
        fo = lay.frame_off_host
        worst = worst_all = 0.0
        for u, w in enumerate(waves):
            p = restate.power_spectrogram(w, n_fft, hop, np.float64)
            ref = restate.amplitude_to_db_power((p.T @ restate.melscale_fbanks_htk(n_fft // 2 + 1, 128)).T)
            got = fm[fo[u]:fo[u + 1]].cpu().numpy().T
            assert got.shape == ref.shape
            e_strong, e_all = logmel_error(got, ref)
            worst, worst_all = max(worst, e_strong), max(worst_all, e_all)
        assert worst < TOL_DB and worst_all < TOL_DB_FLOOR, (n_fft, worst, worst_all)


def test_gradient_stream_and_other_mel_counts(ex, golden_extraction):
    w = golden_extraction["wav4"]
    batch = ex.RaggedAudio.from_list([w])
    got, _ = ex.logmel(batch, n_fft=400, hop=200, deriv=True)
    g = restate.waveform_gradient(w, 1.0).astype(np.float64)
    ref = restate.amplitude_to_db_power((restate.power_spectrogram(g, 400, 200).T @ restate.melscale_fbanks_htk(201, 128)).T)
    assert logmel_error(got.cpu().numpy().T, ref)[0] < TOL_DB
    for n_mels in (40, 64):
        got, _ = ex.logmel(batch, n_fft=800, n_mels=n_mels)
        ref = restate.mel_spectrogram(w[None], 800, n_mels, dtype=np.float64)[0]
        assert logmel_error(got.cpu().numpy().T, ref)[0] < TOL_DB


def test_gradient_stream_every_fft_size(ex):
    """np.gradient stream (deriv=True) through every kernel form: n_fft 800 keeps one straight-line pass 1 per stream kind,
    n_fft 400 / 1600 share one transform behind a run-time switch of the loads (extract.cu: kSharedPass1); 128 bands take the
    tensor-memory table path, 64 bands the shared-memory one.  Ragged batch: interior items difference the staged waveform
    on the fly, edge items (reflection, utterance ends, one-sided differences) stage the gradient itself."""
    from speech_emotion_privacy_trust_b200 import synth
    rng = np.random.default_rng(91)
    waves = [synth.speech_shaped(int(n), rng) for n in (16000, 801, 1700, 23456, 40000)]
    batch = ex.RaggedAudio.from_list(waves)
    for n_fft, hop in ((400, 200), (800, 160), (1600, 160)):
        for n_mels in (128, 64):
            fb = restate.melscale_fbanks_htk(n_fft // 2 + 1, n_mels)
            got, lay = ex.logmel(batch, n_fft=n_fft, hop=hop, n_mels=n_mels, deriv=True)
            fo = lay.frame_off_host
            for u, w in enumerate(waves):
                if len(w) <= n_fft // 2:
                    continue
                g = restate.waveform_gradient(w, 1.0).astype(np.float64)
                ref = restate.amplitude_to_db_power((restate.power_spectrogram(g, n_fft, hop).T @ fb).T)
                e_strong, e_all = logmel_error(got[fo[u]:fo[u + 1]].cpu().numpy().T, ref)
                assert e_strong < TOL_DB and e_all < TOL_DB_FLOOR, (n_fft, n_mels, u, e_strong, e_all)


def test_dropin_callables_keep_reference_types(golden_extraction):
    from speech_emotion_privacy_trust_b200 import dropin
    dropin.install()
    import audio_feature_extraction as afe
    wav = torch.from_numpy(golden_extraction["wav3"])[None]       # CPU tensor, like torchaudio.load returns
    m = afe.mel_spectrogram(wav, n_fft=800, feature_len=128)
    assert isinstance(m, torch.Tensor) and m.device.type == "cpu" and m.dtype == torch.float32
    assert tuple(m.shape) == golden_extraction["mel1_3"].shape
    assert np.max(np.abs(m.numpy() - golden_extraction["mel1_3"])) < TOL_DB
    c = afe.mfcc(wav)
    assert isinstance(c, np.ndarray) and c.dtype == np.float32 and c.shape == golden_extraction["mfcc_3"].shape
    assert np.max(np.abs(c - golden_extraction["mfcc_3"])) / np.max(np.abs(golden_extraction["mfcc_3"])) < TOL_MFCC_REL
    with pytest.raises(ValueError, match="n_fft=1024"):            # the signature default is never used by the reference
        afe.mel_spectrogram(wav)
    with pytest.raises(RuntimeError, match="reflect padding"):     # torch.stft raises for N <= n_fft/2 as well
        afe.mel_spectrogram(torch.zeros(1, 300), n_fft=800)


def test_corpus_scale_properties(ex):
    """Sizes the oracle cannot cover in seconds: size-independent properties on a 600-utterance, ~1-audio-hour batch."""
    from speech_emotion_privacy_trust_b200 import synth
    wav, off = synth.corpus(600, seed=1234)
    batch = ex.RaggedAudio(torch.from_numpy(wav).cuda(), off)
    a, lay = ex.logmel(batch, n_fft=800)
    b, _ = ex.logmel(batch, n_fft=800)
    assert torch.equal(a, b)                                       # deterministic
    assert lay.total_frames == int(sum(1 + (off[u + 1] - off[u]) // 160 for u in range(600)))
    assert bool(torch.isfinite(a).all()) and float(a.min()) >= -100.0
    fo = lay.frame_off_host
    for u in (0, 17, 311, 599):                                    # batch invariance: alone == inside the batch, bit exact
        solo = ex.RaggedAudio(batch.wav[off[u]:off[u + 1]].clone(), np.array([0, off[u + 1] - off[u]]))
        s, _ = ex.logmel(solo, n_fft=800)
        assert torch.equal(s, a[fo[u]:fo[u + 1]])
    # scaling the waveform by 2 shifts every un-floored bin by 20*log10(2) dB
    batch2 = ex.RaggedAudio(batch.wav * 2.0, off)
    c, _ = ex.logmel(batch2, n_fft=800)
    live = a > -99.0
    assert float(((c - a)[live] - 6.020599913).abs().max()) < 1e-4
    # oracle spot check inside the big batch
    u = 311
    ref = restate.mel_spectrogram(wav[off[u]:off[u + 1]][None], 800, 128, dtype=np.float64)[0]
    e_strong, e_all = logmel_error(a[fo[u]:fo[u + 1]].cpu().numpy().T, ref)
    assert e_all < TOL_DB, e_all                                  # corpus-shaped audio: EVERY bin within 1e-3 dB of exact
    # MFCC on the same batch: finite, and the c0 row dominates like an energy term should
    m, mlay = ex.mfcc(batch)
    assert bool(torch.isfinite(m).all())
    blk = ex.split_band_major(m, mlay, 120)[u].cpu().numpy()
    refm = restate.mfcc(wav[off[u]:off[u + 1]][None], dtype=np.float64)[0]
    assert np.max(np.abs(blk - refm)) / np.max(np.abs(refm)) < TOL_MFCC_REL


def test_other_hops_and_mel_counts_fuzz(ex):
    """Parameters the reference never uses but the C ABI accepts: every combination is checked against the fp64 oracle."""
    from speech_emotion_privacy_trust_b200 import synth
    rng = np.random.default_rng(2026)
    combos = [(800, 80, 23), (800, 320, 256), (800, 400, 80), (1600, 100, 64), (1600, 480, 128), (400, 80, 40),
              (400, 160, 128), (400, 400, 96), (800, 160, 1), (1600, 160, 33),
              # the unrolled 128-band path (tables in tensor memory) at hops the reference never uses
              (800, 80, 128), (800, 400, 128), (800, 480, 128), (400, 400, 128), (1600, 100, 128), (1600, 800, 128)]
    for n_fft, hop, n_mels in combos:
        lens = [int(n_fft // 2 + 1 + rng.integers(0, 3 * n_fft)) for _ in range(5)] + [n_fft // 2 + 1, 5 * hop, 5 * hop - 1]
        lens = [max(n, n_fft // 2 + 1) for n in lens]
        waves = [synth.speech_shaped(n, rng) for n in lens]
        batch = ex.RaggedAudio.from_list(waves)
        fm, lay = ex.logmel(batch, n_fft=n_fft, n_mels=n_mels, hop=hop)
        fo = lay.frame_off_host
        fb = restate.melscale_fbanks_htk(n_fft // 2 + 1, n_mels)
        for u, w in enumerate(waves):
            ref = restate.amplitude_to_db_power((restate.power_spectrogram(w, n_fft, hop, np.float64).T @ fb).T)
            got = fm[fo[u]:fo[u + 1]].cpu().numpy().T
            assert got.shape == ref.shape == (n_mels, 1 + len(w) // hop), (n_fft, hop, n_mels, u)
            e_strong, e_all = logmel_error(got, ref)
            assert e_strong < TOL_DB and e_all < TOL_DB_FLOOR, (n_fft, hop, n_mels, u, e_strong, e_all)
    with pytest.raises(ValueError, match="hop"):
        ex.logmel(ex.RaggedAudio.from_list([np.zeros(4000, np.float32)]), n_fft=800, hop=161)


def test_mfcc_fuzz_vs_oracle(ex):
    """MFCC at the one configuration the C ABI accepts (n_fft 400, hop 200, 128 mels, 40 coefficients, three streams), on
    ragged batches that exercise what is special about it: the per-utterance top_db floor (loud + near-silent halves in
    one utterance, whole utterances at the 1e-10 clamp), frame-count boundaries, the shortest legal utterance."""
    from speech_emotion_privacy_trust_b200 import synth
    rng = np.random.default_rng(404)
    lens = [201, 399, 400, 401, 999, 1000, 1001, 1599, 1600] + [int(rng.integers(202, 40000)) for _ in range(15)]
    waves = [synth.speech_shaped(n, rng) for n in lens]
    waves[9][: len(waves[9]) // 2] *= 1e-4                         # half the utterance 80 dB down: sits on the top_db floor
    waves[10] *= 1e-6                                              # every band at the 1e-10 power clamp (-100 dB)
    waves[11][len(waves[11]) // 3:] = 0.0                          # digital silence after speech
    waves.append(np.zeros(777, np.float32))
    batch = ex.RaggedAudio.from_list(waves)
    flat, lay = ex.mfcc(batch)
    blocks = ex.split_band_major(flat, lay, 120)
    for u, w in enumerate(waves):
        ref = restate.mfcc(w[None], dtype=np.float64)[0]
        got = blocks[u].cpu().numpy()
        assert got.shape == ref.shape == (120, 1 + len(w) // 200), u
        assert np.max(np.abs(got - ref)) / max(np.max(np.abs(ref)), 1e-12) < TOL_MFCC_REL, (u, len(w))


def test_against_reference_port_at_corpus_lengths(ex):
    """2-10 s utterances (the corpus shape of BASELINE.json configs[0]) against oracle/ref_port.py -- the reference's own
    callables restated on torchaudio, bit-identical to the reference on the golden vectors -- run on the host CPU."""
    from oracle import ref_port
    from speech_emotion_privacy_trust_b200 import synth
    torch.set_num_threads(4)
    wav, off = synth.corpus(12, seed=77)
    batch = ex.RaggedAudio(torch.from_numpy(wav).cuda(), off)
    m1, lay = ex.logmel(batch, n_fft=800, band_major=True)
    m2, _ = ex.logmel(batch, n_fft=1600, band_major=True)
    mf, mlay = ex.mfcc(batch)
    b1, b2, bm = ex.split_band_major(m1, lay, 128), ex.split_band_major(m2, lay, 128), ex.split_band_major(mf, mlay, 120)
    for u in range(12):
        a = torch.from_numpy(wav[off[u]:off[u + 1]])[None]
        for got, ref, n_fft in ((b1[u], ref_port.mel_spectrogram(a, 800, 128)[0], 800), (b2[u], ref_port.mel_spectrogram(a, 1600, 128)[0], 1600)):
            got, ref = got.cpu().numpy(), ref.numpy()
            assert got.shape == ref.shape
            # corpus-shaped audio has no bin more than 50 dB below its frame's peak: ALL bins within north_star's 1e-3 dB
            # of the reference's own fp32 output, and of fp64-exact arithmetic
            assert np.max(np.abs(got - ref)) < TOL_DB, (u, n_fft, float(np.max(np.abs(got - ref))))
            exact = restate.mel_spectrogram(a.numpy(), n_fft, 128, dtype=np.float64)[0]
            assert np.max(np.abs(got - exact)) < TOL_DB, (u, n_fft, float(np.max(np.abs(got - exact))))
        ref = ref_port.mfcc(a)[0]
        got = bm[u].cpu().numpy()
        assert got.shape == ref.shape
        assert np.max(np.abs(got - ref)) / np.max(np.abs(ref)) < TOL_MFCC_REL


def test_host_buffer_api_float_and_pcm16(ex):
    """extraction.logmel_host: chunked H2D / kernel / D2H pipeline equals the device-resident call bit for bit, for
    float32 input and for 16-bit PCM input (x / 32768 on the device == torchaudio.load's normalisation on the host)."""
    from speech_emotion_privacy_trust_b200 import synth
    wav, off = synth.corpus(40, seed=5, lo_s=0.5, hi_s=3.0)
    pcm = np.round(wav * 32767.0).astype(np.int16)
    wav_q = pcm.astype(np.float32) / 32768.0                      # what torchaudio.load(normalize=True) returns
    ref, lay = ex.logmel(ex.RaggedAudio(torch.from_numpy(wav_q).cuda(), off), n_fft=800)
    for host, tag in ((torch.from_numpy(wav_q).pin_memory(), "float32"), (torch.from_numpy(pcm).pin_memory(), "pcm16")):
        ref_host = ref.cpu()
        out = torch.full((lay.total_frames, 128), float("nan")).pin_memory()
        out, fo = ex.logmel_host(host, off, n_fft=800, out_host=out, chunk_samples=1 << 18, n_streams=3)     # 5+ chunks
        assert torch.equal(out, ref_host), tag                    # read right after the call: no external synchronize
        assert np.array_equal(fo, lay.frame_off_host), tag
        out2, _ = ex.logmel_host(host, off, n_fft=800, chunk_samples=1 << 18, n_streams=3, sync=False)
        torch.cuda.current_stream().synchronize()                 # the async contract: the current stream is ordered after it
        assert torch.equal(out2, ref_host), tag
