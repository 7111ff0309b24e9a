"""End-to-end slice of BASELINE.json configs[4] on synthetic data: CREMA-D-shaped (91 speakers, 1-4 s, 16 kHz) and
MSP-Improv-shaped (12 speakers, 44.1 kHz -> resampled) corpora through resample -> log-mel -> per-speaker statistics ->
window gather -> cloak evaluation sweep over the suppression ratios of adversary_cloak_evaluation.py:167."""
import numpy as np
import pytest
import torch

from oracle import norm as onorm
from oracle import restate

pytestmark = pytest.mark.gpu


def _corpus(n_utts, n_spk, lo_s, hi_s, rate, seed):
    from speech_emotion_privacy_trust_b200 import synth
    rng = np.random.default_rng(seed)
    waves = [synth.speech_shaped(int(rng.uniform(lo_s, hi_s) * rate), rng) for _ in range(n_utts)]
    spk = [f"s{1001 + int(rng.integers(n_spk))}" for _ in range(n_utts)]
    return waves, spk


def test_corpus_shaped_pipeline_and_suppression_sweep():
    from speech_emotion_privacy_trust_b200 import dropin, evaluation, extraction, normalization as nz
    dropin.install()
    import baseline_models
    import cloak_models
    torch.manual_seed(4)
    crema, spk_c = _corpus(40, 91, 1.0, 4.0, 16000, 11)
    msp44, spk_m = _corpus(12, 12, 2.0, 6.0, 44100, 12)
    b_msp = extraction.resample(extraction.RaggedAudio.from_list(msp44), 44100, 16000)
    msp16 = [b_msp.wav[b_msp.utt_off_host[u]:b_msp.utt_off_host[u + 1]].cpu().numpy() for u in range(len(msp44))]
    assert [len(w) for w in msp16] == [restate.resample_length(len(w), 44100, 16000) for w in msp44]   # torchaudio's cut
    waves, spk = crema + msp16, spk_c + [s + "_msp" for s in spk_m]
    batch = extraction.RaggedAudio.from_list(waves)
    mel, lay = extraction.logmel(batch, n_fft=800)
    fo = lay.frame_off_host
    # oracle spot checks: extraction of a resampled utterance, statistics of one speaker
    u = len(crema) + 3
    ref = restate.mel_spectrogram(restate.resample(msp44[3], 44100, 16000)[None], 800, 128, dtype=np.float64)[0]
    got = mel[fo[u]:fo[u + 1]].cpu().numpy().T
    strong = ref > ref.max(axis=0, keepdims=True) - 50.0
    assert np.max(np.abs(got - ref)[strong]) < 1e-3
    whole = [True] * len(waves)                                    # test-split utterances are kept whole (:56-60)
    st = nz.speaker_stats(mel, lay, spk, whole)
    feats = [mel[fo[i]:fo[i + 1]].cpu().numpy() for i in range(len(waves))]
    want = onorm.speaker_stats_f64(feats, spk, whole)
    d = st.as_dict()
    for s in list(want)[:5]:
        assert np.max(np.abs(d[s]["mean"] - want[s]["mean"])) < 1e-3 and np.max(np.abs(d[s]["std"] - want[s]["std"])) < 1e-3
    # random-initialised stand-ins for the checkpoints the reference would load
    mk = lambda pred: baseline_models.two_d_cnn_lstm(1, 128, 5, lstm_hidden_size=64, pred=pred, global_feature=0).cuda().eval()
    base, adv = mk("emotion"), mk("gender")
    layer = cloak_models.cloak_noise(torch.zeros(1, 200, 128), torch.ones(1, 200, 128), 0.01, 5.0, "cuda").cuda()   # eval: max 5 (:205)
    with torch.no_grad():
        layer.rhos.add_(torch.randn(1, 200, 128, device="cuda"))
    n_win = len(evaluation.eval_window_table(lay)[0])
    assert n_win == sum(max(1, (int(fo[i + 1] - fo[i]) - 200) // 50 + 1) for i in range(len(waves)))
    eps = 0.1 * torch.randn(n_win, 200, 128, device="cuda")
    probs = {}
    for ratio in (0, 20, 40, 60, 80):                              # adversary_cloak_evaluation.py:167
        mask = evaluation.suppression_mask(layer, ratio)
        if ratio:
            assert abs(float((mask == 1).float().mean()) - ratio / 100.0) < 0.01
        e_pred, g_pred, e_prob, g_prob = evaluation.cloak_evaluate(layer, base, adv, mel, lay, st, mask=mask, external_eps=eps)
        assert e_pred.shape == (len(waves),) and e_prob.shape == (len(waves), 4) and g_prob.shape == (len(waves), 2)
        assert np.allclose(e_prob.sum(1), 1.0, atol=1e-5) and np.allclose(g_prob.sum(1), 1.0, atol=1e-5)
        assert np.array_equal(e_pred, e_prob.argmax(1)) and np.array_equal(g_pred, g_prob.argmax(1))
        probs[ratio] = e_prob
    again = evaluation.cloak_evaluate(layer, base, adv, mel, lay, st, mask=evaluation.suppression_mask(layer, 40), external_eps=eps)[2]
    assert np.array_equal(again, probs[40])                        # deterministic for a given eps
    assert not np.array_equal(probs[0], probs[80])                 # the mask changes what the classifier sees
