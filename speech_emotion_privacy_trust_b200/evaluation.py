"""Batched cloak evaluation on the device (configs 2 and 5 of BASELINE.json).

The reference evaluates with batch size 1: for every test utterance it slides a 200-frame window with shift 50, runs the
cloak layer (a fresh noise sample per window), then the emotion classifier and the gender adversary on the noisy window,
copies two softmax rows to the host per window, and finally averages them and takes the argmax
(training/adversary_cloak_evaluation.py:60-93).  Here all windows of many utterances go through one forward: windows are
gathered and normalised by sept_normalize_windows_f32, the cloak kernel gives every window its own eps (per_sample), the
softmax rows are averaged per utterance with one index_add, and only the predictions travel to the host.

A waveform cloak (wave_cloak.WaveCloak) is evaluated by wave_cloak_evaluate: the noise goes on the test audio, one fresh
sample per utterance, before extraction; the window loop is the same.
"""
from __future__ import annotations

from typing import Sequence

import numpy as np
import torch

from . import cloak_ops, extraction, normalization
from .extraction import Layout, RaggedAudio

EPS_STD = 0.1


def suppression_mask(noise_layer, ratio: float) -> torch.Tensor | None:
    """Binary mask over (1, W, F): 0 where sigma exceeds the `ratio`-th percentile, 1 elsewhere
    (adversary_cloak_evaluation.py:263-267; np.nanpercentile's linear interpolation == torch.quantile).  The training
    script uses the (100 - ratio)-th percentile instead (training_cloak_with_grl.py:407-408): pass 100 - ratio."""
    if ratio == 0:
        return None
    sigma = noise_layer.scales().detach()
    thr = torch.quantile(sigma.flatten().float(), float(ratio) / 100.0)
    return torch.where(sigma > thr, torch.zeros_like(sigma), torch.ones_like(sigma))


def eval_window_table(lay: Layout, utts: Sequence[int] | None = None, win_len: int = 200, shift_len: int = 50):
    """Windows the reference's test() visits: (T - win_len) // shift + 1 per utterance, one (zero padded) for T < win_len
    (test utterances are stored padded, preprocess_adversary_data.py:29-35)."""
    return normalization.window_table(lay, utts, win_len, shift_len)


@torch.no_grad()
def cloak_evaluate(noise_layer, baseline_model, adversary_model, feat: torch.Tensor, lay: Layout, stats, mask=None,
                   utts: Sequence[int] | None = None, max_windows: int = 512, external_eps: torch.Tensor | None = None,
                   norm_mode: str = "znorm"):
    """Returns (emotion_pred, gender_pred, emotion_prob, gender_prob) per utterance, on the host:
    argmax / mean over the utterance's windows of softmax(baseline(noisy)), softmax(adversary(noisy)).

    feat/lay/stats: frame-major log-mel, its layout and the speaker statistics (normalisation happens in the gather).
    external_eps: optional (n_windows, W, F) noise samples, one per window in window-table order (parity tests).
    Without it the layer's own eps source is honoured: a patched `normal.sample` (the reference's draw site) is called
    once per window, in window order, exactly like the reference's loop; `layer.external_eps` -- ONE (1, W, F) sample --
    would give every window the same noise, which the reference never does, so it is rejected; otherwise eps comes from
    the device Philox stream (one draw per window, counter advanced by the number of windows)."""
    dev = feat.device
    locs, rhos = noise_layer.locs.detach().float().contiguous(), noise_layer.rhos.detach().float().contiguous()
    mask_c = None if mask is None else mask.detach().to(dev).float().contiguous()
    lo, hi = noise_layer._bounds() if hasattr(noise_layer, "_bounds") else (float(noise_layer.min_scale), float(noise_layer.max_scale))
    if external_eps is None and getattr(noise_layer, "external_eps", None) is not None:
        raise ValueError("cloak_evaluate draws one eps per window; layer.external_eps holds a single sample -- pass "
                         "external_eps=(n_windows, W, F) instead")
    sampler = vars(noise_layer.normal).get("sample") if external_eps is None and hasattr(noise_layer, "normal") else None

    def noisy_windows(a, b, wu, wt):
        x = normalization.normalized_windows(feat, lay, stats, wu, wt, mode=norm_mode)
        eps = None
        seed, draw = 0, None
        if external_eps is not None:
            eps = external_eps[a:b].to(dev).float().contiguous().reshape(-1)
        elif sampler is not None:
            eps = torch.cat([sampler(noise_layer.rhos.shape).reshape(1, -1) for _ in range(b - a)]).to(dev).float().contiguous().reshape(-1)
        else:
            _, seed, draw = noise_layer._eps_source()
        noisy, _, _ = cloak_ops.cloak_forward_raw(x, locs, rhos, mask_c, eps, seed, 0, EPS_STD, lo, hi, draw=draw, per_sample=True)
        return noisy

    return _classify_windows(baseline_model, adversary_model, lay, utts, noisy_windows, max_windows, dev)


@torch.no_grad()
def _classify_windows(baseline_model, adversary_model, lay: Layout, utts, windows, max_windows: int, dev):
    """The evaluation loop both evaluators share: the windows of eval_window_table(lay, utts) in chunks of max_windows,
    windows(a, b, win_utt[a:b], win_t0[a:b]) -> the classifiers' (b - a, 1, W, F) input, softmax of both models, the
    per-utterance mean and argmax.  Returns (emotion_pred, gender_pred, emotion_prob, gender_prob) on the host."""
    baseline_model.eval()
    adversary_model.eval()
    utts = list(range(len(lay.frame_off_host) - 1)) if utts is None else list(utts)
    win_utt, win_t0 = eval_window_table(lay, utts)
    n_win, n_utt = len(win_utt), len(utts)
    slot = {u: i for i, u in enumerate(utts)}
    seg_host = np.fromiter((slot[int(u)] for u in win_utt), dtype=np.int64, count=n_win)      # non-decreasing
    counts = torch.from_numpy(np.maximum(np.bincount(seg_host, minlength=n_utt), 1)).to(dev).unsqueeze(1).float()
    emo_sum = gen_sum = None
    for a in range(0, n_win, max_windows):
        b = min(n_win, a + max_windows)
        x = windows(a, b, win_utt[a:b], win_t0[a:b])
        p_emo = torch.softmax(baseline_model(x), dim=1)
        p_gen = torch.softmax(adversary_model(x), dim=1)
        if emo_sum is None:
            emo_sum = torch.zeros((n_utt, p_emo.shape[1]), device=dev)
            gen_sum = torch.zeros((n_utt, p_gen.shape[1]), device=dev)
        # windows of an utterance are contiguous: a segmented sum (no atomics) keeps the result deterministic
        first, last = int(seg_host[a]), int(seg_host[b - 1])
        lengths = torch.from_numpy(np.bincount(seg_host[a:b] - first, minlength=last - first + 1)).to(dev)
        emo_sum[first:last + 1] += torch.segment_reduce(p_emo.float(), "sum", lengths=lengths, axis=0)
        gen_sum[first:last + 1] += torch.segment_reduce(p_gen.float(), "sum", lengths=lengths, axis=0)
    emo_prob, gen_prob = emo_sum / counts, gen_sum / counts
    out = torch.cat([emo_prob.argmax(1, keepdim=True).float(), gen_prob.argmax(1, keepdim=True).float(), emo_prob, gen_prob], 1).cpu()
    ne = emo_prob.shape[1]
    return out[:, 0].long().numpy(), out[:, 1].long().numpy(), out[:, 2:2 + ne].numpy(), out[:, 2 + ne:].numpy()


def _check_stats_source(speaker_of_utt, stats) -> None:
    if (speaker_of_utt is None) == (stats is None):
        raise ValueError("give exactly one of speaker_of_utt (statistics of the noisy test features) and stats")


@torch.no_grad()
def wave_cloak_evaluate(layer, baseline_model, adversary_model, batch: RaggedAudio, speaker_of_utt: Sequence | None = None,
                        stats: normalization.SpeakerStats | None = None, utts: Sequence[int] | None = None, utt_ids=None,
                        n_draws: int | None = None, external_eps: torch.Tensor | None = None, n_fft: int = 800,
                        n_mels: int = 128, norm_mode: str = "znorm", max_windows: int = 512):
    """Evaluation of a waveform cloak (wave_cloak.WaveCloak) on test audio: configs 2 and 5 of BASELINE.json with the
    noise on the signal.  Returns what cloak_evaluate returns, (emotion_pred, gender_pred, emotion_prob, gender_prob) per
    utterance of `utts` (default all), on the host.

    Every utterance gets its own noise sample (layer.noisy_per_utterance: utt_ids, n_draws and external_eps as there), tiled
    from its first sample -- the signal-domain counterpart of the reference's fresh eps per window, whose 200-frame
    windows overlap by 150 frames of audio.  Then log-mel (extraction.logmel, n_fft / n_mels), per-speaker statistics,
    the test windows (eval_window_table) normalised in chunks of max_windows, both classifiers, the per-utterance softmax
    mean and argmax.  Statistics: `stats`, or those of the noisy features of the batch by speaker_of_utt with every
    utterance counted whole (the test split's rule, preprocess_adversary_data.py:56-60); exactly one must be given.  Under
    data parallelism pass speaker_stats_distributed statistics of the noisy features and global utt_ids."""
    _check_stats_source(speaker_of_utt, stats)
    noisy = layer.noisy_per_utterance(batch, utt_ids=utt_ids, n_draws=n_draws, external_eps=external_eps)
    feat, lay = extraction.logmel(noisy, n_fft=n_fft, n_mels=n_mels)
    if stats is None:
        stats = normalization.speaker_stats(feat, lay, speaker_of_utt, whole_utterance=[True] * batch.n_utts)
    return _classify_windows(baseline_model, adversary_model, lay, utts,
                             lambda a, b, wu, wt: normalization.normalized_windows(feat, lay, stats, wu, wt, mode=norm_mode),
                             max_windows, feat.device)
