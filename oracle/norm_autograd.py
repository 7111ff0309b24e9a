"""float64 torch autograd restatement of the per-speaker statistics + normalisation -- TEST INFRASTRUCTURE ONLY.

The reference computes the statistics from a per-speaker list that holds every row of every training window, duplicates
included (preprocess_data/preprocess_adversary_data.py:26-27, 41-48, 357-364), pads short utterances with zeros before
normalising (:29-35) and normalises with znorm or min_max (:377-381).  Here the same computation is written in torch so
that autograd gives its gradient: the rows are gathered with index_select (a frame in k windows is k rows, so its
gradients accumulate k times), mean and ddof-0 std are torch reductions, min / max are torch.amin / amax (which split the
gradient evenly over tied rows), and windows are zero padded.  One rule is added: where a speaker's feature column is
constant (std exactly 0, e.g. digital silence at -100 dB) no gradient flows through the std; torch's sqrt backward
would give 0 * inf = NaN there.
"""
from __future__ import annotations

import torch

from .norm import SHIFT_LEN, WIN_LEN, n_windows


def stacked_rows(n_frames: int, whole: bool = False, win_len: int = WIN_LEN, shift_len: int = SHIFT_LEN) -> torch.Tensor:
    """Frame indices of one utterance in the order :26-27 appends them: every window's rows, or every frame once for
    test-split (whole) and short utterances."""
    if whole or n_frames < win_len:
        return torch.arange(n_frames)
    return torch.cat([torch.arange(i * shift_len, i * shift_len + win_len)
                      for i in range(n_windows(n_frames, win_len, shift_len))])


def speaker_stats(feats, speaker_of_utt, whole_utterance=None, win_len: int = WIN_LEN, shift_len: int = SHIFT_LEN):
    """feats: list of (T_u, F) float64 tensors.  Returns (speakers, stats) with stats (n_spk, 4, F) = mean, std (ddof 0),
    min, max, differentiable with respect to feats; speakers in order of first appearance."""
    speakers = list(dict.fromkeys(speaker_of_utt))
    out = []
    for s in speakers:
        rows = torch.cat([f.index_select(0, stacked_rows(len(f), bool(whole_utterance[u]) if whole_utterance is not None
                                                         else False, win_len, shift_len))
                          for u, f in enumerate(feats) if speaker_of_utt[u] == s])
        mean = rows.mean(0)
        var = ((rows - mean) ** 2).mean(0)
        mn, mx = rows.amin(0), rows.amax(0)
        const = (mn == mx).detach()
        std = torch.where(const, torch.zeros_like(var), torch.sqrt(torch.where(const, torch.ones_like(var), var)))
        out.append(torch.stack([mean, std, mn, mx]))
    return speakers, torch.stack(out)


def normalize(x, st, mode: str = "znorm"):
    """:377-381 for one speaker's (4, F) statistics."""
    if mode == "znorm":
        return (x - st[0]) / (st[1] + 1e-5)
    if mode == "min_max":
        return (x - st[2]) / (st[3] - st[2]) * 2 - 1
    raise ValueError(mode)


def window(feat, t0: int, win_len: int = WIN_LEN):
    """Rows t0 .. t0 + win_len of one utterance, zero padded past its end (:29-35)."""
    T = len(feat)
    rows = feat[min(t0, T):min(t0 + win_len, T)]
    pad = win_len - len(rows)
    if pad:
        rows = torch.cat([rows, torch.zeros((pad, feat.shape[1]), dtype=feat.dtype)])
    return rows


def normalized_windows(feats, stats, spk_row, win_utt, win_t0, mode: str = "znorm", win_len: int = WIN_LEN):
    """(n_windows, win_len, F): window j of utterance win_utt[j] from frame win_t0[j], normalised with the statistics of
    row spk_row[u] of stats (n_spk, 4, F)."""
    return torch.stack([normalize(window(feats[u], int(t0), win_len), stats[spk_row[u]], mode)
                        for u, t0 in zip(win_utt, win_t0)])


def normalize_frames(feats, stats, spk_row, mode: str = "znorm"):
    """Frame-wise normalisation of every utterance (list of (T_u, F))."""
    return [normalize(f, stats[spk_row[u]], mode) for u, f in enumerate(feats)]
