"""Per-speaker normalisation + training-window assembly on the device (csrc/norm.cu via the C ABI).

The reference does this inline in preprocess_data/preprocess_adversary_data.py (:26-27 frame accumulation, :41-48 window
rule, :29-35 zero padding, :357-385 statistics and normalisation); there is no callable to mirror, so this module
defines the API.  Inputs are the frame-major features extraction.logmel() returns.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Sequence

import numpy as np
import torch

from torch.autograd.function import once_differentiable

from . import _lib
from .extraction import Layout

WIN_LEN, SHIFT_LEN = 200, 50      # training_data_preprocess.sh:6-8 ; preprocess_adversary_data.py:131
MODES = {"znorm": 0, "min_max": 1}


@dataclass
class SpeakerStats:
    speakers: list                 # speaker labels, row order of `stats`
    stats: torch.Tensor            # device (n_spk, 5, F): count, mean, std (ddof 0), min, max
    spk_of_utt: torch.Tensor       # device int32 [n_utts] row index per utterance
    spk_lists: tuple | None = None  # device CSR (spk_ptr, spk_utts) the statistics were built with; a backward reuses it

    def as_dict(self) -> dict:
        h = self.stats.detach().cpu().numpy()
        return {s: {"count": h[i, 0], "mean": h[i, 1], "std": h[i, 2], "min": h[i, 3], "max": h[i, 4]}
                for i, s in enumerate(self.speakers)}


def n_windows(n_frames: int, win_len: int = WIN_LEN, shift_len: int = SHIFT_LEN) -> int:
    return 1 if n_frames < win_len else (n_frames - win_len) // shift_len + 1


def _check_feat(feat: torch.Tensor, st: SpeakerStats | None = None) -> None:
    """feat is what the kernels read: a contiguous (total_frames, F) float32 CUDA tensor, with the F of `st`'s statistics
    when they are given."""
    _lib.require_cuda(feat)
    if feat.dtype != torch.float32 or feat.dim() != 2 or not feat.is_contiguous():
        raise ValueError("feat must be a contiguous (total_frames, F) float32 tensor")
    if st is not None and feat.shape[1] != st.stats.shape[2]:
        raise ValueError(f"feat has {feat.shape[1]} features, the statistics {st.stats.shape[2]}")


def _check_window_table(win_utt, win_t0, n_utts: int, win_len: int):
    """(win_utt, win_t0) as int32 arrays.  ValueError for an utterance outside [0, n_utts), or a start below 0 or so large
    that a window's last row (t0 + win_len - 1, int32 in the kernels) would overflow.  Checked before the int32 cast."""
    if win_len <= 0:
        raise ValueError("win_len must be > 0")
    wu = np.asarray(win_utt, dtype=np.int64).reshape(-1)
    wt = np.asarray(win_t0, dtype=np.int64).reshape(-1)
    if len(wu) != len(wt):
        raise ValueError("win_utt and win_t0 must have the same length")
    t_max = np.iinfo(np.int32).max - win_len
    if len(wt) and (wt.min() < 0 or wt.max() > t_max):
        raise ValueError(f"win_t0 must lie in [0, {t_max}]")
    if len(wu) and (wu.min() < 0 or wu.max() >= n_utts):
        raise ValueError(f"win_utt must lie in [0, {n_utts})")
    return wu.astype(np.int32), wt.astype(np.int32)


def speaker_stats(feat: torch.Tensor, lay: Layout, speaker_of_utt: Sequence, whole_utterance: Sequence[bool] | None = None,
                  win_len: int = WIN_LEN, shift_len: int = SHIFT_LEN) -> SpeakerStats:
    """Weighted per-speaker mean/std/min/max: a frame inside k training windows counts k times (:26-27), utterances
    flagged whole (test split, :56-60) count each frame once."""
    speakers, d_spk, spk_lists, d_whole = _speaker_table(feat, lay, speaker_of_utt, whole_utterance)
    stats = _launch_speaker_stats(feat, lay, d_whole, win_len, shift_len, spk_lists)
    return SpeakerStats(speakers, stats, d_spk, spk_lists)


def _speaker_table(feat: torch.Tensor, lay: Layout, speaker_of_utt: Sequence, whole_utterance: Sequence[bool] | None,
                   speakers: Sequence | None = None):
    """What every statistics entry sets up: checks feat and the labels, gives each speaker a row (in first-seen order, or
    in the order of `speakers`, which must hold every label) and returns (speaker rows, device int32 row of each
    utterance, its device CSR, device whole-utterance flags or None)."""
    _check_feat(feat)
    n_utts = len(lay.frame_off_host) - 1
    if len(speaker_of_utt) != n_utts:
        raise ValueError("one speaker label per utterance is required")
    if speakers is None:
        speakers = list(dict.fromkeys(speaker_of_utt))
    else:
        speakers = list(speakers)
        missing = set(speaker_of_utt) - set(speakers)
        if missing:
            raise ValueError(f"speakers missing from all_speakers: {sorted(map(str, missing))}")
    row = {s: i for i, s in enumerate(speakers)}
    spk_idx = np.fromiter((row[s] for s in speaker_of_utt), dtype=np.int32, count=n_utts)
    dev = feat.device
    d_whole = None if whole_utterance is None else torch.from_numpy(np.asarray(whole_utterance, dtype=np.uint8)).to(dev)
    return speakers, torch.from_numpy(spk_idx).to(dev), _speaker_lists(spk_idx, len(speakers), dev), d_whole


def _speaker_lists(spk_idx: np.ndarray, n_spk: int, dev):
    """Device CSR (ptr [n_spk + 1], utterance ids grouped by speaker in utterance order) of a host speaker index."""
    order = np.argsort(spk_idx, kind="stable").astype(np.int32)
    ptr = np.zeros(n_spk + 1, dtype=np.int32)
    np.cumsum(np.bincount(spk_idx, minlength=n_spk), out=ptr[1:])
    return torch.from_numpy(ptr).to(dev), torch.from_numpy(order).to(dev)


def _launch_speaker_stats(feat, lay, d_whole, win_len, shift_len, spk_lists) -> torch.Tensor:
    """(n_spk, 5, F) statistics of the rows of the CSR spk_lists; a row with no utterance gets count, mean and std 0,
    min FLT_MAX and max -FLT_MAX."""
    dev = feat.device
    d_ptr, d_order = spk_lists
    n_utts, n_spk, F = len(lay.frame_off_host) - 1, d_ptr.numel() - 1, feat.shape[1]
    partial = torch.empty((n_utts, 5, F), dtype=torch.float32, device=dev)
    stats = torch.empty((n_spk, 5, F), dtype=torch.float32, device=dev)
    _lib.launch("sept_speaker_stats_f32", feat, lay.frame_off, d_whole, n_utts, F, win_len, shift_len, d_ptr, d_order, n_spk,
                partial, stats, device=dev)
    return stats


def normalize(feat: torch.Tensor, lay: Layout, st: SpeakerStats, mode: str = "znorm") -> torch.Tensor:
    """Frame-wise normalisation with each utterance's speaker statistics (:377-381); same shape as feat."""
    _check_feat(feat, st)
    out = torch.empty_like(feat)
    _lib.launch("sept_normalize_f32", feat, lay.frame_off, st.spk_of_utt, st.stats, len(lay.frame_off_host) - 1, feat.shape[1],
                MODES[mode], out, device=feat.device)
    return out


def window_table(lay: Layout, utts: Sequence[int] | None = None, win_len: int = WIN_LEN, shift_len: int = SHIFT_LEN):
    """(win_utt, win_t0) int32 arrays of every training window of the given utterances (:44-48)."""
    fo = lay.frame_off_host
    utts = range(len(fo) - 1) if utts is None else utts
    wu, wt = [], []
    for u in utts:
        k = n_windows(int(fo[u + 1] - fo[u]), win_len, shift_len)
        wu.append(np.full(k, u, dtype=np.int32))
        wt.append(np.arange(k, dtype=np.int32) * shift_len)
    if not wu:
        return np.zeros(0, np.int32), np.zeros(0, np.int32)
    return np.concatenate(wu), np.concatenate(wt)


def normalized_windows(feat: torch.Tensor, lay: Layout, st: SpeakerStats, win_utt: np.ndarray, win_t0: np.ndarray,
                       mode: str = "znorm", win_len: int = WIN_LEN) -> torch.Tensor:
    """(n_windows, 1, win_len, F) float32 batches for the cloak layer: normalised windows, short utterances zero-padded
    BEFORE normalisation like :29-35.  win_t0 outside [0, 2^31 - 1 - win_len] or win_utt outside [0, n_utts) raises
    ValueError."""
    _check_feat(feat, st)
    wu, wt = _check_window_table(win_utt, win_t0, len(lay.frame_off_host) - 1, win_len)
    dev = feat.device
    n = len(wu)
    F = feat.shape[1]
    out = torch.empty((n, 1, win_len, F), dtype=torch.float32, device=dev)
    d_wu = torch.from_numpy(wu).to(dev)
    d_wt = torch.from_numpy(wt).to(dev)
    _lib.launch("sept_normalize_windows_f32", feat, lay.frame_off, st.spk_of_utt, st.stats, d_wu, d_wt, n, win_len, F,
                MODES[mode], out, device=dev)
    return out


def speaker_stats_distributed(feat: torch.Tensor, lay: Layout, speaker_of_utt: Sequence, all_speakers: Sequence,
                              whole_utterance: Sequence[bool] | None = None, group=None, win_len: int = WIN_LEN,
                              shift_len: int = SHIFT_LEN) -> SpeakerStats:
    """Per-speaker statistics when a speaker's utterances are spread over several ranks (they are under length-bucketed
    sharding, SURVEY 8e): every rank reduces its own utterances with the kernels, then ONE all-gather of the
    (count, mean, M2, min, max) partials and a Chan merge in rank order give every rank the global statistics.
    `all_speakers` fixes the row order on every rank (speakers a rank does not hold contribute empty partials)."""
    speakers, d_spk, spk_lists, d_whole = _speaker_table(feat, lay, speaker_of_utt, whole_utterance, all_speakers)
    stats = _merge_ranks(_launch_speaker_stats(feat, lay, d_whole, win_len, shift_len, spk_lists), spk_lists[0], group)
    return SpeakerStats(speakers, stats, d_spk, spk_lists)


def _merge_ranks(stats: torch.Tensor, spk_ptr: torch.Tensor, group) -> torch.Tensor:
    """The rank's (n_spk, 5, F) statistics over the shared speaker rows (CSR pointer spk_ptr) -> the global ones: one
    all-gather and a Chan merge in rank order (parallel.merge_speaker_partials).  A speaker the rank does not hold enters
    with min +inf and max -inf, so a speaker no rank holds ends as (0, 0, 0, +inf, -inf)."""
    from . import parallel
    held = (spk_ptr[1:] > spk_ptr[:-1]).unsqueeze(1)
    cnt, mean, sd = stats[:, 0], stats[:, 1], stats[:, 2]
    mn, mx = torch.where(held, stats[:, 3], float("inf")), torch.where(held, stats[:, 4], float("-inf"))
    n, mu, sd, lo, hi = parallel.merge_speaker_partials(cnt, mean, sd * sd * cnt, mn, mx, group=group)
    return torch.stack([n, mu, sd, lo, hi], dim=1).contiguous()


# ---- gradients: the same forward launches, with a grad_fn to feat (and to the statistics) ------------------------
class SpeakerStatsFunction(torch.autograd.Function):
    """speaker_stats() or speaker_stats_distributed() with a gradient to (this rank's) feat.  Forward: the
    sept_speaker_stats_f32 launch over the given speaker rows, then, when distributed, the all-gather and Chan merge.
    Backward: when distributed, dstats summed over the ranks in rank order (one all-gather); the rank's min / max tie
    weights against the statistics (sept_speaker_stats_bwd_ties_i32); when distributed, one exact int32 SUM all-reduce of
    them; then sept_speaker_stats_bwd_frames_f32.  The count row gets no gradient; no double backward.  `distributed`,
    not `group`, selects the collectives: group None is the default world group, and the local path must run none even
    when a process group is initialised."""

    @staticmethod
    def forward(ctx, feat, lay, d_whole, win_len, shift_len, d_spk, spk_lists, distributed, group):
        stats = _launch_speaker_stats(feat, lay, d_whole, win_len, shift_len, spk_lists)
        if distributed:
            stats = _merge_ranks(stats, spk_lists[0], group)
        ctx.save_for_backward(feat, stats)
        ctx.cfg = (lay, d_whole, win_len, shift_len, d_spk, spk_lists, distributed, group)
        return stats

    @staticmethod
    @once_differentiable
    def backward(ctx, dstats):
        from . import parallel
        feat, stats = ctx.saved_tensors
        lay, d_whole, win_len, shift_len, d_spk, (d_ptr, d_order), distributed, group = ctx.cfg
        dev, n_utts, n_spk, F = feat.device, len(lay.frame_off_host) - 1, stats.shape[0], feat.shape[1]
        dstats = dstats.contiguous()
        if distributed:
            dstats = parallel.sum_in_rank_order(dstats, group)
        ties = torch.empty((n_spk, 2, F), dtype=torch.int32, device=dev)
        ws = _lib.workspace(_lib.lib().sept_speaker_stats_bwd_ties_workspace_bytes(n_utts, F), dev)
        dfeat = torch.empty_like(feat)
        _lib.launch("sept_speaker_stats_bwd_ties_i32", feat, lay.frame_off, d_whole, n_utts, F, win_len, shift_len, d_spk,
                    d_ptr, d_order, n_spk, stats, ws, ties, device=dev)
        if distributed:
            parallel.allreduce_exact_sum(ties, group)
        _lib.launch("sept_speaker_stats_bwd_frames_f32", feat, lay.frame_off, d_whole, n_utts, F, win_len, shift_len, d_spk,
                    stats, dstats, ties, dfeat, device=dev)
        return dfeat, None, None, None, None, None, None, None, None


def speaker_stats_grad(feat: torch.Tensor, lay: Layout, speaker_of_utt: Sequence,
                       whole_utterance: Sequence[bool] | None = None, win_len: int = WIN_LEN,
                       shift_len: int = SHIFT_LEN) -> SpeakerStats:
    """speaker_stats() with a gradient: `.stats` is bit-identical and carries a grad_fn to feat.

    The gradient is what torch autograd gives through the reference's stacked rows (a frame in k windows is k rows):
    mean and ddof-0 std of the weighted frames, min / max split over tied frames in proportion to their multiplicity.
    The count row gets none; where the std is exactly 0 (a constant feature column) none flows through the std.
    Deterministic (no atomics)."""
    speakers, d_spk, spk_lists, d_whole = _speaker_table(feat, lay, speaker_of_utt, whole_utterance)
    stats = SpeakerStatsFunction.apply(feat, lay, d_whole, win_len, shift_len, d_spk, spk_lists, False, None)
    return SpeakerStats(speakers, stats, d_spk, spk_lists)


def speaker_stats_distributed_grad(feat: torch.Tensor, lay: Layout, speaker_of_utt: Sequence, all_speakers: Sequence,
                                   whole_utterance: Sequence[bool] | None = None, group=None, win_len: int = WIN_LEN,
                                   shift_len: int = SHIFT_LEN) -> SpeakerStats:
    """speaker_stats_distributed() with a gradient: `.stats` is bit-identical and carries a grad_fn to this rank's feat.

    With the ranks' losses summed, the gradient each rank gets is what speaker_stats_grad() gives on one GPU over the
    union of every rank's utterances, restricted to this rank's frames: the statistics, the min / max tie multiplicities
    and the upstream dstats are all global.  The backward is collective (one all-gather of dstats, one int32 all-reduce),
    so every rank of `group` must run it, as with any data-parallel backward.  Without an initialised process group, or
    with one rank, no collective runs.  Deterministic: every rank adds dstats in rank order."""
    speakers, d_spk, spk_lists, d_whole = _speaker_table(feat, lay, speaker_of_utt, whole_utterance, all_speakers)
    stats = SpeakerStatsFunction.apply(feat, lay, d_whole, win_len, shift_len, d_spk, spk_lists, True, group)
    return SpeakerStats(speakers, stats, d_spk, spk_lists)


class NormalizeFunction(torch.autograd.Function):
    """normalize() (win is None) or normalized_windows() with gradients to feat and to the statistics: forward is the
    existing launch, backward one sept_normalize_bwd_f32 call.  The tables the backward needs (each utterance's windows
    sorted by start, built here; each speaker's utterances, the statistics' CSR) are on the device before it, so the
    backward launches kernels only."""

    @staticmethod
    def forward(ctx, feat, stats, lay, st, win, mode):
        st_fwd = SpeakerStats(st.speakers, stats, st.spk_of_utt, st.spk_lists)
        n_utts = len(lay.frame_off_host) - 1
        dev = feat.device
        if win is None:
            out = normalize(feat, lay, st_fwd, mode)
            tables = None
        else:
            wu, wt, win_len = win
            out = normalized_windows(feat, lay, st_fwd, wu, wt, mode, win_len)
            order = np.lexsort((np.arange(len(wu)), wt, wu)).astype(np.int32)     # by utterance, start, window id
            ptr = np.zeros(n_utts + 1, dtype=np.int32)
            np.cumsum(np.bincount(wu, minlength=n_utts), out=ptr[1:])
            tables = (torch.from_numpy(wt).to(dev), torch.from_numpy(ptr).to(dev), torch.from_numpy(order).to(dev),
                      len(wu), win_len)
        spk_lists = st.spk_lists
        if ctx.needs_input_grad[1] and spk_lists is None:                     # a SpeakerStats built by hand
            spk_lists = _speaker_lists(np.asarray(st.spk_of_utt.cpu().numpy(), dtype=np.int32), stats.shape[0], dev)
        ctx.save_for_backward(feat, stats)
        ctx.cfg = (lay, st.spk_of_utt, tables, spk_lists, MODES[mode])
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad):
        feat, stats = ctx.saved_tensors
        lay, spk_of_utt, tables, spk_lists, mode = ctx.cfg
        need_feat, need_stats = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        if not (need_feat or need_stats):
            return None, None, None, None, None, None
        dev, n_utts, F = feat.device, len(lay.frame_off_host) - 1, feat.shape[1]
        dfeat = torch.empty_like(feat) if need_feat else None
        dstats = torch.empty_like(stats) if need_stats else None
        ws = _lib.workspace(_lib.lib().sept_normalize_bwd_workspace_bytes(n_utts, F), dev) if need_stats else None
        d_wt, d_ptr, d_list, n_win, win_len = tables if tables is not None else (None, None, None, 0, 0)
        s_ptr, s_list = spk_lists if need_stats else (None, None)
        _lib.launch("sept_normalize_bwd_f32", feat, lay.frame_off, spk_of_utt, stats, d_wt, d_ptr, d_list, n_win, win_len,
                    n_utts, F, mode, grad.contiguous(), s_ptr, s_list, stats.shape[0], ws, dfeat, dstats, device=dev)
        return dfeat, dstats, None, None, None, None


def normalize_grad(feat: torch.Tensor, lay: Layout, st: SpeakerStats, mode: str = "znorm") -> torch.Tensor:
    """normalize() with a gradient: bit-identical values with a grad_fn to feat and, when st.stats requires grad (from
    speaker_stats_grad), to the statistics.  Deterministic."""
    _lib.require_cuda(feat)
    if mode not in MODES:
        raise ValueError(f"mode must be one of {sorted(MODES)}")
    return NormalizeFunction.apply(feat, st.stats, lay, st, None, mode)


def normalized_windows_grad(feat: torch.Tensor, lay: Layout, st: SpeakerStats, win_utt: np.ndarray, win_t0: np.ndarray,
                            mode: str = "znorm", win_len: int = WIN_LEN) -> torch.Tensor:
    """normalized_windows() with a gradient: bit-identical (n_windows, 1, win_len, F) windows with a grad_fn to feat and,
    when st.stats requires grad (from speaker_stats_grad), to the statistics, padded rows included (they depend on the
    statistics).  Any window table works (subsets, any order, repeated windows); win_t0 outside
    [0, 2^31 - 1 - win_len] or win_utt outside [0, n_utts) raises ValueError.  Deterministic (no atomics)."""
    _lib.require_cuda(feat)
    if mode not in MODES:
        raise ValueError(f"mode must be one of {sorted(MODES)}")
    wu, wt = _check_window_table(win_utt, win_t0, len(lay.frame_off_host) - 1, win_len)
    return NormalizeFunction.apply(feat, st.stats, lay, st, (wu, wt, win_len), mode)
