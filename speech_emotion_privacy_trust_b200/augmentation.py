"""Class-balance noise augmentation of the training windows on the device.

Mirrors preprocess_data/preprocess_adversary_data.py:392-421 of the reference: every class smaller than the largest one
is topped up by re-drawing windows of that class (np.random.randint) and adding N(0, 0.05) noise.  In the reference the
new key aliases the dict of the window it was drawn from and the noisy array is written through the alias, so a window
drawn m times ends up as original + n_1 + ... + n_m and the window and all its copies share that array.  The plan below
reproduces the draws (same order, same RNG calls) and the sharing: `alias_of[k]` is the row that key k -- originals
first, then the new keys in creation order -- reads; the kernel (csrc/augment.cu) adds the samples to the source rows.
"""
from __future__ import annotations

from collections import Counter
from dataclasses import dataclass
from typing import Callable, Optional, Sequence

import numpy as np
import torch

from . import _lib


@dataclass
class BalancePlan:
    alias_of: np.ndarray        # (n + n_aug,) row of every key: originals, then augmented keys in creation order
    draw_rows: np.ndarray       # (n_aug,) source row of every noise sample, in draw order
    labels: list                # label of every key (an augmented key carries its source's label)

    @property
    def n_aug(self) -> int:
        return int(self.draw_rows.size)


def class_balance_plan(labels: Sequence, randint: Optional[Callable] = None) -> BalancePlan:
    """labels[i] is the class (emotion or gender, the reference's --aug choice) of training window i.  randint defaults
    to np.random.randint -- the reference draws from NumPy's global generator -- and is called once per minority class
    in first-occurrence order of the classes, exactly like :398-414."""
    randint = np.random.randint if randint is None else randint
    labels = list(labels)
    counts = Counter(labels)                                       # insertion order = first occurrence (:394, :398)
    max_size = max(counts.values()) if counts else 0
    alias_of = list(range(len(labels)))
    key_labels = list(labels)
    draw_rows = []
    for label in counts:
        if counts[label] == max_size:
            continue
        n_aug = max_size - counts[label]
        # keys of this class in dict order; keys added for earlier classes alias dicts of those classes: never a match
        pool = [k for k in range(len(alias_of)) if key_labels[k] == label]
        for aug_idx in np.asarray(randint(0, len(pool), size=n_aug)).tolist():
            row = alias_of[pool[aug_idx]]
            draw_rows.append(row)
            alias_of.append(row)
            key_labels.append(label)
    return BalancePlan(np.asarray(alias_of, np.int64), np.asarray(draw_rows, np.int64), key_labels)


def apply_plan(windows: torch.Tensor, plan: BalancePlan, std: float = 0.05, seed: int = 0,
               noise: Optional[torch.Tensor] = None, inplace: bool = False) -> torch.Tensor:
    """windows: (n, ...) fp32 CUDA tensor of training windows.  Returns the tensor whose rows carry the accumulated noise
    of their draws; key k of the augmented set is `out[plan.alias_of[k]]`.  noise: optional (n_aug, ...) samples to add
    instead of the device's Philox draws (parity tests)."""
    _lib.require_cuda(windows)
    if windows.dtype != torch.float32 or not windows.is_contiguous():
        raise ValueError("windows must be a contiguous float32 tensor")
    out = windows if inplace else windows.clone()
    if plan.n_aug == 0:
        return out
    row_elems = int(windows[0].numel())
    order = np.argsort(plan.draw_rows, kind="stable")             # draws of one row stay in draw order
    rows, starts = np.unique(plan.draw_rows[order], return_index=True)
    job_ptr = np.concatenate([starts, [order.size]]).astype(np.int32)
    dev = windows.device
    job_row = torch.from_numpy(rows.astype(np.int64)).to(dev)
    job_ptr_t = torch.from_numpy(job_ptr).to(dev)
    draw_id = torch.from_numpy(order.astype(np.int64)).to(dev)
    if noise is not None:
        _lib.require_cuda(noise)
        if noise.dtype != torch.float32 or not noise.is_contiguous() or noise.numel() != plan.n_aug * row_elems:
            raise ValueError("noise must be a contiguous float32 tensor of shape (n_aug, *window shape)")
    for j0 in range(0, rows.size, 65535):
        j1 = min(rows.size, j0 + 65535)
        _lib.launch("sept_add_noise_rows_f32", out, job_row[j0:], job_ptr_t[j0:], draw_id, j1 - j0, row_elems, seed, std, noise,
                    device=dev)
    return out


def class_balance(windows: torch.Tensor, labels: Sequence, std: float = 0.05, seed: int = 0,
                  randint: Optional[Callable] = None):
    """One call: (augmented rows, alias_of, labels of every key)."""
    plan = class_balance_plan(labels, randint)
    return apply_plan(windows, plan, std=std, seed=seed), torch.from_numpy(plan.alias_of), plan.labels
