"""Waveform-domain cloak: a learned noise of period L added to the raw audio of a ragged batch, trained through the
differentiable extraction chain (wav -> wave cloak -> logmel_grad -> speaker_stats_grad -> normalized_windows_grad -> ...).

The signal-domain counterpart of cloak_noise (model/cloak_models.py:24-58): the same mu / rho parameterisation,
sigma = (1 + tanh rho)/2 * (max_scale - min_scale) + min_scale, the same device Philox eps (one (L,) sample per forward,
identical on every rank, fresh on every CUDA-graph replay) and a deterministic backward.  Forward: sept_cloak_fwd_f32 draws
noise = mu + sigma * eps, sept_wave_cloak_fwd_f32 tiles it over every utterance from the utterance's first sample.
Backward: dx = g; sept_wave_cloak_bwd_f32 sums g per phase, sept_cloak_grl_bwd_f32 turns that sum into dlocs and drhos.
Evaluation (WaveCloak.noisy_per_utterance): sept_wave_cloak_eval_f32 gives every utterance its own eps, drawn inside the
add kernel.  Training with that noise (WaveCloak(per_utterance=True)): the same forward, and a backward
(sept_wave_cloak_bwd_per_utt_f32) that draws each utterance's eps again to sum g * eps_u per phase."""
from __future__ import annotations

import numpy as np
import torch
import torch.nn as nn
from torch.autograd.function import once_differentiable

from . import _lib, cloak_ops
from .extraction import RaggedAudio

DEFAULT_PERIOD = 32000     # one 200-frame training window at hop 160
EPS_STD = 0.1              # cloak_noise's Normal(0, 0.1) (cloak_models.py:37)


def _aligned(t: torch.Tensor) -> torch.Tensor:
    """t, or a copy of it at a 16-byte aligned address (the kernels move float4s; a view at an odd offset needs the copy)."""
    return t if t.data_ptr() % 16 == 0 else t.clone()


def new_workspace(device: torch.device, period: int) -> tuple[torch.Tensor, torch.Tensor]:
    """(partial rows of the phase reduction, workspace of the mu / rho backward).  The owner decides their lifetime, as
    with cloak_ops.new_workspace: a WaveCloak layer allocates them on its first forward, before any CUDA-graph capture;
    callers of WaveCloakFunction without one get fresh ones per backward."""
    nbytes = _lib.lib().sept_wave_cloak_bwd_workspace_bytes(period)
    if nbytes == 0:
        raise ValueError(f"period={period} must be a positive multiple of 4")
    return _lib.workspace(nbytes, device), cloak_ops.new_workspace(device, period)


class WaveCloakFunction(torch.autograd.Function):
    """y = wav + noise[(s - utt_off[u]) mod L] over every utterance u of `batch` (samples outside every utterance
    unchanged), noise = locs + sigma(rhos) * eps.  eps: a caller's (L,) sample, or None to draw it on the device from
    Philox(seed, offset) at the draw counter `draw` (advanced by one).  No double backward."""

    @staticmethod
    def forward(ctx, wav, locs, rhos, batch, eps, seed, offset, eps_std, min_scale, max_scale, draw=None, workspace=None):
        _lib.require_cuda(wav)
        period = locs.numel()
        if rhos.numel() != period:
            raise ValueError(f"locs ({period}) and rhos ({rhos.numel()}) must have one element per phase")
        if wav.shape != batch.wav.shape:
            raise ValueError(f"wav of shape {tuple(wav.shape)} is not the batch's buffer {tuple(batch.wav.shape)}")
        tiles = batch.tiles(period)                                  # ValueError unless period is a multiple of 4
        locs_c, rhos_c = cloak_ops._f32c(locs.detach()), cloak_ops._f32c(rhos.detach())
        eps_c = None
        if eps is not None:
            eps_c = cloak_ops._f32c(eps.detach().to(wav.device)).reshape(-1)
            if eps_c.numel() != period:
                raise ValueError(f"eps has {eps_c.numel()} elements; the period is {period}")
        _, eps_used, noise = cloak_ops.cloak_forward_raw(None, locs_c, rhos_c, None, eps_c, seed, offset, eps_std,
                                                         min_scale, max_scale, want_noise=True, draw=draw)
        x = _aligned(wav.detach())
        y = torch.empty_like(x)
        _lib.launch("sept_wave_cloak_fwd_f32", x, batch.utt_off, batch.n_utts, x.numel(), noise, period, y, device=x.device)
        ctx.save_for_backward(eps_used, rhos_c)
        ctx.batch, ctx.tiles, ctx.workspace = batch, tiles, workspace
        ctx.cfg = (float(min_scale), float(max_scale), tuple(locs.shape), tuple(rhos.shape))
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        eps_used, rhos_c = ctx.saved_tensors
        min_scale, max_scale, lshape, rshape = ctx.cfg
        batch, tiles = ctx.batch, ctx.tiles
        period = rhos_c.numel()
        need_wav, need_locs, need_rhos = ctx.needs_input_grad[:3]
        dlocs = drhos = None
        if need_locs or need_rhos:
            gc = _aligned(cloak_ops._f32c(g))
            dev = gc.device
            ws_r, ws_c = ctx.workspace if ctx.workspace is not None else new_workspace(dev, period)
            r = torch.empty(period, dtype=torch.float32, device=dev)
            dlocs = torch.empty(period, dtype=torch.float32, device=dev)
            drhos = torch.empty(period, dtype=torch.float32, device=dev) if need_rhos else None
            _lib.launch("sept_wave_cloak_bwd_f32", gc, batch.utt_off, tiles.tile_off, batch.n_utts, tiles.n_tiles, period, ws_r,
                        r, device=dev)
            _lib.launch("sept_cloak_grl_bwd_f32", r, None, 0.0, eps_used, rhos_c, None, min_scale, max_scale, 1, period, ws_c,
                        dlocs, drhos, None, device=dev)
        return (g if need_wav else None, dlocs.view(lshape) if need_locs else None,
                drhos.view(rshape) if need_rhos else None) + (None,) * 9


def new_per_utt_workspace(device: torch.device, period: int) -> tuple[torch.Tensor, torch.Tensor]:
    """(the two partial-row sets of the per-utterance backward, sigma of the period for the forward), owned as
    new_workspace's are."""
    lib = _lib.lib()
    nbytes = lib.sept_wave_cloak_bwd_per_utt_workspace_bytes(period)
    if nbytes == 0:
        raise ValueError(f"period={period} must be a positive multiple of 4")
    return _lib.workspace(nbytes, device), _lib.workspace(lib.sept_wave_cloak_eval_workspace_bytes(period), device)


class WaveCloakPerUttFunction(torch.autograd.Function):
    """y = wav + (locs + sigma(rhos) * eps_u)[(s - utt_off[u]) mod L] over every utterance u of `batch`, a fresh eps_u per
    utterance (sept_wave_cloak_eval_f32's draw rule).  eps: the caller's (n_utts, L) rows, or None to draw on the device at
    draw index *draw + utt_draw[u] (or + u).  draw is the draw base itself, a device int64 tensor the caller does not move
    afterwards: the backward draws every eps_u again from it.  No double backward."""

    @staticmethod
    def forward(ctx, wav, locs, rhos, batch, eps, seed, draw, utt_draw, eps_std, min_scale, max_scale, workspace=None):
        _lib.require_cuda(wav)
        period = locs.numel()
        if rhos.numel() != period:
            raise ValueError(f"locs ({period}) and rhos ({rhos.numel()}) must have one element per phase")
        if wav.shape != batch.wav.shape:
            raise ValueError(f"wav of shape {tuple(wav.shape)} is not the batch's buffer {tuple(batch.wav.shape)}")
        tiles = batch.tiles(period)                                  # ValueError unless period is a multiple of 4
        dev = wav.device
        ws = workspace if workspace is not None else new_per_utt_workspace(dev, period)
        locs_c, rhos_c = cloak_ops._f32c(locs.detach()), cloak_ops._f32c(rhos.detach())
        if eps is not None:
            eps = _aligned(cloak_ops._f32c(eps.detach().to(dev)))
            if tuple(eps.shape) != (batch.n_utts, period):
                raise ValueError(f"eps must be (n_utts, period) = ({batch.n_utts}, {period}), got {tuple(eps.shape)}")
        x = _aligned(wav.detach())
        y = torch.empty_like(x)
        seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        _lib.launch("sept_wave_cloak_eval_f32", x, batch.utt_off, batch.n_utts, x.numel(), locs_c, rhos_c, eps, seed, 0, draw,
                    utt_draw, eps_std, min_scale, max_scale, period, ws[1], y, device=dev)
        ctx.save_for_backward(rhos_c, eps, draw, utt_draw)
        ctx.batch, ctx.tiles, ctx.workspace = batch, tiles, workspace
        ctx.cfg = (seed, float(eps_std), float(min_scale), float(max_scale), tuple(locs.shape), tuple(rhos.shape))
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        rhos_c, eps, draw, utt_draw = ctx.saved_tensors
        seed, eps_std, min_scale, max_scale, lshape, rshape = ctx.cfg
        batch, tiles = ctx.batch, ctx.tiles
        period = rhos_c.numel()
        need_wav, need_locs, need_rhos = ctx.needs_input_grad[:3]
        dlocs = drhos = None
        if need_locs or need_rhos:
            gc = _aligned(cloak_ops._f32c(g))
            dev = gc.device
            rows = (ctx.workspace if ctx.workspace is not None else new_per_utt_workspace(dev, period))[0]
            dlocs = torch.empty(period, dtype=torch.float32, device=dev)
            if need_rhos:
                drhos = torch.empty(period, dtype=torch.float32, device=dev)
                _lib.launch("sept_wave_cloak_bwd_per_utt_f32", gc, batch.utt_off, tiles.tile_off, batch.n_utts, tiles.n_tiles,
                            period, rhos_c, eps, seed, 0, draw, utt_draw, eps_std, min_scale, max_scale, rows, dlocs, drhos,
                            device=dev)
            else:                                                    # dlocs is the plain phase sum of g
                _lib.launch("sept_wave_cloak_bwd_f32", gc, batch.utt_off, tiles.tile_off, batch.n_utts, tiles.n_tiles, period,
                            rows, dlocs, device=dev)
        return (g if need_wav else None, dlocs.view(lshape) if need_locs else None,
                drhos.view(rshape) if need_rhos else None) + (None,) * 9


class WaveCloak(nn.Module):
    """Learned waveform noise: forward(batch) returns a RaggedAudio with the same utterances whose wav is
    batch.wav + (locs + scales() * eps) tiled from each utterance's first sample, with a grad_fn to locs and rhos (and to
    batch.wav when that requires grad).

    locs, rhos: (period,) parameters, rhos starting at -2 like cloak_noise's (ones - 3).  eps is drawn on the device
    (Philox seeded with torch.initial_seed(), a device draw counter: identical on data-parallel ranks that share the
    seed, fresh on every replay of a captured CUDA graph); set `external_eps` to a (period,) tensor to supply it.

    per_utterance=False (the default): one eps per forward, shared by every utterance of the batch.  per_utterance=True:
    every utterance gets its own eps, drawn as noisy_per_utterance draws it, so the cloak trains on the noise it is
    evaluated with and the rho gradient averages over every utterance of the (global) batch; see forward."""

    def __init__(self, min_scale: float, max_scale: float, period: int = DEFAULT_PERIOD, locs: torch.Tensor | None = None,
                 device=None, per_utterance: bool = False):
        super().__init__()
        if period <= 0 or period % 4:
            raise ValueError(f"period={period} must be a positive multiple of 4")
        self.period = int(period)
        self.per_utterance = bool(per_utterance)
        self.min_scale, self.max_scale = float(min_scale), float(max_scale)
        init = torch.zeros(period) if locs is None else torch.as_tensor(locs, dtype=torch.float32).reshape(-1).clone()
        if init.numel() != period:
            raise ValueError(f"locs has {init.numel()} elements; the period is {period}")
        self.locs = nn.Parameter(init.to(device))
        self.rhos = nn.Parameter(torch.full((period,), -2.0, device=device))
        self.external_eps = None
        self._draws = None            # device counter of samples drawn (the Philox offset lives on the GPU)
        self._workspace = None        # backward workspaces, owned by the layer (allocated on the first forward)
        self._workspace_per_utt = None

    def scales(self) -> torch.Tensor:
        return (1.0 + torch.tanh(self.rhos)) / 2 * (self.max_scale - self.min_scale) + self.min_scale

    def _eps_source(self):
        if self.external_eps is not None:
            if self.external_eps.numel() != self.period:
                raise ValueError(f"external_eps has {self.external_eps.numel()} elements; the period is {self.period}")
            return self.external_eps, 0, None
        if self._draws is None or self._draws.device != self.rhos.device:
            self._draws = torch.zeros(1, dtype=torch.int64, device=self.rhos.device)
        return None, torch.initial_seed(), self._draws

    def _ws(self):
        if self._workspace is None or self._workspace[0].device != self.rhos.device:
            self._workspace = new_workspace(self.rhos.device, self.period)
        return self._workspace

    def _ws_per_utt(self):
        if self._workspace_per_utt is None or self._workspace_per_utt[0].device != self.rhos.device:
            self._workspace_per_utt = new_per_utt_workspace(self.rhos.device, self.period)
        return self._workspace_per_utt

    def _per_utt_draw(self, batch: RaggedAudio, utt_ids, n_draws, external_eps):
        """The per-utterance draw of noisy_per_utterance and of per-utterance training: checks utt_ids, n_draws and
        external_eps (every check before any launch) and returns (eps, seed, draw counter, device ids, n_draws)."""
        n = batch.n_utts
        L = self.period
        n_draws = n if n_draws is None else int(n_draws)
        ids = None
        if utt_ids is not None:
            ids = np.asarray(utt_ids).reshape(-1)
            if ids.size and not np.issubdtype(ids.dtype, np.integer):
                raise ValueError(f"utt_ids must be integers, got {ids.dtype}")
            ids = ids.astype(np.int64)
            if len(ids) != n:
                raise ValueError(f"utt_ids has {len(ids)} entries; the batch has {n} utterances")
            if len(ids) and (ids.min() < 0 or ids.max() >= n_draws):
                raise ValueError(f"utt_ids must lie in [0, n_draws = {n_draws})")
            if len(np.unique(ids)) != len(ids):
                raise ValueError("utt_ids must be distinct: two utterances would share one noise sample")
        elif n > n_draws:
            raise ValueError(f"n_draws = {n_draws} is smaller than the batch's {n} utterances")
        if external_eps is not None:
            if tuple(external_eps.shape) != (n, L):
                raise ValueError(f"external_eps must be (n_utts, period) = ({n}, {L}), got {tuple(external_eps.shape)}")
        elif self.external_eps is not None:
            raise ValueError("per-utterance noise draws one eps per utterance; layer.external_eps holds a single sample -- "
                             "pass external_eps=(n_utts, period) instead")
        _lib.require_cuda(batch.wav)
        dev = batch.wav.device
        if external_eps is not None:
            eps, seed, draw = _aligned(cloak_ops._f32c(external_eps.detach().to(dev))), 0, None
        else:
            eps, seed, draw = self._eps_source()
        return eps, seed, draw, None if ids is None else torch.from_numpy(ids).to(dev), n_draws

    def forward(self, batch: RaggedAudio, utt_ids=None, n_draws: int | None = None,
                external_eps: torch.Tensor | None = None) -> RaggedAudio:
        """Without per_utterance: batch.wav + (locs + scales() * eps) with one eps for the whole batch.

        With per_utterance: utterance u gets its own eps_u, drawn as noisy_per_utterance draws it (draw index = layer
        counter + utt_ids[u]; the same utt_ids / n_draws / external_eps rules), and the layer's counter then advances by
        n_draws.  Under data parallelism every rank passes its utterances' global ids and the global batch size as
        n_draws, so each utterance's noise is the one a single GPU would draw for it.  The backward draws every eps_u
        again from a copy of the counter this forward read, so several forwards before one backward, and every replay
        of a captured CUDA graph, each get the gradient of their own noise."""
        if not self.per_utterance:
            if utt_ids is not None or n_draws is not None or external_eps is not None:
                raise ValueError("utt_ids, n_draws and external_eps apply to per-utterance noise: build the layer with "
                                 "per_utterance=True")
            eps, seed, draw = self._eps_source()
            wav = WaveCloakFunction.apply(batch.wav, self.locs, self.rhos, batch, eps, seed, 0, EPS_STD, self.min_scale,
                                          self.max_scale, draw, self._ws())
            return batch.with_wav(wav)
        eps, seed, draw, d_ids, n_draws = self._per_utt_draw(batch, utt_ids, n_draws, external_eps)
        base = None if draw is None else draw.clone()            # the draw base of this forward, saved for its backward
        wav = WaveCloakPerUttFunction.apply(batch.wav, self.locs, self.rhos, batch, eps, seed, base, d_ids, EPS_STD,
                                            self.min_scale, self.max_scale, self._ws_per_utt())
        if draw is not None:
            _lib.launch("sept_counter_add_u64", draw, n_draws, device=draw.device)
        return batch.with_wav(wav)

    @torch.no_grad()
    def noisy_per_utterance(self, batch: RaggedAudio, utt_ids=None, n_draws: int | None = None,
                            external_eps: torch.Tensor | None = None) -> RaggedAudio:
        """The batch under the cloak with a fresh eps per utterance, as evaluation needs it (the reference never
        evaluates with one noise sample shared by many utterances): utterance u gets locs + scales() * eps_u tiled from
        its first sample, eps_u drawn on the device from draw index (layer counter) + utt_ids[u].  Returns a RaggedAudio
        with the same offsets and cached layouts.

        utt_ids: the utterances' global draw ids (default 0 .. n_utts - 1), non-negative, distinct and below n_draws
        (default n_utts).  With global ids an utterance's noise depends neither on its batch, nor on its position, nor on
        the rank holding it; the layer's draw counter then advances by n_draws, so the ranks of a sharded evaluation stay
        in step.  external_eps: (n_utts, period) samples, one per utterance in batch order (parity tests); the counter does
        not move.  layer.external_eps holds a single sample and is rejected, as cloak_evaluate rejects it."""
        eps, seed, draw, d_ids, n_draws = self._per_utt_draw(batch, utt_ids, n_draws, external_eps)
        L = self.period
        dev = batch.wav.device
        x = _aligned(batch.wav.detach())
        locs_c, rhos_c = cloak_ops._f32c(self.locs.detach()), cloak_ops._f32c(self.rhos.detach())
        ws = _lib.workspace(_lib.lib().sept_wave_cloak_eval_workspace_bytes(L), dev)
        y = torch.empty_like(x)
        _lib.launch("sept_wave_cloak_eval_f32", x, batch.utt_off, batch.n_utts, x.numel(), locs_c, rhos_c, eps,
                    int(seed) & 0xFFFFFFFFFFFFFFFF, 0, draw, d_ids, EPS_STD, self.min_scale, self.max_scale, L, ws, y,
                    device=dev)
        if draw is not None:
            _lib.launch("sept_counter_add_u64", draw, n_draws, device=dev)
        return batch.with_wav(y)
