"""Autograd bindings of the fused cloak / gradient-reversal kernels (csrc/cloak.cu via the C ABI)."""
from __future__ import annotations

import torch

from . import _lib


def new_workspace(device: torch.device, wf: int) -> torch.Tensor:
    """Partial-sum buffer + column counters of the backward kernel (counters start at zero; the kernel leaves them at
    zero again).  The OWNER decides its lifetime: a cloak_noise layer keeps one for as long as it lives -- allocated on
    its first forward, i.e. before any CUDA-graph capture of the step, never inside one -- and callers of the functional
    API get a fresh one per call.  Backward launches that may overlap (different streams) need different workspaces."""
    return _lib.workspace(_lib.lib().sept_cloak_bwd_workspace_bytes(wf), device, zeroed=True)


def _f32c(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


def _alias(t: torch.Tensor) -> torch.Tensor:
    """A second tensor object over the same storage (not an autograd view)."""
    return torch.empty(0, dtype=t.dtype, device=t.device).set_(t.untyped_storage(), t.storage_offset(), t.size(), t.stride())


def cloak_forward_raw(x, locs, rhos, mask, eps, seed, offset, eps_std, min_scale, max_scale, want_noise=False, draw=None,
                      per_sample=False):
    """One launch of sept_cloak_fwd_f32.  Returns (out, eps_used, noise | None).  x may be None (noise only).
    draw: optional device int64 counter of draws so far; it selects the Philox offset on the device and is advanced
    after the launch (CUDA-graph friendly: every replay draws a fresh eps).  per_sample: every batch element gets its own
    eps (eps, when supplied, is (B, wf)); inference only."""
    _lib.require_cuda(locs)
    wf = locs.numel()
    dev = locs.device
    batch = 0 if x is None else x.numel() // wf
    if x is not None and x.numel() != batch * wf:
        raise ValueError(f"input of shape {tuple(x.shape)} does not broadcast against locs of shape {tuple(locs.shape)}")
    out = torch.empty_like(x) if x is not None else None
    eps_used = torch.empty(batch * wf if per_sample else wf, dtype=torch.float32, device=dev) if eps is None else eps
    noise = torch.empty_like(locs) if want_noise else None
    _lib.launch("sept_cloak_fwd_f32", locs if x is None else x, locs, rhos, mask, eps, int(seed) & 0xFFFFFFFFFFFFFFFF,
                int(offset) & 0xFFFFFFFFFFFFFFFF, draw if eps is None else None, int(per_sample), float(eps_std),
                float(min_scale), float(max_scale), batch, wf, locs if out is None else out,
                eps_used if eps is None else None, noise, device=dev)
    if draw is not None and eps is None:
        _lib.launch("sept_counter_add_u64", draw, batch if per_sample else 1, device=dev)
    return out, eps_used, noise


class CloakNoiseFunction(torch.autograd.Function):
    """y = x*mask + locs + sigma(rhos)*eps*mask  (cloak_noise.forward, model/cloak_models.py:52-58).

    twin=True returns the same activations twice, (y, y_rev): gradients that arrive on y_rev are multiplied by
    -grl_lambda inside the one fused backward kernel, i.e. y_rev == GradientReversal(grl_lambda)(y) without the clone,
    the separate -lambda*g launch and autograd's gradient accumulation pass."""

    @staticmethod
    def forward(ctx, x, locs, rhos, mask, eps, seed, offset, eps_std, min_scale, max_scale, twin, grl_lambda, draw=None,
                workspace=None):
        _lib.require_cuda(x)
        x = _f32c(x)
        locs_c, rhos_c = _f32c(locs.detach()), _f32c(rhos.detach())
        mask_c = None if mask is None else _f32c(mask.detach().to(x.device))
        eps_c = None if eps is None else _f32c(eps.detach().to(x.device)).reshape(-1)
        out, eps_used, _ = cloak_forward_raw(x, locs_c, rhos_c, mask_c, eps_c, seed, offset, eps_std, min_scale, max_scale,
                                             draw=draw)
        ctx.save_for_backward(eps_used, rhos_c, mask_c)
        ctx.cfg = (float(min_scale), float(max_scale), float(grl_lambda), bool(twin), tuple(locs.shape))
        ctx.workspace = workspace
        if twin:
            return out, _alias(out)
        return out

    @staticmethod
    def backward(ctx, g_a, g_b=None):
        eps_used, rhos_c, mask_c = ctx.saved_tensors
        min_scale, max_scale, lam, twin, pshape = ctx.cfg
        if g_a is None and g_b is None:
            return (None,) * 14
        if g_a is None:
            g_a = torch.zeros_like(g_b)
        g_a = _f32c(g_a)
        g_b = None if g_b is None else _f32c(g_b)
        dev = g_a.device
        wf = rhos_c.numel()
        batch = g_a.numel() // wf
        need_x, need_locs, need_rhos = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.needs_input_grad[2]
        dlocs = torch.empty(wf, dtype=torch.float32, device=dev)
        drhos = torch.empty(wf, dtype=torch.float32, device=dev) if need_rhos else None
        dx = torch.empty_like(g_a) if need_x else None
        ws = ctx.workspace if ctx.workspace is not None else new_workspace(dev, wf)
        _lib.launch("sept_cloak_grl_bwd_f32", g_a, g_b, lam, eps_used, rhos_c, mask_c, min_scale, max_scale, batch, wf, ws,
                    dlocs, drhos, dx, device=dev)
        return (dx, dlocs.view(pshape) if need_locs else None, drhos.view(pshape) if need_rhos else None,
                None, None, None, None, None, None, None, None, None, None, None)


class GradientReversalFunction(torch.autograd.Function):
    """Identity forward, -lambda * g backward (model/reversal_gradient.py:5-23).  The forward returns a view instead
    of the reference's clone; the backward is one launch of sept_grl_bwd_f32 (no host->device scalar tensor)."""

    @staticmethod
    def forward(ctx, x, lambda_):
        ctx.lambda_ = float(lambda_)
        return x.view_as(x)

    @staticmethod
    def backward(ctx, grads):
        _lib.require_cuda(grads)
        g = _f32c(grads)
        dx = torch.empty_like(g)
        _lib.launch("sept_grl_bwd_f32", g, ctx.lambda_, g.numel(), dx, device=g.device)
        return dx, None
