"""Integrated-gradients attribution of ``CnnGruAttentionModel`` predictions over input channels and time.

For window b with target class c_b, F_b(z) = model(z)[c_b] in eval mode, baseline x0_b (default zeros: the subject
mean of the z-scored windows) and the midpoint rule alpha_k = (k + 1/2) / m, k = 0..m-1:

    A_b     = (x_b - x0_b) * (1/m) sum_k grad_z F_b(x0_b + alpha_k (x_b - x0_b))     float32 [C, T]
    S_b,c   = sum_t A_b,c,t                                                         float64
    delta_b = sum_c S_b,c - (F_b(x_b) - F_b(x0_b))                                  float64, the completeness residual

Eval mode is required: BatchNorm then uses the running statistics, so the B * m interpolation rows are independent
and can be batched freely, and there is no dropout.  The rows are cut into chunks of at most ``max_rows``; each chunk is
one eval forward and one input-gradient-only backward (``mms_cnngru_input_gradient``: no parameter gradient is formed),
with the interpolation and the accumulation in their own kernels.  Every sum over k runs in a fixed order, so A does
not depend on the chunking beyond the last-bit differences of a different GEMM choice at a different chunk size.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _ext
from ._ext import check, ptr, stream


def integrated_gradients(model, x, target=None, baseline=None, steps=32, max_rows=2048):
    """Integrated gradients of ``model`` (``CnnGruAttentionModel``, eval mode, on CUDA) at windows ``x [B, C, T]``.

    ``target``: int64 [B] class per window (default: the argmax of the eval logits, first maximum).
    ``baseline``: [C, T] shared by every window or [B, C, T]; default zeros.
    Returns ``(A, S, delta)``: float32 [B, C, T], float64 [B, C] and float64 [B]."""
    if model.training:
        raise ValueError("integrated_gradients needs model.eval(): BatchNorm must use its running statistics")
    if not isinstance(x, torch.Tensor) or not x.is_cuda:
        raise _ext.MmsError("integrated_gradients: x must be a CUDA tensor (no CPU fallback)")
    if x.dim() != 3 or x.shape[1] != model.in_channels:
        raise ValueError(f"integrated_gradients: expected x of shape [B, {model.in_channels}, T], got {tuple(x.shape)}")
    steps, max_rows = int(steps), int(max_rows)
    if steps < 1 or max_rows < 1:
        raise ValueError("integrated_gradients: steps and max_rows must be >= 1")
    x = x.detach().contiguous().float()
    B, Cc, T = x.shape
    nc = model.num_classes
    if baseline is None:
        x0, per_window = torch.zeros(Cc, T, device=x.device, dtype=torch.float32), 0
    else:
        if not isinstance(baseline, torch.Tensor) or not baseline.is_cuda:
            raise _ext.MmsError("integrated_gradients: the baseline must be a CUDA tensor")
        if tuple(baseline.shape) == (Cc, T):
            per_window = 0
        elif tuple(baseline.shape) == (B, Cc, T):
            per_window = 1
        else:
            raise ValueError(f"integrated_gradients: baseline of shape {tuple(baseline.shape)} does not broadcast to "
                             f"{tuple(x.shape)}; expected [C, T] or [B, C, T]")
        x0 = baseline.detach().contiguous().float()
    with torch.no_grad():
        fx = model(x)
        f0 = model(x0.expand(B, Cc, T).contiguous() if not per_window else x0)
    if target is None:
        target = torch.argmax(fx, dim=1)
    else:
        target = torch.as_tensor(target, device=x.device).to(torch.int64).reshape(-1)
        if target.numel() != B:
            raise ValueError(f"integrated_gradients: {target.numel()} targets for {B} windows")
        if bool(((target < 0) | (target >= nc)).any()):
            raise ValueError(f"integrated_gradients: a target outside [0, {nc})")
    target = target.contiguous()

    lib = _ext.lib()
    model._ensure_flat(x.device)
    A = torch.zeros(B, Cc, T, device=x.device, dtype=torch.float32)
    S = torch.zeros(B, Cc, device=x.device, dtype=torch.float64)
    total = B * steps
    chunk = min(max_rows, total)
    bufs = {}
    for row0 in range(0, total, chunk):
        n = min(chunk, total - row0)
        if n not in bufs:          # one engine (workspace) and one set of buffers per chunk size
            eng = model.engine(n, T, False, True, x.device)
            bufs[n] = (eng, torch.empty(n, Cc, T, device=x.device), torch.empty(n, nc, device=x.device),
                       torch.empty(n, Cc, T, device=x.device))
        eng, z, dl, dx = bufs[n]
        check(lib.mms_ig_interpolate(ptr(x), ptr(x0), per_window, ptr(target), B, Cc, T, nc, steps, row0, n, ptr(z), ptr(dl),
                                     stream()))
        model._rng_calls += 1
        eng.forward(z, model._rng_calls)
        eng.input_gradient(z, dl, dx)
        check(lib.mms_ig_accumulate(ptr(x), ptr(x0), per_window, ptr(dx), B, Cc, T, steps, row0, n, ptr(A), ptr(S), stream()))
    idx = torch.arange(B, device=x.device)
    delta = S.sum(dim=1) - (fx[idx, target].double() - f0[idx, target].double())
    return A, S, delta


def channel_shares(S):
    """|S_b,c| / sum_c' |S_b,c'| per window (float64 [B, C]); a window whose attributions are all zero gets zeros."""
    a = S.abs()
    tot = a.sum(dim=1, keepdim=True)
    return torch.where(tot > 0, a / tot.clamp_min(torch.finfo(torch.float64).tiny), torch.zeros_like(a))
