"""Float64 integrated gradients through the oracle model, with autograd.

TEST INFRASTRUCTURE ONLY (see ``model_oracle``).  The definition is the one of
``multimodalsignal_b200.attribution``: midpoint rule alpha_k = (k + 1/2) / m, target = argmax of the eval
logits unless given, baseline zeros unless given ([C, T] or [B, C, T]).
"""
from __future__ import annotations

import torch

from oracle import model_oracle as mo


def integrated_gradients_fn(f, x, target=None, baseline=None, steps=32):
    """IG of any batched function ``f(z [N, C, T]) -> logits [N, nc]`` whose rows are independent.
    Returns ``(A [B,C,T], S [B,C], delta [B], target [B])`` in the dtype of ``x``."""
    B = x.shape[0]
    x0 = torch.zeros_like(x[0]) if baseline is None else baseline.to(x.dtype)
    x0 = x0.expand_as(x) if x0.dim() == 2 else x0
    with torch.no_grad():
        fx, f0 = f(x), f(x0)
    if target is None:
        target = torch.argmax(fx, dim=1)
    target = torch.as_tensor(target).to(torch.int64)
    alpha = (torch.arange(steps, dtype=x.dtype) + 0.5) / steps
    # all B * m rows at once: row b * m + k
    z = (x0[:, None] + alpha[None, :, None, None] * (x - x0)[:, None]).reshape(B * steps, *x.shape[1:])
    z.requires_grad_(True)
    logits = f(z)
    sel = logits.gather(1, target.repeat_interleave(steps)[:, None]).sum()
    (g,) = torch.autograd.grad(sel, z)
    A = (x - x0) * g.reshape(B, steps, *x.shape[1:]).mean(dim=1)
    S = A.sum(dim=2)
    idx = torch.arange(B)
    delta = S.sum(dim=1) - (fx[idx, target] - f0[idx, target])
    return A.detach(), S.detach(), delta.detach(), target


def integrated_gradients(params, bn_buffers, x, target=None, baseline=None, steps=32, gru_layers=2, attention=True):
    """IG of the eval-mode oracle model (``model_oracle.forward(training=False)``) in float64.
    ``params`` / ``bn_buffers`` map state_dict keys to tensors (converted to float64 here)."""
    p = {k: v.double() for k, v in params.items()}
    bn = {k: v.double() for k, v in bn_buffers.items()}
    f = lambda z: mo.forward(p, z, training=False, bn_buffers=bn, gru_layers=gru_layers, attention=attention, prune=True)[0]
    return integrated_gradients_fn(f, x.double(), target=target, baseline=None if baseline is None else baseline.double(),
                                   steps=steps)
