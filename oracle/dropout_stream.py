"""Host (numpy) port of the kernels' counter-based dropout stream (``DropRng`` in
``multimodalsignal_b200/csrc/mms_common.cuh``).

TEST INFRASTRUCTURE ONLY, like the rest of ``oracle/``.

The stream is a pure function of (seed, offset, element id), so the exact multipliers a
training step drew can be rebuilt here and handed to ``model_oracle.forward(...,
drop_mask_gru=, drop_mask_head=)``: a dropout step is then checked in float64 like any
other.  It is this project's own stream, not torch's Philox stream.

Element-id contract (the project's definition; every kernel that draws a multiplier
computes one of these ids):

* GRU inter-layer site ``l`` (0 <= l < layers - 1), on layer l's output ``[B, L, 2H]``
  (forward direction in columns [0, H), reverse direction in [H, 2H))::

      id = l * 2**40 + (b * L + t) * 2H + j

* head site, on ``relu(classifier.0(last_output))`` ``[B, 64]``::

      id = 2**38 + b * 64 + i

``b`` is the row of the batch a device holds.  With data parallelism every rank uses its
own seed (``DataParallelTrainStep``), so the masks of the global batch are the ranks'
masks concatenated along the batch.

Seeds and offsets: ``CnnGruAttentionModel`` (autograd) uses ``model._rng_seed`` and the
forward call count ``model._rng_calls``; ``FusedTrainStep`` uses
``model._rng_seed ^ 0x5DEECE66D`` and the optimizer's step count before the step
(``FlatAdam.step_dev``, read on the device).
"""
from __future__ import annotations

import numpy as np

LAYER_STRIDE = 1 << 40          # DROP_LAYER_STRIDE in csrc/model.cu
HEAD_BASE = 1 << 38             # HEAD_DROP_BASE in csrc/head_opt.cu
HEAD_HID = 64
_M32 = 0xFFFFFFFF


def gru_seq_len(T):
    """Sequence length L the GRU sees for a window of T samples (reference models.py:46-53: conv 7/2/3, pool 3/2/1,
    conv 5/2/2, pool 3/2/1)."""
    conv = lambda l, k, s, p: (l + 2 * p - k) // s + 1
    pool = lambda l: (l + 2 - 3) // 2 + 1
    return pool(conv(pool(conv(T, 7, 2, 3)), 5, 2, 2))


def fmix32(h):
    """murmur3's 32-bit finaliser on a uint32 array (wrapping arithmetic, as in CUDA)."""
    h = np.asarray(h, dtype=np.uint32).copy()
    h ^= h >> np.uint32(16)
    h *= np.uint32(0x85EBCA6B)
    h ^= h >> np.uint32(13)
    h *= np.uint32(0xC2B2AE35)
    h ^= h >> np.uint32(16)
    return h


def _fmix(v):
    return int(fmix32(np.array([v & _M32], dtype=np.uint32))[0])


def keys(seed, offset):
    """``DropRng::init``: the two 32-bit keys of (seed, offset), both taken modulo 2**64."""
    seed, offset = int(seed) & 0xFFFFFFFFFFFFFFFF, int(offset) & 0xFFFFFFFFFFFFFFFF
    k0 = _fmix((seed & _M32) ^ 0x9E3779B9) ^ _fmix(((offset & _M32) + 0x7F4A7C15) & _M32)
    k1 = (_fmix((seed >> 32) ^ 0x85EBCA6B) + _fmix((offset >> 32) ^ 0xC2B2AE35)) & _M32
    return k0, k1


def uniforms(ids, seed, offset):
    """The float32 uniform u in [0, 1) of every element id (``DropRng::mult`` before the comparison)."""
    ids = np.asarray(ids, dtype=np.uint64)
    k0, k1 = keys(seed, offset)
    lo = (ids & np.uint64(_M32)).astype(np.uint32)
    hi = (ids >> np.uint64(32)).astype(np.uint32)
    h = fmix32(lo ^ np.uint32(k0))
    h = fmix32(h + np.uint32(k1) + hi * np.uint32(0x27D4EB2F))
    return (h >> np.uint32(8)).astype(np.float32) * np.float32(1.0 / 16777216.0)


def scale(p):
    """The kept multiplier 1/(1-p), computed in float32 as the kernels do."""
    p32 = np.float32(p)
    return np.float32(1.0) / (np.float32(1.0) - p32) if p32 < np.float32(1.0) else np.float32(0.0)


def multipliers(ids, p, seed, offset):
    """float32 multipliers of the element ids: 0 where u < float32(p), else float32(1/(1-p))."""
    u = uniforms(ids, seed, offset)
    return np.where(u >= np.float32(p), scale(p), np.float32(0.0)).astype(np.float32)


def gru_site_ids(layer, B, L, H):
    """Element ids [B, L, 2H] of GRU inter-layer site ``layer``."""
    n = np.arange(B * L * 2 * H, dtype=np.uint64)
    return (np.uint64(layer * LAYER_STRIDE) + n).reshape(B, L, 2 * H)


def head_site_ids(B):
    """Element ids [B, 64] of the head site."""
    return (np.uint64(HEAD_BASE) + np.arange(B * HEAD_HID, dtype=np.uint64)).reshape(B, HEAD_HID)


def gru_masks(B, L, H, layers, p, seed, offset):
    """float64 multipliers [layers - 1, B, L, 2H] of every GRU inter-layer site (``drop_mask_gru`` of the oracle);
    index ``l`` is applied to layer l's output."""
    out = np.empty((max(layers - 1, 0), B, L, 2 * H), dtype=np.float64)
    for l in range(layers - 1):
        out[l] = multipliers(gru_site_ids(l, B, L, H), p, seed, offset)
    return out


def head_mask(B, p, seed, offset):
    """float64 multipliers [B, 64] of the head site (``drop_mask_head`` of the oracle)."""
    return multipliers(head_site_ids(B), p, seed, offset).astype(np.float64)
