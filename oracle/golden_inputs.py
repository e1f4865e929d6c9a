"""Inputs of the golden fixtures under ``tests/golden/``, rebuilt from their seeds instead of stored.

TEST INFRASTRUCTURE ONLY.  ``oracle/make_golden.py`` runs the reference on these inputs and stores, beside the
reference's outputs, the SHA-256 of every input; ``tests/conftest.py`` rebuilds the inputs and refuses a fixture whose
digest differs, so a test never compares the reference's outputs with results computed from other inputs.

- model fixtures: windows ``synth.synthetic_windows(B, C, T, seed=C * 100 + B)``; weights initialised after
  ``torch.manual_seed(1234 + C)`` (this package's ``CnnGruAttentionModel`` initialises exactly as the reference's
  does: same modules, same order), then the two BatchNorm layers' affine parameters moved off their trivial values.
- resample fixture: random walks drawn from ``np.random.default_rng(7)``, one per case of ``RESAMPLE_CASES``.

Outputs larger than ``SUBSET`` elements are stored as a fixed seeded subset of their elements (``subset_indices``).
"""
from __future__ import annotations

import hashlib
import warnings
import zlib

import numpy as np

SUBSET = 256

# (n, k, original_fs, target_fs): down-sampling (700 -> 64/128), up-sampling (4, 32 -> 64), identity (64 -> 64),
# even and odd lengths
RESAMPLE_CASES = [
    (7137, 1, 700, 64), (7000, 1, 700, 64), (7001, 3, 700, 128), (6999, 1, 700, 64),
    (240, 1, 4, 64), (241, 1, 4, 64), (1920, 3, 32, 64), (1921, 1, 32, 64),
    (3840, 1, 64, 64), (3841, 1, 64, 64), (21011, 1, 700, 64), (16384, 1, 700, 64),
]


def digest(a) -> str:
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()


def subset_indices(name: str, size: int):
    """Sorted flat indices of the elements kept of an output of ``size`` elements (None: all are kept)."""
    if size <= SUBSET:
        return None
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    return np.sort(rng.choice(size, SUBSET, replace=False)).astype(np.int32)


def model_windows(C, nc, B, T):
    from multimodalsignal_b200 import synth
    return synth.synthetic_windows(B, C, T, seed=C * 100 + B, num_classes=nc)


def perturb_batchnorm(model):
    """Move the BatchNorm affine parameters off their trivial init so the fixtures test them."""
    import torch
    with torch.no_grad():
        for k, v in model.named_parameters():
            if "cnn_encoder.1" in k or "cnn_encoder.5" in k:
                v.add_(0.1 * torch.randn_like(v))


def model_state(C, nc, kwargs):
    """The initial state_dict of a model fixture, as numpy arrays."""
    import torch
    from multimodalsignal_b200.models import CnnGruAttentionModel
    torch.manual_seed(1234 + C)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model = CnnGruAttentionModel(in_channels=C, num_classes=nc, dropout=0.0, **kwargs)
    perturb_batchnorm(model)
    return {k: v.detach().numpy().copy() for k, v in model.state_dict().items()}


def resample_signals():
    rng = np.random.default_rng(7)
    out = []
    for i, (n, k, _, _) in enumerate(RESAMPLE_CASES):
        x = rng.standard_normal((n, k)).cumsum(axis=0) * 0.05 + rng.standard_normal((n, k))
        out.append(x[:, 0] if k == 1 and i % 2 == 0 else x)
    return out
