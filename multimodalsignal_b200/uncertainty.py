"""Monte-Carlo dropout predictive uncertainty of ``CnnGruAttentionModel`` predictions.

BatchNorm stays in eval mode (running statistics), dropout stays on, and each window is run ``samples`` times with
independent masks.  For window b with per-sample softmax p_s (s = 0..m-1):

    probs_b       = (1/m) sum_s p_s                                  the MC predictive distribution
    entropy_b     = H(probs_b) = -sum_c probs log probs              total predictive uncertainty
    mutual_info_b = H(probs_b) - (1/m) sum_s H(p_s)                  its model (epistemic) part, BALD

Sample s of window b is sample row r = b * m + s of the call, and row r draws exactly the multipliers a training-mode
forward of the expanded batch would draw at row r (``oracle/dropout_stream.py``).  No dropout acts before the first GRU
layer's output, so the library runs the encoder and GRU layer 0 once per window and only the layers above and the head
per sample (``mms_cnngru_mc_forward``).  The rows are cut into chunks of whole windows, at most ``max_rows`` sample rows
each; the statistics are summed in float64 in a fixed order (``mms_mc_accumulate``), so they do not depend on the chunking.

``model(x)`` ignores per-submodule ``train()`` / ``eval()`` flags, so the usual torch recipe (``model.eval()`` and then
``.train()`` on the dropout modules) returns m identical samples here: ``mc_dropout`` is the way in.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from . import _ext
from ._ext import CnnGruDesc, check, ptr, stream

SITE0_LIMIT = 1 << 38          # the head site's first dropout id: site-0 ids of the sample rows must stay below it


def gru_seq_len(T):
    """Length L of the sequence the GRU sees for a window of T samples (conv 7/2/3, pool 3/2/1, conv 5/2/2, pool 3/2/1)."""
    conv = lambda l, k, s, p: (l + 2 * p - k) // s + 1
    pool = lambda l: (l + 2 - 3) // 2 + 1
    return pool(conv(pool(conv(int(T), 7, 2, 3)), 5, 2, 2))


@dataclass
class McDropoutResult:
    probs: torch.Tensor          # float64 [B, nc]: mean softmax over the samples
    entropy: torch.Tensor        # float64 [B]: entropy of probs
    mutual_info: torch.Tensor    # float64 [B]: entropy - mean per-sample entropy
    logits: torch.Tensor         # float32 [B, samples, nc]
    prediction: torch.Tensor     # int64 [B]: first argmax of probs
    seed: int
    offset: int


class _McEngine:
    """Descriptor + workspace of one MC chunk size (windows per chunk, window length, samples)."""

    def __init__(self, model, B, T, samples, device):
        self.lib = _ext.lib()
        d = CnnGruDesc()
        d.batch, d.in_channels, d.seq_len, d.num_classes = B, model.in_channels, T, model.num_classes
        d.cnn_out, d.hidden, d.layers = model.cnn_out_channels, model.gru_hidden_size, model.gru_num_layers
        d.training, d.attention, d.need_grad = 0, int(model.attention), 0
        d.dropout_p = float(model.dropout_p)
        self.desc = d
        nbytes = self.lib.mms_cnngru_mc_workspace_bytes(C.byref(d), samples)
        if nbytes < 0:
            check(int(nbytes))
        self.workspace = torch.empty(int(nbytes), dtype=torch.uint8, device=device)

    def forward(self, model, x, samples, row0, seed, offset, logits):
        self.desc.rng_seed, self.desc.rng_offset = seed, offset
        check(self.lib.mms_cnngru_mc_forward(C.byref(self.desc), ptr(x), ptr(model._flat), ptr(model._bn_flat),
                                             ptr(self.workspace), samples, row0, ptr(logits), stream()))


def mc_dropout(model, x, samples=32, seed=None, max_rows=2048):
    """MC-dropout predictive distribution of ``model`` (``CnnGruAttentionModel`` in eval mode, on CUDA) at windows
    ``x [B, C, T]`` with ``samples`` forward samples per window.

    ``seed=None`` draws the masks from ``model._rng_seed`` at offset ``++model._rng_calls`` (a fresh set per call); an
    explicit seed uses offset 0, so the result depends only on the weights, x, samples and the seed.  At most
    ``max_rows`` sample rows (whole windows, ``max_rows // samples`` of them) run at once."""
    if model.training:
        raise ValueError("mc_dropout needs model.eval(): BatchNorm must use its running statistics")
    if not isinstance(x, torch.Tensor) or not x.is_cuda:
        raise _ext.MmsError("mc_dropout: x must be a CUDA tensor (no CPU fallback)")
    if x.dim() != 3 or x.shape[1] != model.in_channels:
        raise ValueError(f"mc_dropout: expected x of shape [B, {model.in_channels}, T], got {tuple(x.shape)}")
    samples, max_rows = int(samples), int(max_rows)
    if samples < 1:
        raise ValueError("mc_dropout: samples must be >= 1")
    if max_rows < samples:
        raise ValueError(f"mc_dropout: max_rows {max_rows} is smaller than one window's {samples} samples")
    B, _, T = x.shape
    L, H = gru_seq_len(T), model.gru_hidden_size
    if B * samples * L * 2 * H >= SITE0_LIMIT:
        raise ValueError(f"mc_dropout: {B} windows x {samples} samples x L = {L} x 2H = {2 * H} reach 2^38, where the "
                         "first GRU dropout site's ids would collide with the head's; split the call")
    if seed is None:
        model._rng_calls += 1
        seed, offset = int(model._rng_seed), int(model._rng_calls)
    else:
        seed, offset = int(seed) & 0xFFFFFFFFFFFFFFFF, 0
    x = x.detach().contiguous().float()
    nc = model.num_classes
    lib = _ext.lib()
    model._ensure_flat(x.device)
    dev = x.device
    logits = torch.empty(B * samples, nc, device=dev, dtype=torch.float32)
    psum = torch.zeros(B, nc, device=dev, dtype=torch.float64)
    hsum = torch.zeros(B, device=dev, dtype=torch.float64)
    probs = torch.empty(B, nc, device=dev, dtype=torch.float64)
    entropy = torch.empty(B, device=dev, dtype=torch.float64)
    mutual_info = torch.empty(B, device=dev, dtype=torch.float64)
    per_chunk = max_rows // samples
    for b0 in range(0, B, per_chunk):
        nb = min(per_chunk, B - b0)
        key = ("mc", nb, T, samples)        # one engine (workspace) per chunk size, kept with the model's engines
        eng = model._engines.get(key)
        if eng is None:
            eng = model._engines[key] = _McEngine(model, nb, T, samples, dev)
        r0, n = b0 * samples, nb * samples
        chunk_logits = logits[r0:r0 + n]
        eng.forward(model, x[b0:b0 + nb], samples, r0, seed, offset, chunk_logits)
        check(lib.mms_mc_accumulate(ptr(chunk_logits), B, nc, samples, r0, n, ptr(psum), ptr(hsum), ptr(probs), ptr(entropy),
                                    ptr(mutual_info), stream()))
    return McDropoutResult(probs=probs, entropy=entropy, mutual_info=mutual_info, logits=logits.view(B, samples, nc),
                           prediction=torch.argmax(probs, dim=1), seed=seed, offset=offset)


def auroc(scores, positive):
    """Area under the ROC curve of ``scores`` as a detector of ``positive`` (bool), by the rank-sum (Mann-Whitney)
    formula with tied scores given their average rank: equal to ``sklearn.metrics.roc_auc_score(positive, scores)``.
    NaN when every window is positive or none is."""
    s = np.asarray(scores, dtype=np.float64).reshape(-1)
    pos = np.asarray(positive, dtype=bool).reshape(-1)
    if s.shape != pos.shape:
        raise ValueError(f"auroc: {s.size} scores for {pos.size} labels")
    n_pos = int(pos.sum())
    n_neg = pos.size - n_pos
    if n_pos == 0 or n_neg == 0:
        return float("nan")
    _, inv, cnt = np.unique(s, return_inverse=True, return_counts=True)
    ranks = (np.cumsum(cnt) - 0.5 * (cnt - 1))[inv]          # 1-based, the average over each run of equal scores
    return float((ranks[pos].sum() - n_pos * (n_pos + 1) / 2.0) / (n_pos * n_neg))


def expected_calibration_error(probs, labels, bins=10):
    """ECE of the predictive distribution ``probs [N, nc]`` against ``labels [N]``: the confidence max_c probs falls
    into one of ``bins`` equal-width bins [k/bins, (k+1)/bins) (the last one closed at 1), and
    ECE = sum_k (n_k / N) |acc_k - conf_k| over the non-empty bins.  0 for N = 0."""
    p = np.asarray(probs, dtype=np.float64)
    y = np.asarray(labels).reshape(-1).astype(np.int64)
    if p.ndim != 2 or p.shape[0] != y.size:
        raise ValueError(f"expected_calibration_error: probs of shape {p.shape} for {y.size} labels")
    if y.size == 0:
        return 0.0
    conf = p.max(axis=1)
    correct = (p.argmax(axis=1) == y).astype(np.float64)
    k = np.minimum((conf * bins).astype(np.int64), bins - 1)
    ece = 0.0
    for b in range(bins):
        sel = k == b
        nb = int(sel.sum())
        if nb:
            ece += nb / y.size * abs(correct[sel].mean() - conf[sel].mean())
    return float(ece)
