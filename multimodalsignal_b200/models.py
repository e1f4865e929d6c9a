"""Drop-in for the reference ``models.py``: same classes, constructor arguments, tensor
shapes and ``state_dict`` layout (``best_model.pt`` files are interchangeable), but
``forward``/``backward`` run hand-written sm_100a kernels through ``libmms_b200.so``.

The ``torch.nn`` sub-modules created here are parameter holders only -- they are
constructed in the same order as reference models.py:42-71 so that a given
``torch.manual_seed`` yields bit-identical initial weights, and so that
``state_dict()`` has the reference's 34 keys.  Their own ``forward`` is never
called; there is no PyTorch / CPU fallback (a CPU tensor raises).

All parameters are views into ONE flat float32 buffer in the segment order of
``mms_cnngru_param_layout`` (include/mms_b200.h), which is what lets Adam and a
gradient all-reduce be single launches.
"""
from __future__ import annotations

import ctypes as C
import itertools

import torch
import torch.nn as nn

from . import _ext
from ._ext import CnnGruDesc, check, ptr, stream

_SEED_COUNTER = itertools.count(1)


class _ChanAttnFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w1, w2):
        lib = _ext.lib()
        x = x.contiguous()
        B, Cc, T = x.shape
        mean = torch.empty(B, Cc, device=x.device, dtype=torch.float32)
        gate = torch.empty_like(mean)
        y = torch.empty_like(x)
        check(lib.mms_chan_attn_fwd(ptr(x), ptr(w1) if w1.numel() else None, ptr(w2) if w2.numel() else None,
                                    B, Cc, T, ptr(mean), ptr(gate), ptr(y), stream()))
        ctx.save_for_backward(x, w1, w2, mean, gate)
        return y

    @staticmethod
    def backward(ctx, dy):
        lib = _ext.lib()
        x, w1, w2, mean, gate = ctx.saved_tensors
        B, Cc, T = x.shape
        dy = dy.contiguous()
        dx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        dw1, dw2 = torch.zeros_like(w1), torch.zeros_like(w2)
        scratch = torch.empty(4 * B * Cc, device=x.device, dtype=torch.float32)
        check(lib.mms_chan_attn_bwd(ptr(x), ptr(dy), ptr(w1) if w1.numel() else None, ptr(w2) if w2.numel() else None,
                                    ptr(mean), ptr(gate), B, Cc, T, ptr(dx),
                                    ptr(dw1) if dw1.numel() else None, ptr(dw2) if dw2.numel() else None,
                                    ptr(scratch), stream()))
        return dx, dw1, dw2


class ChannelAttention(nn.Module):
    """reference models.py:7-31.  ``forward(x[B,C,T]) -> x * sigmoid-gate[B,C,1]``."""

    def __init__(self, in_channels, reduction_ratio=4):
        super().__init__()
        if reduction_ratio != 4:
            raise NotImplementedError("the sm_100a kernels implement the reference's reduction_ratio=4 (models.py:12,42)")
        self.avg_pool = nn.AdaptiveAvgPool1d(1)
        self.fc = nn.Sequential(
            nn.Linear(in_channels, in_channels // reduction_ratio, bias=False),
            nn.ReLU(inplace=True),
            nn.Linear(in_channels // reduction_ratio, in_channels, bias=False),
            nn.Sigmoid(),
        )

    def forward(self, x):
        _require_cuda(x)
        return _ChanAttnFn.apply(x.float(), self.fc[0].weight, self.fc[2].weight)


def _no_flatten():
    """Stands in for ``nn.GRU.flatten_parameters``: the GRU module here only holds parameters (its cuDNN path is
    never run), so ``.to(device)`` must not pay for cuDNN's weight re-packing (and a cuDNN handle)."""


def _require_cuda(x):
    if not x.is_cuda:
        raise _ext.MmsError("multimodalsignal_b200 runs on a B200 only: got a CPU tensor and there is no CPU fallback")


class _Engine:
    """Workspace + descriptor for one (batch, channels, length, mode) configuration."""

    def __init__(self, model, B, T, training, need_grad, device):
        self.lib = _ext.lib()
        self.model = model
        self.key = (B, T, training, need_grad)
        d = CnnGruDesc()
        d.batch, d.in_channels, d.seq_len, d.num_classes = B, model.in_channels, T, model.num_classes
        d.cnn_out, d.hidden, d.layers = model.cnn_out_channels, model.gru_hidden_size, model.gru_num_layers
        d.training, d.attention, d.need_grad = int(training), int(model.attention), int(need_grad)
        d.dropout_p = float(model.dropout_p)
        d.rng_seed, d.rng_offset, d.rng_offset_dev = model._rng_seed, 0, None
        self.desc = d
        nbytes = self.lib.mms_cnngru_workspace_bytes(C.byref(d))
        if nbytes < 0:
            check(int(nbytes))
        self.workspace = torch.empty(int(nbytes), dtype=torch.uint8, device=device)
        self.generation = 0

    def forward(self, x, rng_offset):
        m = self.model
        self.desc.rng_offset = rng_offset
        logits = torch.empty(x.shape[0], m.num_classes, device=x.device, dtype=torch.float32)
        check(self.lib.mms_cnngru_forward(C.byref(self.desc), ptr(x), ptr(m._flat), ptr(m._bn_flat), ptr(m._nbt_flat),
                                          ptr(self.workspace), ptr(logits), stream()))
        self.generation += 1
        return logits

    def backward(self, x, dlogits, want_dx, frozen_segments=0):
        """Parameter gradients (flat, zeros in frozen segments) and optionally dx; the backward stops as early as the
        mask of frozen segments allows (desc.frozen_segments)."""
        m = self.model
        grads = torch.zeros_like(m._flat)
        dx = torch.empty_like(x) if want_dx else None
        self.desc.frozen_segments = frozen_segments
        try:
            check(self.lib.mms_cnngru_backward(C.byref(self.desc), ptr(x), ptr(m._flat), ptr(m._bn_flat), ptr(self.workspace),
                                               ptr(dlogits), ptr(grads), ptr(dx), stream()))
        finally:
            self.desc.frozen_segments = 0
        return grads, dx

    def input_gradient(self, x, dlogits, dx=None):
        """dx only (mms_cnngru_input_gradient) after an eval-mode forward with need_grad on this engine."""
        m = self.model
        if dx is None:
            dx = torch.empty_like(x)
        check(self.lib.mms_cnngru_input_gradient(C.byref(self.desc), ptr(x), ptr(m._flat), ptr(m._bn_flat),
                                                 ptr(self.workspace), ptr(dlogits), ptr(dx), stream()))
        return dx


class _CnnGruFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, model, engine, rng_offset, *params):
        logits = engine.forward(x, rng_offset)
        ctx.model, ctx.engine, ctx.generation = model, engine, engine.generation
        ctx.save_for_backward(x)
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        eng = ctx.engine
        if eng.generation != ctx.generation:
            raise _ext.MmsError("backward() after a newer forward() of the same shape: the activation workspace "
                                "holds one step (the reference trainer does forward->backward per batch, trainer.py:146-148)")
        (x,) = ctx.saved_tensors
        model = ctx.model
        want = ctx.needs_input_grad[4:]
        mask, _ = model.freeze_plan(want)
        if not any(want) and not eng.desc.training:
            # eval mode with every parameter frozen (model.eval().requires_grad_(False)): the input gradient alone, through
            # the eval-mode encoder kernels, no parameter-gradient work at all
            dx = eng.input_gradient(x, dlogits.contiguous().float())
            return (dx, None, None, None, *([None] * len(want)))
        grads, dx = eng.backward(x, dlogits.contiguous().float(), ctx.needs_input_grad[0], mask)
        out = [(grads[o:o + n].view(shape) if n else torch.zeros(shape, device=grads.device)) if w else None
               for (o, n, shape), w in zip(model._param_views, want)]
        return (dx, None, None, None, *out)


class CnnGruAttentionModel(nn.Module):
    """reference models.py:34-81: ChannelAttention -> 2 x [Conv1d, BatchNorm1d, ReLU, MaxPool1d]
    -> bidirectional GRU -> Linear/ReLU/Dropout/Linear.  ``forward(x[B,C,T] float32 cuda)``
    returns ``logits[B,num_classes]``.

    ``attention=False`` (extension, SURVEY D3) gives the ``cnn_gru`` baseline: the same stack
    with the attention gate removed; the (unused) attention parameters keep their
    ``state_dict`` slots so checkpoints stay interchangeable.
    """

    def __init__(self, in_channels, num_classes,
                 cnn_out_channels=32, gru_hidden_size=64, gru_num_layers=2, dropout=0.5, attention=True):
        super().__init__()
        self.in_channels, self.num_classes = int(in_channels), int(num_classes)
        self.cnn_out_channels, self.gru_hidden_size = int(cnn_out_channels), int(gru_hidden_size)
        self.gru_num_layers, self.dropout_p, self.attention = int(gru_num_layers), float(dropout), bool(attention)

        # identical construction order to reference models.py:42-71 (same RNG consumption)
        self.channel_attention = ChannelAttention(in_channels=in_channels)
        self.cnn_encoder = nn.Sequential(
            nn.Conv1d(in_channels, 16, kernel_size=7, stride=2, padding=3, bias=False),
            nn.BatchNorm1d(16),
            nn.ReLU(),
            nn.MaxPool1d(kernel_size=3, stride=2, padding=1),
            nn.Conv1d(16, cnn_out_channels, kernel_size=5, stride=2, padding=2, bias=False),
            nn.BatchNorm1d(cnn_out_channels),
            nn.ReLU(),
            nn.MaxPool1d(kernel_size=3, stride=2, padding=1),
        )
        self.gru = nn.GRU(input_size=cnn_out_channels, hidden_size=gru_hidden_size, num_layers=gru_num_layers,
                          batch_first=True, bidirectional=True, dropout=dropout if gru_num_layers > 1 else 0)
        self.gru.flatten_parameters = _no_flatten
        self.classifier = nn.Sequential(
            nn.Linear(gru_hidden_size * 2, 64),
            nn.ReLU(),
            nn.Dropout(dropout),
            nn.Linear(64, num_classes),
        )
        self._flat = None
        self._bn_flat = None
        self._nbt_flat = None
        self._param_views = None
        self._engines = {}
        self._rng_seed = (torch.initial_seed() * 0x9E3779B97F4A7C15 + next(_SEED_COUNTER)) & 0xFFFFFFFFFFFFFFFF
        self._rng_calls = 0

    def __getstate__(self):
        # the flat buffers / workspaces are rebuilt lazily; never pickle or deep-copy them
        state = dict(self.__dict__)
        state.update(_flat=None, _bn_flat=None, _nbt_flat=None, _param_views=None, _engines={})
        return state

    # ------------------------------------------------------------------ flat storage
    def _segments(self):
        """state_dict parameter name -> (segment index, position inside the segment)."""
        names = ["channel_attention.fc.0.weight", "channel_attention.fc.2.weight", "cnn_encoder.0.weight",
                 "cnn_encoder.1.weight", "cnn_encoder.1.bias", "cnn_encoder.4.weight", "cnn_encoder.5.weight",
                 "cnn_encoder.5.bias"]
        table = {n: (i, 0) for i, n in enumerate(names)}
        seg = len(names)
        for l in range(self.gru_num_layers):
            for kind in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"):
                table[f"gru.{kind}_l{l}"] = (seg, 0)
                table[f"gru.{kind}_l{l}_reverse"] = (seg, 1)
                seg += 1
        for n in ("classifier.0.weight", "classifier.0.bias", "classifier.3.weight", "classifier.3.bias"):
            table[n] = (seg, 0)
            seg += 1
        return table, seg

    def _layout(self):
        lib = _ext.load_library()
        d = CnnGruDesc()
        d.batch, d.in_channels, d.seq_len, d.num_classes = 1, self.in_channels, 64, self.num_classes
        d.cnn_out, d.hidden, d.layers = self.cnn_out_channels, self.gru_hidden_size, self.gru_num_layers
        offs = (C.c_int64 * _ext.MAX_SEGMENTS)()
        sizes = (C.c_int64 * _ext.MAX_SEGMENTS)()
        total = C.c_int64()
        n = check(lib.mms_cnngru_param_layout(C.byref(d), offs, sizes, _ext.MAX_SEGMENTS, C.byref(total)))
        return list(offs[:n]), list(sizes[:n]), int(total.value)

    def flat_layout(self):
        """[(name, offset, numel, shape)] of every parameter inside the flat buffer."""
        offs, sizes, total = self._layout()
        table, nseg = self._segments()
        assert nseg == len(offs), (nseg, len(offs))
        out = []
        for name, p in self.named_parameters():
            seg, half = table[name]
            n = p.numel()
            if half:
                assert sizes[seg] == 2 * n
            out.append((name, offs[seg] + half * n, n, tuple(p.shape)))
        return out, total

    def freeze_plan(self, trainable=None):
        """What fine-tuning with frozen parameters (``requires_grad_(False)``) asks of the library:
        ``(frozen_segments, ranges)``.  ``trainable``: one flag per parameter in ``parameters()`` order (default: the
        parameters' ``requires_grad``).  Bit s of ``frozen_segments`` is set when segment s of the flat layout holds
        elements and every one of its non-empty tensors is frozen -- one GRU direction frozen and the other trainable keeps
        the segment's gradient computed.  ``ranges`` is one ``(offset, count, slot)`` per trainable non-empty tensor, slot =
        the tensor's index in ``parameters()``: the flat ranges Adam updates, each with its own step count.  Host-only."""
        flags = tuple(p.requires_grad for p in self.parameters()) if trainable is None else tuple(bool(t) for t in trainable)
        cache = getattr(self, "_plan_cache", None)
        if cache is not None and cache[0] == flags:
            return cache[1]
        layout, _ = self.flat_layout()
        if len(flags) != len(layout):
            raise ValueError(f"freeze_plan: {len(flags)} flags for {len(layout)} parameters")
        table, nseg = self._segments()
        frozen_only = [None] * nseg              # per segment: True = every non-empty tensor frozen, None = no elements
        ranges = []
        for slot, ((name, off, n, _), t) in enumerate(zip(layout, flags)):
            if n == 0:
                continue
            seg = table[name][0]
            frozen_only[seg] = (frozen_only[seg] is not False) and not t
            if t:
                ranges.append((off, n, slot))
        mask = sum(1 << s for s, f in enumerate(frozen_only) if f)
        plan = (mask, tuple(ranges))
        self._plan_cache = (flags, plan)
        return plan

    def _flatten(self, device):
        layout, total = self.flat_layout()
        flat = torch.zeros(total, dtype=torch.float32, device=device)
        views = []
        with torch.no_grad():
            for (name, off, n, shape), (pname, p) in zip(layout, self.named_parameters()):
                assert name == pname
                if n:
                    flat[off:off + n].copy_(p.detach().reshape(-1).to(device=device, dtype=torch.float32))
                    p.data = flat[off:off + n].view(shape)
                views.append((off, n, shape))
        bn1, bn2 = self.cnn_encoder[1], self.cnn_encoder[5]
        O = self.cnn_out_channels
        bnf = torch.empty(32 + 2 * O, dtype=torch.float32, device=device)
        nbt = torch.empty(2, dtype=torch.int64, device=device)
        with torch.no_grad():
            for buf, lo, hi in ((bn1.running_mean, 0, 16), (bn1.running_var, 16, 32),
                                (bn2.running_mean, 32, 32 + O), (bn2.running_var, 32 + O, 32 + 2 * O)):
                bnf[lo:hi].copy_(buf.to(device))
                buf.data = bnf[lo:hi]
            for i, bn in enumerate((bn1, bn2)):
                nbt[i] = bn.num_batches_tracked.to(device)
                bn.num_batches_tracked.data = nbt[i]
        self._flat, self._bn_flat, self._nbt_flat, self._param_views = flat, bnf, nbt, views
        self._engines = {}

    def _ensure_flat(self, device):
        ok = self._flat is not None and self._flat.device == device
        if ok:
            base = self._flat.data_ptr()
            for (off, n, _), p in zip(self._param_views, self.parameters()):
                if n and p.data_ptr() != base + 4 * off:
                    ok = False
                    break
            ok = ok and self.cnn_encoder[1].running_mean.data_ptr() == self._bn_flat.data_ptr() \
                and self.cnn_encoder[5].num_batches_tracked.data_ptr() == self._nbt_flat.data_ptr() + 8
        if not ok:
            self._flatten(device)

    def _apply(self, fn, recurse=True):
        out = super()._apply(fn, recurse)
        self._flat = None           # .to()/.cuda() re-created the parameter tensors
        self._engines = {}
        return out

    def flat_parameters(self):
        """The flat float32 parameter buffer (device must already be CUDA)."""
        dev = next(self.parameters()).device
        if dev.type != "cuda":
            raise _ext.MmsError("move the model to a CUDA device first (no CPU fallback)")
        self._ensure_flat(dev)
        return self._flat

    def engine(self, B, T, training, need_grad, device):
        key = (B, T, bool(training), bool(need_grad))
        eng = self._engines.get(key)
        if eng is None:
            eng = _Engine(self, B, T, bool(training), bool(need_grad), device)
            self._engines[key] = eng
        return eng

    # ------------------------------------------------------------------------ forward
    def forward(self, x):
        _require_cuda(x)
        if x.dim() != 3 or x.shape[1] != self.in_channels:
            raise ValueError(f"expected x of shape [B, {self.in_channels}, T], got {tuple(x.shape)}")
        if next(self.parameters()).device != x.device:
            raise _ext.MmsError("model and input are on different devices")
        x = x.contiguous().float()
        self._ensure_flat(x.device)
        params = list(self.parameters())
        need_grad = torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in params))
        eng = self.engine(x.shape[0], x.shape[2], self.training, need_grad, x.device)
        self._rng_calls += 1
        if need_grad:
            return _CnnGruFn.apply(x, self, eng, self._rng_calls, *params)
        return eng.forward(x, self._rng_calls)
