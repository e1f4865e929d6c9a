"""Drop-in for the reference ``trainer.py``: ``Trainer(model, fold_output_dir, config)`` with
``.train(train_loader, val_loader)`` / ``.evaluate(loader, is_test, is_val)`` and
``EarlyStopping`` -- same config keys, log lines, ``best_model.pt`` and return values.

What changes is how a step executes (reference trainer.py:144-149): ``zero_grad -> forward ->
CrossEntropyLoss -> backward -> Adam.step`` is ONE C-ABI call (``mms_cnngru_train_step``) that
enqueues the whole kernel chain, replayed as a CUDA graph, with the loss accumulated on the
device (the reference syncs twice per step through ``loss.item()``, trainer.py:152-153).
"""
from __future__ import annotations

import contextlib
import math
import os
import ctypes as C
import threading
import time
from pathlib import Path

import numpy as np
import torch
from torch.optim.lr_scheduler import ReduceLROnPlateau

from . import _ext
from ._ext import CnnGruDesc, check, ptr, stream


class EarlyStopping:
    """reference trainer.py:12-39, bug-for-bug (SURVEY D8): the comparison treats the monitored
    score as higher-is-better although ``Trainer`` feeds it ``val_loss``, so ``best_model.pt`` is
    re-written whenever the validation loss does NOT improve on ``best_score + delta`` and the
    patience counter advances when it does.  ``fixed=True`` (off by default) monitors the loss
    the way the reference's comments intend."""

    def __init__(self, patience=7, delta=0, checkpoint_path='checkpoint.pt', verbose=False, log_func=None, fixed=False):
        self.patience, self.delta = patience, delta
        self.checkpoint_path = checkpoint_path
        self.verbose, self.log_func = verbose, log_func
        self.counter, self.best_score, self.early_stop = 0, None, False
        self.fixed = fixed

    def __call__(self, score, model):
        value = -score if self.fixed else score
        if self.best_score is None:
            self.best_score = value
            self.save_checkpoint(model)
            return
        if value < self.best_score + self.delta:
            self.counter += 1
            if self.verbose and self.log_func:
                self.log_func(f"EarlyStopping counter: {self.counter}/{self.patience}")
            self.early_stop = self.counter >= self.patience
        else:
            self.best_score = value
            self.save_checkpoint(model)
            self.counter = 0

    def save_checkpoint(self, model):
        # plain tensors (not views of the flat buffer) so the file equals the reference's layout
        writer = getattr(model, "_checkpoint_writer", None)
        if writer is not None:
            writer.submit(model, self.checkpoint_path)
        else:
            torch.save({k: v.detach().clone() for k, v in model.state_dict().items()}, self.checkpoint_path)


class CheckpointWriter:
    """``torch.save(model.state_dict(), path)`` (reference trainer.py:38-39) off the training thread.

    ``submit`` snapshots the model's three flat device buffers (parameters, BN running statistics,
    ``num_batches_tracked``) with three stream-ordered device copies and returns; a worker thread
    rebuilds the reference's 34-entry ``state_dict`` as plain tensors from the snapshot and writes the
    file.  Per file only the newest pending snapshot is written ("latest wins": the reference overwrites
    the same file).  ``flush()`` blocks until the file on disk is the last submitted one -- ``Trainer``
    calls it before it re-loads ``best_model.pt`` and before ``train()`` returns."""

    def __init__(self):
        self._cv = threading.Condition()
        self._pending = {}          # path -> newest snapshot for that file (insertion-ordered)
        self._busy = None           # path being written
        self._error = None
        self._thread = None
        self._stream = None

    def submit(self, model, path):
        model.flat_parameters()                                   # make sure the flat views exist
        snap = (model._flat.clone(), model._bn_flat.clone(), model._nbt_flat.clone())
        ready = torch.cuda.Event()
        ready.record(torch.cuda.current_stream())
        layout = self._layout(model)
        with self._cv:
            self._pending.pop(str(path), None)
            self._pending[str(path)] = (snap, ready, layout, Path(path), snap[0].device)
            if self._thread is None:
                self._thread = threading.Thread(target=self._work, name="mms-checkpoint", daemon=True)
                self._thread.start()
            self._cv.notify_all()

    @staticmethod
    def _layout(model):
        """state_dict key -> (buffer index, offset, numel, shape) inside the three flat buffers."""
        cached = getattr(model, "_ckpt_layout", None)
        if cached is not None and cached[0] is model._flat:
            return cached[1]
        bases = (model._flat, model._bn_flat, model._nbt_flat)
        out = []
        for k, v in model.state_dict().items():
            for bi, base in enumerate(bases):
                lo, hi = base.data_ptr(), base.data_ptr() + base.numel() * base.element_size()
                if v.numel() == 0:
                    out.append((k, -1, 0, 0, tuple(v.shape), v.dtype))
                    break
                if v.dtype == base.dtype and lo <= v.data_ptr() < hi:
                    out.append((k, bi, (v.data_ptr() - lo) // base.element_size(), v.numel(), tuple(v.shape), v.dtype))
                    break
            else:
                raise _ext.MmsError(f"state_dict entry {k} does not live in the model's flat buffers")
        model._ckpt_layout = (model._flat, out)
        return out

    def _work(self):
        while True:
            with self._cv:
                while not self._pending:
                    self._cv.wait()
                key = next(iter(self._pending))
                job = self._pending.pop(key)
                self._busy = key
            try:
                snap, ready, layout, path, dev = job
                torch.cuda.set_device(dev)
                if self._stream is None:
                    self._stream = torch.cuda.Stream(device=dev)     # non-blocking: never queues behind the training stream
                with torch.cuda.stream(self._stream):
                    self._stream.wait_event(ready)
                    host = [torch.empty(t.shape, dtype=t.dtype).pin_memory() for t in snap]
                    for h, t in zip(host, snap):
                        h.copy_(t, non_blocking=True)
                    self._stream.synchronize()
                sd = {}
                for k, bi, off, n, shape, dtype in layout:
                    sd[k] = torch.zeros(shape, dtype=dtype) if bi < 0 else host[bi][off:off + n].clone().view(shape)
                torch.save(sd, path)
            except Exception as e:                                   # surfaced by flush()
                self._error = e
            finally:
                with self._cv:
                    self._busy = None
                    self._cv.notify_all()

    def flush(self, path=None):
        """Wait until `path` (default: every submitted file) is on disk."""
        key = None if path is None else str(path)
        with self._cv:
            while (self._pending or self._busy) if key is None else (key in self._pending or self._busy == key):
                self._cv.wait(timeout=0.05)
        if self._error is not None:
            err, self._error = self._error, None
            raise err


_CAPTURE_STREAMS = {}


def capture_graph(enqueue):
    """Record ``enqueue()`` (kernel launches on the current stream) into a ``torch.cuda.CUDAGraph``.

    ``torch.cuda.graph(...)`` is deliberately not used: its ``__enter__`` synchronises the whole device, runs
    ``gc.collect()`` and empties the allocator cache -- tens of milliseconds per capture and a stall for every
    other stream (the concurrently training LOSO folds).  Nothing here allocates during capture, so the bare
    ``capture_begin`` / ``capture_end`` pair on a side stream is enough; ``thread_local`` error mode lets other
    threads (the checkpoint writer) keep issuing CUDA calls."""
    dev = torch.cuda.current_device()
    side = _CAPTURE_STREAMS.get(dev)
    if side is None:
        # MMS_CAPTURE_PRIORITY=-1 (experiment): kernel nodes inherit the priority of the stream they were captured on, so
        # the step's critical chain outranks the library's weight-gradient side streams (default priority) in CTA dispatch
        prio = int(os.environ.get("MMS_CAPTURE_PRIORITY", "0"))
        side = _CAPTURE_STREAMS[dev] = torch.cuda.Stream(device=dev, priority=prio)
    cur = torch.cuda.current_stream()
    side.wait_stream(cur)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        graph.capture_begin(capture_error_mode="thread_local")
        try:
            enqueue()
        finally:
            graph.capture_end()
    cur.wait_stream(side)
    return graph


def check_max_grad_norm(max_norm, norm_type=2.0):
    """``max_norm`` as a float, after the checks of the clipping this package implements: ``norm_type`` 2 only
    (``NotImplementedError`` otherwise), ``max_norm`` finite and > 0 (``ValueError`` otherwise)."""
    try:
        nt = float(norm_type)
    except (TypeError, ValueError):
        nt = None
    if nt != 2.0:
        raise NotImplementedError(f"gradient clipping: only norm_type 2 is implemented, got {norm_type!r}")
    try:
        v = float(max_norm)
    except (TypeError, ValueError):
        raise ValueError(f"gradient clipping: max_norm must be a number, got {max_norm!r}") from None
    if not math.isfinite(v) or v <= 0.0:
        raise ValueError(f"gradient clipping: max_norm must be finite and > 0, got {max_norm!r}")
    return v


class FlatAdam(torch.optim.Optimizer):
    """``torch.optim.Adam(model.parameters(), lr, weight_decay)`` (reference trainer.py:68) over
    the model's flat parameter buffer: one kernel for all 30 tensors.  It is a real
    ``Optimizer`` (``param_groups[0]['lr']`` is what ``ReduceLROnPlateau`` edits, trainer.py:72-77);
    the learning rate and the step count live on the device so the step can be graph-replayed.

    Frozen parameters follow torch: a tensor that is not updated (``step()``: no ``.grad``; ``flat_step()`` and the fused
    steps: ``requires_grad`` False) keeps its value, its moments and its step count, and on unfreezing continues from
    them.  The per-tensor step counts (``tensor_steps``) are used from the first step that leaves a tensor out; until then
    every tensor's count is ``step_dev`` and the single whole-buffer kernel runs.

    ``max_grad_norm`` (None: off) clips the gradient before every update, as
    ``torch.nn.utils.clip_grad_norm_(params, max_grad_norm)`` between ``backward()`` and ``step()`` would: the total 2-norm
    of the gradient of the tensors being updated, and ``coef = min(max_grad_norm / (norm + 1e-6), 1)`` on the gradient
    Adam reads (DESIGN.md, gradient-norm clipping).  ``step()``, ``flat_step()``, ``FusedTrainStep`` and the data-parallel
    steps all clip.  The flat gradient buffer ``grads`` keeps the UNCLIPPED gradient.  ``grad_norm`` is a one-element device
    tensor holding the last update's norm before clipping; ``clip_record`` (float64 [5], device) adds up, per update, the
    finite norms, their maximum, the clipped updates (coef < 1), the non-finite norms and the updates -- zero it with
    ``reset_clip_record()``.  ``set_max_grad_norm`` changes the threshold with a device copy: captured graphs keep working."""

    def __init__(self, model, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, max_grad_norm=None, norm_type=2.0):
        params = [p for p in model.parameters()]
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))
        self.model = model
        flat = model.flat_parameters()
        self.exp_avg = torch.zeros_like(flat)
        self.exp_avg_sq = torch.zeros_like(flat)
        self.grads = torch.zeros_like(flat)
        self.lr_dev = torch.full((1,), float(lr), dtype=torch.float32, device=flat.device)
        self.step_dev = torch.zeros(1, dtype=torch.int64, device=flat.device)
        self.scratch = torch.zeros(1, dtype=torch.int32, device=flat.device)
        self.tensor_steps = torch.zeros(len(params), dtype=torch.int64, device=flat.device)
        self._per_tensor = False            # tensor_steps in use (some step has left a tensor out)
        self._tables = {}                   # ranges -> HOST int64 [n][3] table (kept alive for the library)
        self._lr_on_device = float(lr)
        self.clip_max_norm = torch.zeros(1, dtype=torch.float32, device=flat.device)
        self.clip_record = torch.zeros(5, dtype=torch.float64, device=flat.device)
        self.clip_scratch = torch.zeros(_ext.GRAD_CLIP_SCRATCH_BYTES // 4, dtype=torch.float32, device=flat.device)
        self.grad_norm = self.clip_scratch[0:1]          # written by the norm kernel of every clipped update
        self.clip_coef = self.clip_scratch[1:2]
        self.max_grad_norm = None
        self._norm_tables = {}
        if max_grad_norm is not None:
            self.set_max_grad_norm(max_grad_norm, norm_type)

    def set_max_grad_norm(self, max_norm, norm_type=2.0):
        """Clip to ``max_norm`` from the next update on (None: stop clipping).  A stream-ordered copy to the device value the
        kernels read, so a captured CUDA graph picks it up without re-capture."""
        if max_norm is None:
            self.max_grad_norm = None
            return
        v = check_max_grad_norm(max_norm, norm_type)
        self.clip_max_norm.fill_(v)
        self.max_grad_norm = v

    def reset_clip_record(self):
        self.clip_record.zero_()

    @staticmethod
    def clip_summary(record):
        """``clip_record`` read back to the host (five numbers) as a dict: mean and max of the finite norms (NaN without
        one), clipped / non-finite / total update counts."""
        s, mx, clipped, nonfinite, n = (float(v) for v in record)
        finite = n - nonfinite
        return {'mean': s / finite if finite > 0 else float('nan'), 'max': mx if finite > 0 else float('nan'),
                'clipped': int(clipped), 'nonfinite': int(nonfinite), 'steps': int(n)}

    def norm_table(self, table):
        """The HOST range table the norm is taken over: the Adam range table of the update (``plan()``), or, when the
        update covers the whole buffer, one range per non-empty segment -- never the padding between segments.  Both list
        the same elements in the same order, so the norm has the same bits either way."""
        if table is not None:
            return table
        t = self._norm_tables.get(None)
        if t is None:
            offs, sizes, _ = self.model._layout()
            rows = [(o, n, 0) for o, n in zip(offs, sizes) if n]
            t = self._norm_tables[None] = (C.c_int64 * (3 * len(rows)))(*[v for r in rows for v in r])
        return t

    def sync_lr(self):
        lr = float(self.param_groups[0]['lr'])
        if lr != self._lr_on_device:
            self.lr_dev.fill_(lr)
            self._lr_on_device = lr

    def plan(self, trainable=None):
        """``(frozen_segments, table)`` for a step that updates the tensors flagged in ``trainable`` (default: their
        ``requires_grad``; see ``CnnGruAttentionModel.freeze_plan``).  ``table`` is None while every tensor trains and no
        earlier step left one out (the whole-buffer kernel, ``step_dev`` as every count); otherwise the HOST ctypes array
        of the Adam ranges, ``len(table) // 3`` of them, and from then on the per-tensor counts are in use."""
        mask, ranges = self.model.freeze_plan(trainable)
        everything = len(ranges) == sum(1 for (_, n, _) in self.model._param_views if n)
        if everything and not self._per_tensor:
            return mask, None
        if not self._per_tensor:            # every tensor's count so far is the global one
            self.tensor_steps.copy_(self.step_dev.expand_as(self.tensor_steps))
            self._per_tensor = True
        table = self._tables.get(ranges)
        if table is None:
            table = self._tables[ranges] = (C.c_int64 * max(1, 3 * len(ranges)))(*[v for r in ranges for v in r])
        return mask, table

    @torch.no_grad()
    def step(self, closure=None):
        """Generic path: gather ``p.grad`` into the flat gradient buffer, then one Adam launch over the tensors that have a
        gradient (torch skips the others)."""
        flat = self.model.flat_parameters()
        self.grads.zero_()
        params = list(self.model.parameters())
        for (off, n, _), p in zip(self.model._param_views, params):
            if n and p.grad is not None:
                self.grads[off:off + n].copy_(p.grad.reshape(-1))
        self._update(flat, [p.grad is not None for p in params])

    def flat_step(self, flat=None):
        """Adam over the flat gradient buffer for the parameters that currently require a gradient."""
        self._update(self.model.flat_parameters() if flat is None else flat, None)

    def _update(self, flat, trainable):
        lib = _ext.lib()
        self.sync_lr()
        g = self.param_groups[0]
        _, table = self.plan(trainable)
        if self.max_grad_norm is not None:
            nt = self.norm_table(table)
            check(lib.mms_grad_norm(ptr(self.grads), flat.numel(), nt, len(nt) // 3, ptr(self.clip_max_norm), ptr(self.clip_record),
                                    ptr(self.clip_scratch), stream()))
            if table is None:
                check(lib.mms_adam_flat_clip_step(ptr(flat), ptr(self.grads), ptr(self.exp_avg), ptr(self.exp_avg_sq), flat.numel(),
                                                  ptr(self.lr_dev), g['betas'][0], g['betas'][1], g['eps'], g['weight_decay'],
                                                  ptr(self.step_dev), ptr(self.scratch), ptr(self.clip_coef), stream()))
            else:
                check(lib.mms_adam_ranges_clip_step(ptr(flat), ptr(self.grads), ptr(self.exp_avg), ptr(self.exp_avg_sq), table,
                                                    len(table) // 3, ptr(self.tensor_steps), ptr(self.lr_dev),
                                                    g['betas'][0], g['betas'][1], g['eps'], g['weight_decay'], ptr(self.step_dev),
                                                    ptr(self.scratch), ptr(self.clip_coef), stream()))
            return
        if table is None:
            check(lib.mms_adam_flat_step(ptr(flat), ptr(self.grads), ptr(self.exp_avg), ptr(self.exp_avg_sq), flat.numel(),
                                         ptr(self.lr_dev), g['betas'][0], g['betas'][1], g['eps'], g['weight_decay'],
                                         ptr(self.step_dev), ptr(self.scratch), stream()))
        else:
            check(lib.mms_adam_ranges_step(ptr(flat), ptr(self.grads), ptr(self.exp_avg), ptr(self.exp_avg_sq), table,
                                           len(table) // 3, ptr(self.tensor_steps), ptr(self.lr_dev),
                                           g['betas'][0], g['betas'][1], g['eps'], g['weight_decay'], ptr(self.step_dev),
                                           ptr(self.scratch), stream()))

    def set_plan(self, desc, plan):
        """Writes ``plan`` (from ``plan()``) into a train-step descriptor."""
        mask, table = plan
        desc.frozen_segments = mask
        desc.adam_ranges_host = None if table is None else C.addressof(table)
        desc.adam_steps = None if table is None else self.tensor_steps.data_ptr()
        desc.adam_nranges = 0 if table is None else len(table) // 3
        clip = self.max_grad_norm is not None
        desc.clip_max_norm = self.clip_max_norm.data_ptr() if clip else None
        desc.clip_record = self.clip_record.data_ptr() if clip else None
        desc.clip_scratch = self.clip_scratch.data_ptr() if clip else None


def class_weight_tensor(weight, num_classes, device):
    """``weight`` (a sequence or tensor of ``num_classes`` values) as a contiguous float32 tensor on ``device``."""
    w = torch.as_tensor(weight, dtype=torch.float32).detach().reshape(-1)
    if w.numel() != num_classes:
        raise ValueError(f"class weights: expected {num_classes} values, got {w.numel()}")
    return w.to(device).contiguous()


class FusedTrainStep:
    """One training step = one ``mms_cnngru_train_step`` call, captured once per batch shape into
    a CUDA graph and replayed.  ``__call__(x, y)`` accepts device tensors or pinned host tensors
    (copied into the static graph inputs on the current stream).

    ``class_weight`` (``num_classes`` values) makes the loss ``CrossEntropyLoss(weight=class_weight)``.  The values
    live in a device tensor whose address the graph holds: ``set_class_weight`` changes them with a copy, no re-capture."""

    def __init__(self, model, optimizer: FlatAdam, batch: int, seq_len: int, use_graph: bool = True, source=None, loss_sum=None,
                 class_weight=None):
        self.lib = _ext.lib()
        self.model, self.opt = model, optimizer
        self.source = source            # DeviceBatchSource: the batch is gathered on the device inside the graph
        self.flat = model.flat_parameters()
        dev = self.flat.device
        self.class_weight = None if class_weight is None else class_weight_tensor(class_weight, model.num_classes, dev)
        self.x = torch.zeros(batch, model.in_channels, seq_len, dtype=torch.float32, device=dev)
        self.y = torch.zeros(batch, dtype=torch.int64, device=dev)
        self.logits = torch.zeros(batch, model.num_classes, dtype=torch.float32, device=dev)
        self.loss = torch.zeros(1, dtype=torch.float32, device=dev)
        self.loss_sum = torch.zeros(1, dtype=torch.float64, device=dev) if loss_sum is None else loss_sum
        d = CnnGruDesc()
        d.batch, d.in_channels, d.seq_len, d.num_classes = batch, model.in_channels, seq_len, model.num_classes
        d.cnn_out, d.hidden, d.layers = model.cnn_out_channels, model.gru_hidden_size, model.gru_num_layers
        d.training, d.attention, d.need_grad = 1, int(model.attention), 1
        d.dropout_p = float(model.dropout_p)
        d.rng_seed, d.rng_offset = model._rng_seed ^ 0x5DEECE66D, 0
        d.rng_offset_dev = optimizer.step_dev.data_ptr()      # dropout stream advances with the step count
        d.class_weight = None if self.class_weight is None else self.class_weight.data_ptr()
        self.desc = d
        nbytes = self.lib.mms_cnngru_workspace_bytes(C.byref(d))
        if nbytes < 0:
            check(int(nbytes))
        self.workspace = torch.empty(int(nbytes), dtype=torch.uint8, device=dev)
        self.use_graph = use_graph
        self.graph = None
        self.calls = 0
        self.kernels_per_step = None
        # one graph per freeze plan (requires_grad flags, read at every step): progressive unfreezing switches graphs
        self._graphs, self._eager_done, self._plan = {}, set(), None

    def set_class_weight(self, weight):
        """New class weights for the following steps (a stream-ordered copy into the tensor the graph reads)."""
        if self.class_weight is None:
            raise _ext.MmsError("FusedTrainStep was built without class weights")
        self.class_weight.copy_(class_weight_tensor(weight, self.model.num_classes, self.class_weight.device), non_blocking=True)

    def _enqueue(self):
        m, o, g = self.model, self.opt, self.opt.param_groups[0]
        if self.source is not None:     # trainer.py:130,140-142: next batch of the shuffled epoch, cursor advanced on the device
            src = self.source
            check(self.lib.mms_batch_gather(ptr(src.data), ptr(src.labels), ptr(src.perm), ptr(src.cursor), src.n, src.row_floats,
                                            self.x.shape[0], ptr(self.x), ptr(self.y), 1, ptr(src.scratch), stream()))
        check(self.lib.mms_cnngru_train_step(
            C.byref(self.desc), ptr(self.x), ptr(self.y), ptr(self.flat), ptr(o.grads), ptr(o.exp_avg), ptr(o.exp_avg_sq),
            ptr(m._bn_flat), ptr(m._nbt_flat), ptr(self.workspace), ptr(self.logits), ptr(self.loss), ptr(self.loss_sum),
            ptr(o.lr_dev), g['betas'][0], g['betas'][1], g['eps'], g['weight_decay'], ptr(o.step_dev), ptr(o.scratch),
            stream()))

    def load(self, x, y):
        self.x.copy_(x, non_blocking=True)
        self.y.copy_(y, non_blocking=True)

    # ---- double-buffered input pipeline: the H2D copy of batch i+1 overlaps the step of batch i ----------
    def _pipeline(self):
        if getattr(self, "_copy_stream", None) is None:
            dev = self.x.device
            self._copy_stream = torch.cuda.Stream(device=dev)
            self._stage_x = [torch.empty_like(self.x) for _ in range(2)]
            self._stage_y = [torch.empty_like(self.y) for _ in range(2)]
            self._ready = [torch.cuda.Event() for _ in range(2)]
            self._consumed = [torch.cuda.Event() for _ in range(2)]
            self._queued, self._next_slot = [], 0
        return self._copy_stream

    def prefetch(self, x, y):
        """Enqueue the host->device copy of an upcoming batch on the copy stream (staging slot)."""
        cs = self._pipeline()
        slot = self._next_slot
        cs.wait_event(self._consumed[slot])            # the step that last read this slot has copied it out
        if x.is_cuda:                                  # device-resident batch: produced on the current stream
            cs.wait_stream(torch.cuda.current_stream())
            x.record_stream(cs)
            y.record_stream(cs)
        with torch.cuda.stream(cs):
            self._stage_x[slot].copy_(x, non_blocking=True)
            self._stage_y[slot].copy_(y, non_blocking=True)
            self._ready[slot].record(cs)
        self._queued.append(slot)
        self._next_slot ^= 1

    def run_prefetched(self):
        """Run one step on the oldest prefetched batch (device-to-device hand-over, then the graph)."""
        slot = self._queued.pop(0)
        cur = torch.cuda.current_stream()
        cur.wait_event(self._ready[slot])
        self.x.copy_(self._stage_x[slot], non_blocking=True)
        self.y.copy_(self._stage_y[slot], non_blocking=True)
        self._consumed[slot].record(cur)
        self.run()

    def run(self):
        """Enqueue one step on the static inputs (graph replay after the first two calls of each freeze plan)."""
        if self.model._flat is not self.flat:       # .to() / .cuda() drop the flat buffer (models.py: _apply)
            raise _ext.MmsError("the model's parameter storage moved after FusedTrainStep was built")
        self.opt.sync_lr()
        self.calls += 1
        mask, table = self.opt.plan()
        key = (mask, None if table is None else tuple(table), self.opt.max_grad_norm is not None)
        self.opt.set_plan(self.desc, (mask, table))
        if not self.use_graph or key not in self._eager_done:
            self._eager_done.add(key)
            self._enqueue()                       # first call of a plan eager: sets kernel attributes, warms caches
            return
        self.graph = self._graphs.get(key)
        if self.graph is None:
            self.graph = self._graphs[key] = capture_graph(self._enqueue)
        self.graph.replay()

    def post_loss(self):
        """Enqueue an asynchronous device->host copy of this step's loss into a pinned two-slot ring
        and return a ticket; ``read_loss(ticket)`` waits for exactly that copy.  Lets a caller read
        every step's loss (as reference trainer.py:152 does) one step late, so the GPU never idles
        while Python enqueues the next step."""
        if getattr(self, "_loss_host", None) is None:
            self._loss_host = [torch.zeros(1, dtype=torch.float32).pin_memory() for _ in range(2)]
            self._loss_ev = [torch.cuda.Event() for _ in range(2)]
            self._loss_slot = 0
        k = self._loss_slot
        self._loss_host[k].copy_(self.loss, non_blocking=True)
        self._loss_ev[k].record(torch.cuda.current_stream())
        self._loss_slot ^= 1
        return k

    def read_loss(self, ticket) -> float:
        self._loss_ev[ticket].synchronize()
        return float(self._loss_host[ticket][0])

    def __call__(self, x, y):
        self.load(x, y)
        self.run()

    def last_loss(self) -> float:
        return float(self.loss.item())


class DeviceBatchSource:
    """What ``mms_batch_gather`` reads: a device-resident dataset (float32 ``[N, C, W]`` + int64 labels), the
    epoch's permutation and a cursor, both on the device.  ``start_epoch`` draws the permutation exactly as
    ``DeviceBatchLoader.__iter__`` does (``torch.randperm`` on the CPU generator) and uploads it."""

    def __init__(self, dataset, batch_size):
        self.data, self.labels = dataset.data, dataset.labels
        dev = self.data.device
        self.n = int(self.data.shape[0])
        self.row_floats = int(self.data.shape[1] * self.data.shape[2])
        self.perm = torch.zeros(self.n + batch_size, dtype=torch.int64, device=dev)     # slack: a tail batch never reads past the end
        self.perm_host = torch.zeros(self.n, dtype=torch.int64).pin_memory()
        self.cursor = torch.zeros(1, dtype=torch.int64, device=dev)
        self.scratch = torch.zeros(1, dtype=torch.int32, device=dev)

    def start_epoch(self, shuffle, generator=None):
        if shuffle:
            torch.randperm(self.n, out=self.perm_host, generator=generator)
        else:
            torch.arange(self.n, out=self.perm_host)
        self.perm[:self.n].copy_(self.perm_host, non_blocking=True)
        self.cursor.zero_()


class EvalStep:
    """One evaluation batch (reference trainer.py:213-228) = eval-mode forward + ``mms_eval_accumulate``
    (summed loss, arg-max predictions, confusion counts) on static buffers, replayed as a CUDA graph.

    With ``class_weight`` the loss is ``CrossEntropyLoss(weight=class_weight)`` accumulated per group of ``group``
    consecutive rows (the evaluation loader's batch size; None: the whole batch is one group), each group adding
    ``n * weighted_mean`` as the reference adds ``loss.item() * batch`` per loader batch."""

    def __init__(self, model, batch, seq_len, confusion, loss_sum, use_graph=True, class_weight=None, group=None):
        self.lib = _ext.lib()
        self.model = model
        self.flat = model.flat_parameters()
        dev = self.flat.device
        self.class_weight = None if class_weight is None else class_weight_tensor(class_weight, model.num_classes, dev)
        self.group = int(group) if group else batch
        self.x = torch.zeros(batch, model.in_channels, seq_len, dtype=torch.float32, device=dev)
        self.y = torch.zeros(batch, dtype=torch.int64, device=dev)
        self.logits = torch.zeros(batch, model.num_classes, dtype=torch.float32, device=dev)
        self.pred = torch.zeros(batch, dtype=torch.int64, device=dev)
        self.confusion, self.loss_sum = confusion, loss_sum
        self.engine = model.engine(batch, seq_len, False, False, dev)
        self.use_graph, self.graph, self.calls = use_graph, None, 0

    def _enqueue(self):
        m, e = self.model, self.engine
        check(self.lib.mms_cnngru_forward(C.byref(e.desc), ptr(self.x), ptr(self.flat), ptr(m._bn_flat), ptr(m._nbt_flat),
                                          ptr(e.workspace), ptr(self.logits), stream()))
        if self.class_weight is None:
            check(self.lib.mms_eval_accumulate(ptr(self.logits), ptr(self.y), self.x.shape[0], m.num_classes, ptr(self.pred),
                                               ptr(self.confusion), ptr(self.loss_sum), stream()))
        else:
            check(self.lib.mms_eval_accumulate_weighted(ptr(self.logits), ptr(self.y), self.x.shape[0], m.num_classes,
                                                        ptr(self.class_weight), self.group, ptr(self.pred), ptr(self.confusion),
                                                        ptr(self.loss_sum), stream()))

    def run(self):
        if self.model._flat is not self.flat:
            raise _ext.MmsError("the model's parameter storage moved after EvalStep was built")
        self.calls += 1
        if not self.use_graph or self.calls == 1:
            self._enqueue()
            return
        if self.graph is None:
            self.graph = capture_graph(self._enqueue)
        self.graph.replay()


def metrics_from_confusion(conf):
    """``accuracy_score(y, p)`` and ``f1_score(y, p, average='weighted')`` (reference trainer.py:229-230) as
    functions of the confusion matrix ``conf[true, pred]``: per-class F1 = 2 tp / (2 tp + fp + fn) (0 where
    the denominator is 0, sklearn's zero_division default), weighted by the class support."""
    conf = np.asarray(conf, dtype=np.float64)
    total = conf.sum()
    if total == 0:
        return 0.0, 0.0
    tp = np.diag(conf)
    support = conf.sum(axis=1)
    denom = support + conf.sum(axis=0)                 # 2 tp + fn + fp
    f1 = np.divide(2.0 * tp, denom, out=np.zeros_like(tp), where=denom > 0)
    return float(tp.sum() / total), float((f1 * support).sum() / total)


def balanced_class_weights(labels, num_classes):
    """The class weights ``Trainer`` uses with ``use_class_weights``: sklearn's
    ``compute_class_weight('balanced', classes=range(num_classes), y=labels)``, w_c = N / (num_classes * count_c).
    The reference computes its weights at trainer.py:81-94 in a branch that never runs; its formula is not
    available, so this project defines the option as ``'balanced'``.  ``labels``: numpy array or (CUDA) tensor.
    A class without training windows or a label outside [0, num_classes) raises."""
    if isinstance(labels, torch.Tensor):
        labels = labels.detach().to("cpu").numpy()
    y = np.asarray(labels).reshape(-1).astype(np.int64)
    if y.size == 0:
        raise ValueError("class weights: the training set is empty")
    if y.min() < 0 or y.max() >= num_classes:
        raise ValueError(f"class weights: labels outside [0, {num_classes})")
    counts = np.bincount(y, minlength=num_classes)
    missing = [c for c in range(num_classes) if counts[c] == 0]
    if missing:
        raise ValueError(f"class weights: class {missing[0]} has no training windows"
                         + (f" (nor do classes {missing[1:]})" if len(missing) > 1 else ""))
    return y.size / (num_classes * counts.astype(np.float64))


class _CrossEntropy(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, labels, weight=None):
        lib = _ext.lib()
        logits = logits.contiguous().float()
        loss = torch.empty(1, dtype=torch.float32, device=logits.device)
        dlogits = torch.empty_like(logits)
        if weight is None:
            check(lib.mms_cross_entropy(ptr(logits), ptr(labels.contiguous()), logits.shape[0], logits.shape[1], ptr(loss),
                                        ptr(dlogits), None, stream()))
        else:
            check(lib.mms_cross_entropy_weighted(ptr(logits), ptr(labels.contiguous()), logits.shape[0], logits.shape[1],
                                                 ptr(weight), None, ptr(loss), ptr(dlogits), None, stream()))
        ctx.save_for_backward(dlogits)
        return loss[0]

    @staticmethod
    def backward(ctx, g):
        (dlogits,) = ctx.saved_tensors
        return dlogits * g, None, None


class CrossEntropyLoss(torch.nn.Module):
    """``torch.nn.CrossEntropyLoss()`` (mean reduction, reference trainer.py:69) on the CUDA kernel.

    ``weight`` (``num_classes`` values, a sequence or tensor) is ``CrossEntropyLoss(weight=...)``:
    ``sum_b w[y_b] l_b / sum_b w[y_b]``.  The other options of torch's loss (``ignore_index``, ``label_smoothing``,
    a reduction other than ``'mean'``) are not implemented and raise."""

    def __init__(self, weight=None, size_average=None, ignore_index=-100, reduce=None, reduction='mean', label_smoothing=0.0):
        super().__init__()
        if size_average is not None or reduce is not None or reduction != 'mean':
            raise NotImplementedError("CrossEntropyLoss: only reduction='mean' is implemented")
        if ignore_index != -100:
            raise NotImplementedError("CrossEntropyLoss: ignore_index is not implemented")
        if label_smoothing != 0.0:
            raise NotImplementedError("CrossEntropyLoss: label_smoothing is not implemented")
        self.weight = None if weight is None else torch.as_tensor(weight, dtype=torch.float32).detach().reshape(-1)

    def forward(self, logits, labels):
        if self.weight is None:
            return _CrossEntropy.apply(logits, labels)
        if self.weight.numel() != logits.shape[1]:
            raise ValueError(f"CrossEntropyLoss: {self.weight.numel()} class weights for {logits.shape[1]} classes")
        if self.weight.device != logits.device:
            self.weight = self.weight.to(logits.device).contiguous()
        return _CrossEntropy.apply(logits, labels, self.weight)


_WRITER = None


def _checkpoint_writer():
    global _WRITER
    if _WRITER is None:
        _WRITER = CheckpointWriter()
    return _WRITER


def drive(gen):
    """Run one of the ``*_async`` generators below to completion on the calling thread: wait for every CUDA
    event it yields and return its result."""
    try:
        while True:
            next(gen).synchronize()
    except StopIteration as done:
        return done.value


class Trainer:
    """reference trainer.py:41-247.

    ``train`` / ``evaluate`` keep the reference's blocking signatures.  Underneath they are generators
    (``train_async`` / ``evaluate_async``) that enqueue device work and *yield a CUDA event* wherever the reference
    reads a result back (``loss.item()``, the prediction lists): a caller that owns several trainers -- the LOSO
    folds of ``main.run_simple_experiment(concurrent_folds=K)`` -- resumes whichever one's event has completed, so
    K independent folds keep K CUDA streams busy from ONE host thread.  ``stream`` (optional) is the CUDA stream all
    of this trainer's work is issued on."""

    def __init__(self, model, fold_output_dir: Path, config, stream=None):
        # refuse a bad clipping setting before anything is written or allocated
        grad_clip_norm = config['trainer'].get('grad_clip_norm')
        if grad_clip_norm is not None:
            grad_clip_norm = check_max_grad_norm(grad_clip_norm)
        self.model, self.fold_dir, self.config = model, Path(fold_output_dir), config
        self.fold_dir.mkdir(parents=True, exist_ok=True)
        self.log_file = self.fold_dir / 'training_log.txt'
        with open(self.log_file, 'w') as f:
            f.write(f"Training log for run starting at {time.strftime('%Y-%m-%d %H:%M:%S')}\n")
            f.write("=" * 50 + "\n")
        if not torch.cuda.is_available():
            raise _ext.MmsError("Trainer needs a CUDA device (B200); there is no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device())
        self.stream = stream
        t = config['trainer']
        self.epochs, self.learning_rate = t['epochs'], t['learning_rate']
        self.patience, self.weight_decay = t['early_stopping']['patience'], t['weight_decay']
        # never enabled upstream (SURVEY D9); here an opt-in with the intended behaviour: balanced_class_weights of the
        # training labels, fixed by the first train(), used by every later step and evaluation
        self.use_class_weights = t.get('use_class_weights', False)
        self.class_weights = None                                      # list of num_classes floats once fixed
        self._class_weight = None                                      # the same on the device
        self.use_graph = t.get('cuda_graph', True)
        self.quiet = t.get('quiet', False)                             # log to the file only

        with self._on_stream():
            self.model.to(self.device)
            # gradient-norm clipping (torch.nn.utils.clip_grad_norm_ before every Adam step); None: off
            self.grad_clip_norm = grad_clip_norm
            self.optimizer = FlatAdam(self.model, lr=self.learning_rate, weight_decay=self.weight_decay, max_grad_norm=grad_clip_norm)
            nc = model.num_classes
            self._eval_conf = torch.zeros(nc * nc, dtype=torch.int64, device=self.device)
            self._eval_loss = torch.zeros(1, dtype=torch.float64, device=self.device)
            self._train_loss = torch.zeros(1, dtype=torch.float64, device=self.device)
        self._host_conf = torch.zeros(nc * nc, dtype=torch.int64).pin_memory()
        self._host_loss = torch.zeros(2, dtype=torch.float64).pin_memory()       # [0] training sum, [1] evaluation sum
        self._host_clip = torch.zeros(5, dtype=torch.float64).pin_memory() if grad_clip_norm is not None else None
        self.criterion = CrossEntropyLoss()
        self.scheduler = ReduceLROnPlateau(self.optimizer, mode='min', factor=0.1, patience=3)
        self.early_stopping = None
        if t['early_stopping']['enabled']:
            self.early_stopping = EarlyStopping(patience=self.patience, delta=t['early_stopping']['delta'],
                                                checkpoint_path=self.fold_dir / 'best_model.pt', verbose=True,
                                                log_func=self._log, fixed=t['early_stopping'].get('fixed', False))
        self._steps = {}
        self._eval_steps = {}
        self._sources = {}
        self.async_checkpoint = t.get('async_checkpoint', True)
        if self.async_checkpoint:
            self.model._checkpoint_writer = _checkpoint_writer()
        self.total_start_time = time.time()
        self.windows_trained = 0
        self.timing = {'train_enqueue': 0.0, 'train_wait': 0.0, 'evaluate': 0.0, 'bookkeeping': 0.0}

    def _on_stream(self):
        return torch.cuda.stream(self.stream) if self.stream is not None else contextlib.nullcontext()

    def _event(self):
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream())
        return ev

    def _log(self, message):
        if not self.quiet:
            print(message)
        with open(self.log_file, 'a') as f:
            f.write(message + '\n')

    def _fused(self, batch, seq_len, source=None):
        key = (batch, seq_len, id(source))
        if key not in self._steps:
            self._steps[key] = FusedTrainStep(self.model, self.optimizer, batch, seq_len, use_graph=self.use_graph, source=source,
                                              loss_sum=self._train_loss, class_weight=self._class_weight)
        return self._steps[key]

    def _eval_step(self, batch, seq_len, group=None):
        key = (batch, seq_len, group)
        st = self._eval_steps.get(key)
        if st is None or st.flat is not self.model._flat:
            st = EvalStep(self.model, batch, seq_len, self._eval_conf, self._eval_loss, use_graph=self.use_graph,
                          class_weight=self._class_weight, group=group)
            self._eval_steps[key] = st
        return st

    def _fix_class_weights(self, train_loader):
        """``use_class_weights``: the first ``train()`` fixes sklearn's ``'balanced'`` weights of the training labels."""
        if not self.use_class_weights or self._class_weight is not None:
            return
        labels = getattr(train_loader.dataset, 'labels', None)
        if labels is None:
            raise ValueError("use_class_weights: the training dataset has no .labels to compute class weights from")
        w = balanced_class_weights(labels, self.model.num_classes)
        self.class_weights = [float(v) for v in w]
        with self._on_stream():
            self._class_weight = torch.tensor(self.class_weights, dtype=torch.float32, device=self.device)
        self.criterion = CrossEntropyLoss(weight=self._class_weight)
        self._log("Class weights ('balanced'): " + ", ".join(f"{v:.4f}" for v in self.class_weights))

    @staticmethod
    def _check_batch(batch):
        if isinstance(batch[0], (list, tuple)):
            raise NotImplementedError("HybridDataset inputs (reference void/dataset.py) are out of scope")

    def _train_epoch_host(self, train_loader):
        """trainer.py:130-149 with a one-batch look-ahead: the H2D copy of the next batch runs on a copy
        stream while the current step (one CUDA-graph replay) executes."""
        it = iter(train_loader)
        nxt = next(it, None)
        if nxt is not None:
            self._check_batch(nxt)
            self._fused(nxt[0].shape[0], nxt[0].shape[2]).prefetch(*nxt)
        while nxt is not None:
            inputs, labels = nxt
            step = self._fused(inputs.shape[0], inputs.shape[2])
            nxt = next(it, None)
            if nxt is not None:
                self._check_batch(nxt)
                self._fused(nxt[0].shape[0], nxt[0].shape[2]).prefetch(*nxt)
            step.run_prefetched()
            self.windows_trained += inputs.shape[0]

    def _train_epoch_device(self, loader):
        """The same epoch for a ``DeviceBatchLoader``: the permutation is uploaded once, every step is ONE graph
        replay (batch gather through the device cursor + the fused train step); a ragged last batch (the
        reference's DataLoader keeps it, drop_last=False) replays a second graph of that size."""
        ds = loader.dataset
        src = self._sources.get(id(ds))
        if src is None or src.data is not ds.data:
            src = DeviceBatchSource(ds, loader.batch_size)
            self._sources[id(ds)] = src
        src.start_epoch(loader.shuffle, getattr(loader, "generator", None))
        full, tail = divmod(src.n, loader.batch_size)
        T = int(ds.data.shape[2])
        if full:
            step = self._fused(loader.batch_size, T, src)
            for _ in range(full):
                step.run()
        if tail and not loader.drop_last:
            self._fused(tail, T, src).run()
        self.windows_trained += src.n if not loader.drop_last else full * loader.batch_size

    def _enqueue_train_epoch(self, train_loader):
        from .dataset import DeviceBatchLoader
        self.model.train()
        self._train_loss.zero_()
        if self._host_clip is not None:
            self.optimizer.reset_clip_record()
        if isinstance(train_loader, DeviceBatchLoader):
            self._train_epoch_device(train_loader)
        else:
            self._train_epoch_host(train_loader)
        self._host_loss[0:1].copy_(self._train_loss, non_blocking=True)
        if self._host_clip is not None:                  # read back behind the same event as the loss
            self._host_clip.copy_(self.optimizer.clip_record, non_blocking=True)
        return self._event()

    def train(self, train_loader, val_loader):
        return drive(self.train_async(train_loader, val_loader))

    def _log_frozen(self):
        """One log line when some parameters are frozen (fine-tuning); nothing otherwise."""
        params = list(self.model.parameters())
        if all(p.requires_grad for p in params if p.numel()):
            return
        n = sum(p.numel() for p in params if p.requires_grad)
        self._log(f"Trainable parameters: {n} of {sum(p.numel() for p in params)} (the others are frozen)")

    def train_async(self, train_loader, val_loader):
        self._fix_class_weights(train_loader)
        self._log_frozen()
        best_val_acc = 0
        for epoch in range(self.epochs):
            t0 = time.time()
            with self._on_stream():
                done = self._enqueue_train_epoch(train_loader)
            t1 = time.time()
            yield done                                     # one read-back per epoch instead of two syncs per step
            train_loss = float(self._host_loss[0])
            epoch_duration = time.time() - t0
            self.timing['train_enqueue'] += t1 - t0
            self.timing['train_wait'] += epoch_duration - (t1 - t0)

            val_loss, val_acc, val_f1 = yield from self.evaluate_async(val_loader)
            t2 = time.time()
            self.scheduler.step(val_loss)
            best_val_acc = max(best_val_acc, val_acc)
            self._log(f"Epoch {epoch + 1}/{self.epochs} | "
                      f"耗时: {epoch_duration:.2f}s | "
                      f"训练损失: {train_loss / len(train_loader.dataset):.4f} | "
                      f"验证损失: {val_loss:.4f} | "
                      f"验证Acc: {val_acc:.4f} | "
                      f"验证F1: {val_f1:.4f}")
            if self._host_clip is not None:
                self._log_clipping()
            stop = False
            if self.early_stopping:
                with self._on_stream():
                    self.early_stopping(val_loss, self.model)
                if self.early_stopping.early_stop:
                    self._log("触发早停")
                    stop = True
            self.timing['bookkeeping'] += time.time() - t2
            if stop:
                break
        self._flush_checkpoints()
        if self.early_stopping and self.early_stopping.early_stop:
            self._log(f"加载性能最佳的模型权重从: {self.early_stopping.checkpoint_path}")
            with self._on_stream():
                self.model.load_state_dict(torch.load(self.early_stopping.checkpoint_path, weights_only=True))
        self._log(f"--- 训练完成 --- 总训练时长: {time.time() - self.total_start_time:.2f}秒")

    def _log_clipping(self):
        """The epoch's gradient-norm line (``grad_clip_norm``), plus a warning when a norm was not finite."""
        r = FlatAdam.clip_summary(self._host_clip)
        self._log(f"Gradient norm before clipping: mean {r['mean']:.4f} | max {r['max']:.4f} | "
                  f"clipped {r['clipped']} of {r['steps']} steps")
        if r['nonfinite']:
            self._log(f"Warning: the gradient norm was not finite in {r['nonfinite']} of {r['steps']} steps; "
                      "clipping such a gradient makes the parameters NaN (as torch's clip_grad_norm_ does)")

    def _flush_checkpoints(self):
        writer = getattr(self.model, "_checkpoint_writer", None)
        if writer is not None and self.early_stopping is not None:
            writer.flush(self.early_stopping.checkpoint_path)

    EVAL_CHUNK = 256        # windows per evaluation launch on the device-resident path

    def _enqueue_evaluate(self, data_loader, want_lists):
        from .dataset import DeviceBatchLoader
        self.model.eval()
        self._eval_conf.zero_()
        self._eval_loss.zero_()
        preds, labels_all = [], []
        if isinstance(data_loader, DeviceBatchLoader) and not data_loader.shuffle:
            ds = data_loader.dataset
            n, T = len(ds), int(ds.data.shape[2])
            n_eval = n if not data_loader.drop_last else (n // data_loader.batch_size) * data_loader.batch_size
            chunk, group = self.EVAL_CHUNK, None
            if self._class_weight is not None:
                # the weighted loss is a per-loader-batch mean: slices hold whole loader batches, each one group
                group = data_loader.batch_size
                chunk = group if group > self.EVAL_CHUNK else (self.EVAL_CHUNK // group) * group
            for i in range(0, n_eval, chunk):
                b = min(chunk, n_eval - i)
                st = self._eval_step(b, T, group)
                st.x.copy_(ds.data[i:i + b])
                st.y.copy_(ds.labels[i:i + b])
                st.run()
                if want_lists:
                    preds.append(st.pred.clone())
            if want_lists:
                labels_all.append(ds.labels[:n_eval])
            n_seen = n_eval
        else:
            n_seen = 0
            for inputs, labels in data_loader:
                self._check_batch((inputs, labels))
                st = self._eval_step(inputs.shape[0], inputs.shape[2])
                st.x.copy_(inputs, non_blocking=True)
                st.y.copy_(labels, non_blocking=True)
                st.run()
                n_seen += int(inputs.shape[0])
                if want_lists:
                    preds.append(st.pred.clone())
                    labels_all.append(st.y.clone())
        self._host_conf.copy_(self._eval_conf, non_blocking=True)
        self._host_loss[1:2].copy_(self._eval_loss, non_blocking=True)
        lists = None
        if want_lists:
            lists = []
            for t in (preds, labels_all):
                dev_t = torch.cat(t) if t else torch.zeros(0, dtype=torch.int64, device=self.device)
                host_t = torch.empty(dev_t.shape, dtype=dev_t.dtype).pin_memory()
                lists.append(host_t.copy_(dev_t, non_blocking=True))
        return self._event(), n_seen, lists

    def evaluate_async(self, data_loader, want_lists=False):
        """Generator form of ``evaluate``: yields the CUDA event that marks the read-back, then returns
        ``(loss, acc, f1)`` (plus the prediction / label arrays with ``want_lists``)."""
        if self.use_class_weights and self._class_weight is None:
            raise ValueError("use_class_weights: the class weights are fixed by the first train(); evaluate() cannot run before it")
        t0 = time.time()
        with self._on_stream():
            done, n_seen, lists = self._enqueue_evaluate(data_loader, want_lists)
        self.timing['evaluate'] += time.time() - t0
        yield done
        nc = self.model.num_classes
        conf = self._host_conf.numpy().reshape(nc, nc).copy()
        loss = float(self._host_loss[1]) / len(data_loader.dataset)
        acc, f1 = metrics_from_confusion(conf)
        if int(conf.sum()) != n_seen:
            raise _ext.MmsError(f"evaluation counted {int(conf.sum())} windows, expected {n_seen}")
        if want_lists:
            return loss, acc, f1, lists[0].numpy(), lists[1].numpy()
        return loss, acc, f1

    def evaluate(self, data_loader, is_test=False, is_val=False):
        """reference trainer.py:193-247.  Loss sum, predictions and the confusion matrix are accumulated on
        the device (``mms_eval_accumulate``); accuracy and weighted F1 are computed from the matrix
        (``metrics_from_confusion`` == sklearn's accuracy_score / f1_score(average='weighted')).
        A ``DeviceBatchLoader`` is evaluated in slices of ``EVAL_CHUNK`` windows straight from the
        device-resident array: in eval mode every window's logits are independent of its batch."""
        out = drive(self.evaluate_async(data_loader, want_lists=is_test or is_val))
        if is_test:
            return self.finish_test(*out)
        if is_val:
            loss, acc, f1, all_preds, all_labels = out
            return loss, acc, f1, list(all_preds), list(all_labels)
        return out

    def channel_attribution(self, data_loader, steps=32, channel_names=None, max_rows=2048):
        """Which input channels the model's predictions rest on: integrated gradients (``attribution.py``, eval mode,
        zero baseline, target = the predicted class) over every window of ``data_loader``.  Returns float64
        ``[num_classes, C]``: row k is the mean, over the windows whose TRUE class is k, of |S_b,c| / sum_c' |S_b,c'|
        (zeros for a class without windows).  Also writes ``channel_attribution.txt`` (channels x classes) in the fold
        directory."""
        from .attribution import channel_shares, integrated_gradients
        m = self.model
        nc, Cc = m.num_classes, m.in_channels
        names = list(channel_names) if channel_names is not None else [f"channel_{c}" for c in range(Cc)]
        if len(names) != Cc:
            raise ValueError(f"channel_attribution: {len(names)} channel names for {Cc} channels")
        was_training = m.training
        m.eval()
        sums = torch.zeros(nc, Cc, dtype=torch.float64, device=self.device)
        counts = torch.zeros(nc, dtype=torch.float64, device=self.device)
        try:
            with self._on_stream():
                for batch in data_loader:
                    x, y = batch[0], batch[1]
                    x = x.to(self.device, non_blocking=True).float()
                    y = y.to(self.device, non_blocking=True).long()
                    _, S, _ = integrated_gradients(m, x, steps=steps, max_rows=max_rows)
                    sums.index_add_(0, y, channel_shares(S))
                    counts.index_add_(0, y, torch.ones_like(y, dtype=torch.float64))
                out = (sums / counts.clamp_min(1.0)[:, None]).cpu()
        finally:
            m.train(was_training)
        with open(self.fold_dir / 'channel_attribution.txt', 'w', encoding='utf-8') as f:
            f.write(f"# integrated gradients, {steps} steps, zero baseline, target = predicted class\n")
            f.write("# mean over the windows of each true class of |S_c| / sum_c' |S_c'|\n")
            f.write("channel" + "".join(f"\tclass_{k}" for k in range(nc)) + "\n")
            for c, name in enumerate(names):
                f.write(name + "".join(f"\t{out[k, c].item():.6f}" for k in range(nc)) + "\n")
        return out

    def mc_dropout_uncertainty(self, data_loader, samples=32, max_rows=2048):
        """How sure the model is, window by window: MC dropout (``uncertainty.mc_dropout``, BatchNorm in eval mode,
        ``samples`` dropout samples) over every window of ``data_loader``, as one call with the explicit seed
        ``model._rng_seed``, so the result does not depend on how the loader batches the windows.  Returns a dict: the
        accuracy and weighted F1 of the MC prediction; the mean entropy and mutual information over all, correctly
        classified and misclassified windows (NaN for an empty group); the AUROC of each as a detector of misclassified
        windows (NaN without errors or without correct windows); the ECE of the MC mean and of the plain eval softmax.
        Also writes ``uncertainty.txt`` in the fold directory."""
        from .uncertainty import auroc, expected_calibration_error, mc_dropout
        m = self.model
        nc = m.num_classes
        was_training = m.training
        m.eval()
        try:
            with self._on_stream():
                xs, ys = [], []
                for batch in data_loader:
                    xs.append(batch[0].to(self.device, non_blocking=True).float())
                    ys.append(batch[1].to(self.device, non_blocking=True).long())
                if not xs:
                    raise ValueError("mc_dropout_uncertainty: the loader holds no windows")
                x, y = torch.cat(xs), torch.cat(ys)
                res = mc_dropout(m, x, samples=samples, seed=m._rng_seed, max_rows=max_rows)
                with torch.no_grad():
                    eval_probs = torch.cat([torch.softmax(m(x[i:i + max_rows]).double(), dim=1)
                                            for i in range(0, x.shape[0], max_rows)])
                out = [t.cpu().numpy() for t in (res.probs, res.entropy, res.mutual_info, res.prediction, y, eval_probs)]
        finally:
            m.train(was_training)
        probs, ent, mi, pred, labels, eval_probs = out
        conf = np.zeros((nc, nc), dtype=np.int64)
        np.add.at(conf, (labels, pred), 1)
        acc, f1 = metrics_from_confusion(conf)
        wrong = pred != labels
        mean = lambda v: float(v.mean()) if v.size else float("nan")
        result = {
            'windows': int(labels.size), 'samples': int(samples), 'accuracy': acc, 'f1_score': f1,
            'mean_entropy': mean(ent), 'mean_entropy_correct': mean(ent[~wrong]), 'mean_entropy_wrong': mean(ent[wrong]),
            'mean_mutual_info': mean(mi), 'mean_mutual_info_correct': mean(mi[~wrong]),
            'mean_mutual_info_wrong': mean(mi[wrong]),
            'auroc_entropy': auroc(ent, wrong), 'auroc_mutual_info': auroc(mi, wrong),
            'ece_mc': expected_calibration_error(probs, labels), 'ece_eval': expected_calibration_error(eval_probs, labels),
        }
        with open(self.fold_dir / 'uncertainty.txt', 'w', encoding='utf-8') as f:
            f.write(f"# MC dropout, {samples} samples per window, BatchNorm on running statistics, p = {m.dropout_p}\n")
            f.write("# AUROC: entropy / mutual information as a detector of misclassified windows; ECE: 10 equal-width bins\n")
            for k, v in result.items():
                f.write(f"{k}\t{v:.6f}\n" if isinstance(v, float) else f"{k}\t{v}\n")
        return result

    def finish_test(self, loss, acc, f1, all_preds, all_labels):
        """The is_test tail of reference trainer.py:231-240: confusion-matrix plot + the two log lines."""
        self.plot_confusion_matrix(all_labels, all_preds, filename="test_confusion_matrix.png")
        self._log(f"\n--- 最终测试结果 (模型原始输出) ---")
        self._log(f"测试损失: {loss:.4f} | 测试Acc: {acc:.4f} | 测试F1: {f1:.4f}")
        return loss, acc, f1

    def plot_confusion_matrix(self, true_labels, pred_labels, filename="confusion_matrix.png"):
        """Plotting is out of scope (SURVEY §2); like the reference's own try/except
        (trainer.py:250-273) a missing matplotlib only produces a log line."""
        try:
            from sklearn.metrics import confusion_matrix
            import matplotlib.pyplot as plt
            cm = confusion_matrix(true_labels, pred_labels)
            fig = plt.figure(figsize=(8, 6))
            plt.imshow(cm, cmap='Blues')
            for (i, j), v in np.ndenumerate(cm):
                plt.text(j, i, str(v), ha='center', va='center')
            plt.xlabel('Predicted Label')
            plt.ylabel('True Label')
            plt.title('Confusion Matrix')
            cm_path = self.fold_dir / filename
            plt.savefig(cm_path)
            plt.close(fig)
            self._log(f"混淆矩阵已保存至: {cm_path}")
        except Exception as e:
            self._log(f"保存混淆矩阵失败: {str(e)}")
