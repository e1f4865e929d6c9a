"""Intra-fold data parallelism (SURVEY §8e, BASELINE.json configs[4]): the global batch is split over the
ranks of a process group; every rank holds a replica of the model.

The reference computes BatchNorm statistics over the WHOLE batch on one device (models.py:47,51), so a
faithful data-parallel step needs SyncBN: the float64 batch sums (forward) and the two BN reductions
(backward) are sum-all-reduced between the phases of ``mms_cnngru_{forward,backward}_phase``; the loss is
the global mean (``mms_cross_entropy_partial``); the flat gradient buffer is sum-all-reduced ONCE per
step and the fused Adam kernel then runs on every rank.  All messages are tiny (<= 0.5 MB): latency-bound
on NVLink 5 / NVSwitch, which is why the gradient is one flat buffer and one collective.

The step is written as a generator that yields the tensors to reduce, so the same code runs under
``torch.distributed`` (NCCL) and in the single-process emulation the parity tests use.

``peer=`` selects the B200-native exchange instead: the workspace and the gradient buffer live in symmetric memory
(``torch.distributed._symmetric_memory``: allocation + rendezvous are plumbing), and the five exchange points are OUR
kernels reading the peers' buffers over NVLink -- ``mms_peer_allreduce_f64`` for the SyncBN vectors and
``mms_peer_allreduce_adam``, the gradient all-reduce fused with the Adam update (csrc/peer.cu).  No communication-library
call is left on the data path, and the whole step (kernels + flag barriers) is one CUDA graph per rank.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _ext
from ._ext import CnnGruDesc, check, ptr, stream
from .trainer import FlatAdam


class DataParallelTrainStep:
    """One rank's share of a data-parallel training step.  ``local_batch`` rows of a ``global_batch`` batch."""

    def __init__(self, model, optimizer: FlatAdam, local_batch: int, global_batch: int, seq_len: int, rank: int = 0, group=None,
                 peer=None, use_graph: bool = True, class_weight=None):
        """``peer``: None = ``torch.distributed`` all-reduces (NCCL); ``"symm"`` = symmetric memory + the peer kernels
        (one process per GPU, needs an initialised process group); a ``LocalPeers`` registry = several ranks emulated
        inside one process on one GPU (tests).

        ``class_weight`` (``num_classes`` values, the same on every rank): ``CrossEntropyLoss(weight=...)`` over the
        GLOBAL batch.  Its normaliser sum_b w[y_b] needs every rank's labels; it travels as one more double at the end
        of the BN2 sum vector (``mms_cnngru_sync_offsets``), so the existing exchange sums it and no message is added."""
        from .trainer import class_weight_tensor
        self.lib = _ext.lib()
        self.model, self.opt, self.group = model, optimizer, group
        self.peer, self.rank = peer, rank
        self.flat = model.flat_parameters()
        dev = self.flat.device
        self.class_weight = None if class_weight is None else class_weight_tensor(class_weight, model.num_classes, dev)
        d = CnnGruDesc()
        d.batch, d.in_channels, d.seq_len, d.num_classes = local_batch, model.in_channels, seq_len, model.num_classes
        d.cnn_out, d.hidden, d.layers = model.cnn_out_channels, model.gru_hidden_size, model.gru_num_layers
        d.training, d.attention, d.need_grad = 1, int(model.attention), 1
        d.dropout_p = float(model.dropout_p)
        d.rng_seed, d.rng_offset = (model._rng_seed ^ (0x9E3779B9 * (rank + 1))) & 0xFFFFFFFFFFFFFFFF, 0
        d.rng_offset_dev = optimizer.step_dev.data_ptr()
        d.global_batch = global_batch
        d.class_weight = None if self.class_weight is None else self.class_weight.data_ptr()
        self.desc = d
        self.local_batch, self.global_batch = local_batch, global_batch
        nbytes = self.lib.mms_cnngru_workspace_bytes(C.byref(d))
        if nbytes < 0:
            check(int(nbytes))
        self.workspace = self._alloc(int(nbytes), torch.uint8, dev)
        offs = (C.c_int64 * 4)()
        cnts = (C.c_int64 * 4)()
        check(self.lib.mms_cnngru_sync_offsets(C.byref(d), offs, cnts))
        view = lambda i: self.workspace[offs[i]:offs[i] + 8 * cnts[i]].view(torch.float64)
        self.stats1, self.stats2, self.red1, self.red2 = view(0), view(1), view(2), view(3)
        self.weight_sum = self.stats2[-1:] if self.class_weight is not None else None     # sum_b w[y_b], summed over the ranks
        self.logits = torch.zeros(local_batch, model.num_classes, dtype=torch.float32, device=dev)
        self.dlogits = torch.zeros_like(self.logits)
        self.loss = torch.zeros(1, dtype=torch.float32, device=dev)        # this rank's share of the global mean
        self._sync_offsets = [(int(offs[i]), int(cnts[i])) for i in range(4)]
        self.use_graph, self.graph, self.calls = use_graph, None, 0
        self._graphs, self._eager_done, self._table = {}, set(), None     # peer path: one graph per freeze plan
        self.x = torch.zeros(local_batch, model.in_channels, seq_len, dtype=torch.float32, device=dev)
        self.y = torch.zeros(local_batch, dtype=torch.int64, device=dev)
        if peer is not None:
            self._setup_peer(dev)

    # ------------------------------------------------------------------ peer-memory exchange (csrc/peer.cu)
    def _alloc(self, n, dtype, dev):
        if self.peer == "symm":
            import torch.distributed._symmetric_memory as symm
            t = symm.empty(n, dtype=dtype, device=dev)
            t.zero_()
            return t
        return torch.zeros(n, dtype=dtype, device=dev)

    def _setup_peer(self, dev):
        opt = self.opt
        grads = self._alloc(opt.grads.numel(), torch.float32, dev)          # the gradient buffer the peers read
        opt.grads = grads
        self.signals = self._alloc(256, torch.int32, dev)                   # this rank's signal pad
        self.epoch = torch.zeros(1, dtype=torch.int32, device=dev)
        self.norm_epoch = torch.zeros(1, dtype=torch.int32, device=dev)      # mms_peer_grad_norm's own epoch (clipping)
        self.scratch2 = torch.zeros(2, dtype=torch.int32, device=dev)
        if self.peer == "symm":
            import torch.distributed as dist
            import torch.distributed._symmetric_memory as symm
            group = self.group if self.group is not None else dist.group.WORLD
            self.world = dist.get_world_size(group)
            hw, hg, hs = (symm.rendezvous(t, group) for t in (self.workspace, grads, self.signals))
            self._handles = (hw, hg, hs)
            ws_ptrs, g_ptrs, s_ptrs = list(hw.buffer_ptrs), list(hg.buffer_ptrs), list(hs.buffer_ptrs)
            torch.cuda.synchronize()
            dist.barrier(group)                   # every rank has zeroed its buffers before anybody signals
        else:                                     # LocalPeers: ranks of one process, plain device memory
            self.peer.register(self.rank, self.workspace, grads, self.signals)
            self.world = self.peer.world
            ws_ptrs = g_ptrs = s_ptrs = None
        self._ptrs = (ws_ptrs, g_ptrs, s_ptrs)
        self._tables = None

    def _peer_tables(self):
        """HOST arrays of device pointers (one entry per rank) for the four SyncBN vectors, the gradients and the pads."""
        if self._tables is None:
            ws_ptrs, g_ptrs, s_ptrs = self._ptrs if self._ptrs[0] is not None else self.peer.pointers()
            arr = lambda ps: (C.c_void_p * self.world)(*[int(p) for p in ps])
            self._tables = ([arr([p + off for p in ws_ptrs]) for off, _ in self._sync_offsets], arr(g_ptrs), arr(s_ptrs))
        return self._tables

    def _peer_sum(self, k):
        stats, _, sig = self._peer_tables()
        check(self.lib.mms_peer_allreduce_f64(stats[k], sig, self.world, self.rank, 0, self._sync_offsets[k][1], ptr(self.epoch), stream()))

    def _peer_phases(self):
        """The whole data-parallel step with the peer kernels at the five exchange points, as a generator that yields
        after every exchange kernel has been enqueued (the single-process emulation interleaves the ranks there)."""
        x, y, o, g = self.x, self.y, self.opt, self.opt.param_groups[0]
        self._set_plan()
        o.grads.zero_()                                          # trainer.py:144
        self._fwd(1, x)
        self._weight_sum(y)
        self._peer_sum(0)                                        # SyncBN stage 1
        yield
        self._fwd(2, x)
        self._peer_sum(1)                                        # (+ the weighted loss's normaliser)
        yield
        self._fwd(4, x)                                          # trainer.py:146
        self._loss(y)                                            # :147
        self._bwd(1, x)                                          # trainer.py:148
        self._peer_sum(3)                                        # SyncBN backward, stage 2
        yield
        self._bwd(2, x)
        self._peer_sum(2)
        yield
        self._bwd(4, x)
        _, grads, sig = self._peer_tables()
        if o.max_grad_norm is not None:
            # clip_grad_norm_ on the summed gradient: every rank forms the same norm from the peers' buffers, on pad words
            # [2 world, 3 world) with its own epoch (the Adam kernel below uses [0, 2 world) and self.epoch)
            nt = o.norm_table(self._table)
            check(self.lib.mms_peer_grad_norm(grads, sig, self.world, self.rank, 2 * self.world, self.flat.numel(), nt, len(nt) // 3,
                                              ptr(o.clip_max_norm), ptr(o.clip_record), ptr(o.clip_scratch), ptr(self.norm_epoch),
                                              stream()))
            yield
            if self._table is None:
                check(self.lib.mms_peer_allreduce_adam_clip(ptr(self.flat), grads, sig, self.world, self.rank, 0, ptr(o.exp_avg),
                                                            ptr(o.exp_avg_sq), self.flat.numel(), ptr(o.lr_dev), g['betas'][0],
                                                            g['betas'][1], g['eps'], g['weight_decay'], ptr(o.step_dev), ptr(self.epoch),
                                                            ptr(self.scratch2), ptr(o.clip_coef), stream()))
            else:
                check(self.lib.mms_peer_allreduce_adam_ranges_clip(ptr(self.flat), grads, sig, self.world, self.rank, 0, ptr(o.exp_avg),
                                                                   ptr(o.exp_avg_sq), self._table, len(self._table) // 3,
                                                                   ptr(o.tensor_steps), ptr(o.lr_dev), g['betas'][0], g['betas'][1],
                                                                   g['eps'], g['weight_decay'], ptr(o.step_dev), ptr(self.epoch),
                                                                   ptr(self.scratch2), ptr(o.clip_coef), stream()))
            return
        if self._table is None:
            check(self.lib.mms_peer_allreduce_adam(ptr(self.flat), grads, sig, self.world, self.rank, 0, ptr(o.exp_avg), ptr(o.exp_avg_sq),
                                                   self.flat.numel(), ptr(o.lr_dev), g['betas'][0], g['betas'][1], g['eps'],
                                                   g['weight_decay'], ptr(o.step_dev), ptr(self.epoch), ptr(self.scratch2), stream()))   # :149
        else:                       # frozen parameters: the update (and the sum it reads) over the trainable tensors only
            check(self.lib.mms_peer_allreduce_adam_ranges(ptr(self.flat), grads, sig, self.world, self.rank, 0, ptr(o.exp_avg),
                                                          ptr(o.exp_avg_sq), self._table, len(self._table) // 3, ptr(o.tensor_steps),
                                                          ptr(o.lr_dev), g['betas'][0], g['betas'][1], g['eps'], g['weight_decay'],
                                                          ptr(o.step_dev), ptr(self.epoch), ptr(self.scratch2), stream()))

    def _enqueue_peer(self):
        for _ in self._peer_phases():
            pass

    def _set_plan(self):
        """Reads the parameters' ``requires_grad`` (FlatAdam.plan) into the descriptor; returns the plan's graph key."""
        mask, table = self.opt.plan()
        self.desc.frozen_segments = mask
        self._table = table
        return mask, None if table is None else tuple(table), self.opt.max_grad_norm is not None

    def run_peer(self):
        """One step on the static inputs ``self.x`` / ``self.y`` (graph replay after the first call of each freeze plan)."""
        from .trainer import capture_graph
        self.opt.sync_lr()
        self.calls += 1
        key = self._set_plan()
        if not self.use_graph or key not in self._eager_done:
            self._eager_done.add(key)
            self._enqueue_peer()
            return
        self.graph = self._graphs.get(key)
        if self.graph is None:
            self.graph = self._graphs[key] = capture_graph(self._enqueue_peer)
        self.graph.replay()

    def _weight_sum(self, y):
        """Local sum_b w[y_b] into the extra slot of the BN2 sum vector (after forward phase 1 cleared it)."""
        if self.class_weight is not None:
            check(self.lib.mms_class_weight_sum(ptr(y), self.local_batch, self.model.num_classes, ptr(self.class_weight),
                                                ptr(self.weight_sum), stream()))

    def _loss(self, y):
        """This rank's share of the global mean loss and its dlogits (trainer.py:147)."""
        if self.class_weight is None:
            check(self.lib.mms_cross_entropy_partial(ptr(self.logits), ptr(y), self.local_batch, self.model.num_classes,
                                                     self.global_batch, ptr(self.loss), ptr(self.dlogits), None, stream()))
        else:
            check(self.lib.mms_cross_entropy_weighted(ptr(self.logits), ptr(y), self.local_batch, self.model.num_classes,
                                                      ptr(self.class_weight), ptr(self.weight_sum), ptr(self.loss),
                                                      ptr(self.dlogits), None, stream()))

    def _fwd(self, phases, x):
        m = self.model
        check(self.lib.mms_cnngru_forward_phase(C.byref(self.desc), phases, ptr(x), ptr(self.flat), ptr(m._bn_flat), ptr(m._nbt_flat),
                                                ptr(self.workspace), ptr(self.logits), stream()))

    def _bwd(self, phases, x):
        m, o = self.model, self.opt
        check(self.lib.mms_cnngru_backward_phase(C.byref(self.desc), phases, ptr(x), ptr(self.flat), ptr(m._bn_flat),
                                                 ptr(self.workspace), ptr(self.dlogits), ptr(o.grads), stream()))

    def phases(self, x, y):
        """Generator over the step: yields each tensor that must be sum-reduced over the ranks before it resumes."""
        x = x.contiguous().float()
        y = y.contiguous()
        self._set_plan()
        self.opt.grads.zero_()                                   # trainer.py:144
        self._fwd(1, x)
        self._weight_sum(y)
        yield self.stats1                                        # SyncBN, stage 1: (sum, sum of squares) per channel
        self._fwd(2, x)
        yield self.stats2                                        # (+ sum_b w[y_b] with class weights)
        self._fwd(4, x)                                          # trainer.py:146
        self._loss(y)                                            # :147
        self._bwd(1, x)                                          # trainer.py:148
        yield self.red2                                          # SyncBN backward, stage 2: (sum dy, sum dy*xhat)
        self._bwd(2, x)
        yield self.red1
        self._bwd(4, x)
        yield self.opt.grads                                     # ONE flat gradient all-reduce (~0.5 MB)
        self.opt.flat_step(self.flat)                            # trainer.py:149 (clips the summed gradient if the optimizer does)

    def __call__(self, x, y):
        if self.peer is not None:
            self.x.copy_(x, non_blocking=True)
            self.y.copy_(y, non_blocking=True)
            self.run_peer()
            return
        import torch.distributed as dist
        for t in self.phases(x, y):
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)

    def check_peers(self):
        """Failure detection of the peer-memory path, called wherever results are read back: raises if any bounded wait of the
        peer kernels timed out on this device (a rank died, raised between two phases or made a different number of steps:
        the sums of such a step are meaningless) or if the ranks disagree on the number of steps made."""
        if self.peer is None:
            return
        n = C.c_uint32(0)
        check(self.lib.mms_peer_status(C.byref(n)))
        if n.value:
            raise RuntimeError(f"data-parallel peer exchange: {n.value} wait(s) timed out on rank {self.rank} -- a peer did not reach "
                               "the same exchange point (MMS_PEER_TIMEOUT_MS); the parameters of this fold are no longer valid")
        import torch.distributed as dist
        if self.peer == "symm" and dist.is_available() and dist.is_initialized():
            steps = torch.tensor([self.calls], dtype=torch.int64, device=self.loss.device)
            lo, hi = steps.clone(), steps.clone()
            dist.all_reduce(lo, op=dist.ReduceOp.MIN, group=self.group)
            dist.all_reduce(hi, op=dist.ReduceOp.MAX, group=self.group)
            if int(lo.item()) != int(hi.item()):
                raise RuntimeError(f"data-parallel ranks made different numbers of steps ({int(lo.item())} .. {int(hi.item())}): "
                                   "every rank must see the same number of batches (drop the ragged last batch or pad it)")

    def global_loss(self) -> float:
        """Mean loss over the global batch of the last step (one extra scalar all-reduce; for logging).  Also the point where
        the peer-memory path reports a failed exchange (``check_peers``)."""
        import torch.distributed as dist
        t = self.loss.clone()
        if dist.is_available() and dist.is_initialized():
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
        v = float(t.item())
        self.check_peers()
        return v


class LocalPeers:
    """Registry that lets several ``DataParallelTrainStep`` "ranks" of ONE process (one GPU, one stream per rank) find
    each other's buffers: the single-GPU stand-in for symmetric memory that the peer-kernel tests use."""

    def __init__(self, world):
        self.world = world
        self._bufs = {}

    def register(self, rank, workspace, grads, signals):
        self._bufs[rank] = (workspace, grads, signals)

    def pointers(self):
        assert len(self._bufs) == self.world, "every rank must be constructed before the first step"
        return tuple([self._bufs[r][k].data_ptr() for r in range(self.world)] for k in range(3))


def emulate_peer_ranks(steps, batches, streams):
    """Single-process emulation of the peer exchange: rank r's kernels go to ``streams[r]``; the host interleaves the
    ranks at every exchange point, so that no rank's later work is queued (possibly in the same hardware queue) in front
    of a peer's earlier work that its flag barrier waits for.  Eager only; the graph path is exercised with one process
    per GPU."""
    gens = []
    for s, (x, y), st in zip(steps, batches, streams):
        with torch.cuda.stream(st):
            s.x.copy_(x, non_blocking=True)
            s.y.copy_(y, non_blocking=True)
            s.opt.sync_lr()
        gens.append(s._peer_phases())
    live = list(range(len(gens)))
    while live:
        for r in list(live):
            with torch.cuda.stream(streams[r]):
                try:
                    next(gens[r])
                except StopIteration:
                    live.remove(r)


def emulate_ranks(steps, batches):
    """Run several ranks' ``DataParallelTrainStep`` in lockstep inside ONE process (no collectives):
    at every sync point the yielded tensors are summed and written back to every rank.  This is the
    single-GPU stand-in for NCCL that the parity tests use."""
    gens = [s.phases(x, y) for s, (x, y) in zip(steps, batches)]
    while True:
        tensors = []
        for g in gens:
            try:
                tensors.append(next(g))
            except StopIteration:
                pass
        if not tensors:                      # every rank has run its Adam update
            break
        assert len(tensors) == len(gens), "ranks fell out of lockstep"
        total = torch.stack(tensors).sum(dim=0)
        for t in tensors:
            t.copy_(total)
