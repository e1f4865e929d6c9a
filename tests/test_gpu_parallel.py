"""Intra-fold data parallelism (SyncBN + one flat gradient reduction), emulated on ONE GPU: two ranks'
phase-split steps run in lockstep with their sync tensors summed by hand -- exactly what the NCCL
all-reduce does -- and must reproduce the single-device full-batch step (the reference computes BN
statistics over the whole batch, models.py:47,51)."""
import copy
import time

import numpy as np
import pytest
import torch

from conftest import golden_state, load_golden

pytestmark = pytest.mark.gpu


def _model(meta, sd):
    from multimodalsignal_b200.models import CnnGruAttentionModel
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m = CnnGruAttentionModel(meta["C"], meta["num_classes"], dropout=0.0, **meta["kwargs"])
    m.load_state_dict(sd, strict=True)
    return m.cuda().train()


@pytest.mark.parametrize("case,splits", [("c6_t640", (2, 2)), ("c6_t640", (1, 3)), ("c8_h32_l1", (2, 1))])
def test_two_rank_data_parallel_equals_full_batch(case, splits):
    from multimodalsignal_b200.parallel import DataParallelTrainStep, emulate_ranks
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    z, meta = load_golden(f"model_{case}.npz")
    sd = golden_state(z, "sd")
    x, y = torch.from_numpy(z["x"]).cuda(), torch.from_numpy(z["y"]).cuda()
    B, T = x.shape[0], x.shape[2]
    assert sum(splits) == B
    # single device, full batch (already pinned to the reference's Adam trajectory by test_gpu_model.py)
    ref = _model(meta, sd)
    ref_step = FusedTrainStep(ref, FlatAdam(ref, lr=1e-3, weight_decay=1e-4), B, T, use_graph=False)
    # two emulated ranks
    ranks, steps, lo = [], [], 0
    for r, b in enumerate(splits):
        m = _model(meta, sd)
        ranks.append(m)
        steps.append(DataParallelTrainStep(m, FlatAdam(m, lr=1e-3, weight_decay=1e-4), b, B, T, rank=r))
    losses = []
    for it in range(3):
        ref_step(x, y)
        lo, batches = 0, []
        for b in splits:
            batches.append((x[lo:lo + b], y[lo:lo + b]))
            lo += b
        emulate_ranks(steps, batches)
        losses.append(sum(float(s.loss.item()) for s in steps))
        assert abs(losses[-1] - ref_step.last_loss()) < 2e-5
    ref_sd = ref.state_dict()
    for m in ranks:
        for k, v in m.state_dict().items():
            if v.numel() == 0:
                continue
            np.testing.assert_allclose(v.float().cpu().numpy(), ref_sd[k].float().cpu().numpy(), atol=2e-5, err_msg=k)
    if "adam_losses" in z:        # and therefore also the reference's own trajectory
        np.testing.assert_allclose(losses[:int(z["adam_steps"])], z["adam_losses"][:3], atol=1e-4)


def test_nccl_data_parallel_two_gpus():
    """The same check over real NCCL (skipped on a single-GPU box)."""
    import os
    import subprocess
    import sys
    from conftest import ROOT
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29633", str(ROOT / "tools" / "dp_check.py")],
                       capture_output=True, text=True, timeout=600, env=dict(os.environ))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "dp_check ok" in r.stdout


def test_sharded_preprocess_two_gpus():
    """Subject-sharded resampling + NCCL broadcast of the streams == single-process preprocessing, bit for bit
    (skipped on a single-GPU box)."""
    import os
    import subprocess
    import sys
    from conftest import ROOT
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29637", str(ROOT / "tools" / "shard_check.py")],
                       capture_output=True, text=True, timeout=600, env=dict(os.environ))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "shard_check ok" in r.stdout


@pytest.mark.timeout(120)
@pytest.mark.skipif(__import__("os").environ.get("MMS_TEST_PEER_EMULATION") != "1",
                    reason="kernels of several emulated ranks spin on each other's flags as separate launches on ONE GPU; nothing "
                           "guarantees co-scheduling (B200_PROFILING.md), so this runs only on request: MMS_TEST_PEER_EMULATION=1. "
                           "The default suite covers the peer kernels with world = 1 and, on >= 2 GPUs, one process per GPU.")
@pytest.mark.parametrize("case,splits", [("c6_t640", (2, 2)), ("c6_t640", (1, 3)), ("c6_t640", (1, 1, 2)), ("c8_h32_l1", (2, 1))])
def test_peer_memory_exchange_equals_full_batch(case, splits):
    """The B200-native exchange (csrc/peer.cu): every rank's step -- phase-split forward/backward, SyncBN vectors summed by
    ``mms_peer_allreduce_f64``, gradient all-reduce fused with Adam in ``mms_peer_allreduce_adam``, flag barriers through
    the peers' signal pads -- here with the ranks emulated inside one process (one stream per rank, plain device memory in
    place of symmetric memory).  It must reproduce the single-device full-batch step, and the ranks' parameters must
    stay bit-identical to each other (the gradients are summed in rank order on every rank)."""
    from multimodalsignal_b200.parallel import DataParallelTrainStep, LocalPeers, emulate_peer_ranks
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    z, meta = load_golden(f"model_{case}.npz")
    sd = golden_state(z, "sd")
    x, y = torch.from_numpy(z["x"]).cuda(), torch.from_numpy(z["y"]).cuda()
    B, T = x.shape[0], x.shape[2]
    assert sum(splits) == B
    ref = _model(meta, sd)
    ref_step = FusedTrainStep(ref, FlatAdam(ref, lr=1e-3, weight_decay=1e-4), B, T, use_graph=False)
    # The library's side streams are process-global: with several emulated ranks enqueued one after the other from ONE
    # host thread, rank 0's later side-stream work would queue in front of rank 1's earlier work and wait for a flag that
    # rank 1 can then never set.  (One process per GPU -- the real configuration -- has its own side streams.)
    from multimodalsignal_b200 import _ext
    _ext.lib().mms_set_side_streams(0)
    peers = LocalPeers(len(splits))
    streams = [torch.cuda.Stream() for _ in splits]
    ranks, steps = [], []
    for r, b in enumerate(splits):
        with torch.cuda.stream(streams[r]):
            m = _model(meta, sd)
            ranks.append(m)
            steps.append(DataParallelTrainStep(m, FlatAdam(m, lr=1e-3, weight_decay=1e-4), b, B, T, rank=r, peer=peers, use_graph=False))
    torch.cuda.synchronize()
    for it in range(4):
        ref_step(x, y)
        lo, batches = 0, []
        for b in splits:
            batches.append((x[lo:lo + b], y[lo:lo + b]))
            lo += b
        emulate_peer_ranks(steps, batches, streams)      # rank r on stream r; the peer kernels of the ranks meet on the device
        torch.cuda.synchronize()
        loss = sum(float(s.loss.item()) for s in steps)
        assert abs(loss - ref_step.last_loss()) < 2e-5, (it, loss, ref_step.last_loss())
    ref_sd = ref.state_dict()
    for m in ranks:
        for k, v in m.state_dict().items():
            if v.numel() == 0:
                continue
            np.testing.assert_allclose(v.float().cpu().numpy(), ref_sd[k].float().cpu().numpy(), atol=1e-4, err_msg=k)
    _ext.lib().mms_set_side_streams(1)
    for m in ranks[1:]:
        assert torch.equal(m.flat_parameters(), ranks[0].flat_parameters())
    assert int(steps[0].opt.step_dev.item()) == 4


@pytest.mark.timeout(120)
@pytest.mark.parametrize("case,graph", [("c6_t640", False), ("c6_t640", True), ("c8_h32_l1", True)])
def test_peer_kernels_world_1_equal_fused_step(case, graph):
    """The peer-memory step with a world of ONE rank (its flag barriers are with itself: no kernel ever waits for another
    launch) must equal the fused single-device step: this covers the arithmetic of ``mms_peer_allreduce_f64`` and of the
    fused all-reduce + Adam kernel, the epoch bookkeeping across steps, and CUDA-graph capture / replay of the whole step."""
    from multimodalsignal_b200.parallel import DataParallelTrainStep, LocalPeers
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    z, meta = load_golden(f"model_{case}.npz")
    sd = golden_state(z, "sd")
    x, y = torch.from_numpy(z["x"]).cuda(), torch.from_numpy(z["y"]).cuda()
    B, T = x.shape[0], x.shape[2]
    ref = _model(meta, sd)
    ref_step = FusedTrainStep(ref, FlatAdam(ref, lr=1e-3, weight_decay=1e-4), B, T, use_graph=False)
    m = _model(meta, sd)
    step = DataParallelTrainStep(m, FlatAdam(m, lr=1e-3, weight_decay=1e-4), B, B, T, rank=0, peer=LocalPeers(1), use_graph=graph)
    for it in range(5):
        ref_step(x, y)
        step(x, y)
        torch.cuda.synchronize()
        assert abs(float(step.loss.item()) - ref_step.last_loss()) < 2e-5, it
    assert int(step.epoch.item()) == 25 and int(step.opt.step_dev.item()) == 5      # 5 exchanges per step
    ref_sd = ref.state_dict()
    for k, v in m.state_dict().items():
        if v.numel():
            np.testing.assert_allclose(v.float().cpu().numpy(), ref_sd[k].float().cpu().numpy(), atol=1e-4, err_msg=k)


def test_peer_memory_exchange_two_gpus():
    """The same over real symmetric memory / NVLink, one process per GPU (skipped on a single-GPU box)."""
    import os
    import subprocess
    import sys
    from conftest import ROOT
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29641", str(ROOT / "tools" / "dp_check.py"), "--peer"],
                       capture_output=True, text=True, timeout=600, env=dict(os.environ))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "dp_check ok" in r.stdout


@pytest.mark.timeout(60)
def test_peer_wait_is_bounded_and_reported():
    """csrc/peer.cu failure behaviour: a peer that never signals (a dead or diverged rank) must not hang the kernel.  World of
    two ranks of which only rank 0 ever runs: its waits run into the deadline (MMS_PEER_TIMEOUT_MS), the kernels finish,
    and mms_peer_status reports -- and clears -- the timeouts."""
    import ctypes as C
    from multimodalsignal_b200 import _ext
    lib = _ext.lib()
    dev = torch.device("cuda")
    bufs = [torch.ones(8, dtype=torch.float64, device=dev), torch.full((8,), 2.0, dtype=torch.float64, device=dev)]
    sigs = [torch.zeros(256, dtype=torch.int32, device=dev) for _ in range(2)]
    epoch = torch.zeros(1, dtype=torch.int32, device=dev)
    arr = lambda ts: (C.c_void_p * 2)(*[t.data_ptr() for t in ts])
    n = C.c_uint32(7)
    _ext.check(lib.mms_peer_status(C.byref(n)))          # clear whatever earlier tests left
    prev = lib.mms_get_option(b"PEER_TIMEOUT_MS", -1)
    _ext.check(lib.mms_set_option(b"PEER_TIMEOUT_MS", 20))
    try:
        t0 = time.perf_counter()
        _ext.check(lib.mms_peer_allreduce_f64(arr(bufs), arr(sigs), 2, 0, 0, 8, epoch.data_ptr(), torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        assert time.perf_counter() - t0 < 5.0
        _ext.check(lib.mms_peer_status(C.byref(n)))
        assert n.value >= 1                                # both barriers of the call timed out on the silent peer's word
        _ext.check(lib.mms_peer_status(C.byref(n)))
        assert n.value == 0                                # read-and-clear
        # the fused gradient all-reduce + Adam: every CTA waits for itself, none for another CTA of the launch
        N = 4096
        p, m, v = (torch.zeros(N, device=dev) for _ in range(3))
        g = [torch.ones(N, device=dev), torch.ones(N, device=dev)]
        lr = torch.full((1,), 1e-3, device=dev)
        step = torch.zeros(1, dtype=torch.int64, device=dev)
        scratch = torch.zeros(2, dtype=torch.int32, device=dev)
        _ext.check(lib.mms_peer_allreduce_adam(p.data_ptr(), arr(g), arr(sigs), 2, 0, 8, m.data_ptr(), v.data_ptr(), N, lr.data_ptr(),
                                               0.9, 0.999, 1e-8, 0.0, step.data_ptr(), epoch.data_ptr(), scratch.data_ptr(),
                                               torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        _ext.check(lib.mms_peer_status(C.byref(n)))
        assert n.value >= 1
    finally:
        _ext.check(lib.mms_set_option(b"PEER_TIMEOUT_MS", prev) if prev >= 0 else lib.mms_clear_option(b"PEER_TIMEOUT_MS"))
