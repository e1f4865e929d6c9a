"""Training with dropout against the float64 oracle, with the exact masks the kernels drew.

Seven kernels draw dropout multipliers from the counter-based stream of csrc/mms_common.cuh, each computing its own element
ids, and model.cu picks which of them run from the shapes and the options.  The stream is a pure function of (seed, offset,
element id), so oracle/dropout_stream.py rebuilds the masks of a step on the host and the whole step -- logits, loss, every
gradient, the BatchNorm running statistics -- is checked against model_oracle in float64, at the tolerances of
test_gpu_model.py.  The seed and the offset are read from what the kernels were given (the engine's or the step's
descriptor, the optimizer's device step count), not recomputed.

First the port is pinned bit for bit to mms_dropout_apply; then every path model.cu can take under dropout is run on a shape
that reaches it, through autograd and through FusedTrainStep with and without the fused head; negative controls show that
the comparison catches wrong masks."""
import contextlib

import numpy as np
import pytest
import torch

from oracle import dropout_stream as ds
from oracle import model_oracle as mo

pytestmark = pytest.mark.gpu

LOGIT_ATOL = 1e-4
LOSS_ATOL = 1e-4
GRAD_RTOL = 1e-3
PARAM_ATOL = 5e-5


def _lib():
    from multimodalsignal_b200 import _ext
    return _ext.lib()


def _check(rc):
    from multimodalsignal_b200 import _ext
    _ext.check(rc)


@contextlib.contextmanager
def _options(opts):
    """Set run-time options (mms_set_option) for the block; restore each one afterwards."""
    lib = _lib()
    prev = {k: lib.mms_get_option(k.encode(), -1) for k in opts}
    try:
        for k, v in opts.items():
            _check(lib.mms_set_option(k.encode(), v))
        yield
    finally:
        for k, v in prev.items():
            _check(lib.mms_set_option(k.encode(), v) if v >= 0 else lib.mms_clear_option(k.encode()))


# ------------------------------------------------------------------------------------------------ a. the port, bit for bit
SEEDS = [0x0000000000000007, 0xDEADBEEF12345678, (99 * 0x9E3779B97F4A7C15 + 3) & 0xFFFFFFFFFFFFFFFF]


@pytest.mark.parametrize("p", [0.1, 0.5, 0.8])
@pytest.mark.parametrize("base", [0, 1 << 38, (1 << 40) + 12345, 2 << 40])
def test_port_matches_dropout_apply_bit_for_bit(p, base):
    """A ones input through mms_dropout_apply returns the multipliers themselves: they must equal the host port's, bit for
    bit.  n = 1, 3 (no full float4), 1 000 003 (float4 body + tail); the pointer shifted by one float takes the scalar path;
    seeds with the high word set; offsets past 2^32 given on the host and through rng_offset_dev (which wins over the host
    value)."""
    lib = _lib()
    st = torch.cuda.current_stream().cuda_stream
    off_dev = torch.zeros(1, dtype=torch.int64, device="cuda")
    draws = [(SEEDS[0], 5, None), (SEEDS[1], (1 << 32) + 3, None), (SEEDS[2], 0, (2 << 32) + 7)]
    for n in (1, 3, 1_000_003):
        ids = np.uint64(base) + np.arange(n, dtype=np.uint64)
        for seed, off_host, off_device in draws:
            ref = ds.multipliers(ids, p, seed, off_host if off_device is None else off_device)
            if off_device is not None:
                off_dev.fill_(off_device)
            for shift in (0, 1):
                src = torch.ones(n + 1, device="cuda")
                dst = torch.full((n + 1,), -1.0, device="cuda")
                _check(lib.mms_dropout_apply(src.data_ptr() + 4 * shift, dst.data_ptr() + 4 * shift, n, base, p, seed, off_host,
                                             None if off_device is None else off_dev.data_ptr(), st))
                got = dst[shift:shift + n].cpu().numpy()
                assert np.array_equal(got.view(np.uint32), ref.view(np.uint32)), (n, seed, off_host, off_device, shift,
                                                                                   int(np.sum(got != ref)))
                assert dst[n if shift == 0 else 0].item() == -1.0       # nothing written outside the n elements
    assert np.unique(ref).size == 2


# ------------------------------------------------------------------------------------------------ b. the whole step
def _state(C, nc, H, layers, seed, O=32):
    """Reference-shaped parameters (oracle/cpu_port.make_state) with non-trivial BatchNorm affine values."""
    from oracle import cpu_port
    p, bufs = cpu_port.make_state(C=C, num_classes=nc, cnn_out=O, H=H, layers=layers, seed=seed)
    g = torch.Generator().manual_seed(seed + 100)
    for k in ("cnn_encoder.1", "cnn_encoder.5"):
        p[f"{k}.weight"] = p[f"{k}.weight"] + 0.1 * torch.randn(p[f"{k}.weight"].shape, generator=g)
        p[f"{k}.bias"] = p[f"{k}.bias"] + 0.1 * torch.randn(p[f"{k}.bias"].shape, generator=g)
    return p, bufs


def _model(p, bufs, C, nc, H, layers, dropout, O=32, attention=True):
    from multimodalsignal_b200.models import CnnGruAttentionModel
    m = CnnGruAttentionModel(C, nc, cnn_out_channels=O, gru_hidden_size=H, gru_num_layers=layers, dropout=dropout,
                             attention=attention)
    sd = dict(p)
    sd.update(bufs)
    sd["cnn_encoder.1.num_batches_tracked"] = torch.zeros((), dtype=torch.int64)
    sd["cnn_encoder.5.num_batches_tracked"] = torch.zeros((), dtype=torch.int64)
    m.load_state_dict(sd, strict=True)
    return m.cuda().train()


def _masks(B, T, H, layers, p, seed, offset):
    """(GRU site masks [layers-1, B, L, 2H], head mask [B, 64]) of one device's step, float64."""
    return ds.gru_masks(B, ds.gru_seq_len(T), H, layers, p, seed, offset), ds.head_mask(B, p, seed, offset)


def _oracle(p64, x, y, layers, masks):
    gru, head = masks
    return mo.loss_and_grads(p64, x.double(), y, training=True, prune=True, gru_layers=layers,
                             drop_mask_gru=torch.from_numpy(gru) if len(gru) else None,
                             drop_mask_head=None if head is None else torch.from_numpy(head))


def _assert_nontrivial(masks, p):
    gru, head = masks
    for m in [*gru, head]:
        kept = float(np.mean(m != 0))
        assert 0.0 < kept < 1.0, kept
        assert set(np.unique(m).tolist()) == {0.0, float(ds.scale(p))}


def _mismatches(got, ref, bufs):
    """Every quantity of a GPU step outside the tolerance of the oracle step ``ref``: [] when the step agrees."""
    ref_loss, ref_logits, ref_grads, aux = ref
    bad = []
    e = float(np.abs(got["logits"] - ref_logits.numpy()).max())
    if e > LOGIT_ATOL:
        bad.append(("logits", e))
    e = abs(got["loss"] - float(ref_loss))
    if e > LOSS_ATOL:
        bad.append(("loss", e))
    for k, g in ref_grads.items():
        ref = g.numpy()
        if ref.size == 0:
            continue
        e, scale = float(np.abs(got["grads"][k] - ref).max()), max(float(np.abs(ref).max()), 1e-6)
        if e > GRAD_RTOL * scale:
            bad.append((k, e, scale))
    for prefix, key in (("cnn_encoder.1", "s1"), ("cnn_encoder.5", "s2")):
        n = aux[f"{key}_conv"].shape[0] * aux[f"{key}_conv"].shape[2]
        rm, rv = mo.running_stats_update(bufs[f"{prefix}.running_mean"].double(), bufs[f"{prefix}.running_var"].double(),
                                         aux[f"{key}_mean"].detach(), aux[f"{key}_var"].detach(), n)
        for name, r in (("running_mean", rm.numpy()), ("running_var", rv.numpy())):
            g = got["running"][f"{prefix}.{name}"]
            if not np.all(np.abs(g - r) <= 2e-6 + 1e-5 * np.abs(r)):
                bad.append((f"{prefix}.{name}", float(np.abs(g - r).max())))
    return bad


def _running(m):
    return {k: v.detach().cpu().numpy() for k, v in m.state_dict().items() if "running" in k}


def _run_autograd(m, x, y):
    """m(x) -> CE -> backward.  Returns the step's results and the (seed, offset) the kernels were given."""
    out = m(x)
    loss = torch.nn.functional.cross_entropy(out, y)
    loss.backward()
    desc = m._engines[(x.shape[0], x.shape[2], True, True)].desc
    got = dict(logits=out.detach().cpu().numpy(), loss=float(loss.item()),
               grads={k: q.grad.detach().cpu().numpy() for k, q in m.named_parameters()}, running=_running(m))
    return got, int(desc.rng_seed), int(desc.rng_offset)


def _flat_grads(m, flat):
    return {k: flat[o:o + n].view(shape).cpu().numpy() if n else np.zeros(shape, np.float32)
            for (k, _), (o, n, shape) in zip(m.named_parameters(), m._param_views)}


def _run_fused(m, x, y, head_fused):
    """One FusedTrainStep (eager) with MMS_HEAD_FUSED = head_fused; the gradients are read from the flat buffer the
    Adam update consumed."""
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    opt = FlatAdam(m, lr=1e-3, weight_decay=1e-4)
    with _options({"HEAD_FUSED": head_fused}):
        step = FusedTrainStep(m, opt, batch=x.shape[0], seq_len=x.shape[2], use_graph=False)
        offset = int(opt.step_dev.item())                  # the kernels read the step count before Adam advances it
        step(x, y)
        torch.cuda.synchronize()
    got = dict(logits=step.logits.cpu().numpy(), loss=float(step.loss.item()), grads=_flat_grads(m, opt.grads),
               running=_running(m))
    assert int(opt.step_dev.item()) == offset + 1
    return got, int(step.desc.rng_seed), offset


# B, C, T, O, H, layers, p, num_classes, options: the path each reaches (model.cu)
STEP_CASES = {
    # M = 320 < TC_MIN_ROWS: separate dropout pass, SIMT products, forward skinny product on the dropped tensor, skinny
    # drop-on-C in the backward, head_fwd2
    "b8_t640": (8, 6, 640, 32, 64, 2, 0.5, 2, {}),
    # the bench configuration: tcgen05 A-operand dropout (forward), skinny drop-on-A (forward), epilogue dropout (backward)
    "b64_t3840": (64, 6, 3840, 32, 64, 2, 0.5, 2, {}),
    # the same with the fusions off: separate pass, gemm_nn + dropout_rows
    "b64_t3840_unfused": (64, 6, 3840, 32, 64, 2, 0.5, 2, {"DROP_FUSED": 0, "GEMM_SKINNY": 0}),
    # H = 128: N = 384 split into tiles
    "b16_h128": (16, 6, 3840, 32, 128, 2, 0.5, 2, {}),
    # H = 32, 3 classes, p = 0.2
    "b16_h32_c3": (16, 8, 3840, 32, 32, 2, 0.2, 3, {}),
    # two sites: layer 0 by a separate pass, layer 1 on the A operand
    "b8_l3": (8, 6, 3840, 32, 64, 3, 0.5, 2, {}),
    # B > 256: skinny refused -> forward gemm_nt on the dropped tensor, backward gemm_nn + dropout_rows; M = 6321 on tcgen05
    "b301_t336": (301, 3, 336, 32, 64, 2, 0.5, 2, {}),
    # odd L = 63, p = 0.8 (scale 5)
    "b5_t1004_p08": (5, 6, 1004, 32, 64, 2, 0.8, 2, {}),
    # one layer: the head site only
    "b8_l1": (8, 6, 640, 32, 64, 1, 0.5, 2, {}),
    # O = 64 (per-layer BN-folded encoder backward), four GRU sites at offsets l * 2^40 on tcgen05 (M = 3840), 8 classes
    "b16_o64_l5_c8": (16, 6, 3840, 64, 64, 5, 0.5, 8, {}),
    # O = 16 at H = 128: bottom-layer weight gradient with N2 = 16 on the SIMT TN product, in tn_split's row halves
    "b16_o16_h128": (16, 6, 3840, 16, 128, 2, 0.5, 3, {}),
    # eight layers at M = 320: seven GRU sites on the separate pass and the SIMT products
    "b8_t640_l8": (8, 6, 640, 32, 64, 8, 0.5, 2, {}),
}


@pytest.mark.parametrize("case", list(STEP_CASES))
def test_dropout_step_vs_float64_oracle_with_drawn_masks(case):
    from multimodalsignal_b200.synth import synthetic_windows
    B, C, T, O, H, layers, p, nc, opts = STEP_CASES[case]
    params, bufs = _state(C, nc, H, layers, seed=20 + C + H, O=O)
    x, y = synthetic_windows(B, C, T, seed=7 + B, num_classes=nc)
    xt, yt = torch.from_numpy(x), torch.from_numpy(y)
    p64 = {k: v.double() for k, v in params.items()}
    runs = []
    with _options(opts):
        runs.append(("autograd",) + _run_autograd(_model(params, bufs, C, nc, H, layers, p, O=O), xt.cuda(), yt.cuda()))
        for head_fused in (1, 0):
            runs.append((f"fused_step/HEAD_FUSED={head_fused}",)
                        + _run_fused(_model(params, bufs, C, nc, H, layers, p, O=O), xt.cuda(), yt.cuda(), head_fused))
    assert len({(seed, off) for _, _, seed, off in runs}) == len(runs)      # three different streams
    for name, got, seed, offset in runs:
        masks = _masks(B, T, H, layers, p, seed, offset)
        assert len(masks[0]) == layers - 1
        _assert_nontrivial(masks, p)
        bad = _mismatches(got, _oracle(p64, xt, yt, layers, masks), bufs)
        assert not bad, (name, bad)


# ------------------------------------------------------------------------------------------------ c. negative controls
def test_wrong_masks_are_caught():
    """The comparison above would catch a kernel that drew the wrong multipliers: the bench-configuration step is outside
    tolerance of the oracle run with the masks of the next offset, with the layer mask's direction halves swapped, and
    without the head mask."""
    from multimodalsignal_b200.synth import synthetic_windows
    B, C, T, _, H, layers, p, nc, _ = STEP_CASES["b64_t3840"]
    params, bufs = _state(C, nc, H, layers, seed=20 + C + H)
    x, y = synthetic_windows(B, C, T, seed=7 + B, num_classes=nc)
    xt, yt = torch.from_numpy(x), torch.from_numpy(y)
    p64 = {k: v.double() for k, v in params.items()}
    got, seed, offset = _run_autograd(_model(params, bufs, C, nc, H, layers, p), xt.cuda(), yt.cuda())
    gru, head = _masks(B, T, H, layers, p, seed, offset)
    assert not _mismatches(got, _oracle(p64, xt, yt, layers, (gru, head)), bufs)
    swapped = np.concatenate([gru[..., H:], gru[..., :H]], axis=-1)
    wrong = {"offset + 1": _masks(B, T, H, layers, p, seed, offset + 1), "halves swapped": (swapped, head),
             "no head mask": (gru, None)}
    for what, masks in wrong.items():
        assert _mismatches(got, _oracle(p64, xt, yt, layers, masks), bufs), what


# ------------------------------------------------------------------------------------------------ d. graph replay
@pytest.mark.parametrize("B,C,T", [(8, 6, 640), (16, 6, 3840)])
def test_graph_replayed_dropout_trajectory_vs_float64_oracle(B, C, T):
    """FusedTrainStep replayed as a CUDA graph for 5 steps on new batches: step k draws its masks at offset k (the device
    step count), so a graph that baked in the offset of its capture would fail at step 2.  Reference: the float64 oracle
    step with those masks, then Adam (torch.optim.Adam rule) and the running-statistics update."""
    from multimodalsignal_b200.synth import synthetic_windows
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    H, layers, p, nc, steps = 64, 2, 0.5, 2, 5
    params, bufs = _state(C, nc, H, layers, seed=40 + T)
    m = _model(params, bufs, C, nc, H, layers, p)
    opt = FlatAdam(m, lr=1e-3, weight_decay=1e-4)
    step = FusedTrainStep(m, opt, batch=B, seq_len=T, use_graph=True)
    seed = int(step.desc.rng_seed)
    ref_p = {k: v.double() for k, v in params.items()}
    ref_m = {k: torch.zeros_like(v) for k, v in ref_p.items()}
    ref_v = {k: torch.zeros_like(v) for k, v in ref_p.items()}
    prev = None
    for k in range(steps):
        x, y = synthetic_windows(B, C, T, seed=300 + k, num_classes=nc)
        xt, yt = torch.from_numpy(x), torch.from_numpy(y)
        assert int(opt.step_dev.item()) == k
        step(xt.cuda(), yt.cuda())
        loss = step.last_loss()
        masks = _masks(B, T, H, layers, p, seed, k)
        if prev is not None:
            assert not np.array_equal(masks[0], prev[0]) and not np.array_equal(masks[1], prev[1])
        prev = masks
        ref_loss, _, ref_grads, _ = _oracle(ref_p, xt, yt, layers, masks)
        assert abs(loss - float(ref_loss)) <= LOSS_ATOL, (k, loss, float(ref_loss))
        for name in ref_p:
            if ref_p[name].numel():
                ref_p[name], ref_m[name], ref_v[name] = mo.adam_step(ref_p[name], ref_grads[name], ref_m[name], ref_v[name],
                                                                     k + 1, lr=1e-3, weight_decay=1e-4)
    assert step.graph is not None
    sd = m.state_dict()
    for name, ref in ref_p.items():
        np.testing.assert_allclose(sd[name].cpu().numpy(), ref.numpy(), atol=PARAM_ATOL, rtol=0, err_msg=name)
    assert int(sd["cnn_encoder.1.num_batches_tracked"].item()) == steps
    assert int(sd["cnn_encoder.5.num_batches_tracked"].item()) == steps


# ------------------------------------------------------------------------------------------------ e. data parallelism
@pytest.mark.parametrize("T,splits", [(3840, (8, 8)), (3840, (4, 6, 6)), (640, (3, 5))])
def test_data_parallel_dropout_step_vs_float64_oracle(T, splits):
    """Emulated ranks (emulate_ranks: the sync tensors summed as the all-reduce would).  Each rank draws its masks with
    its own seed for its local rows, so the full-batch reference uses the ranks' masks concatenated along the batch."""
    from multimodalsignal_b200.parallel import DataParallelTrainStep, emulate_ranks
    from multimodalsignal_b200.synth import synthetic_windows
    from multimodalsignal_b200.trainer import FlatAdam
    C, H, layers, p, nc = 6, 64, 2, 0.5, 2
    B = sum(splits)
    params, bufs = _state(C, nc, H, layers, seed=60 + len(splits))
    x, y = synthetic_windows(B, C, T, seed=70 + B, num_classes=nc)
    xt, yt = torch.from_numpy(x), torch.from_numpy(y)
    xc, yc = xt.cuda(), yt.cuda()
    ranks, steps, batches, lo = [], [], [], 0
    for r, b in enumerate(splits):
        m = _model(params, bufs, C, nc, H, layers, p)
        ranks.append(m)
        steps.append(DataParallelTrainStep(m, FlatAdam(m, lr=1e-3, weight_decay=1e-4), b, B, T, rank=r))
        batches.append((xc[lo:lo + b], yc[lo:lo + b]))
        lo += b
    offsets = [int(s.opt.step_dev.item()) for s in steps]
    emulate_ranks(steps, batches)
    torch.cuda.synchronize()
    seeds = [int(s.desc.rng_seed) for s in steps]
    assert len(set(seeds)) == len(seeds)
    per_rank = [_masks(b, T, H, layers, p, s, o) for b, s, o in zip(splits, seeds, offsets)]
    masks = (np.concatenate([g for g, _ in per_rank], axis=1), np.concatenate([h for _, h in per_rank], axis=0))
    _assert_nontrivial(masks, p)
    p64 = {k: v.double() for k, v in params.items()}
    ref_loss, _, ref_grads, _ = _oracle(p64, xt, yt, layers, masks)
    loss = sum(float(s.loss.item()) for s in steps)
    assert abs(loss - float(ref_loss)) <= LOSS_ATOL, (loss, float(ref_loss))
    for k, g in _flat_grads(ranks[0], steps[0].opt.grads).items():          # the all-reduced gradient
        ref = ref_grads[k].numpy()
        if ref.size:
            assert np.abs(g - ref).max() <= GRAD_RTOL * max(np.abs(ref).max(), 1e-6), k
    flat0 = ranks[0].flat_parameters()
    for m in ranks[1:]:
        assert torch.equal(m.flat_parameters(), flat0)
    sd = ranks[0].state_dict()
    for k, v in p64.items():
        if v.numel():
            new, _, _ = mo.adam_step(v, ref_grads[k], torch.zeros_like(v), torch.zeros_like(v), 1, lr=1e-3, weight_decay=1e-4)
            np.testing.assert_allclose(sd[k].cpu().numpy(), new.numpy(), atol=PARAM_ATOL, rtol=0, err_msg=k)


# ------------------------------------------------------------------------------------------------ f. eval mode
def test_eval_ignores_dropout_and_training_masks_follow_the_offset():
    """In eval mode p = 0.5 draws nothing: the logits are bit-equal to those of the same weights at p = 0 and match the
    oracle's eval forward (running statistics).  In training mode the masks are a function of the forward count alone:
    two forwards at the same _rng_calls give identical logits, the next count different ones."""
    from multimodalsignal_b200.synth import synthetic_windows
    B, C, T, H, layers, nc = 16, 6, 3840, 64, 2, 2
    params, bufs = _state(C, nc, H, layers, seed=80)
    bufs = {k: (v + 0.05 if "mean" in k else v * 1.5) for k, v in bufs.items()}      # non-trivial running statistics
    x, _ = synthetic_windows(B, C, T, seed=81, num_classes=nc)
    xt = torch.from_numpy(x)
    xc = xt.cuda()
    drop = _model(params, bufs, C, nc, H, layers, 0.5).eval()
    plain = _model(params, bufs, C, nc, H, layers, 0.0).eval()
    with torch.no_grad():
        a, b = drop(xc), plain(xc)
    assert torch.equal(a, b)
    ref, _ = mo.forward({k: v.double() for k, v in params.items()}, xt.double(), training=False,
                        bn_buffers={k: v.double() for k, v in bufs.items()}, gru_layers=layers, prune=True)
    np.testing.assert_allclose(a.cpu().numpy(), ref.numpy(), atol=LOGIT_ATOL)

    drop.train()
    outs = []
    for calls in (40, 40, 41):
        drop._rng_calls = calls
        outs.append(drop(xc).detach().clone())
    assert torch.equal(outs[0], outs[1])
    assert not torch.allclose(outs[0], outs[2], atol=LOGIT_ATOL)
