"""Whole-model parity on a B200: the drop-in ``CnnGruAttentionModel`` (CUDA kernels through the
C ABI) against fixtures produced by the unmodified reference ``models.py`` (tests/golden) and
against the float64 oracle.

Stated tolerances (north star / SURVEY §7): fp32 path, dropout disabled --
|logit error| <= 1e-4 absolute; gradients <= 1e-3 of the tensor's max magnitude."""
import numpy as np
import pytest
import torch

from conftest import MODEL_CASES, golden_kept, golden_state, load_golden
from oracle import model_oracle as mo

pytestmark = pytest.mark.gpu

LOGIT_ATOL = 1e-4
GRAD_RTOL = 1e-3


def build(meta, sd, dropout=0.0, attention=True):
    from multimodalsignal_b200.models import CnnGruAttentionModel
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m = CnnGruAttentionModel(meta["C"], meta["num_classes"], dropout=dropout, attention=attention, **meta["kwargs"])
    missing = m.load_state_dict(sd, strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    return m.cuda()


@pytest.mark.parametrize("case", MODEL_CASES)
def test_state_dict_layout_matches_reference(case):
    z, meta = load_golden(f"model_{case}.npz")
    sd = golden_state(z, "sd")
    m = build(meta, sd)
    mine = m.state_dict()
    assert list(mine.keys()) == list(sd.keys())
    for k in sd:
        assert tuple(mine[k].shape) == tuple(sd[k].shape), k
        assert mine[k].dtype == sd[k].dtype, k
    # after the first CUDA forward every parameter is a view of the flat buffer and still round-trips
    x = torch.from_numpy(z["x"]).cuda()
    m.eval()
    with torch.no_grad():
        m(x)
    for k, v in m.state_dict().items():
        assert torch.equal(v.cpu(), sd[k]), k


@pytest.mark.parametrize("case", MODEL_CASES)
def test_train_forward_backward_vs_reference(case):
    z, meta = load_golden(f"model_{case}.npz")
    sd = golden_state(z, "sd")
    m = build(meta, sd)
    m.train()
    x, y = torch.from_numpy(z["x"]).cuda(), torch.from_numpy(z["y"]).cuda()
    logits = m(x)
    np.testing.assert_allclose(logits.detach().cpu().numpy(), z["train_logits"], atol=LOGIT_ATOL)
    loss = torch.nn.functional.cross_entropy(logits, y)
    assert abs(loss.item() - float(z["train_loss"])) < 1e-4
    loss.backward()
    for k, p in m.named_parameters():
        got, ref = golden_kept(z, f"grad/{k}", p.grad.detach().cpu().numpy())
        if ref.size == 0:
            continue
        scale = max(float(z[f"absmax/grad/{k}"]), 1e-6)
        assert np.abs(got - ref).max() <= GRAD_RTOL * scale, (k, np.abs(got - ref).max(), scale)
    for k, v in m.state_dict().items():
        if "running" in k:
            np.testing.assert_allclose(v.cpu().numpy(), z[f"sd_after_fwd/{k}"], atol=2e-6, rtol=1e-5, err_msg=k)
        if "num_batches" in k:
            assert int(v.item()) == 1
    m.eval()
    with torch.no_grad():
        ev = m(x)
    np.testing.assert_allclose(ev.cpu().numpy(), z["eval_logits"], atol=LOGIT_ATOL)


@pytest.mark.parametrize("case", MODEL_CASES)
def test_gradients_vs_float64_oracle(case):
    """Tighter than the float32 reference allows: compare with the oracle evaluated in float64."""
    z, meta = load_golden(f"model_{case}.npz")
    sd = golden_state(z, "sd")
    params = {k: v.double() for k, v in sd.items() if "running" not in k and "num_batches" not in k}
    x, y = torch.from_numpy(z["x"]), torch.from_numpy(z["y"])
    loss, logits, grads, _ = mo.loss_and_grads(params, x.double(), y, training=True,
                                               gru_layers=meta["kwargs"].get("gru_num_layers", 2), prune=True)
    m = build(meta, sd)
    m.train()
    out = m(x.cuda())
    np.testing.assert_allclose(out.detach().cpu().numpy(), logits.numpy(), atol=5e-5)
    torch.nn.functional.cross_entropy(out, y.cuda()).backward()
    for k, p in m.named_parameters():
        ref = grads[k].numpy()
        if ref.size == 0:
            continue
        got = p.grad.detach().cpu().numpy()
        scale = max(np.abs(ref).max(), 1e-6)
        assert np.abs(got - ref).max() <= 3e-4 * scale, (k, np.abs(got - ref).max(), scale)


def test_input_gradient_matches_oracle():
    z, meta = load_golden("model_c6_t640.npz")
    sd = golden_state(z, "sd")
    params = {k: v.double() for k, v in sd.items() if "running" not in k and "num_batches" not in k}
    x, y = torch.from_numpy(z["x"]), torch.from_numpy(z["y"])
    xr = x.double().requires_grad_()
    logits, _ = mo.forward(params, xr, training=True)
    mo.cross_entropy_mean(logits, y).backward()
    m = build(meta, sd)
    m.train()
    xc = x.cuda().requires_grad_()
    torch.nn.functional.cross_entropy(m(xc), y.cuda()).backward()
    ref = xr.grad.numpy()
    assert np.abs(xc.grad.cpu().numpy() - ref).max() <= 3e-4 * np.abs(ref).max()


def test_cnn_gru_baseline_variant():
    """configs[0]: ``cnn_gru`` = the stack without attention (SURVEY D3), vs the oracle."""
    z, meta = load_golden("model_c6_t640.npz")
    sd = golden_state(z, "sd")
    params = {k: v.double() for k, v in sd.items() if "running" not in k and "num_batches" not in k}
    x, y = torch.from_numpy(z["x"]), torch.from_numpy(z["y"])
    loss, logits, grads, _ = mo.loss_and_grads(params, x.double(), y, training=True, attention=False, prune=True)
    m = build(meta, sd, attention=False)
    m.train()
    out = m(x.cuda())
    np.testing.assert_allclose(out.detach().cpu().numpy(), logits.numpy(), atol=5e-5)
    torch.nn.functional.cross_entropy(out, y.cuda()).backward()
    for k, p in m.named_parameters():
        ref = grads[k].numpy()
        got = p.grad.detach().cpu().numpy()
        scale = max(np.abs(ref).max(), 1e-6)
        assert np.abs(got - ref).max() <= 3e-4 * scale + 1e-9, k


@pytest.mark.parametrize("case", ["c6_t640", "c8_h32_l1", "c6_t3840_b8"])
def test_fused_train_step_follows_reference_adam_trajectory(case):
    """mms_cnngru_train_step (zero_grad+forward+CE+backward+Adam in one call, CUDA-graph replayed)
    against the reference's torch.optim.Adam trajectory (trainer.py:68,144-149)."""
    from multimodalsignal_b200.trainer import FusedTrainStep, FlatAdam
    z, meta = load_golden(f"model_{case}.npz")
    sd = golden_state(z, "sd")
    m = build(meta, sd)
    m.train()
    x, y = torch.from_numpy(z["x"]).cuda(), torch.from_numpy(z["y"]).cuda()
    opt = FlatAdam(m, lr=1e-3, weight_decay=1e-4)
    step = FusedTrainStep(m, opt, batch=x.shape[0], seq_len=x.shape[2])
    losses = []
    for _ in range(int(z["adam_steps"])):
        step(x, y)
        losses.append(step.last_loss())
    np.testing.assert_allclose(losses, z["adam_losses"], atol=1e-4)
    mine = m.state_dict()
    for k in sd:
        got, ref = golden_kept(z, f"sd_adam/{k}", mine[k].cpu().numpy())
        if ref.size == 0 or "num_batches" in k:
            continue
        np.testing.assert_allclose(got, ref, atol=5e-5, err_msg=k)
    assert int(mine["cnn_encoder.1.num_batches_tracked"].item()) == int(z["adam_steps"])


def _random_state(C, seed):
    """Reference-shaped parameters with non-trivial BN affine values (oracle/cpu_port.make_state: same keys / shapes as the
    reference state_dict)."""
    from oracle import cpu_port
    p, bufs = cpu_port.make_state(C=C, seed=seed)
    g = torch.Generator().manual_seed(seed + 100)
    for k in ("cnn_encoder.1", "cnn_encoder.5"):
        p[f"{k}.weight"] = p[f"{k}.weight"] + 0.1 * torch.randn(p[f"{k}.weight"].shape, generator=g)
        p[f"{k}.bias"] = p[f"{k}.bias"] + 0.1 * torch.randn(p[f"{k}.bias"].shape, generator=g)
    return p, bufs


def _model_from(p, bufs, C):
    from multimodalsignal_b200.models import CnnGruAttentionModel
    m = CnnGruAttentionModel(C, 2, dropout=0.0)
    sd = dict(p)
    sd.update(bufs)
    sd["cnn_encoder.1.num_batches_tracked"] = torch.zeros((), dtype=torch.int64)
    sd["cnn_encoder.5.num_batches_tracked"] = torch.zeros((), dtype=torch.int64)
    m.load_state_dict(sd, strict=True)
    return m.cuda().train()


# The configurations the numbers are QUOTED on (BASELINE.json configs[1], the as-shipped RAW_FS = 128 window of
# preprocess.py:21 -> T = 7680 / L = 480 with the shipped 3 channels, and the all-channel ablation): the whole step
# (forward, CE, backward) through the C ABI against the float64 oracle.  M = B*L = 15 360 / 30 720 rows: every GEMM of
# the GRU runs on the tcgen05 kernels here, which the small golden cases never reach.
@pytest.mark.parametrize("B,C,T", [(64, 6, 3840), (64, 3, 7680), (64, 14, 3840)])
def test_whole_step_at_quoted_configs_vs_float64_oracle(B, C, T):
    _whole_step_case(B, C, T)


# Edge shapes of the fused encoder kernels (conv_fused.cu takes T % 8 == 0, conv_bwd.cu T % 64 == 0): the shortest sequence (one
# partial tile everywhere, L = 4), one and sixteen channels, tile counts that do not divide (T = 4032: L2 = 504 = 3.9 tiles of
# 128, L1 = 2016 = 4.2 chunks of 480), a single batch row -- and lengths that take the per-layer backward kernels (T % 64 != 0)
# or the per-layer kernels throughout (T % 8 != 0).
@pytest.mark.parametrize("B,C,T", [(1, 1, 64), (3, 5, 128), (2, 16, 1088), (5, 6, 4032), (4, 8, 320), (3, 5, 96), (4, 8, 352),
                                   (2, 6, 100), (3, 4, 1004)])
def test_whole_step_edge_shapes_vs_float64_oracle(B, C, T):
    _whole_step_case(B, C, T)


def _whole_step_case(B, C, T):
    from multimodalsignal_b200.synth import synthetic_windows
    p, bufs = _random_state(C, seed=11 + C)
    x, y = synthetic_windows(B, C, T, seed=5 + C)
    xt, yt = torch.from_numpy(x), torch.from_numpy(y)
    params = {k: v.double() for k, v in p.items()}
    ref_loss, ref_logits, ref_grads, aux = mo.loss_and_grads(params, xt.double(), yt, training=True, prune=True)
    m = _model_from(p, bufs, C)
    out = m(xt.cuda())
    np.testing.assert_allclose(out.detach().cpu().numpy(), ref_logits.numpy(), atol=LOGIT_ATOL)
    loss = torch.nn.functional.cross_entropy(out, yt.cuda())
    assert abs(loss.item() - ref_loss.item()) < 1e-4
    loss.backward()
    for k, prm in m.named_parameters():
        ref = ref_grads[k].numpy()
        if ref.size == 0:
            continue
        got = prm.grad.detach().cpu().numpy()
        scale = max(np.abs(ref).max(), 1e-6)
        assert np.abs(got - ref).max() <= GRAD_RTOL * scale, (k, np.abs(got - ref).max(), scale)
    # BatchNorm running statistics after one training forward (momentum 0.1, unbiased variance)
    for prefix, key in (("cnn_encoder.1", "s1"), ("cnn_encoder.5", "s2")):
        n = aux[f"{key}_conv"].shape[0] * aux[f"{key}_conv"].shape[2]
        rm, rv = mo.running_stats_update(bufs[f"{prefix}.running_mean"].double(), bufs[f"{prefix}.running_var"].double(),
                                         aux[f"{key}_mean"].detach(), aux[f"{key}_var"].detach(), n)
        sd = m.state_dict()
        np.testing.assert_allclose(sd[f"{prefix}.running_mean"].cpu().numpy(), rm.numpy(), atol=2e-6, rtol=1e-5)
        np.testing.assert_allclose(sd[f"{prefix}.running_var"].cpu().numpy(), rv.numpy(), atol=2e-6, rtol=1e-5)


def test_whole_step_c14_batch256_vs_library_cpu_step():
    """cfg5's largest single-GPU batch in the parity suite (C = 14, B = 256, M = 61 440 rows).  The float64 oracle's
    Python recurrence needs minutes at this size, so the checker is oracle/cpu_port.py (float32 ATen CPU kernels,
    pinned to the reference fixtures by tests/test_oracle_model.py::test_cpu_port_*)."""
    from oracle import cpu_port
    from multimodalsignal_b200.synth import synthetic_windows
    B, C, T = 256, 14, 3840
    p, bufs = _random_state(C, seed=31)
    x, y = synthetic_windows(B, C, T, seed=17)
    xt, yt = torch.from_numpy(x), torch.from_numpy(y)
    leaves = {k: v.clone().requires_grad_(True) for k, v in p.items()}
    ref_logits = cpu_port.forward(leaves, {k: v.clone() for k, v in bufs.items()}, xt, training=True, dropout=0.0)
    ref_loss = torch.nn.functional.cross_entropy(ref_logits, yt)
    ref_loss.backward()
    m = _model_from(p, bufs, C)
    out = m(xt.cuda())
    np.testing.assert_allclose(out.detach().cpu().numpy(), ref_logits.detach().numpy(), atol=LOGIT_ATOL)
    torch.nn.functional.cross_entropy(out, yt.cuda()).backward()
    for k, prm in m.named_parameters():
        ref = leaves[k].grad.numpy()
        got = prm.grad.detach().cpu().numpy()
        scale = max(np.abs(ref).max(), 1e-6)
        assert np.abs(got - ref).max() <= GRAD_RTOL * scale, (k, np.abs(got - ref).max(), scale)


def test_dropout_training_runs_and_is_stochastic():
    z, meta = load_golden("model_c6_t640.npz")
    sd = golden_state(z, "sd")
    m = build(meta, sd, dropout=0.5)
    m.train()
    x = torch.from_numpy(z["x"]).cuda()
    a = m(x).detach().clone()
    b = m(x).detach().clone()
    assert torch.isfinite(a).all() and not torch.allclose(a, b)
    y = torch.from_numpy(z["y"]).cuda()
    out = m(x)
    torch.nn.functional.cross_entropy(out, y).backward()
    assert all(torch.isfinite(p.grad).all() for p in m.parameters() if p.numel())
    m.eval()
    with torch.no_grad():
        np.testing.assert_allclose(m(x).cpu().numpy(), m(x).cpu().numpy())


def test_cpu_input_is_refused():
    """No CPU fallback: the product path fails loudly."""
    from multimodalsignal_b200.models import CnnGruAttentionModel
    from multimodalsignal_b200._ext import MmsError
    m = CnnGruAttentionModel(6, 2)
    with pytest.raises(MmsError):
        m(torch.zeros(2, 6, 640))


def test_overlong_window_is_refused_up_front():
    """seq_len > 16384 (the BatchNorm / pool kernels stage whole rows in shared memory): a clear error from the descriptor check,
    not a failed launch somewhere inside the chain."""
    from multimodalsignal_b200.models import CnnGruAttentionModel
    from multimodalsignal_b200._ext import MmsError
    m = CnnGruAttentionModel(3, 2).cuda().eval()
    with pytest.raises(MmsError, match="16384"):
        with torch.no_grad():
            m(torch.zeros(1, 3, 16400, device="cuda"))


def test_dropout_gradient_fused_into_gemm_epilogue_equals_separate_pass():
    """The gradient through nn.GRU's inter-layer dropout (models.py:62) is applied by the epilogue of the tensor-core product that
    forms it (MMS_DROP_FUSED=1, default) -- the same multipliers as a separate dropout_apply pass over the result
    (MMS_DROP_FUSED=0); in the forward the multipliers ride on the A operand of the top layer's input projection.  Same RNG
    offset in both runs: equal logits and gradients up to rounding / atomic ordering."""
    from multimodalsignal_b200 import _ext
    from multimodalsignal_b200.models import CnnGruAttentionModel
    lib = _ext.lib()
    torch.manual_seed(11)
    B, C, T = 8, 6, 3840                      # M = B * L = 1920 rows: the tcgen05 products
    m = CnnGruAttentionModel(C, 2, dropout=0.5).cuda().train()
    x = torch.randn(B, C, T, device="cuda")
    y = torch.randint(0, 2, (B,), device="cuda")
    prev = lib.mms_get_option(b"DROP_FUSED", -1)
    grads = {}
    try:
        for mode in (1, 0):
            _ext.check(lib.mms_set_option(b"DROP_FUSED", mode))
            m.zero_grad()
            m._rng_calls = 100                # the same dropout masks in both runs
            out = m(x)
            torch.nn.functional.cross_entropy(out, y).backward()
            grads[mode] = {k: p.grad.detach().clone() for k, p in m.named_parameters() if p.numel()}
            grads[mode]["__logits__"] = out.detach().clone()
    finally:
        _ext.check(lib.mms_set_option(b"DROP_FUSED", prev) if prev >= 0 else lib.mms_clear_option(b"DROP_FUSED"))
    for k in grads[1]:
        scale = max(grads[0][k].abs().max().item(), 1e-8)
        assert (grads[1][k] - grads[0][k]).abs().max().item() <= 2e-5 * scale, k
