"""Pin ``oracle/model_oracle.py`` to fixtures produced by the unmodified reference
``models.py`` (tests/golden/model_*.npz, made by oracle/make_golden.py)."""
import numpy as np
import pytest
import torch

from conftest import MODEL_CASES, golden_kept, golden_state, load_golden
from oracle import model_oracle as mo


def _layers(meta):
    return meta["kwargs"].get("gru_num_layers", 2)


@pytest.mark.parametrize("case", MODEL_CASES)
@pytest.mark.parametrize("prune", [False, True])
def test_forward_backward_matches_reference(case, prune):
    z, meta = load_golden(f"model_{case}.npz")
    sd = golden_state(z, "sd")
    params = {k: v for k, v in sd.items() if "running" not in k and "num_batches" not in k}
    x, y = torch.from_numpy(z["x"]), torch.from_numpy(z["y"])
    loss, logits, grads, aux = mo.loss_and_grads(params, x, y, training=True,
                                                 gru_layers=_layers(meta), prune=prune)
    np.testing.assert_allclose(logits.numpy(), z["train_logits"], atol=2e-5, rtol=1e-4)
    assert abs(loss.item() - float(z["train_loss"])) < 2e-5
    for k in params:
        got, ref = golden_kept(z, f"grad/{k}", grads[k].numpy())
        if ref.size == 0:
            continue
        scale = max(1e-6, float(z[f"absmax/grad/{k}"]))
        assert np.abs(got - ref).max() <= 2e-4 * scale + 1e-7, k


@pytest.mark.parametrize("case", MODEL_CASES)
def test_float64_oracle_close_to_reference_float32(case):
    z, meta = load_golden(f"model_{case}.npz")
    sd = golden_state(z, "sd")
    params = {k: v.double() for k, v in sd.items() if "running" not in k and "num_batches" not in k}
    x, y = torch.from_numpy(z["x"]).double(), torch.from_numpy(z["y"])
    loss, logits, grads, _ = mo.loss_and_grads(params, x, y, training=True, gru_layers=_layers(meta), prune=True)
    np.testing.assert_allclose(logits.numpy(), z["train_logits"], atol=5e-5)


@pytest.mark.parametrize("case", MODEL_CASES)
def test_running_stats_and_eval(case):
    z, meta = load_golden(f"model_{case}.npz")
    sd = golden_state(z, "sd")
    params = {k: v for k, v in sd.items() if "running" not in k and "num_batches" not in k}
    x = torch.from_numpy(z["x"])
    _, aux = mo.forward(params, x, training=True, gru_layers=_layers(meta))
    bufs = {}
    for prefix, key in (("cnn_encoder.1", "s1"), ("cnn_encoder.5", "s2")):
        n = aux[f"{key}_conv"].shape[0] * aux[f"{key}_conv"].shape[2]
        rm, rv = mo.running_stats_update(sd[f"{prefix}.running_mean"], sd[f"{prefix}.running_var"],
                                         aux[f"{key}_mean"], aux[f"{key}_var"], n)
        np.testing.assert_allclose(rm.numpy(), z[f"sd_after_fwd/{prefix}.running_mean"], atol=1e-6)
        np.testing.assert_allclose(rv.numpy(), z[f"sd_after_fwd/{prefix}.running_var"], atol=1e-6, rtol=1e-5)
        assert int(z[f"sd_after_fwd/{prefix}.num_batches_tracked"]) == 1
        bufs[f"{prefix}.running_mean"], bufs[f"{prefix}.running_var"] = rm, rv
    logits, _ = mo.forward(params, x, training=False, bn_buffers=bufs, gru_layers=_layers(meta), prune=True)
    np.testing.assert_allclose(logits.numpy(), z["eval_logits"], atol=2e-5, rtol=1e-4)


@pytest.mark.parametrize("case", ["c6_t640", "c8_h32_l1"])
def test_adam_trajectory(case):
    """oracle forward/backward + oracle Adam reproduce the reference's
    ``torch.optim.Adam(lr=1e-3, weight_decay=1e-4)`` trajectory (trainer.py:68)."""
    z, meta = load_golden(f"model_{case}.npz")
    sd = golden_state(z, "sd")
    params = {k: v.clone() for k, v in sd.items() if "running" not in k and "num_batches" not in k}
    x, y = torch.from_numpy(z["x"]), torch.from_numpy(z["y"])
    m = {k: torch.zeros_like(v) for k, v in params.items()}
    v2 = {k: torch.zeros_like(v) for k, v in params.items()}
    steps = int(z["adam_steps"])
    losses = []
    for step in range(1, steps + 1):
        loss, _, grads, _ = mo.loss_and_grads(params, x, y, training=True, gru_layers=_layers(meta), prune=True)
        losses.append(loss.item())
        for k in params:
            if params[k].numel():
                params[k], m[k], v2[k] = mo.adam_step(params[k], grads[k], m[k], v2[k], step)
    np.testing.assert_allclose(losses, z["adam_losses"], atol=5e-5)
    for k in params:
        np.testing.assert_allclose(*golden_kept(z, f"sd_adam/{k}", params[k].numpy()), atol=3e-5, err_msg=k)


def test_cnn_gru_baseline_is_attention_identity():
    """SURVEY D3: the ``cnn_gru`` baseline = same stack with the attention removed."""
    z, meta = load_golden("model_c6_t640.npz")
    sd = golden_state(z, "sd")
    params = {k: v for k, v in sd.items() if "running" not in k and "num_batches" not in k}
    x = torch.from_numpy(z["x"])
    la, _ = mo.forward(params, x, training=True, attention=True)
    lb, aux = mo.forward(params, x, training=True, attention=False)
    assert aux["x_scaled"] is x
    assert not np.allclose(la.numpy(), lb.numpy())


def test_degenerate_attention_gate_is_half():
    """SURVEY D5: C=3 -> C//4 == 0 -> zero-sized linears -> gate == 0.5."""
    z, _ = load_golden("model_c3_t336_ternary.npz")
    sd = golden_state(z, "sd")
    assert sd["channel_attention.fc.0.weight"].numel() == 0
    x = torch.from_numpy(z["x"])
    _, gate, _ = mo.channel_attention(x, sd["channel_attention.fc.0.weight"], sd["channel_attention.fc.2.weight"])
    assert torch.all(gate == 0.5)


@pytest.mark.parametrize("case", MODEL_CASES)
def test_cpu_port_matches_reference(case):
    """oracle/cpu_port.py (the CPU baseline bench.py times) against the reference fixtures."""
    from oracle import cpu_port
    z, meta = load_golden(f"model_{case}.npz")
    sd = golden_state(z, "sd")
    p = {k: v.clone().requires_grad_(v.numel() > 0) for k, v in sd.items() if "running" not in k and "num_batches" not in k}
    bufs = {k: v.clone() for k, v in sd.items() if "running" in k}
    x, y = torch.from_numpy(z["x"]), torch.from_numpy(z["y"])
    logits = cpu_port.forward(p, bufs, x, training=True, dropout=0.0, layers=_layers(meta))
    np.testing.assert_allclose(logits.detach().numpy(), z["train_logits"], atol=2e-5, rtol=1e-4)
    loss = torch.nn.functional.cross_entropy(logits, y)
    loss.backward()
    for k, v in p.items():
        if v.numel():
            got, ref = golden_kept(z, f"grad/{k}", v.grad.numpy())
            assert np.abs(got - ref).max() <= 2e-4 * max(1e-6, float(z[f"absmax/grad/{k}"])) + 1e-7, k
    for k, v in bufs.items():
        np.testing.assert_allclose(v.numpy(), z[f"sd_after_fwd/{k}"], atol=1e-6, rtol=1e-5)
