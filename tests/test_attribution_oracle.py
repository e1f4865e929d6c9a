"""The float64 integrated-gradients oracle (oracle/attribution_oracle.py) on the CPU: exact for a linear model, and on the
eval-mode model its completeness residual shrinks as the number of steps grows."""
import warnings

import torch

from oracle import attribution_oracle as ao


def test_oracle_ig_is_exact_for_a_linear_model():
    g = torch.Generator().manual_seed(0)
    B, C_, T, nc = 3, 4, 50, 3
    W = torch.randn(nc, C_, T, generator=g, dtype=torch.float64)
    bias = torch.randn(nc, generator=g, dtype=torch.float64)
    f = lambda z: torch.einsum("bct,kct->bk", z, W) + bias
    x = torch.randn(B, C_, T, generator=g, dtype=torch.float64)
    x0 = torch.randn(C_, T, generator=g, dtype=torch.float64)
    for steps in (1, 5):
        A, S, delta, target = ao.integrated_gradients_fn(f, x, baseline=x0, steps=steps)
        assert torch.equal(target, torch.argmax(f(x), dim=1))
        torch.testing.assert_close(A, (x - x0) * W[target], rtol=1e-12, atol=1e-12)
        torch.testing.assert_close(S, A.sum(dim=2))
        assert delta.abs().max().item() < 1e-10
    A, S, delta, target = ao.integrated_gradients_fn(f, x, target=torch.tensor([2, 2, 0]), steps=3)
    torch.testing.assert_close(A, x * W[torch.tensor([2, 2, 0])], rtol=1e-12, atol=1e-12)


def test_oracle_ig_residual_shrinks_with_steps_on_the_model():
    from multimodalsignal_b200.models import CnnGruAttentionModel
    torch.manual_seed(4)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m = CnnGruAttentionModel(6, 2, gru_num_layers=1, dropout=0.0)
    sd = m.state_dict()
    params = {k: v for k, v in sd.items() if "running" not in k and "num_batches" not in k}
    bn = {k: v for k, v in sd.items() if "running" in k}
    x = 2.0 * torch.randn(2, 6, 336, generator=torch.Generator().manual_seed(5))
    res = []
    for steps in (1, 4, 32):
        _, _, delta, _ = ao.integrated_gradients(params, bn, x, steps=steps, gru_layers=1)
        res.append(delta.abs().max().item())
    assert res[2] < res[1] < res[0], res
    assert res[2] < 0.25 * res[0], res
