"""Input-gradient-only backward (mms_cnngru_input_gradient), eval-mode autograd and integrated gradients on a B200, against
the float64 oracle (oracle/model_oracle.py, oracle/attribution_oracle.py).

Tolerances as elsewhere in the suite: |logit error| <= 1e-4 absolute, gradients <= 1e-3 of the tensor's max magnitude."""
import ctypes as C
import warnings

import numpy as np
import pytest
import torch

from oracle import attribution_oracle as ao
from oracle import model_oracle as mo

pytestmark = pytest.mark.gpu

LOGIT_ATOL = 1e-4
GRAD_RTOL = 1e-3


@pytest.fixture(scope="module")
def lib():
    from multimodalsignal_b200 import _ext
    return _ext.lib()


def make_model(C_, nc=2, H=64, layers=2, attention=True, seed=0, O=32):
    """A model with random weights AND random BatchNorm running statistics / affine parameters, so that the eval-mode
    BatchNorm is a non-trivial affine map."""
    from multimodalsignal_b200.models import CnnGruAttentionModel
    torch.manual_seed(seed)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m = CnnGruAttentionModel(C_, nc, cnn_out_channels=O, gru_hidden_size=H, gru_num_layers=layers, dropout=0.5,
                                 attention=attention)
    g = torch.Generator().manual_seed(seed + 1000)
    with torch.no_grad():
        for bn in (m.cnn_encoder[1], m.cnn_encoder[5]):
            n = bn.running_mean.numel()
            bn.running_mean.copy_(0.3 * torch.randn(n, generator=g))
            bn.running_var.copy_(0.5 + 1.5 * torch.rand(n, generator=g))
            bn.weight.copy_(1.0 + 0.3 * torch.randn(n, generator=g))
            bn.bias.copy_(0.2 * torch.randn(n, generator=g))
    return m.cuda().eval()


def oracle_state(m):
    sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    params = {k: v.double() for k, v in sd.items() if "running" not in k and "num_batches" not in k}
    bn = {k: v.double() for k, v in sd.items() if "running" in k}
    return params, bn


def oracle_forward(m, params, bn):
    return lambda z: mo.forward(params, z, training=False, bn_buffers=bn, gru_layers=m.gru_num_layers,
                                attention=m.attention, prune=True)[0]


def make_x(B, C_, T, seed=1):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, C_, T, generator=g)


def oracle_input_grad(m, x, target):
    params, bn = oracle_state(m)
    xd = x.double().requires_grad_(True)
    logits = oracle_forward(m, params, bn)(xd)
    (dx,) = torch.autograd.grad(logits.gather(1, target[:, None]).sum(), xd)
    return logits.detach(), dx


def assert_grad_close(got, ref, what):
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    scale = max(np.abs(ref).max(), 1e-12)
    err = np.abs(got - ref).max()
    assert err <= GRAD_RTOL * scale, (what, err, scale)


# ---- mms_cnngru_input_gradient through autograd (frozen parameters) against the float64 oracle ---------------------------

SHAPES = [(6, 3840), (3, 7680), (14, 3840), (6, 336), (6, 4040)]
CASES = [(B, C_, T, 64, 2, att) for (C_, T) in SHAPES for B in (1, 7, 64) for att in (True, False)]
CASES += [(7, 6, 3840, H, layers, True) for H in (32, 64, 128) for layers in (1, 2, 3)]
CASES += [(64, 6, 3840, 128, 2, False), (7, 14, 4040, 32, 3, True), (64, 3, 336, 128, 1, True)]


@pytest.mark.parametrize("B,C_,T,H,layers,attention", CASES)
def test_input_gradient_matches_oracle(B, C_, T, H, layers, attention):
    m = make_model(C_, nc=3, H=H, layers=layers, attention=attention, seed=B + T + H + layers)
    m.requires_grad_(False)
    x = make_x(B, C_, T, seed=B * 7 + C_)
    xg = x.cuda().requires_grad_(True)
    logits = m(xg)
    target = torch.argmax(logits.detach(), dim=1)
    logits.gather(1, target[:, None]).sum().backward()
    ref_logits, ref_dx = oracle_input_grad(m, x, target.cpu())
    np.testing.assert_allclose(logits.detach().cpu().numpy(), ref_logits.numpy(), atol=LOGIT_ATOL)
    assert_grad_close(xg.grad.cpu().numpy(), ref_dx.numpy(), "dx")


@pytest.mark.parametrize("O", [16, 64])
def test_input_gradient_other_cnn_widths(O):
    m = make_model(6, nc=2, O=O, seed=O)
    m.requires_grad_(False)
    x = make_x(7, 6, 3840, seed=O)
    xg = x.cuda().requires_grad_(True)
    logits = m(xg)
    target = torch.tensor([k % 2 for k in range(7)], device="cuda")
    logits.gather(1, target[:, None]).sum().backward()
    ref_logits, ref_dx = oracle_input_grad(m, x, target.cpu())
    np.testing.assert_allclose(logits.detach().cpu().numpy(), ref_logits.numpy(), atol=LOGIT_ATOL)
    assert_grad_close(xg.grad.cpu().numpy(), ref_dx.numpy(), "dx")


# ---- eval-mode autograd with live parameters: the full backward in eval mode --------------------------------------------

@pytest.mark.parametrize("B,C_,T,attention", [(7, 6, 3840, True), (64, 3, 7680, True), (5, 6, 336, False), (7, 14, 4040, True)])
def test_eval_mode_autograd_with_and_without_parameter_gradients(B, C_, T, attention):
    m = make_model(C_, nc=2, attention=attention, seed=3 * B + C_)
    x = make_x(B, C_, T, seed=B + 11)
    params, bn = oracle_state(m)
    # frozen parameters: input-gradient path
    m.requires_grad_(False)
    xg = x.cuda().requires_grad_(True)
    out = m(xg)
    target = torch.argmax(out.detach(), dim=1)
    out.gather(1, target[:, None]).sum().backward()
    dx_frozen = xg.grad.detach().cpu().clone()
    # live parameters: the full backward (mms_cnngru_backward) in eval mode
    m.requires_grad_(True)
    m.zero_grad(set_to_none=True)
    xg = x.cuda().requires_grad_(True)
    out = m(xg)
    out.gather(1, target[:, None]).sum().backward()
    # oracle
    leaves = {k: v.clone().requires_grad_(v.numel() > 0) for k, v in params.items()}
    xd = x.double().requires_grad_(True)
    logits = mo.forward(leaves, xd, training=False, bn_buffers=bn, gru_layers=m.gru_num_layers, attention=attention,
                        prune=True)[0]
    names = [k for k, v in leaves.items() if v.requires_grad]
    grads = torch.autograd.grad(logits.gather(1, target.cpu()[:, None]).sum(), [xd] + [leaves[k] for k in names],
                                allow_unused=True)
    np.testing.assert_allclose(out.detach().cpu().numpy(), logits.detach().numpy(), atol=LOGIT_ATOL)
    assert_grad_close(dx_frozen.numpy(), grads[0].numpy(), "dx (frozen parameters)")
    assert_grad_close(xg.grad.cpu().numpy(), grads[0].numpy(), "dx (live parameters)")
    by = dict(m.named_parameters())
    for k, g in zip(names, grads[1:]):
        ref = torch.zeros_like(leaves[k]) if g is None else g
        if not attention and k.startswith("channel_attention"):
            continue
        assert_grad_close(by[k].grad.cpu().numpy(), ref.numpy(), k)


# ---- the launch list of the input-gradient path ------------------------------------------------------------------------

def _profiled(lib, fn):
    buf = C.create_string_buffer(16384)
    torch.cuda.synchronize()
    lib.mms_profile_enable(1)
    try:
        fn()
        torch.cuda.synchronize()
        lib.mms_profile_report(buf, 16384)
    finally:
        lib.mms_profile_enable(0)
    out = {}
    for line in buf.value.decode().strip().splitlines():
        name, cnt, _ = line.rsplit(" ", 2)
        out[name] = int(cnt)
    return out


FORBIDDEN = ("gemm_tn", "tn_batch", "wgrad", "adam", "head_bwd", "chan_param", "conv1_bwd", "conv2_bwd", "bn_bwd_apply",
             "pool_relu_bwd", "pool_bwd")


@pytest.mark.parametrize("B,C_,T,layers", [(64, 6, 3840, 2), (7, 3, 336, 1), (64, 14, 4040, 3)])
def test_input_gradient_launch_list_has_no_weight_gradient_work(lib, B, C_, T, layers):
    m = make_model(C_, layers=layers, seed=5)
    m.requires_grad_(False)
    x = make_x(B, C_, T).cuda()
    m.flat_parameters()
    eng = m.engine(B, T, False, True, x.device)
    eng.forward(x, 1)
    dl = torch.zeros(B, m.num_classes, device="cuda")
    dl[:, 0] = 1
    names = _profiled(lib, lambda: eng.input_gradient(x, dl))
    for n in names:
        assert not any(f in n for f in FORBIDDEN), (n, names)
    assert "encoder_eval_bwd_kernel" in names and "head_input_grad_kernel" in names, names
    assert "attn_input_grad_kernel" in names and "conv1d_dgrad_kernel" in names, names


# ---- integrated gradients against attribution_oracle --------------------------------------------------------------------

def _check_ig(got, ref):
    A, S, delta = (t.cpu().double().numpy() for t in got)
    rA, rS, rdelta, _ = ref
    rA, rS, rdelta = rA.numpy(), rS.numpy(), rdelta.numpy()
    assert np.abs(A - rA).max() <= 1e-3 * np.abs(rA).max(), np.abs(A - rA).max()
    assert np.abs(S - rS).max() <= 1e-3 * np.abs(rS).max(), (S, rS)
    return A, S, delta


@pytest.mark.parametrize("steps", [1, 8, 32])
@pytest.mark.parametrize("given_target", [False, True])
@pytest.mark.parametrize("baseline", ["zero", "shared", "per_window"])
def test_integrated_gradients_vs_oracle(steps, given_target, baseline):
    from multimodalsignal_b200.attribution import integrated_gradients
    B, C_, T = 4, 6, 3840
    m = make_model(C_, nc=3, seed=steps)
    m.requires_grad_(False)
    x = make_x(B, C_, T, seed=steps + 1)
    g = torch.Generator().manual_seed(9)
    x0 = {"zero": None, "shared": 0.5 * torch.randn(C_, T, generator=g), "per_window": 0.5 * torch.randn(B, C_, T, generator=g)}[baseline]
    target = torch.tensor([2, 0, 1, 2]) if given_target else None
    got = integrated_gradients(m, x.cuda(), target=None if target is None else target.cuda(),
                               baseline=None if x0 is None else x0.cuda(), steps=steps)
    params, bn = oracle_state(m)
    ref = ao.integrated_gradients(params, bn, x, target=target, baseline=x0, steps=steps, gru_layers=m.gru_num_layers)
    A, S, delta = _check_ig(got, ref)
    # completeness residual: the same quantity as the oracle's, to 1e-4 + 1e-3 |F(x) - F(x0)|
    f = oracle_forward(m, params, bn)
    with torch.no_grad():
        fx = f(x.double())
        f0 = f(torch.zeros_like(x.double()) if x0 is None else x0.double().expand_as(x))
    t = ref[3]
    gap = (fx[torch.arange(B), t] - f0[torch.arange(B), t]).numpy()
    assert np.all(np.abs(delta - ref[2].numpy()) <= 1e-4 + 1e-3 * np.abs(gap)), (delta, ref[2], gap)


def test_integrated_gradients_chunking_does_not_change_the_result():
    from multimodalsignal_b200.attribution import integrated_gradients
    B, C_, T, steps = 9, 6, 3840, 8
    m = make_model(C_, seed=21)
    m.requires_grad_(False)
    x = make_x(B, C_, T, seed=22).cuda()
    outs = [integrated_gradients(m, x, steps=steps, max_rows=r) for r in (1 * steps, 7 * steps, 2048)]
    A0, S0, d0 = outs[-1]
    for A, S, d in outs[:-1]:
        assert (A - A0).abs().max().item() <= 1e-6 * A0.abs().max().item()
        assert (S - S0).abs().max().item() <= 1e-6 * S0.abs().max().item()
        assert (d - d0).abs().max().item() <= 1e-6 * max(d0.abs().max().item(), S0.abs().max().item())
    # rows that do not split evenly into windows: a chunk boundary inside a window
    A, S, _ = integrated_gradients(m, x, steps=steps, max_rows=5)
    assert (A - A0).abs().max().item() <= 1e-6 * A0.abs().max().item()
    assert (S - S0).abs().max().item() <= 1e-6 * S0.abs().max().item()


# ---- refusals ---------------------------------------------------------------------------------------------------------

def test_refusals(lib):
    from multimodalsignal_b200 import _ext
    from multimodalsignal_b200.attribution import integrated_gradients
    m = make_model(6, seed=3)
    x = make_x(2, 6, 336).cuda()
    m.flat_parameters()
    m.train()
    with pytest.raises(ValueError, match="eval"):
        integrated_gradients(m, x, steps=2)
    m.eval()
    with pytest.raises(ValueError, match="target"):
        integrated_gradients(m, x, target=torch.tensor([0, 2], device="cuda"), steps=2)
    with pytest.raises(ValueError, match="target"):
        integrated_gradients(m, x, target=torch.tensor([-1, 0], device="cuda"), steps=2)
    with pytest.raises(ValueError, match="broadcast"):
        integrated_gradients(m, x, baseline=torch.zeros(3, 6, 336, device="cuda"), steps=2)
    with pytest.raises(ValueError, match="broadcast"):
        integrated_gradients(m, x, baseline=torch.zeros(6, 335, device="cuda"), steps=2)
    with pytest.raises(_ext.MmsError):
        integrated_gradients(m, x.cpu(), steps=2)
    # the ABI refuses anything but training = 0, need_grad = 1
    for training, need_grad in ((1, 1), (0, 0), (1, 0)):
        eng = m.engine(2, 336, bool(training), bool(need_grad), x.device)
        eng.forward(x, 1)
        dl = torch.zeros(2, 2, device="cuda")
        dx = torch.empty_like(x)
        rc = lib.mms_cnngru_input_gradient(C.byref(eng.desc), x.data_ptr(), m._flat.data_ptr(), m._bn_flat.data_ptr(),
                                           eng.workspace.data_ptr(), dl.data_ptr(), dx.data_ptr(), _ext.stream())
        assert rc == -1 and b"eval-mode forward" in lib.mms_last_error()


# ---- Trainer.channel_attribution and main.ATTRIBUTION_STEPS -------------------------------------------------------------

class _Loader:
    def __init__(self, x, y, bs):
        self.x, self.y, self.bs = x, y, bs

    def __iter__(self):
        for i in range(0, len(self.y), self.bs):
            yield self.x[i:i + self.bs], self.y[i:i + self.bs]


def _trainer(tmp_path, m):
    from multimodalsignal_b200.main import trainer_config
    from multimodalsignal_b200.trainer import Trainer
    cfg = trainer_config()
    cfg['trainer']['quiet'] = True
    return Trainer(m, tmp_path, cfg)


def test_trainer_channel_attribution_equals_recomputation(tmp_path):
    from multimodalsignal_b200.attribution import channel_shares, integrated_gradients
    m = make_model(3, nc=3, seed=31)
    x = make_x(21, 3, 3840, seed=32)
    y = torch.tensor([k % 3 for k in range(21)])
    tr = _trainer(tmp_path, m)
    att = tr.channel_attribution(_Loader(x, y, 8), steps=4, channel_names=["ECG", "EDA", "Resp"])
    assert att.shape == (3, 3) and att.dtype == torch.float64
    m.eval()
    _, S, _ = integrated_gradients(m, x.cuda(), steps=4)
    sh = channel_shares(S).cpu()
    for k in range(3):
        ref = sh[y == k].mean(dim=0)
        torch.testing.assert_close(att[k], ref, rtol=1e-6, atol=1e-9)
        assert abs(att[k].sum().item() - 1.0) < 1e-9
    text = (tmp_path / "channel_attribution.txt").read_text().splitlines()
    assert text[2].split("\t") == ["channel", "class_0", "class_1", "class_2"]
    assert [line.split("\t")[0] for line in text[3:]] == ["ECG", "EDA", "Resp"]


def _run_synthetic_fold(tmp_path, monkeypatch, steps):
    """One fold of main.run_fold_async on a tiny synthetic data set (file path): returns the fold's files and result."""
    import multimodalsignal_b200.main as main
    from multimodalsignal_b200 import dataset
    from multimodalsignal_b200.trainer import drive

    class _DS(torch.utils.data.Dataset):
        def __init__(self, n, seed):
            g = torch.Generator().manual_seed(seed)
            self.x = torch.randn(n, 3, 336, generator=g)
            self.labels = np.array([k % 2 for k in range(n)])

        def __len__(self):
            return len(self.labels)

        def __getitem__(self, i):
            return self.x[i], int(self.labels[i])

    made = iter([_DS(24, 1), _DS(8, 2), _DS(10, 3)])
    monkeypatch.setattr(dataset, "WesadDataset", lambda *a, **k: next(made))
    monkeypatch.setattr(main, "EPOCHS", 1)
    monkeypatch.setattr(main, "BATCH_SIZE", 8)
    monkeypatch.setattr(main, "ATTRIBUTION_STEPS", steps)
    out = tmp_path / f"run_{steps}"
    res = drive(main.run_fold_async(0, "S2", out, ["chest_ECG", "chest_EDA", "chest_Resp"], quiet=True))
    files = sorted(p.name for p in (out / "fold_test_on_S2").iterdir())
    return files, res, out


def test_main_attribution_switch(tmp_path, monkeypatch):
    import multimodalsignal_b200.main as main
    files_off, res_off, _ = _run_synthetic_fold(tmp_path, monkeypatch, 0)
    assert "channel_attribution.txt" not in files_off and "channel_attribution" not in res_off
    files_on, res_on, out = _run_synthetic_fold(tmp_path, monkeypatch, 4)
    assert sorted(set(files_on) - set(files_off)) == ["channel_attribution.txt"]
    att = np.array(res_on["channel_attribution"])
    assert att.shape == (2, 3)
    np.testing.assert_allclose(att.sum(axis=1), 1.0, atol=1e-9)
    res2 = dict(res_on, subject="S3")
    path = main.write_attribution_summary(out, [res_on, res2])
    lines = path.read_text(encoding="utf-8").splitlines()
    assert lines[2].split("\t") == ["channel", "class_0", "class_1"]
    assert [ln.split("\t")[0] for ln in lines[3:]] == main.CHANNELS_TO_USE
