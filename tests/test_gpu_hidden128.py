"""gru_hidden_size = 128 on a B200: the recurrence kernels through the C ABI against the float64 oracle, the whole training step
against oracle/model_oracle.py (float64) and oracle/cpu_port.py, every Python entry point (autograd, FusedTrainStep, EvalStep /
Trainer.evaluate, DataParallelTrainStep, best_model.pt), and the refusal of the sizes that stay unsupported.

Tolerances as at hidden size 64 (tests/test_gpu_ops.py, tests/test_gpu_model.py): |logit error| <= 1e-4 absolute, gradients
<= 1e-3 of the tensor's max magnitude."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import cpu_port
from oracle import model_oracle as mo
from test_gpu_ops import _gru_case

pytestmark = pytest.mark.gpu

H = 128
LOGIT_ATOL = 1e-4
GRAD_RTOL = 1e-3


@pytest.fixture(scope="module")
def lib():
    from multimodalsignal_b200 import _ext
    return _ext.lib()


class _option:
    """mms_set_option for the duration of a with-block."""

    def __init__(self, lib, name, value):
        self.lib, self.name, self.value = lib, name.encode(), value

    def __enter__(self):
        from multimodalsignal_b200 import _ext
        self.prev = self.lib.mms_get_option(self.name, -1)
        _ext.check(self.lib.mms_set_option(self.name, self.value))

    def __exit__(self, *exc):
        from multimodalsignal_b200 import _ext
        _ext.check(self.lib.mms_set_option(self.name, self.prev) if self.prev >= 0 else self.lib.mms_clear_option(self.name))


# ---- recurrence kernels ---------------------------------------------------------------------------------------------------

# B = 301 (x 1 direction here, x 2 in the model) is past the 296 CTAs of two waves: at H = 128 it runs one row per CTA over
# several waves instead of the multi-row kernels
@pytest.mark.parametrize("reverse", [False, True])
@pytest.mark.parametrize("L", [1, 3, 40, 240])
@pytest.mark.parametrize("B", [1, 5, 150, 301])
def test_gru_recurrence_h128(lib, B, L, reverse):
    _gru_case(lib, B, L, H, 256 if B <= 5 else 32, reverse)


def test_gru_single_reverse_step_h128(lib):
    """The top layer's reverse direction is observed after one step only; with and without an upstream gradient."""
    _gru_case(lib, 4, 20, H, 256, True, steps=1)
    _gru_case(lib, 4, 20, H, 256, True, steps=1, with_dout=False)
    _gru_case(lib, 4, 20, H, 256, False, steps=3)


@pytest.mark.parametrize("depth", [4, 8])
def test_gru_backward_ring_depths_h128(lib, depth):
    with _option(lib, "GRU_BWD_RING", depth):
        for case in [(5, 40, H, 64, False), (5, 40, H, 64, True), (7, 2, H, 32, True), (301, 9, H, 32, True)]:
            _gru_case(lib, *case)
        _gru_case(lib, 4, 20, H, 256, True, steps=depth + 1)
        _gru_case(lib, 4, 20, H, 64, False, steps=depth, with_dout=False)


def test_gru_h128_refuses_the_kernels_it_has_no_instantiation_of(lib):
    """The register-ring backward and the multi-row forward are not built at H = 128: selecting them is an error, not a
    launch of a spilling kernel."""
    from multimodalsignal_b200._ext import MmsError
    with _option(lib, "GRU_BWD_RING", 0):
        with pytest.raises(MmsError, match="GRU_BWD_RING=0"):
            _gru_case(lib, 3, 5, H, 32, False)
    with _option(lib, "GRU_FWD_V2", 0):
        with pytest.raises(MmsError, match="GRU_FWD_V2=0"):
            _gru_case(lib, 3, 5, H, 32, False)
    # an h sequence that is not 16-byte aligned (row stride H + 1 floats)
    from multimodalsignal_b200._ext import GruDirBwd
    w = torch.zeros(3 * H, H, device="cuda")
    stash = torch.zeros(2, 3, 4 * H, device="cuda")
    hs = torch.zeros(2, 3, H + 1, device="cuda")
    D = torch.zeros(2, 3, 4 * H, device="cuda")
    bd = GruDirBwd()
    bd.w_hh = w.data_ptr()
    bd.stash, bd.st_bs, bd.st_ts = stash.data_ptr(), 3 * 4 * H, 4 * H
    bd.hs, bd.hs_bs, bd.hs_ts = hs.data_ptr(), 3 * (H + 1), H + 1
    bd.D, bd.d_bs, bd.d_ts = D.data_ptr(), 3 * 4 * H, 4 * H
    bd.t0, bd.dt, bd.nsteps = 0, 1, 3
    from multimodalsignal_b200 import _ext
    with pytest.raises(MmsError, match="16-byte aligned"):
        _ext.check(lib.mms_gru_recur_bwd(C.byref(bd), 1, 2, H, 0.0, 0, 0, None, torch.cuda.current_stream().cuda_stream))


@pytest.mark.parametrize("bad", [48, 96, 256])
def test_gru_recurrence_refuses_other_hidden_sizes(lib, bad):
    from multimodalsignal_b200._ext import MmsError
    with pytest.raises(MmsError, match="32, 64 or 128"):
        _gru_case(lib, 2, 3, bad, 32, False)


# ---- whole model --------------------------------------------------------------------------------------------------------

def _state(C, layers, seed, num_classes=3):
    """Reference-shaped parameters at H = 128 with non-trivial BatchNorm affine values."""
    p, bufs = cpu_port.make_state(C=C, num_classes=num_classes, H=H, layers=layers, seed=seed)
    g = torch.Generator().manual_seed(seed + 100)
    for k in ("cnn_encoder.1", "cnn_encoder.5"):
        p[f"{k}.weight"] = p[f"{k}.weight"] + 0.1 * torch.randn(p[f"{k}.weight"].shape, generator=g)
        p[f"{k}.bias"] = p[f"{k}.bias"] + 0.1 * torch.randn(p[f"{k}.bias"].shape, generator=g)
    return p, bufs


def _model(p, bufs, C, layers, num_classes=3, dropout=0.0, attention=False):
    from multimodalsignal_b200.models import CnnGruAttentionModel
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m = CnnGruAttentionModel(C, num_classes, gru_hidden_size=H, gru_num_layers=layers, dropout=dropout, attention=attention)
    sd = dict(p)
    sd.update(bufs)
    sd["cnn_encoder.1.num_batches_tracked"] = torch.zeros((), dtype=torch.int64)
    sd["cnn_encoder.5.num_batches_tracked"] = torch.zeros((), dtype=torch.int64)
    m.load_state_dict(sd, strict=True)
    return m.cuda().train()


def _check_grads(m, ref_grads):
    for k, prm in m.named_parameters():
        ref = ref_grads[k].detach().numpy()
        if ref.size == 0:
            continue
        got = prm.grad.detach().cpu().numpy()
        scale = max(np.abs(ref).max(), 1e-6)
        assert np.abs(got - ref).max() <= GRAD_RTOL * scale + 1e-9, (k, np.abs(got - ref).max(), scale)


@pytest.mark.parametrize("layers", [1, 2, 3])
@pytest.mark.parametrize("B,C,T", [(64, 6, 3840), (64, 3, 7680), (1, 1, 64), (3, 5, 96), (5, 6, 4032)])
def test_whole_step_h128_vs_float64_oracle(B, C, T, layers):
    from multimodalsignal_b200.synth import synthetic_windows
    p, bufs = _state(C, layers, seed=11 + C + layers)
    x, y = synthetic_windows(B, C, T, seed=5 + C, num_classes=3)
    xt, yt = torch.from_numpy(x), torch.from_numpy(y)
    params = {k: v.double() for k, v in p.items()}
    ref_loss, ref_logits, ref_grads, aux = mo.loss_and_grads(params, xt.double(), yt, training=True, gru_layers=layers,
                                                             attention=False, prune=True)
    m = _model(p, bufs, C, layers)
    out = m(xt.cuda())
    np.testing.assert_allclose(out.detach().cpu().numpy(), ref_logits.numpy(), atol=LOGIT_ATOL)
    loss = torch.nn.functional.cross_entropy(out, yt.cuda())
    assert abs(loss.item() - ref_loss.item()) < 1e-4
    loss.backward()
    _check_grads(m, ref_grads)
    sd = m.state_dict()
    for prefix, key in (("cnn_encoder.1", "s1"), ("cnn_encoder.5", "s2")):
        n = aux[f"{key}_conv"].shape[0] * aux[f"{key}_conv"].shape[2]
        rm, rv = mo.running_stats_update(bufs[f"{prefix}.running_mean"].double(), bufs[f"{prefix}.running_var"].double(),
                                         aux[f"{key}_mean"].detach(), aux[f"{key}_var"].detach(), n)
        np.testing.assert_allclose(sd[f"{prefix}.running_mean"].cpu().numpy(), rm.numpy(), atol=2e-6, rtol=1e-5)
        np.testing.assert_allclose(sd[f"{prefix}.running_var"].cpu().numpy(), rv.numpy(), atol=2e-6, rtol=1e-5)


def test_whole_step_h128_c14_batch256_vs_library_cpu_step():
    """B = 256, C = 14 (M = 61 440 rows): checked against oracle/cpu_port.py, as at hidden size 64."""
    from multimodalsignal_b200.synth import synthetic_windows
    B, C, T = 256, 14, 3840
    p, bufs = _state(C, 2, seed=31, num_classes=2)
    x, y = synthetic_windows(B, C, T, seed=17)
    xt, yt = torch.from_numpy(x), torch.from_numpy(y)
    leaves = {k: v.clone().requires_grad_(True) for k, v in p.items()}
    ref_logits = cpu_port.forward(leaves, {k: v.clone() for k, v in bufs.items()}, xt, training=True, dropout=0.0)
    torch.nn.functional.cross_entropy(ref_logits, yt).backward()
    m = _model(p, bufs, C, 2, num_classes=2, attention=True)
    out = m(xt.cuda())
    np.testing.assert_allclose(out.detach().cpu().numpy(), ref_logits.detach().numpy(), atol=LOGIT_ATOL)
    torch.nn.functional.cross_entropy(out, yt.cuda()).backward()
    _check_grads(m, {k: v.grad for k, v in leaves.items()})


def test_fused_train_step_h128_follows_float64_adam_trajectory(tmp_path):
    """FusedTrainStep (CUDA graph, Adam with weight decay) for six steps against model_oracle.adam_step on the float64
    oracle; then the eval-mode forward, and the state_dict saved and loaded into oracle/cpu_port, give the same logits."""
    from multimodalsignal_b200.synth import synthetic_windows
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    B, C, T, layers, steps = 8, 6, 3840, 2, 6
    p, bufs = _state(C, layers, seed=3, num_classes=2)
    x, y = synthetic_windows(B, C, T, seed=9)
    xt, yt = torch.from_numpy(x), torch.from_numpy(y)
    m = _model(p, bufs, C, layers, num_classes=2, attention=True)
    step = FusedTrainStep(m, FlatAdam(m, lr=1e-3, weight_decay=1e-4), batch=B, seq_len=T)
    xc, yc = xt.cuda(), yt.cuda()
    losses = []
    for _ in range(steps):
        step(xc, yc)
        losses.append(step.last_loss())

    ref = {k: v.double() for k, v in p.items()}
    m1 = {k: torch.zeros_like(v) for k, v in ref.items()}
    m2 = {k: torch.zeros_like(v) for k, v in ref.items()}
    ref_losses = []
    for s in range(1, steps + 1):
        loss, _, grads, _ = mo.loss_and_grads(ref, xt.double(), yt, training=True, gru_layers=layers, prune=True)
        ref_losses.append(loss.item())
        for k in ref:
            ref[k], m1[k], m2[k] = mo.adam_step(ref[k], grads[k], m1[k], m2[k], s)
    np.testing.assert_allclose(losses, ref_losses, atol=1e-4)
    mine = m.state_dict()
    for k, v in ref.items():
        np.testing.assert_allclose(mine[k].cpu().numpy(), v.numpy(), atol=5e-5, err_msg=k)
    assert int(mine["cnn_encoder.1.num_batches_tracked"].item()) == steps

    m.eval()
    with torch.no_grad():
        ev = m(xc).cpu()
    torch.save({k: v.detach().cpu().clone() for k, v in mine.items()}, tmp_path / "sd.pt")
    sd = torch.load(tmp_path / "sd.pt")
    cp = {k: v for k, v in sd.items() if "running" not in k and "num_batches" not in k}
    cb = {k: v for k, v in sd.items() if "running" in k}
    with torch.no_grad():
        ref_ev = cpu_port.forward(cp, cb, xt, training=False, dropout=0.0, layers=layers)
    np.testing.assert_allclose(ev.numpy(), ref_ev.numpy(), atol=LOGIT_ATOL)


def test_trainer_evaluate_and_best_model_h128(tmp_path):
    """Trainer.train (fused graph-replayed steps, best_model.pt) and Trainer.evaluate (EvalStep) at H = 128: the checkpoint has
    the reference's keys and shapes and, loaded into oracle/cpu_port, gives the loss Trainer.evaluate reports."""
    from torch.utils.data import DataLoader, TensorDataset
    from multimodalsignal_b200.models import CnnGruAttentionModel
    from multimodalsignal_b200.synth import synthetic_windows
    from multimodalsignal_b200.trainer import Trainer
    C, T = 3, 640
    x, y = synthetic_windows(48, C, T, seed=21)
    ds = TensorDataset(torch.from_numpy(x), torch.from_numpy(y))
    tl = DataLoader(ds, batch_size=16, shuffle=False, num_workers=0)
    torch.manual_seed(0)
    model = CnnGruAttentionModel(in_channels=C, num_classes=2, gru_hidden_size=H, dropout=0.0)
    ref_keys = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    cfg = {'trainer': {'epochs': 1, 'learning_rate': 1e-3, 'early_stopping': {'enabled': True, 'patience': 20, 'delta': 0},
                       'weight_decay': 1e-4}}
    trainer = Trainer(model, tmp_path / "fold", cfg)
    trainer.train(tl, tl)
    loss, acc, f1 = trainer.evaluate(tl)
    sd = torch.load(tmp_path / "fold" / "best_model.pt", map_location="cpu")
    assert {k: tuple(v.shape) for k, v in sd.items()} == ref_keys and list(sd.keys()) == list(ref_keys)
    cp = {k: v.float() for k, v in sd.items() if "running" not in k and "num_batches" not in k}
    cb = {k: v.float() for k, v in sd.items() if "running" in k}
    with torch.no_grad():
        logits = cpu_port.forward(cp, cb, torch.from_numpy(x), training=False, dropout=0.0)
    ref_loss = torch.nn.functional.cross_entropy(logits, torch.from_numpy(y)).item()
    assert abs(loss - ref_loss) < 1e-4, (loss, ref_loss)
    assert abs(acc - (logits.argmax(1).numpy() == y).mean()) < 1e-12


def test_data_parallel_world_1_equals_fused_step_h128():
    """The peer-memory data-parallel step with a world of one rank equals the fused single-device step at H = 128."""
    from multimodalsignal_b200.parallel import DataParallelTrainStep, LocalPeers
    from multimodalsignal_b200.synth import synthetic_windows
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    B, C, T = 8, 6, 3840
    p, bufs = _state(C, 2, seed=5, num_classes=2)
    x, y = synthetic_windows(B, C, T, seed=13)
    xc, yc = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    ref = _model(p, bufs, C, 2, num_classes=2, attention=True)
    ref_step = FusedTrainStep(ref, FlatAdam(ref, lr=1e-3, weight_decay=1e-4), B, T, use_graph=False)
    m = _model(p, bufs, C, 2, num_classes=2, attention=True)
    step = DataParallelTrainStep(m, FlatAdam(m, lr=1e-3, weight_decay=1e-4), B, B, T, rank=0, peer=LocalPeers(1), use_graph=True)
    for it in range(5):
        ref_step(xc, yc)
        step(xc, yc)
        torch.cuda.synchronize()
        assert abs(float(step.loss.item()) - ref_step.last_loss()) < 2e-5, it
    ref_sd = ref.state_dict()
    for k, v in m.state_dict().items():
        if v.numel():
            np.testing.assert_allclose(v.float().cpu().numpy(), ref_sd[k].float().cpu().numpy(), atol=1e-4, err_msg=k)


def test_dropout_training_runs_and_is_stochastic_h128():
    from multimodalsignal_b200.synth import synthetic_windows
    p, bufs = _state(6, 2, seed=2, num_classes=2)
    x, y = synthetic_windows(8, 6, 640, seed=4)
    m = _model(p, bufs, 6, 2, num_classes=2, dropout=0.5, attention=True)
    xc = torch.from_numpy(x).cuda()
    a = m(xc).detach().clone()
    b = m(xc).detach().clone()
    assert torch.isfinite(a).all() and not torch.allclose(a, b)
    torch.nn.functional.cross_entropy(m(xc), torch.from_numpy(y).cuda()).backward()
    assert all(torch.isfinite(q.grad).all() for q in m.parameters() if q.numel())
    m.eval()
    with torch.no_grad():
        np.testing.assert_allclose(m(xc).cpu().numpy(), m(xc).cpu().numpy())


def _launches(lib, hidden):
    """Kernel name -> launch count of one eager training step (forward + backward) at B = 64, C = 6, T = 3840."""
    from multimodalsignal_b200.models import CnnGruAttentionModel
    from multimodalsignal_b200.synth import synthetic_windows
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m = CnnGruAttentionModel(6, 2, gru_hidden_size=hidden, dropout=0.5).cuda().train()
    x, y = synthetic_windows(64, 6, 3840, seed=1)
    xc, yc = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    torch.nn.functional.cross_entropy(m(xc), yc).backward()          # first call: engine and workspace set-up
    torch.cuda.synchronize()
    buf = (C.c_char * 16384)()
    lib.mms_profile_enable(1)                                         # records eager launches from here on
    try:
        torch.nn.functional.cross_entropy(m(xc), yc).backward()
        lib.mms_profile_report(buf, 16384)
    finally:
        lib.mms_profile_enable(0)
    out = {}
    for line in buf.value.decode().strip().splitlines():
        name, cnt, _ = line.rsplit(" ", 2)
        out[name] = int(cnt)
    return out


def test_weight_gradients_h128_run_on_tensor_cores(lib):
    """At B*L >= 1024 every weight-gradient product of the B*L rows runs on the tcgen05 TN kernels at H = 128, as at H = 64.
    The only SIMT TN launches left are the two B-row products of the top layer's single reverse step (M = B = 64 rows), which
    take gemm_tn_acc_kernel at H = 64 as well."""
    k128, k64 = _launches(lib, 128), _launches(lib, 64)
    assert k128.get("gru_fwd_v2_kernel") and k128.get("gru_bwd_ring_kernel")
    assert k128.get("gemm_tn_acc_kernel", 0) == k64.get("gemm_tn_acc_kernel", 0) <= 2, (k128, k64)
    tc = k128.get("tc_gemm_tn_batch_kernel", 0) + k128.get("tc_gemm_tn_kernel", 0)
    assert tc >= 4, k128


@pytest.mark.parametrize("bad", [48, 256])
def test_other_hidden_sizes_are_refused(bad):
    from multimodalsignal_b200.models import CnnGruAttentionModel
    from multimodalsignal_b200._ext import MmsError
    m = CnnGruAttentionModel(6, 2, gru_hidden_size=bad).cuda().eval()
    with pytest.raises(MmsError, match=r"not in \{32,64,128\}"):
        with torch.no_grad():
            m(torch.zeros(2, 6, 640, device="cuda"))
