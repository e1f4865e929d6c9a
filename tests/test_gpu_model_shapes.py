"""Training at the model shapes the library accepts beyond the suite's usual corner, against the float64 oracle.

make_dims (csrc/model.cu) takes cnn_out_channels O in {16, 32, 64}, 1..8 classes and 1..8 GRU layers.  O != 32 changes
which kernels run, not only their sizes: the fused encoder backward (conv_bwd.cu) takes O = 32 only, so at O = 16 / 64
every training backward goes down the per-layer path (time-major bn_relu_pool_bwd, conv1d_wgrad / conv1d_dgrad with the
BatchNorm backward folded in), the forward runs bn_pool_conv2_fwd_kernel<16|64>, and the bottom GRU layer's products have
K = O (input projection) and N2 = O (weight gradient; N2 = 16 fails tc_gemm_tn_supported and takes the SIMT product).  The
head kernels size their arrays by MAX_NC = 8; the workspace, the W_ih^T copies, the dropout sites and the Adam range table
grow with the depth.

Every case is compared with oracle/model_oracle.py in float64 (prune=True) at the suite's tolerances: |logit error| <= 1e-4,
loss within 1e-4, every gradient within 1e-3 of its tensor's max magnitude, BatchNorm running statistics within
2e-6 + 1e-5 |ref|.  Parameters: oracle/cpu_port.make_state with non-trivial BatchNorm affine values (test_gpu_dropout._state)."""
import ctypes as C
import warnings

import numpy as np
import pytest
import torch

from oracle import cpu_port
from oracle import model_oracle as mo
from test_gpu_dropout import _mismatches, _model, _running, _state

pytestmark = pytest.mark.gpu

LOGIT_ATOL = 1e-4
LOSS_ATOL = 1e-4
PARAM_ATOL = 5e-5


def _lib():
    from multimodalsignal_b200 import _ext
    return _ext.lib()


def _inputs(B, C_, T, nc, seed):
    """Synthetic windows; with 8 classes the labels are arange(B) % 8 so every class appears."""
    from multimodalsignal_b200.synth import synthetic_windows
    x, y = synthetic_windows(B, C_, T, seed=seed, num_classes=nc)
    if nc == 8:
        y = np.arange(B, dtype=np.int64) % 8
    return torch.from_numpy(x), torch.from_numpy(y)


def _oracle_step(p64, x, y, layers, attention, want_dx):
    """model_oracle forward -> CE -> backward in float64: (loss, logits, grads, aux) as mo.loss_and_grads, and dx."""
    leaves = {k: v.detach().clone().requires_grad_(v.numel() > 0) for k, v in p64.items()}
    xd = x.double().requires_grad_(want_dx)
    logits, aux = mo.forward(leaves, xd, training=True, gru_layers=layers, attention=attention, prune=True)
    loss = mo.cross_entropy_mean(logits, y)
    names = [k for k, v in leaves.items() if v.requires_grad]
    grads = torch.autograd.grad(loss, [leaves[k] for k in names] + ([xd] if want_dx else []), allow_unused=True)
    out = {k: torch.zeros_like(leaves[k]) for k in leaves}
    out.update({k: g for k, g in zip(names, grads) if g is not None})
    return (loss.detach(), logits.detach(), out, aux), (grads[-1] if want_dx else None)


def _pool_near_ties(p64, aux, rel=2e-6):
    """Max-pool windows of either stage whose two largest (positive) values are within ``rel`` of each other.  The max-pool
    gradient is discontinuous there: float32 may pick the other element than float64, which moves a whole position's gradient
    and shifts the conv2 / stage-1 / attention gradients by percents (the BatchNorm-2 affine and GRU gradients do not see
    it).  A case is only a test of the kernels when its data has no such window."""
    n = 0
    for key, bn in (("s1", "cnn_encoder.1"), ("s2", "cnn_encoder.5")):
        y = aux[f"{key}_conv"].detach()
        mean, var = aux[f"{key}_mean"].detach()[None, :, None], aux[f"{key}_var"].detach()[None, :, None]
        z = torch.relu((y - mean) / torch.sqrt(var + mo.BN_EPS) * p64[f"{bn}.weight"][None, :, None]
                       + p64[f"{bn}.bias"][None, :, None])
        zp = torch.nn.functional.pad(z, (1, 1), value=-1.0)
        win = zp.unfold(2, 3, 2)[:, :, :(z.shape[2] - 1) // 2 + 1]
        top = torch.topk(win, 2, dim=3).values
        n += int(((top[..., 0] > 0) & (top[..., 0] - top[..., 1] < rel * top[..., 0])).sum())
    return n


def _tie_free_inputs(p64, B, C_, T, nc, seed, attention=True):
    """_inputs at the first of seed, seed + 1, ... whose windows have no max-pool near-tie under the parameters p64."""
    for s in range(seed, seed + 8):
        xt, yt = _inputs(B, C_, T, nc, s)
        with torch.no_grad():
            _, aux = mo.forward(p64, xt.double(), training=True, gru_layers=1, attention=attention)
        if not _pool_near_ties(p64, aux):
            return xt, yt
    raise AssertionError(f"no tie-free inputs at seeds {seed}..{seed + 7}")


def _oracle_running(bufs, aux):
    """The BatchNorm running statistics after the oracle's training step."""
    out = {}
    for prefix, key in (("cnn_encoder.1", "s1"), ("cnn_encoder.5", "s2")):
        n = aux[f"{key}_conv"].shape[0] * aux[f"{key}_conv"].shape[2]
        rm, rv = mo.running_stats_update(bufs[f"{prefix}.running_mean"].double(), bufs[f"{prefix}.running_var"].double(),
                                         aux[f"{key}_mean"].detach(), aux[f"{key}_var"].detach(), n)
        out[f"{prefix}.running_mean"], out[f"{prefix}.running_var"] = rm, rv
    return out


# ---- 1. the whole training step -----------------------------------------------------------------------------------------

# B, C, T, O, H, layers, num_classes, extras: the path each reaches (model.cu, conv_fused.cu, tc_gemm.cu, head_opt.cu).
# extras: attention (default True), dx (request the input gradient).  M = B * L rows, L = T / 16.
STEP_CASES = {
    # fused forward bn_pool_conv2_fwd<16>; per-layer BN-folded backward (conv1d_wgrad / dgrad <16>); tcgen05 NT input
    # projection with K = 16; bottom-layer weight gradient on the SIMT TN product with N2 = 16 at M = 15 360
    "b64_o16": (64, 6, 3840, 16, 64, 2, 2, {}),
    # the same at <64>; the bottom-layer weight gradient on tcgen05 TN with N2 = 64
    "b64_o64": (64, 6, 3840, 64, 64, 2, 2, {}),
    # H = 128: tn_split cuts N1 = 384 into two row halves, both falling back to SIMT with N2 = 16
    "b16_o16_h128": (16, 6, 3840, 16, 128, 2, 3, {}),
    # H = 128: tn_split's row halves with N2 = 64 on tcgen05; 5 classes
    "b16_o64_h128_c5": (16, 6, 3840, 64, 128, 2, 5, {}),
    # partial tiles (T = 4032, B = 5) at O = 16; input gradient requested
    "b5_t4032_o16_dx": (5, 6, 4032, 16, 64, 2, 3, {"dx": True}),
    # fused forward with T % 64 != 0 at O = 64; 4 classes; input gradient requested
    "b4_t352_o64_c4_dx": (4, 8, 352, 64, 64, 2, 4, {"dx": True}),
    # per-layer forward (T % 8 != 0) at O = 16, H = 32, one layer
    "b3_t100_o16": (3, 5, 100, 16, 32, 1, 2, {}),
    # the same without the attention gate
    "b3_t100_o16_noattn": (3, 5, 100, 16, 32, 1, 2, {"attention": False}),
    # C = 16 at O = 64, three layers
    "b2_c16_o64_l3": (2, 16, 1088, 64, 32, 3, 2, {}),
    # B = 1, the shortest window (L = 4) at O = 64
    "b1_t64_o64": (1, 1, 64, 64, 64, 2, 2, {}),
    # one class: loss 0 and every gradient exactly 0 in the oracle
    "b8_c1": (8, 6, 640, 32, 64, 2, 1, {}),
    # eight classes (every class present): the head forward and backward at MAX_NC
    "b16_c8": (16, 6, 3840, 32, 64, 2, 8, {}),
    # B > 256 with 8 classes: the head kernels over more rows than a CTA has threads; the skinny products refused
    "b301_t336_c8": (301, 3, 336, 32, 64, 2, 8, {}),
    # four layers on tcgen05 (M = 1920)
    "b8_l4": (8, 6, 3840, 32, 64, 4, 2, {}),
    # eight layers (MAX_LAYERS), SIMT products (M = 320), fifteen W_ih^T jobs
    "b8_t640_h32_l8": (8, 6, 640, 32, 32, 8, 3, {}),
    # eight layers on tcgen05 (M = 3840) with O = 64 and 8 classes
    "b16_o64_l8_c8": (16, 6, 3840, 64, 64, 8, 8, {}),
    # a deep stack at H = 128 with O = 16
    "b8_o16_h128_l5": (8, 6, 3840, 16, 128, 5, 4, {}),
}


@pytest.mark.parametrize("case", list(STEP_CASES))
def test_training_step_vs_float64_oracle(case):
    """Autograd forward -> CE -> backward: logits, loss, every parameter gradient (and dx where requested), both BatchNorm
    layers' running statistics; then the eval-mode forward against the oracle's with the updated running statistics."""
    B, C_, T, O, H, layers, nc, extras = STEP_CASES[case]
    attention, want_dx = extras.get("attention", True), extras.get("dx", False)
    params, bufs = _state(C_, nc, H, layers, seed=30 + C_ + O + layers, O=O)
    p64 = {k: v.double() for k, v in params.items()}
    xt, yt = _tie_free_inputs(p64, B, C_, T, nc, seed=B + T + O, attention=attention)
    ref, ref_dx = _oracle_step(p64, xt, yt, layers, attention, want_dx)

    m = _model(params, bufs, C_, nc, H, layers, 0.0, O=O, attention=attention)
    xc = xt.cuda().requires_grad_(want_dx)
    out = m(xc)
    loss = torch.nn.functional.cross_entropy(out, yt.cuda())
    loss.backward()
    got = dict(logits=out.detach().cpu().numpy(), loss=float(loss.item()),
               grads={k: q.grad.detach().cpu().numpy() for k, q in m.named_parameters()}, running=_running(m))
    bad = _mismatches(got, ref, bufs)         # a gradient whose reference is all zeros must be within 1e-9 of zero
    assert not bad, bad
    if nc == 1:
        assert float(ref[0]) == 0.0 and all(not g.any() for g in ref[2].values())
    if want_dx:
        e, scale = float(np.abs(xc.grad.cpu().numpy() - ref_dx.numpy()).max()), float(ref_dx.abs().max())
        assert e <= 1e-3 * scale, ("dx", e, scale)

    m.eval()
    with torch.no_grad():
        ev = m(xt.cuda()).cpu().numpy()
    ref_ev, _ = mo.forward(p64, xt.double(), training=False, bn_buffers=_oracle_running(bufs, ref[3]), gru_layers=layers,
                           attention=attention, prune=True)
    np.testing.assert_allclose(ev, ref_ev.numpy(), atol=LOGIT_ATOL, rtol=0)


# ---- 2. the kernels the O != 32 cases reach -----------------------------------------------------------------------------

def _step_launches(O):
    """Kernel name -> launch count of one eager training step (forward + backward) at B = 64, C = 6, T = 3840."""
    lib = _lib()
    params, bufs = _state(6, 2, 64, 2, seed=1, O=O)
    m = _model(params, bufs, 6, 2, 64, 2, 0.0, O=O)
    xt, yt = _inputs(64, 6, 3840, 2, seed=1)
    xc, yc = xt.cuda(), yt.cuda()
    torch.nn.functional.cross_entropy(m(xc), yc).backward()          # first call: engine and workspace set-up
    torch.cuda.synchronize()
    buf = C.create_string_buffer(16384)
    lib.mms_profile_enable(1)
    try:
        torch.nn.functional.cross_entropy(m(xc), yc).backward()
        torch.cuda.synchronize()
        lib.mms_profile_report(buf, 16384)
    finally:
        lib.mms_profile_enable(0)
    out = {}
    for line in buf.value.decode().strip().splitlines():
        name, cnt, _ = line.rsplit(" ", 2)
        out[name] = int(cnt)
    return out


@pytest.mark.parametrize("O", [16, 32, 64])
def test_cnn_width_selects_the_encoder_backward(O):
    """The fused forward (bn_pool_conv2_fwd_kernel) runs at every width; the fused encoder backward (conv2_bwd_kernel) at
    O = 32 only, the per-layer conv1d_wgrad / conv1d_dgrad kernels at O = 16 and 64.  This keeps the O != 32 rows of
    STEP_CASES on the per-layer path they claim to cover."""
    k = _step_launches(O)
    assert k.get("bn_pool_conv2_fwd_kernel"), k
    if O == 32:
        assert k.get("conv2_bwd_kernel") and not k.get("conv1d_wgrad_kernel") and not k.get("conv1d_dgrad_kernel"), k
    else:
        assert not k.get("conv2_bwd_kernel") and k.get("conv1d_wgrad_kernel") and k.get("conv1d_dgrad_kernel"), k


# ---- 3. the fused, graph-replayed training step over several steps ------------------------------------------------------

@pytest.mark.parametrize("B,C_,T,O,H,layers,nc", [
    (8, 6, 3840, 16, 64, 2, 3),
    (8, 6, 3840, 64, 64, 2, 2),
    (8, 6, 640, 64, 32, 8, 8),       # 76 Adam ranges (limit 96), 44 flat segments (limit 64)
])
def test_fused_train_step_follows_float64_adam_trajectory(tmp_path, B, C_, T, O, H, layers, nc):
    """FusedTrainStep (CUDA graph, FlatAdam with weight decay) for five steps against model_oracle.adam_step on the float64
    oracle; then the eval-mode forward, and the state_dict saved and loaded into oracle/cpu_port, give the same logits."""
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    steps = 5
    params, bufs = _state(C_, nc, H, layers, seed=50 + O + layers, O=O)
    xt, yt = _tie_free_inputs({k: v.double() for k, v in params.items()}, B, C_, T, nc, seed=60 + O)
    m = _model(params, bufs, C_, nc, H, layers, 0.0, O=O)
    step = FusedTrainStep(m, FlatAdam(m, lr=1e-3, weight_decay=1e-4), batch=B, seq_len=T)
    xc, yc = xt.cuda(), yt.cuda()
    losses = []
    for _ in range(steps):
        step(xc, yc)
        losses.append(step.last_loss())
    assert step.graph is not None

    ref = {k: v.double() for k, v in params.items()}
    m1 = {k: torch.zeros_like(v) for k, v in ref.items()}
    m2 = {k: torch.zeros_like(v) for k, v in ref.items()}
    ref_losses = []
    for s in range(1, steps + 1):
        loss, _, grads, _ = mo.loss_and_grads(ref, xt.double(), yt, training=True, gru_layers=layers, prune=True)
        ref_losses.append(loss.item())
        for k in ref:
            ref[k], m1[k], m2[k] = mo.adam_step(ref[k], grads[k], m1[k], m2[k], s)
    np.testing.assert_allclose(losses, ref_losses, atol=LOSS_ATOL)
    mine = m.state_dict()
    for k, v in ref.items():
        np.testing.assert_allclose(mine[k].cpu().numpy(), v.numpy(), atol=PARAM_ATOL, err_msg=k)
    assert int(mine["cnn_encoder.5.num_batches_tracked"].item()) == steps

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


# ---- 5. data parallelism ------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("T,O,layers,nc", [(3840, 64, 4, 5), (640, 16, 2, 8)])
def test_two_rank_data_parallel_equals_full_batch(T, O, layers, nc):
    """Two emulated ranks (3 + 5 windows, sync tensors summed as the all-reduce would: the 2 * O SyncBN vectors of stage 2)
    for three steps equal the full-batch FusedTrainStep."""
    from multimodalsignal_b200.parallel import DataParallelTrainStep, emulate_ranks
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    splits, C_, H = (3, 5), 6, 64
    B = sum(splits)
    params, bufs = _state(C_, nc, H, layers, seed=70 + O, O=O)
    xt, yt = _inputs(B, C_, T, nc, seed=80 + O)
    xc, yc = xt.cuda(), yt.cuda()
    ref = _model(params, bufs, C_, nc, H, layers, 0.0, O=O)
    ref_step = FusedTrainStep(ref, FlatAdam(ref, lr=1e-3, weight_decay=1e-4), B, T, use_graph=False)
    ranks, steps, batches, lo = [], [], [], 0
    for r, b in enumerate(splits):
        m = _model(params, bufs, C_, nc, H, layers, 0.0, O=O)
        ranks.append(m)
        steps.append(DataParallelTrainStep(m, FlatAdam(m, lr=1e-3, weight_decay=1e-4), b, B, T, rank=r))
        batches.append((xc[lo:lo + b], yc[lo:lo + b]))
        lo += b
    for it in range(3):
        ref_step(xc, yc)
        emulate_ranks(steps, batches)
        loss = sum(float(s.loss.item()) for s in steps)
        assert abs(loss - ref_step.last_loss()) < 2e-5, (it, loss, ref_step.last_loss())
    # parameters within 1e-4 as in the peer-step comparisons: the split batch sums in another order, and Adam turns a
    # rounding-level difference of a near-zero gradient into up to lr per step
    ref_sd = ref.state_dict()
    for m in ranks:
        for k, v in m.state_dict().items():
            if v.numel():
                np.testing.assert_allclose(v.float().cpu().numpy(), ref_sd[k].float().cpu().numpy(), atol=1e-4, err_msg=k)
    for m in ranks[1:]:
        assert torch.equal(m.flat_parameters(), ranks[0].flat_parameters())


@pytest.mark.timeout(120)
def test_peer_kernels_world_1_equal_fused_step_o64():
    """The peer-memory data-parallel step with a world of one rank (its barriers are with itself) equals the fused
    single-device step at O = 64, graph-replayed."""
    from multimodalsignal_b200.parallel import DataParallelTrainStep, LocalPeers
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    B, C_, T, O, H, layers, nc = 8, 6, 3840, 64, 64, 2, 3
    params, bufs = _state(C_, nc, H, layers, seed=90, O=O)
    xt, yt = _inputs(B, C_, T, nc, seed=91)
    xc, yc = xt.cuda(), yt.cuda()
    ref = _model(params, bufs, C_, nc, H, layers, 0.0, O=O)
    ref_step = FusedTrainStep(ref, FlatAdam(ref, lr=1e-3, weight_decay=1e-4), B, T, use_graph=False)
    m = _model(params, bufs, C_, nc, H, layers, 0.0, O=O)
    step = DataParallelTrainStep(m, FlatAdam(m, lr=1e-3, weight_decay=1e-4), B, B, T, rank=0, peer=LocalPeers(1), use_graph=True)
    for it in range(5):
        ref_step(xc, yc)
        step(xc, yc)
        torch.cuda.synchronize()
        assert abs(float(step.loss.item()) - ref_step.last_loss()) < 2e-5, it
    assert int(step.opt.step_dev.item()) == 5
    ref_sd = ref.state_dict()
    for k, v in m.state_dict().items():
        if v.numel():
            np.testing.assert_allclose(v.float().cpu().numpy(), ref_sd[k].float().cpu().numpy(), atol=1e-4, err_msg=k)


# ---- 6. Trainer and the refusals ----------------------------------------------------------------------------------------

def test_trainer_evaluate_and_best_model_o64_l4_c3(tmp_path):
    """Trainer.train (fused graph-replayed steps, best_model.pt) and Trainer.evaluate (EvalStep) with cnn_out_channels = 64,
    3 classes and 4 GRU layers: the checkpoint has the reference's keys and shapes and, loaded into oracle/cpu_port, gives
    the loss Trainer.evaluate reports."""
    from torch.utils.data import DataLoader, TensorDataset
    from multimodalsignal_b200.models import CnnGruAttentionModel
    from multimodalsignal_b200.trainer import Trainer
    C_, T, nc, layers = 3, 640, 3, 4
    xt, yt = _inputs(48, C_, T, nc, seed=21)
    tl = DataLoader(TensorDataset(xt, yt), batch_size=16, shuffle=False, num_workers=0)
    torch.manual_seed(0)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model = CnnGruAttentionModel(in_channels=C_, num_classes=nc, cnn_out_channels=64, gru_num_layers=layers, dropout=0.0)
    ref_keys = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    cfg = {'trainer': {'epochs': 1, 'learning_rate': 1e-3, 'early_stopping': {'enabled': True, 'patience': 20, 'delta': 0},
                       'weight_decay': 1e-4}}
    trainer = Trainer(model, tmp_path / "fold", cfg)
    trainer.train(tl, tl)
    loss, acc, _ = trainer.evaluate(tl)
    sd = torch.load(tmp_path / "fold" / "best_model.pt", map_location="cpu")
    assert {k: tuple(v.shape) for k, v in sd.items()} == ref_keys and list(sd.keys()) == list(ref_keys)
    assert sd["cnn_encoder.4.weight"].shape == (64, 16, 5) and sd["classifier.3.weight"].shape == (nc, 64)
    cp = {k: v.float() for k, v in sd.items() if "running" not in k and "num_batches" not in k}
    cb = {k: v.float() for k, v in sd.items() if "running" in k}
    with torch.no_grad():
        logits = cpu_port.forward(cp, cb, xt, training=False, dropout=0.0, layers=layers)
    ref_loss = torch.nn.functional.cross_entropy(logits, yt).item()
    assert abs(loss - ref_loss) < 1e-4, (loss, ref_loss)
    assert abs(acc - (logits.argmax(1) == yt).double().mean().item()) < 1e-12


@pytest.mark.parametrize("arg,value,msg", [
    ("cnn_out_channels", 8, r"cnn_out_channels 8 not in \{16,32,64\}"),
    ("cnn_out_channels", 48, r"cnn_out_channels 48 not in \{16,32,64\}"),
    ("cnn_out_channels", 128, r"cnn_out_channels 128 not in \{16,32,64\}"),
    ("num_classes", 0, r"num_classes 0 outside \[1,8\]"),
    ("num_classes", 9, r"num_classes 9 outside \[1,8\]"),
    ("gru_num_layers", 9, r"gru_num_layers 9 outside \[1,8\]"),
])
def test_unsupported_shapes_are_refused_before_any_launch(arg, value, msg):
    """A shape make_dims does not accept raises MmsError naming the argument at the first forward, before any kernel is
    launched (training and eval mode)."""
    from multimodalsignal_b200._ext import MmsError
    from multimodalsignal_b200.models import CnnGruAttentionModel
    kw = dict(in_channels=6, num_classes=2, dropout=0.0)
    kw[arg] = value
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m = CnnGruAttentionModel(**kw).cuda()
    lib = _lib()
    x = torch.zeros(2, 6, 640, device="cuda")
    buf = C.create_string_buffer(16384)
    torch.cuda.synchronize()
    lib.mms_profile_enable(1)
    try:
        for train in (True, False):
            m.train(train)
            with pytest.raises(MmsError, match=msg):
                m(x)
        torch.cuda.synchronize()
        lib.mms_profile_report(buf, 16384)
    finally:
        lib.mms_profile_enable(0)
    assert buf.value.decode().strip() == "", buf.value.decode()
