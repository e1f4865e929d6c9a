"""Class-weighted cross entropy (``CrossEntropyLoss(weight=w)``, ``use_class_weights``): the weighted forms of the loss
kernels against torch / the float64 oracle, the training step on both head paths, the Adam trajectory, the evaluation
grouping, data parallelism and the ``Trainer`` option.  The host-only cases at the top run without a GPU."""
import ctypes as C
import re
import warnings

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import model_oracle as mo

LOGIT_ATOL = 1e-4
GRAD_RTOL = 3e-4


# ----------------------------------------------------------------------------------------------- host-only
def test_balanced_weights_equal_sklearn():
    from sklearn.utils.class_weight import compute_class_weight
    from multimodalsignal_b200.trainer import balanced_class_weights
    rng = np.random.default_rng(0)
    for nc, n in ((2, 301), (3, 1000), (8, 97)):
        y = rng.integers(0, nc, n)
        y[:nc] = np.arange(nc)
        ref = compute_class_weight('balanced', classes=np.arange(nc), y=y)
        np.testing.assert_allclose(balanced_class_weights(y, nc), ref, rtol=1e-12)
        np.testing.assert_allclose(balanced_class_weights(torch.from_numpy(y), nc), ref, rtol=1e-12)


def test_balanced_weights_refuse_a_missing_class_and_bad_labels():
    from multimodalsignal_b200.trainer import balanced_class_weights
    with pytest.raises(ValueError, match="class 1 has no training windows"):
        balanced_class_weights(np.array([0, 0, 2, 2]), 3)
    with pytest.raises(ValueError, match="outside"):
        balanced_class_weights(np.array([0, 1, 2]), 2)


def test_cross_entropy_loss_refuses_unimplemented_options():
    from multimodalsignal_b200.trainer import CrossEntropyLoss
    CrossEntropyLoss()
    CrossEntropyLoss(weight=[1.0, 2.0])
    for kw in ({"ignore_index": 0}, {"label_smoothing": 0.1}, {"reduction": "sum"}, {"reduction": "none"}):
        with pytest.raises(NotImplementedError):
            CrossEntropyLoss(**kw)


# ---- float64 references of the weighted loss, built on the unweighted oracle (oracle/model_oracle.py, oracle/cpu_port.py)
def _weighted_ce(logits, labels, weight):
    """CrossEntropyLoss(weight=w), mean reduction, as an explicit formula: sum_b w[y_b] l_b / sum_b w[y_b]."""
    lse = torch.logsumexp(logits, dim=1)
    picked = logits.gather(1, labels[:, None]).squeeze(1)
    wy = weight.to(logits.dtype)[labels]
    return (wy * (lse - picked)).sum() / wy.sum()


def _weighted_loss_and_grads(params, x, labels, weight, **fw):
    """oracle/model_oracle.loss_and_grads with the weighted loss: (loss, logits, grads_by_name)."""
    leaves = {k: v.detach().clone().requires_grad_(v.numel() > 0 and v.is_floating_point()) for k, v in params.items()}
    logits, _ = mo.forward(leaves, x, **fw)
    loss = _weighted_ce(logits, labels, weight)
    names = [k for k, v in leaves.items() if v.requires_grad]
    grads = torch.autograd.grad(loss, [leaves[k] for k in names], allow_unused=True)
    out = {k: torch.zeros_like(v) for k, v in leaves.items()}
    out.update({k: g for k, g in zip(names, grads) if g is not None})
    return loss.detach(), logits.detach(), out


def _weighted_cpu_step(p, bufs, weight, **kw):
    """oracle/cpu_port.CpuTrainStep (float32 ATen CPU kernels, torch.optim.Adam) with CrossEntropyLoss(weight=...);
    ``.weight`` may be changed between steps."""
    from oracle import cpu_port

    class Step(cpu_port.CpuTrainStep):
        def __call__(self, x, y):
            self.opt.zero_grad()
            logits = cpu_port.forward(self.p, self.bufs, x, training=True, dropout=self.dropout, layers=self.layers,
                                      attention=self.attention)
            loss = F.cross_entropy(logits, y, weight=self.weight)
            loss.backward()
            self.opt.step()
            return loss.item()

    step = Step(p, bufs, **kw)
    step.weight = torch.as_tensor(weight, dtype=torch.float32)
    return step


def test_weighted_reference_equals_torch():
    g = torch.Generator().manual_seed(3)
    logits = torch.randn(37, 3, generator=g, dtype=torch.float64)
    y = torch.randint(0, 3, (37,), generator=g)
    w = torch.tensor([0.3, 2.0, 0.0], dtype=torch.float64)
    ref = F.cross_entropy(logits, y, weight=w)
    assert abs(_weighted_ce(logits, y, w).item() - ref.item()) < 1e-14
    assert abs(_weighted_ce(logits, y, torch.ones(3, dtype=torch.float64)).item() - mo.cross_entropy_mean(logits, y).item()) < 1e-14


def _desc(weighted, O=32):
    from multimodalsignal_b200._ext import CnnGruDesc
    d = CnnGruDesc()
    d.batch, d.in_channels, d.seq_len, d.num_classes = 4, 6, 640, 2
    d.cnn_out, d.hidden, d.layers, d.training, d.attention, d.need_grad = O, 64, 2, 1, 1, 1
    d.global_batch = 8
    d.class_weight = 0x1000 if weighted else None          # only its presence matters to the layout queries
    return d


@pytest.mark.parametrize("O", [16, 32, 64])
def test_sync_offsets_grow_by_one_double_only_with_class_weights(O):
    """Layout queries are host-only.  Without weights the exchanged vectors are the BN sums alone; with weights the BN2
    vector carries one more double, and nothing else moves."""
    from multimodalsignal_b200 import _ext
    from multimodalsignal_b200.build import build
    build()
    lib = _ext.load_library()
    out = {}
    for weighted in (False, True):
        offs, cnts = (C.c_int64 * 4)(), (C.c_int64 * 4)()
        assert lib.mms_cnngru_sync_offsets(C.byref(_desc(weighted, O)), offs, cnts) == 0
        out[weighted] = (list(offs), list(cnts))
    assert out[False][1] == [32, 2 * O, 32, 2 * O]
    assert out[True][1] == [32, 2 * O + 1, 32, 2 * O]
    assert out[True][0] == out[False][0]
    assert out[False][0][1] == out[False][0][0] + 8 * 32


# ----------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def lib():
    from multimodalsignal_b200 import _ext
    return _ext.lib()


def P(t):
    return None if t is None else t.data_ptr()


def ST():
    return torch.cuda.current_stream().cuda_stream


def ok(rc):
    from multimodalsignal_b200 import _ext
    return _ext.check(rc)


def _weights(nc, seed, zero=True):
    g = torch.Generator().manual_seed(seed)
    w = torch.rand(nc, generator=g) * 2 + 0.1
    if zero and nc > 2:
        w[1] = 0.0
    return w


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 7, 64, 301, 1024])
@pytest.mark.parametrize("nc", [1, 2, 3, 8])
def test_weighted_cross_entropy_vs_torch(lib, B, nc):
    g = torch.Generator().manual_seed(B * 10 + nc)
    logits = torch.randn(B, nc, generator=g) * 3
    y = torch.randint(0, nc, (B,), generator=g)
    y[0] = nc - 1
    w = _weights(nc, B + nc)
    ref_loss = F.cross_entropy(logits.double(), y, weight=w.double())
    lg = logits.double().requires_grad_(True)
    F.cross_entropy(lg, y, weight=w.double()).backward()
    ld, yd, wd = logits.cuda(), y.cuda(), w.cuda()
    loss = torch.zeros(1, device="cuda")
    dl = torch.zeros(B, nc, device="cuda")
    acc = torch.zeros(1, dtype=torch.float64, device="cuda")
    ok(lib.mms_cross_entropy_weighted(P(ld), P(yd), B, nc, P(wd), None, P(loss), P(dl), P(acc), ST()))
    assert abs(loss.item() - ref_loss.item()) <= 1e-5 * max(1.0, abs(ref_loss.item()))
    np.testing.assert_allclose(dl.cpu().numpy(), lg.grad.numpy(), atol=1e-6, rtol=1e-5)
    assert abs(acc.item() - loss.item() * B) <= 1e-6 * max(1.0, abs(acc.item()))
    # the same with an external normaliser equal to the local sum
    norm = torch.tensor([float(w.double()[y].sum())], dtype=torch.float64, device="cuda")
    loss2 = torch.zeros(1, device="cuda")
    dl2 = torch.zeros_like(dl)
    ok(lib.mms_cross_entropy_weighted(P(ld), P(yd), B, nc, P(wd), P(norm), P(loss2), P(dl2), None, ST()))
    assert abs(loss2.item() - ref_loss.item()) <= 1e-5 * max(1.0, abs(ref_loss.item()))
    np.testing.assert_allclose(dl2.cpu().numpy(), lg.grad.numpy(), atol=1e-6, rtol=1e-5)
    # all-ones weights == the unweighted entry point
    ones = torch.ones(nc, device="cuda")
    lu, du = torch.zeros(1, device="cuda"), torch.zeros_like(dl)
    ok(lib.mms_cross_entropy(P(ld), P(yd), B, nc, P(lu), P(du), None, ST()))
    ok(lib.mms_cross_entropy_weighted(P(ld), P(yd), B, nc, P(ones), None, P(loss), P(dl), None, ST()))
    assert abs(loss.item() - lu.item()) <= 1e-6 * max(1e-6, abs(lu.item()))
    np.testing.assert_allclose(dl.cpu().numpy(), du.cpu().numpy(), rtol=1e-6, atol=1e-9)
    # NULL weights: exactly mms_cross_entropy
    ok(lib.mms_cross_entropy_weighted(P(ld), P(yd), B, nc, None, None, P(loss), P(dl), None, ST()))
    assert loss.item() == lu.item() and torch.equal(dl, du)
    # an out-of-range label: NaN loss, that row adds no gradient
    if B > 1:
        yb = yd.clone()
        yb[B // 2] = nc
        ok(lib.mms_cross_entropy_weighted(P(ld), P(yb), B, nc, P(wd), None, P(loss), P(dl), None, ST()))
        assert np.isnan(loss.item())
        assert torch.all(dl[B // 2] == 0)


@pytest.mark.gpu
def test_weighted_cross_entropy_refusals_and_zero_weight_sum(lib):
    ld = torch.randn(4, 3, device="cuda")
    yd = torch.tensor([0, 0, 2, 2], device="cuda")
    loss, dl = torch.zeros(1, device="cuda"), torch.zeros(4, 3, device="cuda")
    norm = torch.ones(1, dtype=torch.float64, device="cuda")
    assert lib.mms_cross_entropy_weighted(P(ld), P(yd), 4, 3, None, P(norm), P(loss), P(dl), None, ST()) < 0
    w = torch.tensor([0.0, 1.0, 0.0], device="cuda")            # sum_b w[y_b] == 0: NaN, as torch
    ok(lib.mms_cross_entropy_weighted(P(ld), P(yd), 4, 3, P(w), None, P(loss), P(dl), None, ST()))
    assert np.isnan(loss.item())
    assert np.isnan(F.cross_entropy(ld.cpu(), yd.cpu(), weight=w.cpu()).item())
    out = torch.full((1,), -1.0, dtype=torch.float64, device="cuda")
    w2 = torch.tensor([0.5, 1.0, 3.0], device="cuda")
    ok(lib.mms_class_weight_sum(P(yd), 4, 3, P(w2), P(out), ST()))
    assert out.item() == 7.0


@pytest.mark.gpu
@pytest.mark.parametrize("B,group,nc", [(301, 48, 2), (301, 64, 3), (256, 256, 2), (7, 0, 8), (1000, 300, 2)])
def test_eval_accumulate_weighted_groups(lib, B, group, nc):
    g = torch.Generator().manual_seed(B + group)
    logits = torch.randn(B, nc, generator=g) * 2
    y = torch.randint(0, nc, (B,), generator=g)
    w = _weights(nc, 7, zero=False)
    ld, yd, wd = logits.cuda(), y.cuda(), w.cuda()
    preds = torch.zeros(B, dtype=torch.int64, device="cuda")
    conf = torch.zeros(nc * nc, dtype=torch.int64, device="cuda")
    loss = torch.zeros(1, dtype=torch.float64, device="cuda")
    ok(lib.mms_eval_accumulate_weighted(P(ld), P(yd), B, nc, P(wd), group, P(preds), P(conf), P(loss), ST()))
    gs = group if group > 0 else B
    ref = sum(len(y[i:i + gs]) * F.cross_entropy(logits[i:i + gs].double(), y[i:i + gs], weight=w.double()).item()
              for i in range(0, B, gs))
    assert abs(loss.item() - ref) <= 1e-6 * abs(ref)
    p2 = torch.zeros_like(preds)
    c2 = torch.zeros_like(conf)
    ok(lib.mms_eval_accumulate(P(ld), P(yd), B, nc, P(p2), P(c2), None, ST()))
    assert torch.equal(preds, p2) and torch.equal(conf, c2)


# ---- whole training step against the float64 oracle
def _state(C, H, seed):
    from oracle import cpu_port
    p, bufs = cpu_port.make_state(C=C, H=H, seed=seed)
    g = torch.Generator().manual_seed(seed + 100)
    for k in ("cnn_encoder.1", "cnn_encoder.5"):
        p[f"{k}.weight"] = p[f"{k}.weight"] + 0.1 * torch.randn(p[f"{k}.weight"].shape, generator=g)
        p[f"{k}.bias"] = p[f"{k}.bias"] + 0.1 * torch.randn(p[f"{k}.bias"].shape, generator=g)
    return p, bufs


def _model(p, bufs, C, H=64, nc=2):
    from multimodalsignal_b200.models import CnnGruAttentionModel
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m = CnnGruAttentionModel(C, nc, dropout=0.0, gru_hidden_size=H)
    sd = dict(p)
    sd.update(bufs)
    sd["cnn_encoder.1.num_batches_tracked"] = torch.zeros((), dtype=torch.int64)
    sd["cnn_encoder.5.num_batches_tracked"] = torch.zeros((), dtype=torch.int64)
    m.load_state_dict(sd, strict=True)
    return m.cuda().train()


def _labels(B, seed):
    """Skewed binary labels (about a quarter positive, as WESAD stress_binary), at least one of each when B > 1."""
    g = torch.Generator().manual_seed(seed)
    y = (torch.rand(B, generator=g) < 0.25).long()
    if B > 1:
        y[0], y[1] = 0, 1
    return y


@pytest.mark.gpu
@pytest.mark.parametrize("B,C,T,H", [(64, 6, 3840, 64), (8, 3, 336, 64), (1, 6, 640, 64), (4, 6, 640, 128)])
def test_weighted_train_step_vs_float64_oracle(lib, B, C, T, H):
    """One mms_cnngru_train_step with class weights, fused head (HEAD_FUSED=1) and separate cross entropy (HEAD_FUSED=0):
    loss, logits and every gradient against the float64 oracle's CrossEntropyLoss(weight=w)."""
    from multimodalsignal_b200.synth import synthetic_windows
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    p, bufs = _state(C, H, seed=21 + C)
    x, _ = synthetic_windows(B, C, T, seed=9 + C)
    xt, yt = torch.from_numpy(x), _labels(B, B + T)
    w = torch.tensor([0.6, 2.5])
    params = {k: v.double() for k, v in p.items()}
    ref_loss, ref_logits, ref_grads = _weighted_loss_and_grads(params, xt.double(), yt, w.double(), training=True, prune=True)
    try:
        for fused in (1, 0):
            ok(lib.mms_set_option(b"HEAD_FUSED", fused))
            m = _model(p, bufs, C, H)
            opt = FlatAdam(m, lr=1e-3, weight_decay=1e-4)
            step = FusedTrainStep(m, opt, B, T, use_graph=False, class_weight=w)
            step(xt.cuda(), yt.cuda())
            torch.cuda.synchronize()
            np.testing.assert_allclose(step.logits.cpu().numpy(), ref_logits.numpy(), atol=LOGIT_ATOL)
            assert abs(step.last_loss() - ref_loss.item()) < 1e-4, (fused, step.last_loss(), ref_loss.item())
            assert abs(step.loss_sum.item() - step.last_loss() * B) <= 1e-6 * max(1.0, abs(step.loss_sum.item()))
            grads = opt.grads.cpu()
            for (off, n, shape), (k, _) in zip(m._param_views, m.named_parameters()):
                ref = ref_grads[k].numpy()
                if ref.size == 0:
                    continue
                got = grads[off:off + n].view(shape).numpy()
                scale = max(np.abs(ref).max(), 1e-6)
                assert np.abs(got - ref).max() <= GRAD_RTOL * scale, (fused, k, np.abs(got - ref).max(), scale)
    finally:
        lib.mms_clear_option(b"HEAD_FUSED")


@pytest.mark.gpu
def test_weighted_fused_step_follows_cpu_adam_trajectory_and_weights_change_without_recapture():
    """Graph-replayed FusedTrainStep with class weights against oracle/cpu_port.CpuTrainStep with the weighted loss on the same batches
    (dropout 0).  Halfway the weights change by set_class_weight: the captured graph reads them from the same tensor."""
    from multimodalsignal_b200.synth import synthetic_windows
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    B, C, T = 8, 6, 640
    p, bufs = _state(C, 64, seed=4)
    m = _model(p, bufs, C)
    opt = FlatAdam(m, lr=1e-3, weight_decay=1e-4)
    w1, w2 = [0.7, 1.9], [3.0, 0.4]
    step = FusedTrainStep(m, opt, B, T, class_weight=w1)
    ref = _weighted_cpu_step(p, bufs, w1, dropout=0.0)
    losses, ref_losses = [], []
    for it in range(6):
        x, _ = synthetic_windows(B, C, T, seed=100 + it)
        xt, yt = torch.from_numpy(x), _labels(B, 200 + it)
        if it == 3:
            step.set_class_weight(w2)
            ref.weight = torch.tensor(w2)
        step(xt.cuda(), yt.cuda())
        losses.append(step.last_loss())
        ref_losses.append(ref(xt, yt))
    assert step.graph is not None                       # replays from the second call on; one capture
    np.testing.assert_allclose(losses, ref_losses, atol=1e-4)
    mine = m.state_dict()
    for k, v in ref.p.items():
        if v.numel():
            np.testing.assert_allclose(mine[k].cpu().numpy(), v.detach().numpy(), atol=5e-5, err_msg=k)


# ---- evaluation grouping
class _TensorSet(torch.utils.data.Dataset):
    def __init__(self, data, labels):
        self.data, self.labels = data.cpu(), labels.cpu()

    def __len__(self):
        return len(self.labels)

    def __getitem__(self, i):
        return self.data[i], self.labels[i]


class _DevSet:
    def __init__(self, data, labels):
        self.data, self.labels = data.cuda(), labels.cuda()

    def __len__(self):
        return int(self.labels.shape[0])


def _cfg(epochs, weighted=True):
    return {'trainer': {'epochs': epochs, 'learning_rate': 1e-3, 'use_class_weights': weighted,
                        'early_stopping': {'enabled': False, 'patience': 20, 'delta': 0}, 'weight_decay': 1e-4}}


def _new_model(seed, C=3):
    from multimodalsignal_b200.models import CnnGruAttentionModel
    torch.manual_seed(seed)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return CnnGruAttentionModel(in_channels=C, num_classes=2, dropout=0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("bs", [48, 64])
def test_weighted_evaluation_groups_by_loader_batch(tmp_path, bs):
    """Trainer.evaluate with class weights adds n_k * CE_w(batch k) per loader batch (reference trainer.py:217-228), for a
    host DataLoader and a DeviceBatchLoader (301 windows: a ragged last batch).  The labels make that value differ from
    the global weighted mean and from a per-256-slice grouping, so a wrong grouping fails.  Accuracy and F1 are those of
    the unweighted evaluation."""
    from torch.utils.data import DataLoader
    from multimodalsignal_b200.dataset import DeviceBatchLoader
    from multimodalsignal_b200.trainer import Trainer
    N, Cc, T = 301, 3, 640
    g = torch.Generator().manual_seed(bs)
    y = torch.zeros(N, dtype=torch.int64)
    y[::3] = 1
    y[:40] = 1                                  # label mix varies from batch to batch
    x = torch.randn(N, Cc, T, generator=g) + y[:, None, None].float() * torch.sin(torch.arange(T) / 5.0)
    train_y = torch.tensor([0, 0, 0, 1] * 8)
    train_x = torch.randn(len(train_y), Cc, T, generator=g)
    model = _new_model(3)
    tr = Trainer(model, tmp_path / "w", _cfg(0))
    with pytest.raises(ValueError, match="before it"):
        tr.evaluate(DataLoader(_TensorSet(x, y), batch_size=bs))
    tr.train(DataLoader(_TensorSet(train_x, train_y), batch_size=8), None)      # 0 epochs: fixes the weights only
    w = torch.tensor(tr.class_weights, dtype=torch.float64)
    np.testing.assert_allclose(tr.class_weights, [32 / (2 * 24), 32 / (2 * 8)], rtol=1e-12)
    model.eval()
    with torch.no_grad():
        logits = model(x.cuda()).double().cpu()
    ce = lambda a, b: F.cross_entropy(logits[a:b], y[a:b], weight=w).item()
    ref = sum((min(i + bs, N) - i) * ce(i, i + bs) for i in range(0, N, bs)) / N
    glob = ce(0, N)
    per256 = (256 * ce(0, 256) + (N - 256) * ce(256, N)) / N
    assert abs(ref - glob) > 1e-4 * abs(ref) and abs(ref - per256) > 1e-4 * abs(ref)
    tr_u = Trainer(model, tmp_path / "u", _cfg(0, weighted=False))
    for loader in (DataLoader(_TensorSet(x, y), batch_size=bs), DeviceBatchLoader(_DevSet(x, y), bs, shuffle=False)):
        loss, acc, f1 = tr.evaluate(loader)
        assert abs(loss - ref) <= 1e-6 * abs(ref), (type(loader).__name__, loss, ref, glob, per256)
        _, acc_u, f1_u = tr_u.evaluate(loader)
        assert acc == acc_u and f1 == f1_u


# ---- data parallelism
@pytest.mark.gpu
@pytest.mark.parametrize("splits", [(3, 5), (2, 2, 4)])
def test_weighted_data_parallel_equals_full_batch(lib, splits):
    """emulate_ranks with ranks whose label mixes differ: the summed normaliser makes the ranks' weighted losses and
    gradients add up to the weighted full-batch step.  Each rank normalising by its own labels does not."""
    from multimodalsignal_b200.parallel import DataParallelTrainStep, emulate_ranks
    from multimodalsignal_b200.synth import synthetic_windows
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    B, C, T = sum(splits), 6, 640
    p, bufs = _state(C, 64, seed=8)
    w = [0.4, 2.2]
    ref = _model(p, bufs, C)
    ref_step = FusedTrainStep(ref, FlatAdam(ref, lr=1e-3, weight_decay=1e-4), B, T, use_graph=False, class_weight=w)
    ranks, steps = [], []
    for r, b in enumerate(splits):
        m = _model(p, bufs, C)
        ranks.append(m)
        steps.append(DataParallelTrainStep(m, FlatAdam(m, lr=1e-3, weight_decay=1e-4), b, B, T, rank=r, class_weight=w))
    for it in range(3):
        x, _ = synthetic_windows(B, C, T, seed=50 + it)
        xt = torch.from_numpy(x).cuda()
        yt = torch.zeros(B, dtype=torch.int64)
        yt[:splits[0]] = 1                                  # rank 0 mostly positive, the others negative
        yt[0] = 0
        yt[-1] = 1
        yt = yt.cuda()
        ref_step(xt, yt)
        lo, batches = 0, []
        for b in splits:
            batches.append((xt[lo:lo + b], yt[lo:lo + b]))
            lo += b
        emulate_ranks(steps, batches)
        loss = sum(float(s.loss.item()) for s in steps)
        assert abs(loss - ref_step.last_loss()) < 2e-5, (it, loss, ref_step.last_loss())
        # each rank normalising by its local labels (its share of the batch weighting its local mean) is not the same loss
        wd = torch.tensor(w, device="cuda")
        local = 0.0
        for s, (_, yb) in zip(steps, batches):
            out = torch.zeros(1, device="cuda")
            ok(lib.mms_cross_entropy_weighted(P(s.logits), P(yb), yb.shape[0], 2, P(wd), None, P(out), None, None, ST()))
            local += out.item() * yb.shape[0] / B
        assert abs(local - ref_step.last_loss()) > 1e-3
    ref_sd = ref.state_dict()
    for m in ranks:
        for k, v in m.state_dict().items():
            if v.numel():
                np.testing.assert_allclose(v.float().cpu().numpy(), ref_sd[k].float().cpu().numpy(), atol=2e-5, err_msg=k)


@pytest.mark.gpu
@pytest.mark.timeout(120)
@pytest.mark.parametrize("graph", [False, True])
def test_weighted_peer_kernels_world_1_equal_fused_step(graph):
    """The peer-memory step with one rank and class weights (the normaliser travels in the BN2 vector through
    mms_peer_allreduce_f64) equals the weighted fused single-device step."""
    from multimodalsignal_b200.parallel import DataParallelTrainStep, LocalPeers
    from multimodalsignal_b200.synth import synthetic_windows
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    B, C, T = 6, 6, 640
    p, bufs = _state(C, 64, seed=9)
    w = [0.5, 1.7]
    ref = _model(p, bufs, C)
    ref_step = FusedTrainStep(ref, FlatAdam(ref, lr=1e-3, weight_decay=1e-4), B, T, use_graph=False, class_weight=w)
    m = _model(p, bufs, C)
    step = DataParallelTrainStep(m, FlatAdam(m, lr=1e-3, weight_decay=1e-4), B, B, T, rank=0, peer=LocalPeers(1),
                                 use_graph=graph, class_weight=w)
    for it in range(4):
        x, _ = synthetic_windows(B, C, T, seed=70 + it)
        xt, yt = torch.from_numpy(x).cuda(), _labels(B, 80 + it).cuda()
        ref_step(xt, yt)
        step(xt, yt)
        torch.cuda.synchronize()
        assert abs(float(step.loss.item()) - ref_step.last_loss()) < 2e-5, it
    ref_sd = ref.state_dict()
    for k, v in m.state_dict().items():
        if v.numel():
            np.testing.assert_allclose(v.float().cpu().numpy(), ref_sd[k].float().cpu().numpy(), atol=1e-4, err_msg=k)


@pytest.mark.gpu
@pytest.mark.timeout(120)
@pytest.mark.skipif(__import__("os").environ.get("MMS_TEST_PEER_EMULATION") != "1",
                    reason="several emulated ranks spin on each other's flags on ONE GPU; runs only with MMS_TEST_PEER_EMULATION=1 "
                           "(as tests/test_gpu_parallel.py::test_peer_memory_exchange_equals_full_batch)")
def test_weighted_peer_exchange_emulated_ranks_equal_full_batch():
    from multimodalsignal_b200 import _ext
    from multimodalsignal_b200.parallel import DataParallelTrainStep, LocalPeers, emulate_peer_ranks
    from multimodalsignal_b200.synth import synthetic_windows
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    splits, C, T = (2, 4), 6, 640
    B = sum(splits)
    p, bufs = _state(C, 64, seed=10)
    w = [0.5, 1.7]
    ref = _model(p, bufs, C)
    ref_step = FusedTrainStep(ref, FlatAdam(ref, lr=1e-3, weight_decay=1e-4), B, T, use_graph=False, class_weight=w)
    _ext.lib().mms_set_side_streams(0)
    try:
        peers = LocalPeers(len(splits))
        streams = [torch.cuda.Stream() for _ in splits]
        steps = []
        for r, b in enumerate(splits):
            with torch.cuda.stream(streams[r]):
                m = _model(p, bufs, C)
                steps.append(DataParallelTrainStep(m, FlatAdam(m, lr=1e-3, weight_decay=1e-4), b, B, T, rank=r, peer=peers,
                                                   use_graph=False, class_weight=w))
        torch.cuda.synchronize()
        for it in range(3):
            x, _ = synthetic_windows(B, C, T, seed=90 + it)
            xt, yt = torch.from_numpy(x).cuda(), _labels(B, 95 + it).cuda()
            ref_step(xt, yt)
            emulate_peer_ranks(steps, [(xt[:2], yt[:2]), (xt[2:], yt[2:])], streams)
            torch.cuda.synchronize()
            assert abs(sum(float(s.loss.item()) for s in steps) - ref_step.last_loss()) < 2e-5
    finally:
        _ext.lib().mms_set_side_streams(1)


@pytest.mark.gpu
def test_weights_off_leave_the_launch_list_unchanged(lib):
    """A step without class weights launches what it always did; with weights the fused head path adds no launch and the
    separate cross entropy path none either (the normaliser is reduced inside the loss kernels)."""
    from multimodalsignal_b200.synth import synthetic_windows
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    B, C, T = 8, 6, 640
    p, bufs = _state(C, 64, seed=12)
    x, _ = synthetic_windows(B, C, T, seed=1)
    xt, yt = torch.from_numpy(x).cuda(), _labels(B, 2).cuda()
    counts = {}
    for cw in (None, [0.5, 2.0]):
        m = _model(p, bufs, C)
        step = FusedTrainStep(m, FlatAdam(m), B, T, use_graph=False, class_weight=cw)
        step(xt, yt)
        torch.cuda.synchronize()
        n0 = lib.mms_launch_count()
        step(xt, yt)
        torch.cuda.synchronize()
        counts[cw is None] = lib.mms_launch_count() - n0
    assert counts[True] == counts[False]


# ---- Trainer
EPOCH_RE = re.compile(r"训练损失: ([\d.]+) \|")


@pytest.mark.gpu
def test_trainer_use_class_weights_matches_cpu_replica(tmp_path):
    """Two epochs with use_class_weights = True (dropout 0, no shuffling): the logged training loss of every epoch
    against a CPU replica of the same batches through oracle/cpu_port.CpuTrainStep with the weighted loss ('balanced' weights)."""
    from sklearn.utils.class_weight import compute_class_weight
    from torch.utils.data import DataLoader
    from multimodalsignal_b200.trainer import Trainer
    g = torch.Generator().manual_seed(17)
    n_tr, n_va, Cc, T, bs = 150, 40, 3, 640, 64
    def mk(n):
        y = (torch.rand(n, generator=g) < 0.25).long()
        x = torch.randn(n, Cc, T, generator=g) + y[:, None, None].float() * torch.sin(torch.arange(T) / 7.0)
        return x, y
    (xtr, ytr), (xva, yva) = mk(n_tr), mk(n_va)
    model = _new_model(5)
    sd0 = {k: v.detach().clone() for k, v in model.state_dict().items()}
    tr = Trainer(model, tmp_path / "t", _cfg(2))
    tl = DataLoader(_TensorSet(xtr, ytr), batch_size=bs, shuffle=False)
    tr.train(tl, DataLoader(_TensorSet(xva, yva), batch_size=bs))
    ref_w = compute_class_weight('balanced', classes=np.arange(2), y=ytr.numpy())
    np.testing.assert_allclose(tr.class_weights, ref_w, rtol=1e-12)
    log = (tmp_path / "t" / "training_log.txt").read_text(encoding="utf-8")
    assert "Class weights ('balanced')" in log
    got = [float(v) for v in EPOCH_RE.findall(log)]
    p = {k: v.float() for k, v in sd0.items() if "running" not in k and "num_batches" not in k}
    bufs = {k: v.float() for k, v in sd0.items() if "running" in k}
    cpu = _weighted_cpu_step(p, bufs, ref_w, lr=1e-3, weight_decay=1e-4, dropout=0.0)
    ref = []
    for _ in range(2):
        s = 0.0
        for i in range(0, n_tr, bs):
            s += cpu(xtr[i:i + bs], ytr[i:i + bs]) * len(ytr[i:i + bs])
        ref.append(s / n_tr)
    assert len(got) == 2
    np.testing.assert_allclose(got, ref, atol=2e-3)
    # the test evaluation uses the weights too
    loss, _, _ = tr.evaluate(DataLoader(_TensorSet(xva, yva), batch_size=bs))
    model.eval()
    with torch.no_grad():
        lg = model(xva.cuda()).double().cpu()
    wt = torch.tensor(ref_w)
    exp = sum(len(yva[i:i + bs]) * F.cross_entropy(lg[i:i + bs], yva[i:i + bs], weight=wt).item() for i in range(0, n_va, bs)) / n_va
    assert abs(loss - exp) <= 1e-6 * abs(exp)


@pytest.mark.gpu
def test_trainer_refuses_missing_class_and_missing_labels(tmp_path):
    from torch.utils.data import DataLoader, TensorDataset
    from multimodalsignal_b200.trainer import Trainer
    x = torch.randn(8, 3, 640)
    tr = Trainer(_new_model(1), tmp_path / "a", _cfg(1))
    with pytest.raises(ValueError, match="class 1 has no training windows"):
        tr.train(DataLoader(_TensorSet(x, torch.zeros(8, dtype=torch.int64)), batch_size=4), None)
    tr = Trainer(_new_model(1), tmp_path / "b", _cfg(1))
    with pytest.raises(ValueError, match="no .labels"):
        tr.train(DataLoader(TensorDataset(x, torch.zeros(8, dtype=torch.int64)), batch_size=4), None)
