"""MC dropout (uncertainty.mc_dropout, mms_cnngru_mc_forward, mms_mc_accumulate) on a B200 against the float64 oracle.

The masks are exact: sample row r = b * samples + s draws the multipliers of row r of a training-mode forward of the
expanded batch (oracle/dropout_stream.py), so every sample is compared with ``model_oracle.forward`` of x repeated per
sample row, BatchNorm on its running statistics, with those masks.  |logit error| <= 1e-4 as elsewhere in the suite."""
import ctypes as C
import warnings

import numpy as np
import pytest
import torch

from oracle import dropout_stream as ds
from oracle import model_oracle as mo

pytestmark = pytest.mark.gpu

LOGIT_ATOL = 1e-4


def make_model(C_, nc=2, H=64, layers=2, attention=True, seed=0, p=0.5, O=32):
    """Random weights and random BatchNorm running statistics / affine parameters (eval BatchNorm is a non-trivial map)."""
    from multimodalsignal_b200.models import CnnGruAttentionModel
    torch.manual_seed(seed)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m = CnnGruAttentionModel(C_, nc, cnn_out_channels=O, gru_hidden_size=H, gru_num_layers=layers, dropout=p,
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


def make_x(B, C_, T, seed=1):
    return torch.randn(B, C_, T, generator=torch.Generator().manual_seed(seed))


def masks(m, R, T, seed, offset):
    L = ds.gru_seq_len(T)
    return (ds.gru_masks(R, L, m.gru_hidden_size, m.gru_num_layers, m.dropout_p, seed, offset),
            ds.head_mask(R, m.dropout_p, seed, offset))


def oracle_logits(m, x, samples, gru, head, windows_per_call=4):
    """float64 logits [B*samples, nc] of x repeated per sample row with the given masks; the rows are run a few windows at
    a time (each row depends on its own input and mask only)."""
    sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    params = {k: v.double() for k, v in sd.items() if "running" not in k and "num_batches" not in k}
    bn = {k: v.double() for k, v in sd.items() if "running" in k}
    xr = x.double().repeat_interleave(samples, dim=0)
    out = []
    step = windows_per_call * samples
    for r0 in range(0, xr.shape[0], step):
        sl = slice(r0, r0 + step)
        out.append(mo.forward(params, xr[sl], training=False, bn_buffers=bn, gru_layers=m.gru_num_layers,
                              drop_mask_gru=torch.from_numpy(gru[:, sl]) if len(gru) else None,
                              drop_mask_head=None if head is None else torch.from_numpy(head[sl]),
                              attention=m.attention, prune=True)[0])
    return torch.cat(out).numpy()


def stats_np(logits, samples):
    """probs, entropy, mutual information in float64 numpy from logits [B*samples, nc]."""
    lg = np.asarray(logits, dtype=np.float64)
    lg = lg.reshape(-1, samples, lg.shape[-1])
    e = np.exp(lg - lg.max(axis=2, keepdims=True))
    ps = e / e.sum(axis=2, keepdims=True)
    plogp = lambda q: np.where(q > 0, q * np.log(np.where(q > 0, q, 1.0)), 0.0)
    probs = ps.mean(axis=1)
    ent = -plogp(probs).sum(axis=1)
    return probs, ent, ent - (-plogp(ps).sum(axis=2)).mean(axis=1)


def run(m, x, samples, seed=1234, max_rows=2048):
    from multimodalsignal_b200.uncertainty import mc_dropout
    res = mc_dropout(m, x.cuda(), samples=samples, seed=seed, max_rows=max_rows)
    torch.cuda.synchronize()
    return res


# ---- every sample against the float64 oracle ----------------------------------------------------------------------------

CASES = [  # B, C, T, H, layers, nc, attention, samples
    (64, 6, 3840, 64, 2, 2, True, 32),       # the north-star shape: 2048 sample rows
    (7, 3, 336, 32, 1, 3, True, 5),          # 1 layer: only the head's mask varies
    (5, 8, 640, 128, 3, 8, False, 4),        # a middle layer on the sample rows
    (3, 6, 4040, 64, 2, 2, True, 7),         # T % 64 != 0
    (1, 14, 3840, 64, 2, 2, True, 1),
    (64, 6, 3840, 128, 2, 2, True, 32),
]

# cnn_out_channels O != 32: the per-window encoder workspace and the bottom layer's input projection (K = O)
CNN_WIDTH_CASES = [  # O, B, C, T, H, layers, nc, attention, samples
    (16, 8, 6, 3840, 64, 2, 3, True, 16),    # 128 sample rows
    (64, 6, 6, 3840, 64, 3, 5, True, 8),     # a middle layer on the sample rows
]


@pytest.mark.parametrize("B,C_,T,H,layers,nc,attention,samples", CASES)
def test_every_sample_matches_oracle(B, C_, T, H, layers, nc, attention, samples):
    _check_every_sample(B, C_, T, H, layers, nc, attention, samples)


@pytest.mark.parametrize("O,B,C_,T,H,layers,nc,attention,samples", CNN_WIDTH_CASES)
def test_every_sample_matches_oracle_other_cnn_widths(O, B, C_, T, H, layers, nc, attention, samples):
    _check_every_sample(B, C_, T, H, layers, nc, attention, samples, O=O)


def _check_every_sample(B, C_, T, H, layers, nc, attention, samples, O=32):
    m = make_model(C_, nc=nc, H=H, layers=layers, attention=attention, seed=B + T + H, O=O)
    x = make_x(B, C_, T, seed=B + layers)
    res = run(m, x, samples)
    assert res.offset == 0 and res.seed == 1234
    got = res.logits.reshape(B * samples, nc).cpu().numpy().astype(np.float64)
    gru, head = masks(m, B * samples, T, res.seed, res.offset)
    ref = oracle_logits(m, x, samples, gru, head)
    err = float(np.abs(got - ref).max())
    assert err <= LOGIT_ATOL, err
    if samples > 1:      # the samples of a window differ: dropout is on
        assert float(np.abs(np.diff(got.reshape(B, samples, nc), axis=1)).max()) > 1e-3
    # statistics: float64 formulas on the returned logits, and on the oracle's
    probs, ent, mi = (t.cpu().numpy() for t in (res.probs, res.entropy, res.mutual_info))
    rp, re_, rm = stats_np(got, samples)
    np.testing.assert_allclose(probs, rp, rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(ent, re_, rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(mi, rm, rtol=1e-12, atol=1e-14)
    op, oe, om = stats_np(ref, samples)
    for a, b in ((probs, op), (ent, oe), (mi, om)):
        assert float(np.abs(a - b).max()) <= 2e-4
    assert float(mi.min()) >= -1e-12
    assert torch.equal(res.prediction.cpu(), torch.argmax(res.probs, dim=1).cpu())
    assert res.probs.dtype == torch.float64 and res.logits.dtype == torch.float32 and res.prediction.dtype == torch.int64


# ---- chunking -----------------------------------------------------------------------------------------------------------

def test_chunking_gives_the_same_samples_and_statistics():
    B, samples = 11, 6
    m = make_model(6, nc=3, H=64, layers=3, seed=5)
    x = make_x(B, 6, 3840, seed=6)
    runs = [run(m, x, samples, max_rows=mr) for mr in (samples, 3 * samples + 1, B * samples)]
    bitwise = []
    for r in runs[:-1]:
        for a, b in ((r.logits, runs[-1].logits), (r.probs, runs[-1].probs), (r.entropy, runs[-1].entropy),
                     (r.mutual_info, runs[-1].mutual_info)):
            assert float((a.double() - b.double()).abs().max()) <= 1e-6
            bitwise.append(torch.equal(a, b))
    print(f"chunked results bit-identical: {all(bitwise)} ({sum(bitwise)}/{len(bitwise)})")
    # and the chunked call is still the oracle's
    gru, head = masks(m, B * samples, 3840, 1234, 0)
    ref = oracle_logits(m, x, samples, gru, head)
    assert float(np.abs(runs[0].logits.reshape(-1, 3).cpu().numpy() - ref).max()) <= LOGIT_ATOL


# ---- negative controls: the ids and the sharing are what the contract says ---------------------------------------------

def test_negative_controls_fail_the_oracle():
    B, samples, T = 5, 4, 3840
    m = make_model(6, nc=2, H=64, layers=2, seed=9)
    x = make_x(B, 6, T, seed=10)
    res = run(m, x, samples, max_rows=2 * samples)            # chunks of 2 windows: rows 8.. have a non-zero base
    got = res.logits.reshape(B * samples, 2).cpu().numpy()
    R, L, H = B * samples, ds.gru_seq_len(T), 64
    gru, head = masks(m, R, T, 1234, 0)
    assert float(np.abs(got - oracle_logits(m, x, samples, gru, head)).max()) <= LOGIT_ATOL

    def err(g, h):
        return float(np.abs(got - oracle_logits(m, x, samples, g, h)).max())

    # masks drawn with chunk-local rows (row0 ignored)
    n = 2 * samples
    local_g = np.concatenate([masks(m, n, T, 1234, 0)[0][:, :min(n, R - r0)] for r0 in range(0, R, n)], axis=1)
    local_h = np.concatenate([masks(m, n, T, 1234, 0)[1][:min(n, R - r0)] for r0 in range(0, R, n)], axis=0)
    assert err(local_g, local_h) > 1e-2
    g1, h1 = masks(m, R, T, 1234, 1)                          # offset + 1
    assert err(g1, h1) > 1e-2
    assert err(gru, None) > 1e-2                              # no head mask
    # the first site's rows per window instead of per sample row
    per_window = ds.gru_masks(B, L, H, 2, m.dropout_p, 1234, 0).repeat(samples, axis=1)
    assert err(per_window, head) > 1e-2


# ---- p = 0 --------------------------------------------------------------------------------------------------------------

def test_p0_samples_equal_the_eval_forward():
    B, samples = 9, 5
    for layers in (1, 2, 3):
        m = make_model(6, nc=3, H=64, layers=layers, seed=20 + layers, p=0.0)
        x = make_x(B, 6, 3840, seed=21).cuda()
        with torch.no_grad():
            ev = m(x).double()
        res = run(m, x, samples)
        diff = (res.logits.double() - ev[:, None, :]).abs().max().item()
        assert diff <= 1e-6, (layers, diff)
        assert float(res.mutual_info.abs().max()) <= 1e-12
        torch.testing.assert_close(res.probs, torch.softmax(res.logits[:, 0].double(), dim=1), rtol=1e-12, atol=1e-15)
        torch.testing.assert_close(res.probs, torch.softmax(ev, dim=1), rtol=0, atol=1e-6)


# ---- seeds --------------------------------------------------------------------------------------------------------------

def test_seeds():
    from multimodalsignal_b200.uncertainty import mc_dropout
    m = make_model(6, nc=2, seed=30)
    x = make_x(6, 6, 3840, seed=31).cuda()
    a, b = run(m, x, 8, seed=77), run(m, x, 8, seed=77)
    for f in ("logits", "probs", "entropy", "mutual_info", "prediction"):
        assert torch.equal(getattr(a, f), getattr(b, f)), f
    assert not torch.equal(run(m, x, 8, seed=78).logits, a.logits)
    calls = m._rng_calls
    c = mc_dropout(m, x, samples=8)
    assert m._rng_calls == calls + 1 and c.seed == m._rng_seed and c.offset == calls + 1
    d = mc_dropout(m, x, samples=8)
    assert d.offset == calls + 2 and not torch.equal(c.logits, d.logits)
    gru, head = masks(m, 48, 3840, c.seed, c.offset)
    assert float(np.abs(c.logits.reshape(48, 2).cpu().numpy() - oracle_logits(m, x.cpu(), 8, gru, head)).max()) <= LOGIT_ATOL


# ---- refusals and untouched state ---------------------------------------------------------------------------------------

def test_refusals():
    from multimodalsignal_b200 import _ext
    from multimodalsignal_b200.uncertainty import _McEngine, mc_dropout
    m = make_model(6, nc=2, seed=40)
    x = make_x(2, 6, 3840, seed=41)
    with pytest.raises(_ext.MmsError):
        mc_dropout(m, x, samples=4)                            # CPU tensor
    xc = x.cuda()
    with pytest.raises(ValueError):
        mc_dropout(m, xc, samples=4, max_rows=3)               # max_rows < samples
    with pytest.raises(ValueError):
        mc_dropout(m, xc, samples=0)
    with pytest.raises(ValueError):
        mc_dropout(m, xc[:, :3], samples=4)                    # wrong shape
    with pytest.raises(ValueError):
        mc_dropout(m, xc, samples=2 ** 23, max_rows=2 ** 23)  # 2 * 2^23 rows * L = 240 * 2H = 128 >= 2^38
    m.train()
    with pytest.raises(ValueError):
        mc_dropout(m, xc, samples=4)
    m.eval()
    # the C ABI: a row0 whose site-0 ids would reach the head site, and a row0 inside a window
    m._ensure_flat(xc.device)
    eng = _McEngine(m, 2, 3840, 4, xc.device)
    logits = torch.empty(8, 2, device="cuda")
    limit = (1 << 38) // (240 * 128)
    with pytest.raises(_ext.MmsError, match="2\\^38"):
        eng.forward(m, xc, 4, (limit // 4) * 4, 1, 0, logits)
    with pytest.raises(_ext.MmsError, match="window boundary"):
        eng.forward(m, xc, 4, 2, 1, 0, logits)
    eng.forward(m, xc, 4, 0, 1, 0, logits)                     # the same engine still works


def test_state_untouched():
    m = make_model(6, nc=2, seed=50)
    x = make_x(5, 6, 3840, seed=51)
    before = {k: v.detach().clone() for k, v in m.state_dict().items()}
    run(m, x, 6)
    for k, v in m.state_dict().items():
        assert torch.equal(v, before[k]), k
    assert not m.training


# ---- Trainer and main ---------------------------------------------------------------------------------------------------

def _trainer(tmp_path, m):
    from multimodalsignal_b200.main import trainer_config
    from multimodalsignal_b200.trainer import Trainer
    cfg = trainer_config()
    cfg['trainer']['quiet'] = True
    return Trainer(m, tmp_path, cfg)


def test_trainer_uncertainty_on_both_loader_types(tmp_path):
    from multimodalsignal_b200.dataset import DeviceBatchLoader
    from multimodalsignal_b200.uncertainty import auroc, mc_dropout
    m = make_model(3, nc=2, seed=60)
    x = make_x(23, 3, 3840, seed=61)
    y = torch.tensor([k % 2 for k in range(23)])

    class _DevDS:
        data, labels = x.cuda(), y.cuda()

        def __len__(self):
            return 23

    m.train()
    out = []
    for k, loader in enumerate((DeviceBatchLoader(_DevDS(), 8),
                                torch.utils.data.DataLoader(torch.utils.data.TensorDataset(x, y), batch_size=5))):
        d = tmp_path / str(k)
        out.append(_trainer(d, m).mc_dropout_uncertainty(loader, samples=6, max_rows=20))
        assert m.training                                      # the train / eval state is restored
        text = (d / "uncertainty.txt").read_text(encoding="utf-8")
        assert "auroc_entropy" in text and "ece_mc" in text
    a, b = out
    assert a.keys() == b.keys()
    for k in a:
        assert (np.isnan(a[k]) and np.isnan(b[k])) or a[k] == b[k], k
    m.eval()
    res = mc_dropout(m, x.cuda(), samples=6, seed=m._rng_seed, max_rows=20)
    wrong = (res.prediction.cpu() != y).numpy()
    assert a["accuracy"] == pytest.approx(1.0 - wrong.mean(), abs=1e-12)
    ent = res.entropy.cpu().numpy()
    assert a["mean_entropy"] == pytest.approx(ent.mean(), rel=1e-12)
    ref_auc = auroc(ent, wrong)
    assert (np.isnan(ref_auc) and np.isnan(a["auroc_entropy"])) or a["auroc_entropy"] == pytest.approx(ref_auc, abs=1e-12)
    assert 0.0 <= a["ece_mc"] <= 1.0 and 0.0 <= a["ece_eval"] <= 1.0


def test_run_fold_with_mc_dropout(tmp_path, monkeypatch):
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
    monkeypatch.setattr(main, "MC_DROPOUT_SAMPLES", 4)
    out = tmp_path / "run"
    res = drive(main.run_fold_async(0, "S2", out, ["chest_ECG", "chest_EDA", "chest_Resp"], quiet=True))
    u = res["uncertainty"]
    assert u["windows"] == 10 and u["samples"] == 4 and 0.0 <= u["accuracy"] <= 1.0
    assert (out / "fold_test_on_S2" / "uncertainty.txt").exists()
    path = main.write_uncertainty_summary(out, [res, dict(res, subject="S3")])
    lines = path.read_text(encoding="utf-8").splitlines()
    assert lines[1].startswith("accuracy\t")
