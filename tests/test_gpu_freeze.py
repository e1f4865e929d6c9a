"""Fine-tuning with frozen parameters (``requires_grad_(False)``): the mask / range helper and the descriptor layout on
the host, then on a B200 the fused training step against torch's per-parameter Adam (oracle/cpu_port.CpuTrainStep with
the same leaves frozen), the masked backward, the launches a freeze pattern removes, ``Trainer`` and the data-parallel
paths."""
import ctypes as C
import shutil
import subprocess
import warnings
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parents[1]

ENCODER = ("channel_attention.", "cnn_encoder.")


def _model(C_in=6, **kw):
    from multimodalsignal_b200.models import CnnGruAttentionModel
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return CnnGruAttentionModel(C_in, 2, dropout=0.0, **kw)


def _plan(m, frozen):
    names = [n for n, _ in m.named_parameters()]
    return m.freeze_plan([not frozen(n) for n in names])


# ------------------------------------------------------------------------------------------------------------ host only
def test_freeze_plan_default_model():
    m = _model()
    names = [n for n, _ in m.named_parameters()]
    assert len(m.state_dict()) == 34 and len(names) == 28
    layout, _ = m.flat_layout()
    assert m.freeze_plan() == (0, tuple((off, n, i) for i, (_, off, n, _) in enumerate(layout)))
    # encoder frozen: segments 0-7
    mask, ranges = _plan(m, lambda n: n.startswith(ENCODER))
    assert mask == 0xFF and [r[2] for r in ranges] == list(range(8, 28))
    # head only: everything but the last four segments (8 + 4*2 .. 8 + 4*2 + 3)
    mask, ranges = _plan(m, lambda n: not n.startswith("classifier."))
    assert mask == (1 << 16) - 1 and [r[2] for r in ranges] == [24, 25, 26, 27]
    # one GRU direction frozen: the segment still computes its gradient, the range of the frozen half is left out
    mask, ranges = _plan(m, lambda n: n == "gru.weight_ih_l0")
    assert mask == 0
    by = {name: (off, n) for name, off, n, _ in layout}
    assert by["gru.weight_ih_l0"] not in [r[:2] for r in ranges] and by["gru.weight_ih_l0_reverse"] in [r[:2] for r in ranges]
    mask, _ = _plan(m, lambda n: n.startswith("gru.weight_ih_l0"))
    assert mask == 1 << 8
    mask, ranges = _plan(m, lambda n: True)
    assert mask == (1 << 20) - 1 and ranges == ()


def test_freeze_plan_small_and_c3_models():
    m = _model(8, gru_hidden_size=32, gru_num_layers=1)
    # the forward direction of the only GRU layer frozen: its four segments keep their gradients (the reverse halves train)
    mask, ranges = _plan(m, lambda n: n.startswith(ENCODER) or n.endswith("_l0"))
    assert mask == 0xFF
    assert [r[2] for r in ranges] == [i for i, (n, _) in enumerate(m.named_parameters()) if not n.startswith(ENCODER) and not n.endswith("_l0")]
    assert _plan(m, lambda n: n.startswith(ENCODER) or "_l0" in n)[0] == (1 << 12) - 1
    # C = 3: the attention weights are empty; they never count as frozen or as ranges
    m3 = _model(3)
    assert m3.freeze_plan()[0] == 0
    assert all(r[1] > 0 for r in m3.freeze_plan()[1])
    assert _plan(m3, lambda n: n.startswith("cnn_encoder."))[0] == 0xFC     # segments 0-1 hold nothing
    assert _plan(m3, lambda n: n.startswith(ENCODER))[0] == 0xFC


def test_descriptor_layout_matches_ctypes(tmp_path):
    if shutil.which("gcc") is None:
        pytest.skip("gcc not on PATH")
    from multimodalsignal_b200._ext import CnnGruDesc
    fields = ["frozen_segments", "adam_ranges_host", "adam_steps", "adam_nranges", "class_weight", "global_batch"]
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "mms_b200.h"\nint main(void) {\n'
                   + "".join(f'  printf("%zu\\n", offsetof(mms_cnngru_desc, {f}));\n' for f in fields)
                   + '  printf("%zu\\n", sizeof(mms_cnngru_desc));\n  printf("%d\\n", MMS_MAX_ADAM_RANGES);\n  return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", str(ROOT / "include"), str(src), "-o", str(exe)], check=True)
    out = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    from multimodalsignal_b200 import _ext
    assert out[:-2] == [getattr(CnnGruDesc, f).offset for f in fields]
    assert out[-2] == C.sizeof(CnnGruDesc) and out[-1] == _ext.MAX_ADAM_RANGES


# ---------------------------------------------------------------------------------------------------------- on the B200
PATTERNS = {
    "head_only": lambda n, top: not n.startswith("classifier."),
    "top_and_head": lambda n, top: not (n.startswith("classifier.") or (n.startswith("gru.") and f"_l{top}" in n)),
    "encoder_frozen": lambda n, top: n.startswith(ENCODER),
    "encoder_only": lambda n, top: not n.startswith(ENCODER),
    "bn_affine_frozen": lambda n, top: n.startswith(("cnn_encoder.1.", "cnn_encoder.5.")),
    "ih_l0_forward_frozen": lambda n, top: n == "gru.weight_ih_l0",
    "all_frozen": lambda n, top: True,
}
CONFIGS = {"default": dict(B=8, C=6, T=640, H=64, layers=2), "c3_t336": dict(B=8, C=3, T=336, H=64, layers=2),
           "h32_l1": dict(B=8, C=8, T=640, H=32, layers=1)}


def _setup(cfg, seed=0):
    """The same random state as a GPU model and as the CPU port (dropout 0), plus one batch."""
    from oracle import cpu_port
    p, bufs = cpu_port.make_state(C=cfg["C"], H=cfg["H"], layers=cfg["layers"], seed=seed)
    g = torch.Generator().manual_seed(seed + 100)
    for k in ("cnn_encoder.1", "cnn_encoder.5"):
        p[f"{k}.weight"] = p[f"{k}.weight"] + 0.1 * torch.randn(p[f"{k}.weight"].shape, generator=g)
        p[f"{k}.bias"] = p[f"{k}.bias"] + 0.1 * torch.randn(p[f"{k}.bias"].shape, generator=g)
    m = _model(cfg["C"], gru_hidden_size=cfg["H"], gru_num_layers=cfg["layers"])
    sd = dict(p)
    sd.update(bufs)
    sd["cnn_encoder.1.num_batches_tracked"] = torch.zeros((), dtype=torch.int64)
    sd["cnn_encoder.5.num_batches_tracked"] = torch.zeros((), dtype=torch.int64)
    m.load_state_dict(sd, strict=True)
    m = m.cuda().train()
    ref = cpu_port.CpuTrainStep(p, bufs, lr=1e-3, weight_decay=1e-4, dropout=0.0, layers=cfg["layers"])
    x = torch.randn(cfg["B"], cfg["C"], cfg["T"], generator=g)
    y = torch.randint(0, 2, (cfg["B"],), generator=g)
    x[:, 0, :] += y[:, None].float()
    return m, ref, x, y


def _freeze(m, ref, pattern, top):
    for n, q in m.named_parameters():
        f = pattern(n, top)
        q.requires_grad_(not f)
        if ref.p[n].numel():
            ref.p[n].requires_grad_(not f)


def _ref_step(ref, x, y):
    """CpuTrainStep; with every parameter frozen torch has nothing to differentiate: the forward alone (BN statistics)."""
    from oracle import cpu_port
    if any(v.requires_grad for v in ref.p.values()):
        ref(x, y)
        return
    with torch.no_grad():
        cpu_port.forward(ref.p, ref.bufs, x, training=True, dropout=0.0, layers=ref.layers, attention=ref.attention)


def _compare(m, ref, init, pattern, top):
    mine = m.state_dict()
    for n, v in ref.p.items():
        got = mine[n].cpu()
        if v.numel() == 0:
            continue
        if pattern(n, top):
            assert torch.equal(got, init[n]), f"frozen {n} moved"
        else:
            np.testing.assert_allclose(got.numpy(), v.detach().numpy(), atol=5e-5, err_msg=n)
    for n, v in ref.bufs.items():
        np.testing.assert_allclose(mine[n].cpu().numpy(), v.numpy(), atol=2e-6, rtol=1e-5, err_msg=n)


@pytest.mark.gpu
@pytest.mark.parametrize("config", list(CONFIGS))
@pytest.mark.parametrize("pattern", list(PATTERNS))
def test_fused_step_with_frozen_parameters_follows_torch_adam(pattern, config):
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    cfg = CONFIGS[config]
    top = cfg["layers"] - 1
    m, ref, x, y = _setup(cfg)
    pat = PATTERNS[pattern]
    _freeze(m, ref, pat, top)
    init = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    opt = FlatAdam(m, lr=1e-3, weight_decay=1e-4)
    step = FusedTrainStep(m, opt, batch=cfg["B"], seq_len=cfg["T"])
    xc, yc = x.cuda(), y.cuda()
    for _ in range(4):                 # eager, capture, two replays
        step(xc, yc)
        _ref_step(ref, x, y)
    torch.cuda.synchronize()
    _compare(m, ref, init, pat, top)


@pytest.mark.gpu
def test_progressive_unfreezing_keeps_per_tensor_step_counts():
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    cfg = CONFIGS["default"]
    m, ref, x, y = _setup(cfg, seed=3)
    enc = PATTERNS["encoder_frozen"]
    _freeze(m, ref, enc, 1)
    opt = FlatAdam(m, lr=1e-3, weight_decay=1e-4)
    step = FusedTrainStep(m, opt, batch=cfg["B"], seq_len=cfg["T"])
    xc, yc = x.cuda(), y.cuda()
    for _ in range(3):
        step(xc, yc)
        _ref_step(ref, x, y)
    _freeze(m, ref, lambda n, top: False, 1)
    for _ in range(3):
        step(xc, yc)
        _ref_step(ref, x, y)
    torch.cuda.synchronize()
    _compare(m, ref, None, lambda n, top: False, 1)
    steps = opt.tensor_steps.cpu().tolist()
    names = [n for n, _ in m.named_parameters()]
    assert [s for s, n in zip(steps, names) if n.startswith(ENCODER) and m.state_dict()[n].numel()] == [3] * 8
    assert all(s == 6 for s, n in zip(steps, names) if not n.startswith(ENCODER))
    assert int(opt.step_dev.item()) == 6


def _profile_names(lib):
    buf = C.create_string_buffer(1 << 16)
    assert lib.mms_profile_report(buf, len(buf)) == 0
    return [line.split()[0] for line in buf.value.decode().splitlines() if line.strip()]


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", ["encoder_frozen", "head_only", "bn_affine_frozen", "ih_l0_forward_frozen", "encoder_only"])
def test_masked_backward_leaves_frozen_slots_and_skips_launches(pattern):
    from multimodalsignal_b200 import _ext
    from multimodalsignal_b200._ext import check, ptr, stream
    B, Cc, T = 16, 6, 3840            # B*L = 3840 rows: the tensor-core products and the fused encoder kernels
    m, _, x, y = _setup(dict(B=B, C=Cc, T=T, H=64, layers=2), seed=5)
    lib = _ext.lib()
    xc = x.cuda()
    flat = m.flat_parameters()
    eng = m.engine(B, T, True, True, xc.device)
    dl = torch.randn(B, 2, device="cuda") / B
    mask, ranges = _plan(m, lambda n: PATTERNS[pattern](n, 1))
    offs, sizes, total = m._layout()
    frozen_idx = torch.zeros(total, dtype=torch.bool)
    for s in range(len(offs)):
        if (mask >> s) & 1:
            frozen_idx[offs[s]:offs[s] + sizes[s]] = True

    def run(msk, sentinel, profile=False):
        eng.forward(xc, 7)
        torch.cuda.synchronize()
        lib.mms_profile_enable(1 if profile else 0)       # the backward's launches only
        g = torch.where(frozen_idx.cuda(), torch.full_like(flat, sentinel), torch.zeros_like(flat)) if msk else torch.zeros_like(flat)
        eng.desc.frozen_segments = msk
        try:
            check(lib.mms_cnngru_backward(C.byref(eng.desc), ptr(xc), ptr(flat), ptr(m._bn_flat), ptr(eng.workspace), ptr(dl),
                                          ptr(g), None, stream()))
        finally:
            eng.desc.frozen_segments = 0
        torch.cuda.synchronize()
        return g

    full = run(0, 0.0)
    masked = run(mask, 1234.5, profile=True)
    names = _profile_names(lib)
    lib.mms_profile_enable(0)
    fi = frozen_idx.cuda()
    assert bool((masked[fi] == 1234.5).all())
    tr = ~fi
    scale = full[tr].abs().max().item()
    assert (masked[tr] - full[tr]).abs().max().item() <= 1e-5 * max(scale, 1e-6)
    enc_bwd = ("conv2_bwd_kernel", "conv1_bwd_kernel", "pool_bwd_tm_kernel", "pool_bwd_ncl_kernel", "wgrad_reduce_kernel")
    if pattern in ("encoder_frozen", "head_only"):
        assert not any(n.startswith(enc_bwd) for n in names), names
    if pattern == "head_only":
        assert not any("gru_bwd" in n for n in names), names
        assert not any("gemm" in n for n in names), names


@pytest.mark.gpu
def test_nothing_frozen_launches_what_it_did():
    """With every parameter trainable the step takes the whole-buffer Adam and no mask: the launch sequence of a step is the
    same as that of a descriptor without the new fields."""
    from multimodalsignal_b200 import _ext
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    cfg = dict(B=16, C=6, T=3840, H=64, layers=2)
    m, _, x, y = _setup(cfg, seed=9)
    opt = FlatAdam(m)
    step = FusedTrainStep(m, opt, batch=16, seq_len=3840, use_graph=False)
    lib = _ext.lib()
    step(x.cuda(), y.cuda())
    assert step.desc.frozen_segments == 0 and not step.desc.adam_steps and step.desc.adam_nranges == 0
    lib.mms_profile_enable(1)
    step(x.cuda(), y.cuda())
    names = _profile_names(lib)
    lib.mms_profile_enable(0)
    assert "adam_flat_kernel" in names and "adam_ranges_kernel" not in names


class _DevDS:
    def __init__(self, x, y):
        self.data, self.labels = x, y

    def __len__(self):
        return int(self.data.shape[0])


@pytest.mark.gpu
@pytest.mark.parametrize("device_loader", [True, False])
def test_trainer_keeps_frozen_encoder_and_unfreezes(tmp_path, device_loader):
    from torch.utils.data import DataLoader, TensorDataset
    from multimodalsignal_b200.dataset import DeviceBatchLoader
    from multimodalsignal_b200.trainer import Trainer
    torch.manual_seed(0)
    m = _model(3)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(96, 3, 640, generator=g)
    y = torch.randint(0, 2, (96,), generator=g)
    x[:, 0, :] += y[:, None].float()
    for n, p in m.named_parameters():
        p.requires_grad_(not n.startswith(ENCODER))
    init = {k: v.detach().clone() for k, v in m.state_dict().items()}
    cfg = {'trainer': {'epochs': 2, 'learning_rate': 1e-3, 'early_stopping': {'enabled': True, 'patience': 20, 'delta': 0},
                       'weight_decay': 1e-4, 'quiet': True}}
    tr = Trainer(m, tmp_path / "fold", cfg)
    if device_loader:
        tl = DeviceBatchLoader(_DevDS(x.cuda(), y.cuda()), 32, shuffle=True)
        vl = DeviceBatchLoader(_DevDS(x.cuda(), y.cuda()), 32, shuffle=False)
    else:
        tl = DataLoader(TensorDataset(x, y), batch_size=32, shuffle=True)
        vl = DataLoader(TensorDataset(x, y), batch_size=32, shuffle=False)
    tr.train(tl, vl)
    log = (tmp_path / "fold" / "training_log.txt").read_text(encoding="utf-8")
    n_train = sum(p.numel() for n, p in m.named_parameters() if not n.startswith(ENCODER))
    assert f"Trainable parameters: {n_train} of " in log
    best = torch.load(tmp_path / "fold" / "best_model.pt", weights_only=True)
    for k, v in best.items():
        if k.startswith(ENCODER) and "running" not in k and "num_batches" not in k:
            assert torch.equal(v, init[k].cpu()), k
    assert any(not torch.equal(best[k], init[k].cpu()) for k in best if k.startswith("classifier."))
    for p in m.parameters():
        p.requires_grad_(True)
    tr.train(tl, vl)
    now = m.state_dict()
    assert not torch.equal(now["cnn_encoder.0.weight"].cpu(), init["cnn_encoder.0.weight"].cpu())


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", ["encoder_frozen", "head_only"])
def test_data_parallel_paths_with_frozen_parameters(pattern):
    from multimodalsignal_b200.parallel import DataParallelTrainStep, LocalPeers, emulate_peer_ranks, emulate_ranks
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    cfg = dict(B=16, C=6, T=640, H=64, layers=2)
    pat = PATTERNS[pattern]

    def fresh():
        m, _, x, y = _setup(cfg, seed=11)
        for n, p in m.named_parameters():
            p.requires_grad_(not pat(n, 1))
        return m, x.cuda(), y.cuda()

    m0, x, y = fresh()
    init = {k: v.detach().clone() for k, v in m0.state_dict().items()}
    fused = FusedTrainStep(m0, FlatAdam(m0), 16, 640, use_graph=False)
    for _ in range(2):
        fused(x, y)
    # world-1 peer path (the whole batch on one rank)
    m1, _, _ = fresh()
    st = DataParallelTrainStep(m1, FlatAdam(m1), 16, 16, 640, rank=0, peer=LocalPeers(1), use_graph=False)
    for _ in range(2):
        emulate_peer_ranks([st], [(x, y)], [torch.cuda.current_stream()])
    # two ranks, NCCL-style exchange emulated in one process
    m2a, _, _ = fresh()
    m2b, _, _ = fresh()
    ranks = [DataParallelTrainStep(mm, FlatAdam(mm), 8, 16, 640, rank=r) for r, mm in enumerate((m2a, m2b))]
    for _ in range(2):
        emulate_ranks(ranks, [(x[:8], y[:8]), (x[8:], y[8:])])
    torch.cuda.synchronize()
    a, b, c = m0.state_dict(), m1.state_dict(), m2a.state_dict()
    for n, _ in m0.named_parameters():
        if pat(n, 1):
            assert torch.equal(b[n], init[n]) and torch.equal(c[n], init[n]), n
        else:
            np.testing.assert_allclose(b[n].cpu().numpy(), a[n].cpu().numpy(), atol=2e-6, err_msg=n)
            np.testing.assert_allclose(c[n].cpu().numpy(), a[n].cpu().numpy(), atol=1e-4, err_msg=n)
