"""Gradient-norm clipping (``FlatAdam(max_grad_norm=...)``, ``Trainer`` ``grad_clip_norm``): torch's
``clip_grad_norm_`` (norm_type 2) between the backward and Adam.  On the host: the refusals and the descriptor layout.  On
a B200: the norm kernel, the clipped Adam kernels against ``clip_grad_norm_`` + ``torch.optim.Adam``, the fused step against
a CPU reference, the launches it adds, the data-parallel paths and ``Trainer``."""
import ctypes as C
import os
import re
import shutil
import subprocess
import sys
import warnings
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.nn.functional as F

ROOT = Path(__file__).resolve().parents[1]
ENCODER = ("channel_attention.", "cnn_encoder.")


def _model(C_in=6, **kw):
    from multimodalsignal_b200.models import CnnGruAttentionModel
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return CnnGruAttentionModel(C_in, 2, dropout=0.0, **kw)


# ------------------------------------------------------------------------------------------------------------ host only
@pytest.mark.parametrize("bad", [0, 0.0, -1.0, float("nan"), float("inf"), -float("inf"), "x", None])
def test_bad_max_norm_is_refused(bad):
    from multimodalsignal_b200.trainer import check_max_grad_norm
    with pytest.raises(ValueError):
        check_max_grad_norm(bad)


@pytest.mark.parametrize("norm_type", [1, 1.0, 3, float("inf"), "fro", None])
def test_other_norm_types_are_refused(norm_type):
    from multimodalsignal_b200.trainer import check_max_grad_norm
    with pytest.raises(NotImplementedError):
        check_max_grad_norm(1.0, norm_type)
    assert check_max_grad_norm(0.5, 2) == 0.5 and check_max_grad_norm(2, 2.0) == 2.0


def test_trainer_refuses_a_bad_setting_before_touching_the_fold_directory(tmp_path):
    from multimodalsignal_b200.trainer import Trainer
    cfg = {'trainer': {'epochs': 1, 'learning_rate': 1e-3, 'early_stopping': {'enabled': False, 'patience': 1, 'delta': 0},
                       'weight_decay': 0.0, 'grad_clip_norm': -1.0}}
    with pytest.raises(ValueError):
        Trainer(_model(), tmp_path / "fold", cfg)
    assert not (tmp_path / "fold").exists()


def test_main_passes_the_setting_through():
    from multimodalsignal_b200 import main
    assert main.GRAD_CLIP_NORM is None and main.trainer_config()['trainer']['grad_clip_norm'] is None


def test_descriptor_clip_fields_match_the_header(tmp_path):
    if shutil.which("gcc") is None:
        pytest.skip("gcc not on PATH")
    from multimodalsignal_b200 import _ext
    from multimodalsignal_b200._ext import CnnGruDesc
    fields = ["adam_nranges", "clip_max_norm", "clip_record", "clip_scratch"]
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "mms_b200.h"\nint main(void) {\n'
                   + "".join(f'  printf("%zu\\n", offsetof(mms_cnngru_desc, {f}));\n' for f in fields)
                   + '  printf("%zu\\n", sizeof(mms_cnngru_desc));\n  printf("%d\\n", MMS_GRAD_CLIP_SCRATCH_BYTES);\n  return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", str(ROOT / "include"), str(src), "-o", str(exe)], check=True)
    out = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert out[:-2] == [getattr(CnnGruDesc, f).offset for f in fields]
    assert out[-2] == C.sizeof(CnnGruDesc) and out[-1] == _ext.GRAD_CLIP_SCRATCH_BYTES


# ---------------------------------------------------------------------------------------------------------- on the B200
def _torch_coef(norm_f32, max_norm):
    """torch.nn.utils.clip_grad_norm_'s coefficient for a given fp32 total norm, on the GPU."""
    t = torch.tensor([norm_f32], dtype=torch.float32, device="cuda")
    return torch.clamp(max_norm / (t + 1e-6), max=1.0)


class _Clip:
    """The device state FlatAdam keeps, for the raw entry points."""

    def __init__(self, max_norm):
        from multimodalsignal_b200 import _ext
        self.max_norm = torch.tensor([max_norm], dtype=torch.float32, device="cuda")
        self.record = torch.zeros(5, dtype=torch.float64, device="cuda")
        self.scratch = torch.zeros(_ext.GRAD_CLIP_SCRATCH_BYTES // 4, dtype=torch.float32, device="cuda")

    def norm(self, g, table=None):
        from multimodalsignal_b200 import _ext
        from multimodalsignal_b200._ext import check, ptr, stream
        n = 0 if table is None else len(table) // 3
        check(_ext.lib().mms_grad_norm(ptr(g), g.numel(), table, n, ptr(self.max_norm), ptr(self.record), ptr(self.scratch), stream()))
        torch.cuda.synchronize()
        return self.scratch[0].item(), self.scratch[1:2].clone()


def _table(rows):
    return (C.c_int64 * (3 * len(rows)))(*[v for r in rows for v in (r[0], r[1], 0)])


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 3, 1021, 1025, 131077, 700003])
def test_norm_kernel_whole_buffer(n):
    g = torch.randn(n, generator=torch.Generator().manual_seed(n)).cuda() * 1e-2
    c = _Clip(0.7)
    norm, _ = c.norm(g)
    ref = g.double().norm().item()
    assert abs(norm - ref) <= 1e-6 * ref
    for _ in range(3):
        assert c.norm(g)[0] == norm                    # bit-reproducible


@pytest.mark.gpu
def test_norm_kernel_by_ranges_ignores_padding():
    """A range table over a buffer with garbage between the ranges gives the bits of the same elements packed contiguously."""
    rows = [(5, 100), (200, 37), (240, 1), (1000, 2001), (4000, 131077)]
    n = rows[-1][0] + rows[-1][1] + 9
    g = torch.full((n,), 1e30, device="cuda")
    pieces = [torch.randn(cnt, generator=torch.Generator().manual_seed(k)).cuda() for k, (_, cnt) in enumerate(rows)]
    for (off, cnt), p in zip(rows, pieces):
        g[off:off + cnt] = p
    packed = torch.cat(pieces)
    c = _Clip(1.0)
    norm_r, _ = c.norm(g, _table(rows))
    norm_p, _ = c.norm(packed)
    assert norm_r == norm_p
    ref = packed.double().norm().item()
    assert abs(norm_r - ref) <= 1e-6 * ref


@pytest.mark.gpu
def test_coefficient_is_torch_bit_for_bit_around_max_norm():
    max_norm = 0.7
    c = _Clip(max_norm)
    base = torch.randn(4099, generator=torch.Generator().manual_seed(0)).cuda()
    base = base / base.double().norm().float()
    for s in np.linspace(0.5, 2.0, 301):
        norm, coef = c.norm(base * float(s * max_norm))
        assert torch.equal(coef, _torch_coef(norm, max_norm)), (s, norm)
    rec = c.record.cpu().numpy()
    assert rec[4] == 301 and rec[3] == 0 and 0 < rec[2] < 301 and rec[1] <= 2.0 * max_norm * 1.0001


@pytest.mark.gpu
def test_non_finite_totals_behave_as_in_torch():
    c = _Clip(0.7)
    g = torch.randn(5000, generator=torch.Generator().manual_seed(1)).cuda()
    g[1234] = float("nan")
    norm, coef = c.norm(g)
    assert np.isnan(norm) and torch.isnan(coef).all()
    g[1234] = float("inf")
    norm, coef = c.norm(g)
    assert np.isinf(norm) and coef.item() == 0.0
    assert torch.equal(coef, _torch_coef(norm, 0.7))
    rec = c.record.cpu().numpy()
    assert rec[3] == 2 and rec[4] == 2 and rec[2] == 1 and rec[0] == 0.0


def _adam_state(n, seed):
    g = torch.Generator().manual_seed(seed)
    p = torch.randn(n, generator=g).cuda()
    grads = [torch.randn(n, generator=g).cuda() * 0.1 for _ in range(3)]
    return p, grads


@pytest.mark.gpu
@pytest.mark.parametrize("ranges", [False, True])
def test_clipped_adam_follows_clip_grad_norm_and_torch_adam(ranges):
    """Three updates on the GPU in fp32: mms_grad_norm + the clipped Adam against clip_grad_norm_ + torch.optim.Adam."""
    from multimodalsignal_b200 import _ext
    from multimodalsignal_b200._ext import check, ptr, stream
    lib = _ext.lib()
    n = 10007
    rows = [(3, 2000), (2100, 5), (4000, 6007)] if ranges else None
    p0, grads = _adam_state(n, 7)
    lr, wd, max_norm = 1e-3, 1e-4, 0.3
    p, m, v = p0.clone(), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    lr_dev = torch.tensor([lr], device="cuda")
    step, scratch = torch.zeros(1, dtype=torch.int64, device="cuda"), torch.zeros(1, dtype=torch.int32, device="cuda")
    steps = torch.zeros(3, dtype=torch.int64, device="cuda")
    c = _Clip(max_norm)
    coef = c.scratch[1:2]
    tref = [p0[o:o + k].clone().requires_grad_(True) for o, k in rows] if ranges else [p0.clone().requires_grad_(True)]
    opt = torch.optim.Adam(tref, lr=lr, weight_decay=wd)
    for g in grads:
        c.norm(g, _table(rows) if ranges else None)
        if ranges:
            t = (C.c_int64 * 9)(*[v for k, (o, cnt) in enumerate(rows) for v in (o, cnt, k)])
            check(lib.mms_adam_ranges_clip_step(ptr(p), ptr(g), ptr(m), ptr(v), t, 3, ptr(steps), ptr(lr_dev), 0.9, 0.999, 1e-8, wd,
                                                ptr(step), ptr(scratch), ptr(coef), stream()))
            for q, (o, cnt) in zip(tref, rows):
                q.grad = g[o:o + cnt].clone()
        else:
            check(lib.mms_adam_flat_clip_step(ptr(p), ptr(g), ptr(m), ptr(v), n, ptr(lr_dev), 0.9, 0.999, 1e-8, wd, ptr(step),
                                              ptr(scratch), ptr(coef), stream()))
            tref[0].grad = g.clone()
        tn = torch.nn.utils.clip_grad_norm_(tref, max_norm)
        opt.step()
        torch.cuda.synchronize()
        assert abs(c.scratch[0].item() - tn.item()) <= 1e-5 * tn.item()
        assert coef.item() < 1.0
    got = [p[o:o + k] for o, k in rows] if ranges else [p]
    for a, b in zip(got, tref):
        torch.testing.assert_close(a, b.detach(), rtol=1e-5, atol=1e-7)
    if ranges:                                   # elements outside the ranges are never touched
        assert torch.equal(p[:3], p0[:3]) and torch.equal(p[2005:2100], p0[2005:2100])


@pytest.mark.gpu
@pytest.mark.parametrize("ranges", [False, True])
def test_clipped_adam_with_coef_one_is_bit_identical_to_adam(ranges):
    from multimodalsignal_b200 import _ext
    from multimodalsignal_b200._ext import check, ptr, stream
    lib = _ext.lib()
    n = 70001
    p0, grads = _adam_state(n, 3)
    rows = [(0, 30000), (30016, 39985)]
    t = (C.c_int64 * 6)(0, 30000, 0, 30016, 39985, 1)

    def run(clip):
        p, m, v = p0.clone(), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
        lr = torch.tensor([1e-3], device="cuda")
        step, scratch = torch.zeros(1, dtype=torch.int64, device="cuda"), torch.zeros(1, dtype=torch.int32, device="cuda")
        steps = torch.zeros(2, dtype=torch.int64, device="cuda")
        c = _Clip(1e30)
        for g in grads:
            if clip:
                c.norm(g, _table(rows) if ranges else None)
                assert c.scratch[1].item() == 1.0
            a = (ptr(p), ptr(g), ptr(m), ptr(v))
            if ranges:
                tail = (t, 2, ptr(steps), ptr(lr), 0.9, 0.999, 1e-8, 1e-4, ptr(step), ptr(scratch))
                check(lib.mms_adam_ranges_clip_step(*a, *tail, ptr(c.scratch[1:2]), stream()) if clip else
                      lib.mms_adam_ranges_step(*a, *tail, stream()))
            else:
                tail = (n, ptr(lr), 0.9, 0.999, 1e-8, 1e-4, ptr(step), ptr(scratch))
                check(lib.mms_adam_flat_clip_step(*a, *tail, ptr(c.scratch[1:2]), stream()) if clip else
                      lib.mms_adam_flat_step(*a, *tail, stream()))
        torch.cuda.synchronize()
        return p, m, v

    for a, b in zip(run(False), run(True)):
        assert torch.equal(a, b)


# ---- the fused step against a CPU reference -------------------------------------------------------------------------
CONFIGS = {"default": dict(B=8, C=6, T=640, H=64, layers=2), "c3_t336": dict(B=8, C=3, T=336, H=64, layers=2),
           "h32_l1": dict(B=8, C=8, T=640, H=32, layers=1), "h128": dict(B=8, C=6, T=640, H=128, layers=2)}
PATTERNS = {"none": lambda n: False, "encoder_frozen": lambda n: n.startswith(ENCODER),
            "head_only": lambda n: not n.startswith("classifier.")}


def _setup(cfg, seed=0):
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
    x = torch.randn(cfg["B"], cfg["C"], cfg["T"], generator=g)
    y = torch.randint(0, 2, (cfg["B"],), generator=g)
    x[:, 0, :] += y[:, None].float()
    return m.cuda().train(), p, bufs, x, y


class _RefStep:
    """cpu_port.forward + F.cross_entropy + clip_grad_norm_ + torch.optim.Adam (fp32, CPU, dropout 0)."""

    def __init__(self, p, bufs, layers, max_norm, frozen=lambda n: False, weight=None):
        self.p = {k: v.clone().requires_grad_(v.numel() > 0 and not frozen(k)) for k, v in p.items()}
        self.bufs = {k: v.clone() for k, v in bufs.items()}
        self.layers, self.max_norm, self.weight = layers, max_norm, weight
        self.opt = torch.optim.Adam([v for v in self.p.values() if v.requires_grad], lr=1e-3, weight_decay=1e-4)

    def grad_norm(self, x, y):
        """The pre-clip norm of a step from the current state, without stepping (the BN buffers are left alone)."""
        from oracle import cpu_port
        bufs = {k: v.clone() for k, v in self.bufs.items()}
        logits = cpu_port.forward(self.p, bufs, x, training=True, dropout=0.0, layers=self.layers)
        F.cross_entropy(logits, y, weight=self.weight).backward()
        n = torch.linalg.vector_norm(torch.stack([v.grad.norm() for v in self.p.values() if v.grad is not None])).item()
        self.opt.zero_grad()
        return n

    def __call__(self, x, y):
        from oracle import cpu_port
        self.opt.zero_grad()
        logits = cpu_port.forward(self.p, self.bufs, x, training=True, dropout=0.0, layers=self.layers)
        F.cross_entropy(logits, y, weight=self.weight).backward()
        n = torch.nn.utils.clip_grad_norm_([v for v in self.p.values() if v.grad is not None], self.max_norm)
        self.opt.step()
        return float(n)


def _compare(m, ref, atol=5e-5):
    mine = m.state_dict()
    for n, v in ref.p.items():
        if v.numel():
            np.testing.assert_allclose(mine[n].cpu().numpy(), v.detach().numpy(), atol=atol, err_msg=n)
    for n, v in ref.bufs.items():
        np.testing.assert_allclose(mine[n].cpu().numpy(), v.numpy(), atol=2e-6, rtol=1e-5, err_msg=n)


@pytest.mark.gpu
@pytest.mark.parametrize("config,pattern,weighted", [("default", "none", False), ("c3_t336", "none", False), ("h32_l1", "none", False),
                                                     ("h128", "none", False), ("default", "encoder_frozen", False),
                                                     ("default", "head_only", False), ("default", "none", True)])
def test_fused_step_clips_like_torch(config, pattern, weighted):
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    cfg = CONFIGS[config]
    m, p, bufs, x, y = _setup(cfg)
    frozen = PATTERNS[pattern]
    for n, q in m.named_parameters():
        q.requires_grad_(not frozen(n))
    w = [0.7, 1.9] if weighted else None
    ref = _RefStep(p, bufs, cfg["layers"], 1.0, frozen, None if w is None else torch.tensor(w))
    ref.max_norm = max_norm = 0.1 * ref.grad_norm(x, y)
    opt = FlatAdam(m, lr=1e-3, weight_decay=1e-4, max_grad_norm=max_norm)
    step = FusedTrainStep(m, opt, batch=cfg["B"], seq_len=cfg["T"], class_weight=w)
    xc, yc = x.cuda(), y.cuda()
    got, want = [], []
    for _ in range(4):                 # eager, capture, two replays
        step(xc, yc)
        want.append(ref(x, y))
        torch.cuda.synchronize()
        got.append(opt.grad_norm.item())
        assert torch.equal(opt.clip_coef, _torch_coef(got[-1], max_norm))
    np.testing.assert_allclose(got, want, rtol=2e-4)
    assert all(n > max_norm for n in want)
    _compare(m, ref)
    rec = opt.clip_record.cpu().numpy()
    assert rec[4] == 4 and rec[2] == 4 and rec[3] == 0
    assert abs(rec[0] - sum(got)) <= 1e-6 * sum(got) and rec[1] == max(got)


@pytest.mark.gpu
def test_inactive_clipping_equals_the_unclipped_step():
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    cfg = CONFIGS["default"]
    out = []
    for clip in (None, 1e30):
        m, _, _, x, y = _setup(cfg, seed=4)
        opt = FlatAdam(m, lr=1e-3, weight_decay=1e-4, max_grad_norm=clip)
        step = FusedTrainStep(m, opt, batch=cfg["B"], seq_len=cfg["T"])
        for _ in range(3):
            step(x.cuda(), y.cuda())
        torch.cuda.synchronize()
        out.append(m.flat_parameters().clone())
        if clip:
            assert opt.clip_coef.item() == 1.0 and opt.clip_record[2].item() == 0 and opt.clip_record[4].item() == 3
    assert (out[0] - out[1]).abs().max().item() <= 1e-5


@pytest.mark.gpu
def test_set_max_grad_norm_between_replays_needs_no_recapture():
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    cfg = CONFIGS["default"]
    m, _, _, x, y = _setup(cfg, seed=2)
    opt = FlatAdam(m, max_grad_norm=1e30)
    step = FusedTrainStep(m, opt, batch=cfg["B"], seq_len=cfg["T"])
    xc, yc = x.cuda(), y.cuda()
    for _ in range(3):
        step(xc, yc)
    assert len(step._graphs) == 1
    torch.cuda.synchronize()
    assert opt.clip_coef.item() == 1.0
    small = 0.25 * opt.grad_norm.item()
    opt.set_max_grad_norm(small)
    step(xc, yc)
    torch.cuda.synchronize()
    assert len(step._graphs) == 1
    assert opt.clip_coef.item() < 1.0 and torch.equal(opt.clip_coef, _torch_coef(opt.grad_norm.item(), small))
    opt.set_max_grad_norm(None)                      # off again: the unclipped graph
    step(xc, yc)
    step(xc, yc)
    assert len(step._graphs) == 2


def _profile_names(lib):
    buf = C.create_string_buffer(1 << 16)
    assert lib.mms_profile_report(buf, len(buf)) == 0
    return [line.split()[0] for line in buf.value.decode().splitlines() if line.strip()]


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", ["none", "encoder_frozen"])
def test_clipping_adds_the_norm_kernel_and_swaps_adam(pattern):
    from multimodalsignal_b200 import _ext
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    lib = _ext.lib()
    cfg = dict(B=16, C=6, T=3840, H=64, layers=2)
    names = {}
    for clip in (None, 1.0):
        m, _, _, x, y = _setup(cfg, seed=9)
        for n, q in m.named_parameters():
            q.requires_grad_(not PATTERNS[pattern](n))
        step = FusedTrainStep(m, FlatAdam(m, max_grad_norm=clip), batch=16, seq_len=3840, use_graph=False)
        step(x.cuda(), y.cuda())
        lib.mms_profile_enable(1)
        step(x.cuda(), y.cuda())
        names[clip] = _profile_names(lib)
        lib.mms_profile_enable(0)
    adam = "adam_flat_kernel" if pattern == "none" else "adam_ranges_kernel"
    off, on = names[None], names[1.0]
    assert adam in off and "grad_norm_kernel" not in off and not any("clip" in n for n in off)
    assert [n for n in on if n not in ("grad_norm_kernel", adam.replace("_kernel", "_clip_kernel"))] == [n for n in off if n != adam]
    assert on.index("grad_norm_kernel") < on.index(adam.replace("_kernel", "_clip_kernel"))


# ---- data parallelism ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_emulated_ranks_with_clipping_equal_the_full_batch_step():
    from multimodalsignal_b200.parallel import DataParallelTrainStep, emulate_ranks
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    cfg = dict(B=16, C=6, T=640, H=64, layers=2)
    m0, _, _, x, y = _setup(cfg, seed=11)
    xc, yc = x.cuda(), y.cuda()
    opt0 = FlatAdam(m0, lr=1e-3, weight_decay=1e-4, max_grad_norm=0.05)
    fused = FusedTrainStep(m0, opt0, 16, 640, use_graph=False)
    ms = [_setup(cfg, seed=11)[0] for _ in range(2)]
    ranks = [DataParallelTrainStep(mm, FlatAdam(mm, lr=1e-3, weight_decay=1e-4, max_grad_norm=0.05), 8, 16, 640, rank=r)
             for r, mm in enumerate(ms)]
    for _ in range(3):
        fused(xc, yc)
        emulate_ranks(ranks, [(xc[:8], yc[:8]), (xc[8:], yc[8:])])
        torch.cuda.synchronize()
        assert opt0.clip_coef.item() < 1.0
        for s in ranks:
            assert abs(s.opt.grad_norm.item() - opt0.grad_norm.item()) <= 1e-4 * opt0.grad_norm.item()
    a = m0.flat_parameters()
    for mm in ms:
        assert (mm.flat_parameters() - a).abs().max().item() <= 2e-5


@pytest.mark.gpu
@pytest.mark.timeout(120)
@pytest.mark.parametrize("graph,pattern", [(False, "none"), (True, "none"), (True, "encoder_frozen")])
def test_peer_world_1_with_clipping_equals_the_fused_step(graph, pattern):
    from multimodalsignal_b200.parallel import DataParallelTrainStep, LocalPeers
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    cfg = dict(B=16, C=6, T=640, H=64, layers=2)

    def fresh():
        m, _, _, x, y = _setup(cfg, seed=12)
        for n, q in m.named_parameters():
            q.requires_grad_(not PATTERNS[pattern](n))
        return m, x.cuda(), y.cuda()

    m0, x, y = fresh()
    ref = FusedTrainStep(m0, FlatAdam(m0, lr=1e-3, weight_decay=1e-4, max_grad_norm=0.05), 16, 640, use_graph=False)
    m1, _, _ = fresh()
    st = DataParallelTrainStep(m1, FlatAdam(m1, lr=1e-3, weight_decay=1e-4, max_grad_norm=0.05), 16, 16, 640, rank=0,
                               peer=LocalPeers(1), use_graph=graph)
    for it in range(4):
        ref(x, y)
        st(x, y)
        torch.cuda.synchronize()
        assert abs(st.opt.grad_norm.item() - ref.opt.grad_norm.item()) <= 1e-5 * ref.opt.grad_norm.item(), it
        assert st.opt.clip_coef.item() < 1.0
    st.check_peers()
    assert int(st.norm_epoch.item()) == 4 and int(st.epoch.item()) == 20
    assert st.opt.clip_record[4].item() == 4
    np.testing.assert_allclose(m1.flat_parameters().cpu().numpy(), m0.flat_parameters().cpu().numpy(), atol=2e-6)


@pytest.mark.gpu
@pytest.mark.timeout(120)
@pytest.mark.skipif(os.environ.get("MMS_TEST_PEER_EMULATION") != "1",
                    reason="several emulated ranks spin on each other's flags on ONE GPU; runs only with MMS_TEST_PEER_EMULATION=1 "
                           "(tests/test_gpu_parallel.py)")
def test_peer_emulated_ranks_with_clipping_equal_the_full_batch_step():
    from multimodalsignal_b200 import _ext
    from multimodalsignal_b200.parallel import DataParallelTrainStep, LocalPeers, emulate_peer_ranks
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    cfg = dict(B=16, C=6, T=640, H=64, layers=2)
    m0, _, _, x, y = _setup(cfg, seed=13)
    xc, yc = x.cuda(), y.cuda()
    ref = FusedTrainStep(m0, FlatAdam(m0, lr=1e-3, weight_decay=1e-4, max_grad_norm=0.05), 16, 640, use_graph=False)
    _ext.lib().mms_set_side_streams(0)
    try:
        peers, streams, ms, steps = LocalPeers(2), [torch.cuda.Stream() for _ in range(2)], [], []
        for r in range(2):
            with torch.cuda.stream(streams[r]):
                mm = _setup(cfg, seed=13)[0]
                ms.append(mm)
                steps.append(DataParallelTrainStep(mm, FlatAdam(mm, lr=1e-3, weight_decay=1e-4, max_grad_norm=0.05), 8, 16, 640, rank=r,
                                                   peer=peers, use_graph=False))
        torch.cuda.synchronize()
        for _ in range(3):
            ref(xc, yc)
            emulate_peer_ranks(steps, [(xc[:8], yc[:8]), (xc[8:], yc[8:])], streams)
            torch.cuda.synchronize()
        for s in steps:
            s.check_peers()
    finally:
        _ext.lib().mms_set_side_streams(1)
    assert steps[0].opt.grad_norm.item() == steps[1].opt.grad_norm.item()
    assert torch.equal(ms[0].flat_parameters(), ms[1].flat_parameters())
    assert (ms[0].flat_parameters() - m0.flat_parameters()).abs().max().item() <= 1e-4


@pytest.mark.gpu
def test_peer_memory_exchange_with_clipping_two_gpus():
    """Symmetric memory over NVLink, one process per GPU: the parameters stay bit-identical on both ranks (skipped on one GPU)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29643", str(ROOT / "tools" / "dp_check.py"), "--peer", "--clip"],
                       capture_output=True, text=True, timeout=600, env=dict(os.environ))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "dp_check ok" in r.stdout


# ---- Trainer ---------------------------------------------------------------------------------------------------------
class _DevDS:
    def __init__(self, x, y):
        self.data, self.labels = x, y

    def __len__(self):
        return int(self.data.shape[0])


EPOCH_LINE = re.compile(r"^Epoch \d+/\d+ \| 耗时: [\d.]+s \| 训练损失: [-\d.naif]+ \| 验证损失: [-\d.naif]+ \| 验证Acc: [\d.]+ \| 验证F1: [\d.]+$")


@pytest.mark.gpu
@pytest.mark.parametrize("device_loader", [True, False])
def test_trainer_clips_logs_and_matches_a_hand_driven_loop(tmp_path, device_loader):
    from torch.utils.data import DataLoader, TensorDataset
    from multimodalsignal_b200.dataset import DeviceBatchLoader
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep, Trainer
    g = torch.Generator().manual_seed(1)
    x = torch.randn(96, 3, 640, generator=g)
    y = torch.randint(0, 2, (96,), generator=g)
    x[:, 0, :] += y[:, None].float()
    torch.manual_seed(0)
    m = _model(3)
    init = {k: v.detach().clone() for k, v in m.state_dict().items()}
    max_norm = 0.05
    cfg = {'trainer': {'epochs': 2, 'learning_rate': 1e-3, 'early_stopping': {'enabled': False, 'patience': 20, 'delta': 0},
                       'weight_decay': 1e-4, 'quiet': True, 'grad_clip_norm': max_norm}}
    tr = Trainer(m, tmp_path / "fold", cfg)
    if device_loader:
        tl = DeviceBatchLoader(_DevDS(x.cuda(), y.cuda()), 32, shuffle=False)
        vl = DeviceBatchLoader(_DevDS(x.cuda(), y.cuda()), 32, shuffle=False)
    else:
        tl = DataLoader(TensorDataset(x, y), batch_size=32, shuffle=False)
        vl = DataLoader(TensorDataset(x, y), batch_size=32, shuffle=False)
    tr.train(tl, vl)
    lines = (tmp_path / "fold" / "training_log.txt").read_text(encoding="utf-8").splitlines()
    clip_lines = [l for l in lines if l.startswith("Gradient norm before clipping")]
    assert len(clip_lines) == 2 and not any(l.startswith("Warning") for l in lines)
    # the same six steps by hand, with the norms read after every step
    m2 = _model(3)
    m2.load_state_dict(init)
    m2 = m2.cuda().train()
    opt = FlatAdam(m2, lr=1e-3, weight_decay=1e-4, max_grad_norm=max_norm)
    step = FusedTrainStep(m2, opt, 32, 640)
    norms = []
    for _ in range(2):
        for i in range(0, 96, 32):
            step(x[i:i + 32].cuda(), y[i:i + 32].cuda())
            torch.cuda.synchronize()
            norms.append(opt.grad_norm.item())
    np.testing.assert_allclose(m.flat_parameters().cpu().numpy(), m2.flat_parameters().cpu().numpy(), atol=1e-5)
    for e, line in enumerate(clip_lines):
        mean, mx, k, n = re.match(r"Gradient norm before clipping: mean ([\d.]+) \| max ([\d.]+) \| clipped (\d+) of (\d+) steps$",
                                  line).groups()
        ep = norms[3 * e:3 * e + 3]
        assert int(n) == 3 and int(k) == sum(v > max_norm for v in ep)
        assert abs(float(mean) - np.mean(ep)) <= 1e-4 + 1e-3 * np.mean(ep) and abs(float(mx) - max(ep)) <= 1e-4 + 1e-3 * max(ep)


@pytest.mark.gpu
def test_trainer_without_clipping_logs_what_it_did(tmp_path):
    from torch.utils.data import DataLoader, TensorDataset
    from multimodalsignal_b200.trainer import Trainer
    g = torch.Generator().manual_seed(2)
    x = torch.randn(64, 3, 640, generator=g)
    y = torch.randint(0, 2, (64,), generator=g)
    cfg = {'trainer': {'epochs': 2, 'learning_rate': 1e-3, 'early_stopping': {'enabled': False, 'patience': 20, 'delta': 0},
                       'weight_decay': 1e-4, 'quiet': True, 'grad_clip_norm': None}}
    tr = Trainer(_model(3), tmp_path / "fold", cfg)
    assert tr.optimizer.max_grad_norm is None
    tr.train(DataLoader(TensorDataset(x, y), batch_size=32), DataLoader(TensorDataset(x, y), batch_size=32))
    lines = (tmp_path / "fold" / "training_log.txt").read_text(encoding="utf-8").splitlines()
    assert not any("Gradient norm" in l or l.startswith("Warning") for l in lines)
    epoch = [l for l in lines if l.startswith("Epoch ")]
    assert len(epoch) == 2 and all(EPOCH_LINE.match(l) for l in epoch), epoch
    assert lines[2:4] == epoch and lines[4].startswith("--- 训练完成 --- 总训练时长: ") and len(lines) == 5
