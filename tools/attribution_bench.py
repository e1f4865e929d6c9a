"""Integrated-gradients timings on one GPU, recorded with the card's name and power limit from the same run.

(a) IG per attributed window: ``attribution.integrated_gradients`` (eval forward + ``mms_cnngru_input_gradient`` per chunk)
    against the same IG through stock PyTorch / cuDNN in strict fp32 -- the reference model restated with torch.nn modules,
    BatchNorm in eval mode, the GRU in train mode with dropout 0 (cuDNN's RNN backward refuses eval mode) and
    ``torch.autograd.grad`` over the same chunks, with frozen parameters.
(b) ``mms_cnngru_input_gradient`` against ``mms_cnngru_backward`` after the same eval forward, alternated.
(c) with ``--parent DIR``: ``bench.py`` of DIR (an older checkout, already built) and of this tree, alternated.

    python tools/attribution_bench.py [--parent DIR] [--out profiles/attribution_bench.json]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
import warnings
from pathlib import Path

import torch
import torch.nn as nn

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    idx = torch.cuda.current_device()
    lines = q.stdout.strip().splitlines()
    return lines[idx].strip() if idx < len(lines) else q.stdout.strip()


class _RefAttention(nn.Module):
    def __init__(self, C):
        super().__init__()
        self.avg_pool = nn.AdaptiveAvgPool1d(1)
        self.fc = nn.Sequential(nn.Linear(C, C // 4, bias=False), nn.ReLU(inplace=True), nn.Linear(C // 4, C, bias=False),
                                nn.Sigmoid())

    def forward(self, x):
        b, c, _ = x.size()
        y = self.avg_pool(x).view(b, c)
        return x * self.fc(y).view(b, c, 1)


class RefModel(nn.Module):
    """The reference CnnGruAttentionModel in stock torch.nn modules (same state_dict keys)."""

    def __init__(self, C, nc, O=32, H=64, layers=2):
        super().__init__()
        self.channel_attention = _RefAttention(C)
        self.cnn_encoder = nn.Sequential(
            nn.Conv1d(C, 16, 7, 2, 3, bias=False), nn.BatchNorm1d(16), nn.ReLU(), nn.MaxPool1d(3, 2, 1),
            nn.Conv1d(16, O, 5, 2, 2, bias=False), nn.BatchNorm1d(O), nn.ReLU(), nn.MaxPool1d(3, 2, 1))
        self.gru = nn.GRU(O, H, layers, batch_first=True, bidirectional=True, dropout=0.0)
        self.classifier = nn.Sequential(nn.Linear(2 * H, 64), nn.ReLU(), nn.Dropout(0.5), nn.Linear(64, nc))

    def forward(self, x):
        x = self.channel_attention(x)
        x = self.cnn_encoder(x).permute(0, 2, 1)
        out, _ = self.gru(x)
        return self.classifier(out[:, -1, :])


def timed(fn, reps):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps


def stock_ig(ref, x, target, steps, max_rows):
    B = x.shape[0]
    A = torch.zeros_like(x)
    total = B * steps
    alpha = (torch.arange(steps, device=x.device, dtype=torch.float32) + 0.5) / steps
    rows_b = torch.arange(total, device=x.device) // steps
    rows_a = alpha.repeat(B)
    for r0 in range(0, total, max_rows):
        rb, ra = rows_b[r0:r0 + max_rows], rows_a[r0:r0 + max_rows]
        z = (ra[:, None, None] * x[rb]).requires_grad_(True)          # zero baseline
        logits = ref(z)
        (g,) = torch.autograd.grad(logits.gather(1, target[rb][:, None]).sum(), z)
        A.index_add_(0, rb, g / steps)
    return A * x


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--channels", type=int, default=6)
    ap.add_argument("--seq-len", type=int, default=3840)
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--bwd-batch", type=int, default=2048)
    ap.add_argument("--parent", default=None, help="an older, built checkout: bench.py of both trees, alternated")
    ap.add_argument("--bench-rounds", type=int, default=3)
    ap.add_argument("--bench-steps", type=int, default=300)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "attribution_bench.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("attribution_bench needs a CUDA device")
    from multimodalsignal_b200.attribution import integrated_gradients
    from multimodalsignal_b200.models import CnnGruAttentionModel

    res = {"card": card(), "batch": a.batch, "channels": a.channels, "seq_len": a.seq_len, "hidden": 64, "layers": 2,
           "ig_steps": a.steps}
    torch.manual_seed(0)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m = CnnGruAttentionModel(a.channels, 2).cuda().eval().requires_grad_(False)
    x = torch.randn(a.batch, a.channels, a.seq_len, device="cuda")

    # (a) IG per window, ours against stock PyTorch / cuDNN (strict fp32)
    run = lambda: integrated_gradients(m, x, steps=a.steps, max_rows=2048)
    A_ours, _, _ = run()
    t_ours = timed(run, a.reps)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    ref = RefModel(a.channels, 2).cuda()
    ref.load_state_dict({k: v.detach().clone() for k, v in m.state_dict().items()})
    ref.eval().requires_grad_(False)
    ref.gru.train()                       # cuDNN's RNN backward needs train mode; dropout is 0
    with torch.no_grad():
        target = torch.argmax(m(x), dim=1)
    srun = lambda: stock_ig(ref, x, target, a.steps, 2048)
    A_stock = srun()
    t_stock = timed(srun, a.reps)
    res["a_ig"] = {"ours_ms_per_window": 1e3 * t_ours / a.batch, "stock_ms_per_window": 1e3 * t_stock / a.batch,
                   "speedup": t_stock / t_ours,
                   "max_abs_diff_A_over_max_A": (A_ours - A_stock).abs().max().item() / A_stock.abs().max().item()}
    print(json.dumps(res["a_ig"]), flush=True)

    # (b) input-gradient-only backward against the full backward after the same eval forward
    B2 = a.bwd_batch
    x2 = torch.randn(B2, a.channels, a.seq_len, device="cuda")
    eng = m.engine(B2, a.seq_len, False, True, x2.device)
    eng.forward(x2, 1)
    dl = torch.zeros(B2, 2, device="cuda")
    dl[:, 0] = 1
    dx = torch.empty_like(x2)
    ig_fn = lambda: eng.input_gradient(x2, dl, dx)
    bwd_fn = lambda: eng.backward(x2, dl, True)
    ig_fn(); bwd_fn()
    t_ig, t_bwd = [], []
    for _ in range(10):
        t_ig.append(timed(ig_fn, 3))
        t_bwd.append(timed(bwd_fn, 3))
    t_ig.sort(); t_bwd.sort()
    res["b_backward"] = {"batch": B2, "input_gradient_ms_median": 1e3 * t_ig[5], "full_backward_ms_median": 1e3 * t_bwd[5],
                         "input_gradient_ms_min": 1e3 * t_ig[0], "full_backward_ms_min": 1e3 * t_bwd[0],
                         "ratio": t_bwd[5] / t_ig[5]}
    print(json.dumps(res["b_backward"]), flush=True)

    # (c) bench.py headline, parent against this tree, alternated
    if a.parent:
        def bench(tree):
            out = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", str(a.bench_steps), "--warmup", "50",
                                  "--no-cpu-baseline", "--no-library-baseline"], cwd=tree, capture_output=True, text=True)
            lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
            return json.loads(lines[-1]) if lines else {"error": out.stderr[-2000:]}
        rounds = []
        for _ in range(a.bench_rounds):
            rounds.append({"parent": bench(a.parent), "branch": bench(str(ROOT))})
        res["c_bench"] = rounds
        print(json.dumps(rounds), flush=True)
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(res, indent=1))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
