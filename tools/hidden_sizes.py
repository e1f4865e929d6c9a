"""Training-step time at gru_hidden_size 32, 64 and 128 on one GPU, and the same model at 128 through stock PyTorch / cuDNN.

Workload: B = 64, C = 6, T = 3840 (L = 240 GRU steps), 2 GRU layers, fp32, dropout 0.5, Adam (lr 1e-3, weight decay 1e-4),
one CUDA graph per step (FusedTrainStep).  Every size is warmed up, then timed in `--repeats` rounds of `--steps` steps with
the sizes alternated inside each round, so that drift of the shared machine falls on all of them alike.  Afterwards one
eager run per size with mms_profile_enable(1) and side streams off gives the per-launch time of each recurrence kernel,
reported also per GRU time step.  The stock arm runs oracle/cpu_port.forward (the reference model written with
torch.nn.functional / torch._VF.gru, i.e. cuDNN's GRU) on the GPU with torch.optim.Adam, TF32 off for matmul and cuDNN
(strict fp32, the arithmetic the library's kernels match).  The card's name and power limit are read in the same run.

    python tools/hidden_sizes.py --out /tmp/hidden_sizes.json
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

B, CH, T, LAYERS, NC, P = 64, 6, 3840, 2, 2, 0.5
SIZES = (32, 64, 128)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [s.strip() for s in q.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def timed(fn, steps):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=30)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()

    import torch
    from multimodalsignal_b200 import _ext
    from multimodalsignal_b200.models import CnnGruAttentionModel
    from multimodalsignal_b200.synth import synthetic_windows
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    from oracle import cpu_port

    if not torch.cuda.is_available():
        raise SystemExit("hidden_sizes.py measures on a GPU; none is visible")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lib = _ext.lib()
    xs, ys = [], []
    for i in range(4):
        x, y = synthetic_windows(B, CH, T, seed=100 + i)
        xs.append(torch.from_numpy(x).to(dev))
        ys.append(torch.from_numpy(y).to(dev))
    L = T // 16

    steps = {}
    for H in SIZES:
        torch.manual_seed(0)
        m = CnnGruAttentionModel(CH, NC, gru_hidden_size=H, gru_num_layers=LAYERS, dropout=P).to(dev).train()
        st = FusedTrainStep(m, FlatAdam(m, lr=1e-3, weight_decay=1e-4), B, T)
        for i in range(args.warmup):
            st(xs[i % 4], ys[i % 4])
        torch.cuda.synchronize()
        steps[H] = st

    ms = {H: [] for H in SIZES}
    for _ in range(args.repeats):
        for H in SIZES:
            st = steps[H]
            ms[H].append(timed(lambda i: st(xs[i % 4], ys[i % 4]), args.steps))

    recur = {}
    lib.mms_set_side_streams(0)
    for H in SIZES:
        st = steps[H]
        lib.mms_profile_enable(1)
        n = 20
        for i in range(n):
            st.load(xs[i % 4], ys[i % 4])
            st._enqueue()
        buf = (C.c_char * 16384)()
        lib.mms_profile_report(buf, 16384)
        lib.mms_profile_enable(0)
        kern = {}
        for line in buf.value.decode().strip().splitlines():
            name, cnt, tot = line.rsplit(" ", 2)
            kern[name] = (int(cnt), float(tot))
        recur[H] = {}
        for name in ("gru_fwd_v2_kernel", "gru_bwd_ring_kernel"):
            cnt, tot = kern[name]
            us = 1e3 * tot / cnt
            # one launch runs both directions of a layer side by side, L steps long
            recur[H][name] = {"launches_per_step": cnt / n, "us_per_launch": us, "ns_per_time_step": 1e3 * us / L}
    lib.mms_set_side_streams(1)

    # stock PyTorch / cuDNN, strict fp32, same model at H = 128
    saved = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = False, False
    try:
        p, bufs = cpu_port.make_state(C=CH, num_classes=NC, H=128, layers=LAYERS, seed=0)
        leaves = {k: v.to(dev).requires_grad_(True) for k, v in p.items()}
        bufs = {k: v.to(dev) for k, v in bufs.items()}
        opt = torch.optim.Adam(list(leaves.values()), lr=1e-3, weight_decay=1e-4)

        def ref_step(i):
            opt.zero_grad()
            out = cpu_port.forward(leaves, bufs, xs[i % 4], training=True, dropout=P, layers=LAYERS)
            torch.nn.functional.cross_entropy(out, ys[i % 4]).backward()
            opt.step()
        for i in range(args.warmup):
            ref_step(i)
        torch.cuda.synchronize()
        ref_ms = [timed(ref_step, args.steps) for _ in range(args.repeats)]
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = saved

    res = {
        "card": card(),
        "workload": {"batch": B, "channels": CH, "seq_len": T, "gru_steps": L, "gru_num_layers": LAYERS, "num_classes": NC,
                     "dropout": P, "optimizer": "Adam lr 1e-3 wd 1e-4", "precision": "fp32",
                     "steps_per_repeat": args.steps, "warmup": args.warmup, "repeats": args.repeats,
                     "timing": "CUDA events around --steps graph replays, sizes alternated inside every repeat"},
        "recurrence_design_h128": "gru_fwd_v2_kernel<128> / gru_bwd_ring_kernel<128, 8>: the kernels of H = 32 / 64 instantiated "
                                  "at H = 128 (256 threads, W_hh in registers, one CTA per SM); no other H = 128 design is built",
        "ours": {str(H): {"ms_per_step": min(ms[H]), "ms_per_step_all": ms[H], "windows_per_s": B / (min(ms[H]) * 1e-3),
                          "recurrence": recur[H]} for H in SIZES},
        "stock_pytorch_fp32_strict_h128": {"ms_per_step": min(ref_ms), "ms_per_step_all": ref_ms,
                                           "windows_per_s": B / (min(ref_ms) * 1e-3), "torch": torch.__version__,
                                           "cudnn": torch.backends.cudnn.version(),
                                           "model": "oracle/cpu_port.forward on cuda (cuDNN GRU), torch.optim.Adam"},
    }
    res["speedup_h128_vs_stock_fp32"] = res["stock_pytorch_fp32_strict_h128"]["ms_per_step"] / res["ours"]["128"]["ms_per_step"]
    out = Path(args.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    out.write_text(json.dumps(res, indent=1))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
