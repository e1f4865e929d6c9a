"""Training-step time with and without class weights (CrossEntropyLoss(weight=w), Trainer's use_class_weights).

Workload: the bench configuration, B = 64, C = 6, T = 3840, 2 GRU layers of 64, 2 classes, fp32, dropout 0.5, Adam
(lr 1e-3, weight decay 1e-4), one CUDA graph per step (FusedTrainStep, fused head).  Both arms are warmed up, then timed
with CUDA events in `--repeats` rounds of `--steps` graph replays, the two arms alternated inside every round so that
drift of the shared machine falls on both alike.  With weights, each of the B head CTAs also reads the B labels and
their weights to form the normaliser.  The card's name and power limit are read in the same run.

    python tools/class_weights_step.py --out /tmp/class_weights_step.json
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

B, CH, T, NC, P = 64, 6, 3840, 2, 0.5


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
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()

    import torch
    from multimodalsignal_b200.models import CnnGruAttentionModel
    from multimodalsignal_b200.synth import synthetic_windows
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep, balanced_class_weights

    if not torch.cuda.is_available():
        raise SystemExit("class_weights_step.py measures on a GPU; none is visible")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    xs, ys = [], []
    for i in range(4):
        x, y = synthetic_windows(B, CH, T, seed=100 + i)
        xs.append(torch.from_numpy(x).to(dev))
        ys.append(torch.from_numpy(y).to(dev))
    weights = [float(v) for v in balanced_class_weights(torch.cat(ys), NC)]

    arms = {}
    for name, cw in (("unweighted", None), ("weighted", weights)):
        torch.manual_seed(0)
        m = CnnGruAttentionModel(CH, NC, dropout=P).to(dev).train()
        st = FusedTrainStep(m, FlatAdam(m, lr=1e-3, weight_decay=1e-4), B, T, class_weight=cw)
        for i in range(args.warmup):
            st(xs[i % 4], ys[i % 4])
        torch.cuda.synchronize()
        arms[name] = st

    ms = {name: [] for name in arms}
    for _ in range(args.repeats):
        for name, st in arms.items():
            ms[name].append(timed(lambda i: st(xs[i % 4], ys[i % 4]), args.steps))

    res = {
        "card": card(),
        "workload": {"batch": B, "channels": CH, "seq_len": T, "num_classes": NC, "dropout": P, "precision": "fp32",
                     "optimizer": "Adam lr 1e-3 wd 1e-4", "class_weights": weights, "steps_per_repeat": args.steps,
                     "warmup": args.warmup, "repeats": args.repeats,
                     "timing": "CUDA events around --steps graph replays, arms alternated inside every repeat"},
        "ms_per_step": {name: {"min": min(v), "median": sorted(v)[len(v) // 2], "all": v} for name, v in ms.items()},
    }
    res["weighted_over_unweighted_min"] = min(ms["weighted"]) / min(ms["unweighted"])
    out = Path(args.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    out.write_text(json.dumps(res, indent=1))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
