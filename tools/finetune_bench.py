"""Step time of fine-tuning with frozen parameters: the fused training step (graph-replayed) at B = 64, C = 6, T = 3840 for
four freeze patterns -- all trainable, encoder frozen, encoder + GRU layer 0 frozen, head only -- alternated round by
round after warm-up, with the launches of one step and the card's name and power limit read in the same process.

    python tools/finetune_bench.py [--rounds 5] [--steps 200] [--out profiles/finetune_bench.json]
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

ENCODER = ("channel_attention.", "cnn_encoder.")
PATTERNS = {
    "all_trainable": lambda n: False,
    "encoder_frozen": lambda n: n.startswith(ENCODER),
    "encoder_gru_l0_frozen": lambda n: n.startswith(ENCODER) or "_l0" in n,
    "head_only": lambda n: not n.startswith("classifier."),
}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--channels", type=int, default=6)
    ap.add_argument("--seq-len", type=int, default=3840)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("finetune_bench needs a CUDA device (B200)")
    from multimodalsignal_b200 import _ext
    from multimodalsignal_b200.models import CnnGruAttentionModel
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    lib = _ext.lib()
    B, Cc, T = args.batch, args.channels, args.seq_len
    torch.manual_seed(42)
    dev = torch.device("cuda")
    model = CnnGruAttentionModel(Cc, 2, dropout=0.5).to(dev).train()
    names = [n for n, _ in model.named_parameters()]
    # one optimizer and one step per pattern: each keeps its own graph; the model is shared, so the patterns see the same
    # weights' magnitudes (the step time does not depend on their values)
    steps = {}
    for k in PATTERNS:
        opt = FlatAdam(model, lr=1e-4, weight_decay=1e-4)
        steps[k] = FusedTrainStep(model, opt, B, T)
    gen = torch.Generator(device=dev).manual_seed(1234)
    NB = 16
    xs = torch.randn(NB, B, Cc, T, device=dev, generator=gen)
    ys = torch.randint(0, 2, (NB, B), device=dev, generator=gen)

    def freeze(k):
        for n, p in model.named_parameters():
            p.requires_grad_(not PATTERNS[k](n))

    info = {}
    for k, st in steps.items():            # warm-up: eager step (launch count), capture, replays
        freeze(k)
        l0 = lib.mms_launch_count()
        st(xs[0], ys[0])
        torch.cuda.synchronize()
        launches = int(lib.mms_launch_count() - l0)
        for i in range(1, 20):
            st(xs[i % NB], ys[i % NB])
        torch.cuda.synchronize()
        n_train = sum(p.numel() for n, p in model.named_parameters() if not PATTERNS[k](n))
        info[k] = {"launches_per_step": launches, "trainable_params": n_train,
                   "frozen_segments": hex(st.desc.frozen_segments), "ms": []}
    for r in range(args.rounds):
        for k, st in steps.items():
            freeze(k)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(args.steps):
                st(xs[i % NB], ys[i % NB])
            e1.record()
            torch.cuda.synchronize()
            info[k]["ms"].append(e0.elapsed_time(e1) / args.steps)
    for k in info:
        v = sorted(info[k]["ms"])
        info[k]["median_ms_per_step"] = v[len(v) // 2]
    res = {"card": card(), "device": torch.cuda.get_device_name(), "batch": B, "channels": Cc, "seq_len": T,
           "rounds": args.rounds, "steps_per_round": args.steps, "cuda_graph": True, "patterns": info}
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
