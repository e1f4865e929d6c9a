"""Cost of gradient-norm clipping in the fused training step (graph-replayed) at B = 64, C = 6, T = 3840: the same step with
clipping off and on (``FlatAdam(max_grad_norm=...)``), alternated round by round after warm-up, with the launches of one step
and the card's name and power limit read in the same process.  With ``--peer`` on >= 2 GPUs (torchrun, one process per GPU)
it times the symmetric-memory data-parallel step instead, at B = 256, C = 14.

    python tools/grad_clip_bench.py [--rounds 7] [--steps 200] [--out profiles/grad_clip_bench.json]
    python -m torch.distributed.run --nproc-per-node 2 tools/grad_clip_bench.py --peer [--out ...]
"""
import argparse
import json
import os
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

MAX_NORM = 1.0          # below the gradient norm of these random batches: every step clips


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--channels", type=int, default=None)
    ap.add_argument("--seq-len", type=int, default=3840)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--peer", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("grad_clip_bench needs a CUDA device (B200)")
    from multimodalsignal_b200 import _ext
    from multimodalsignal_b200.models import CnnGruAttentionModel
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    rank, world = 0, 1
    if args.peer:
        import torch.distributed as dist
        rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = _ext.lib()
    B = args.batch or (256 if args.peer else 64)
    Cc = args.channels or (14 if args.peer else 6)
    T = args.seq_len
    dev = torch.device("cuda")
    steps = {}
    for k, clip in (("off", None), ("on", MAX_NORM)):
        torch.manual_seed(42)
        model = CnnGruAttentionModel(Cc, 2, dropout=0.5).to(dev).train()
        opt = FlatAdam(model, lr=1e-4, weight_decay=1e-4, max_grad_norm=clip)
        if args.peer:
            from multimodalsignal_b200.parallel import DataParallelTrainStep
            steps[k] = DataParallelTrainStep(model, opt, B // world, B, T, rank=rank, peer="symm")
        else:
            steps[k] = FusedTrainStep(model, opt, B, T)
    b = B // world
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    NB = 16
    xs = torch.randn(NB, b, Cc, T, device=dev, generator=gen)
    ys = torch.randint(0, 2, (NB, b), device=dev, generator=gen)
    info = {}
    for k, st in steps.items():            # warm-up: eager step (launch count), capture, replays
        l0 = lib.mms_launch_count()
        st(xs[0], ys[0])
        torch.cuda.synchronize()
        launches = int(lib.mms_launch_count() - l0)
        for i in range(1, 30):
            st(xs[i % NB], ys[i % NB])
        torch.cuda.synchronize()
        info[k] = {"launches_per_step": launches, "ms": []}
    for _ in range(args.rounds):
        for k, st in steps.items():
            if args.peer:
                torch.distributed.barrier()
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
    on = steps["on"].opt
    info["on"]["clipped_steps"] = int(on.clip_record[2].item())
    info["on"]["steps_recorded"] = int(on.clip_record[4].item())
    info["on"]["last_grad_norm"] = float(on.grad_norm.item())
    if args.peer:
        steps["on"].check_peers()
        steps["off"].check_peers()
    res = {"card": card(), "device": torch.cuda.get_device_name(), "world": world, "path": "peer" if args.peer else "fused",
           "batch": B, "channels": Cc, "seq_len": T, "max_grad_norm": MAX_NORM, "rounds": args.rounds,
           "steps_per_round": args.steps, "cuda_graph": True, "clipping": info,
           "overhead_ms": info["on"]["median_ms_per_step"] - info["off"]["median_ms_per_step"]}
    if rank == 0:
        line = json.dumps(res)
        print(line)
        if args.out:
            Path(args.out).parent.mkdir(parents=True, exist_ok=True)
            Path(args.out).write_text(line + "\n")
    if args.peer:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
