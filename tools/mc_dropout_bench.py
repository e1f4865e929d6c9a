"""MC-dropout timings on one GPU, recorded with the card's name, power limit and max SM clock from the same run.

Shape: B windows (default 64), C = 6, T = 3840, H = 64, 2 GRU layers, m samples (default 32): B*m = 2048 sample rows,
one chunk.  Alternated, median of --reps rounds after a warm-up:

(1) ``uncertainty.mc_dropout``: the shared prefix (encoder + GRU layer 0 per window), the expansion of layer 0's output
    to the sample rows, the per-sample top layer and head, and the statistics.  The split comes from one extra call with
    the library's launch timeline on (device timestamps around each launch), as shares of that call.
(2) this library's eval forward of the replicated [B*m, C, T] batch: the same rows without the shared prefix (no dropout:
    the eval forward has none, so this is the cost of the rows alone).
(3) the torch recipe: the reference model in stock torch.nn modules, strict fp32 (no TF32), BatchNorm in eval mode,
    the GRU and the classifier's Dropout in train mode, one forward of the B*m replicated rows.
(4) with ``--parent DIR`` (an older checkout, already built): ``bench.py`` of DIR and of this tree, alternated, and
    ``bench.py --dump-outputs`` of each tree, twice, compared array by array (the parent against itself shows what a
    rerun of unchanged code changes).

    python tools/mc_dropout_bench.py [--parent DIR] [--out profiles/r5_mc_dropout_bench.json]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import subprocess
import sys
import tempfile
import time
import warnings
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    idx = torch.cuda.current_device()
    lines = q.stdout.strip().splitlines()
    return lines[idx].strip() if idx < len(lines) else q.stdout.strip()


def timed(fn, reps=3):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps


def timeline_split(lib, fn):
    """Shares of one call of ``fn`` between the shared prefix, the expansion, the per-sample layers + head and the
    statistics, from the library's launch timeline (ns device timestamps, launches in enqueue order)."""
    lib.mms_timeline_enable(1)
    fn()
    buf = C.create_string_buffer(1 << 20)
    lib.mms_timeline_report(buf, len(buf))
    lib.mms_timeline_enable(0)
    recs = []
    for ln in buf.value.decode().splitlines():
        name, _, t0, t1 = ln.split()
        recs.append((name, int(t0), int(t1)))
    first = min(r[1] for r in recs)
    exp = [r for r in recs if r[0] == "mc_expand_kernel"]
    acc = [r for r in recs if r[0] == "mc_accumulate_kernel"]
    start_exp, end_exp = exp[0][1], exp[-1][2]
    start_acc, end_acc = acc[0][1], acc[-1][2]
    total = end_acc - first
    parts = {"prefix": start_exp - first, "expansion": end_exp - start_exp, "per_sample_layers_and_head": start_acc - end_exp,
             "statistics": end_acc - start_acc}
    return {"launches": len(recs), "call_us_timeline": total / 1e3,
            "share": {k: v / total for k, v in parts.items()}, "us": {k: v / 1e3 for k, v in parts.items()}}


def bench_json(tree, args):
    out = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", str(args.bench_steps), "--warmup", "50",
                          *args.bench_extra.split()], cwd=tree, capture_output=True, text=True)
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    if not lines:
        return {"error": out.stderr[-2000:]}
    r = json.loads(lines[-1])
    return {k: r.get(k) for k in ("value", "unit", "ms_per_step", "kernels_per_step", "clocks")}


def dump(tree, out_dir):
    out = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", "20", "--warmup", "5",
                          "--dump-outputs", str(out_dir), *"--no-cpu-baseline --no-library-baseline".split()],
                         cwd=tree, capture_output=True, text=True)
    return out.returncode, out.stderr[-1500:]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--samples", type=int, default=32)
    ap.add_argument("--reps", type=int, default=11)
    ap.add_argument("--parent", default=None, help="an older, built checkout: bench.py of both trees, alternated")
    ap.add_argument("--bench-rounds", type=int, default=3)
    ap.add_argument("--bench-steps", type=int, default=300)
    ap.add_argument("--bench-extra", default="--no-cpu-baseline --no-library-baseline")
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r5_mc_dropout_bench.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mc_dropout_bench needs a CUDA device")
    from multimodalsignal_b200 import _ext
    from multimodalsignal_b200.models import CnnGruAttentionModel
    from multimodalsignal_b200.uncertainty import mc_dropout
    from attribution_bench import RefModel

    Cc, T, B, m_ = 6, 3840, a.batch, a.samples
    res = {"card_name_power_limit_max_sm_clock": card(), "batch": B, "samples": m_, "rows": B * m_, "channels": Cc,
           "seq_len": T, "hidden": 64, "layers": 2, "dropout": 0.5, "reps": a.reps, "statistic": "median"}
    torch.manual_seed(0)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model = CnnGruAttentionModel(Cc, 2).cuda().eval()
    x = torch.randn(B, Cc, T, device="cuda")
    xr = x.repeat_interleave(m_, dim=0).contiguous()
    lib = _ext.lib()

    mc = lambda: mc_dropout(model, x, samples=m_, seed=1, max_rows=B * m_)

    def ev():
        with torch.no_grad():
            return model(xr)

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    ref = RefModel(Cc, 2).cuda()
    ref.gru.dropout = 0.5
    ref.load_state_dict({k: v.detach().clone() for k, v in model.state_dict().items()})
    ref.eval()
    ref.gru.train()
    ref.classifier[2].train()

    def recipe():
        with torch.no_grad():
            return ref(xr)

    for f in (mc, ev, recipe):          # warm every shape
        f(); f()
    t = {"mc": [], "eval_replicated": [], "torch_recipe": []}
    for _ in range(a.reps):
        t["mc"].append(timed(mc))
        t["eval_replicated"].append(timed(ev))
        t["torch_recipe"].append(timed(recipe))
    med = {k: float(np.median(v)) for k, v in t.items()}
    res["ms_per_call"] = {k: 1e3 * v for k, v in med.items()}
    res["ms_per_window"] = {k: 1e3 * v / B for k, v in med.items()}
    res["ms_per_call_min_max"] = {k: [1e3 * min(v), 1e3 * max(v)] for k, v in t.items()}
    res["speedup_vs_eval_replicated"] = med["eval_replicated"] / med["mc"]
    res["speedup_vs_torch_recipe"] = med["torch_recipe"] / med["mc"]
    res["mc_split"] = timeline_split(lib, mc)
    print(json.dumps(res), flush=True)

    if a.parent:
        rounds = []
        for _ in range(a.bench_rounds):
            rounds.append({"parent": bench_json(a.parent, a), "branch": bench_json(str(ROOT), a)})
        res["bench_alternated"] = rounds
        # --dump-outputs twice per tree: parent against parent shows what a rerun of the same code changes
        with tempfile.TemporaryDirectory() as td:
            dirs = {k: Path(td) / k for k in ("parent_a", "branch_a", "parent_b", "branch_b")}
            rc = {k: dump(a.parent if k.startswith("parent") else str(ROOT), d) for k, d in dirs.items()}

            def compare(x, y):
                names = sorted(p.name for p in dirs[x].glob("*.npy"))
                diff = {}
                for f in names:
                    u, v = np.load(dirs[x] / f), np.load(dirs[y] / f)
                    if u.shape != v.shape or u.tobytes() != v.tobytes():
                        diff[f] = float(np.abs(u.astype(np.float64) - v.astype(np.float64)).max()) if u.shape == v.shape else "shape"
                return {"arrays": len(names), "bit_identical": len(names) - len(diff),
                        "max_abs_diff": max([d for d in diff.values() if d != "shape"], default=0.0), "different": diff}
            res["dump_outputs"] = {"returncodes": {k: v[0] for k, v in rc.items()},
                                   "parent_vs_branch": compare("parent_a", "branch_a"),
                                   "parent_vs_parent": compare("parent_a", "parent_b"),
                                   "branch_vs_branch": compare("branch_a", "branch_b")}
            if any(v[0] for v in rc.values()):
                res["dump_outputs"]["stderr"] = {k: v[1] for k, v in rc.items()}
        print(json.dumps({k: res[k] for k in ("bench_alternated", "dump_outputs")}), flush=True)
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
