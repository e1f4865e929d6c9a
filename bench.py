#!/usr/bin/env python
"""Headline benchmark: CnnGruAttention training throughput (windows/s, fwd+bwd+Adam).

``python bench.py --gpus N --steps K --warmup W`` -- one process per GPU (torchrun for N > 1).
Workload = BASELINE.json configs[1]: cnn_gru_attention, 6 channels, B=64 windows of T=3840
(64 Hz x 60 s), one LOSO fold per GPU, dropout 0.5 as the reference trains, synthetic data.
With N > 1 every rank trains its own fold (LOSO folds are independent: weak scaling, no
collective on the data path).

One JSON line on rank 0:
  value        windows/s, inputs resident in HBM (a pool larger than L2 is cycled);
  e2e          the same step driven through the public step API with HOST data, as reference
               trainer.py:140-153 does: pinned host batch -> H2D copy (copy stream, one batch ahead) ->
               step -> every step's loss read back on the host (async D2H, consumed one step late);
  roofline     the dominant kernel of the step, timed live with CUDA events (eager replay of the
               same step through the library's event hooks);
  cpu_baseline oracle/cpu_port.py (the reference's step through the same ATen CPU kernels) on the
               host cores, bounded sample, rank 0 at N=1 only.
``--impl reference`` times that CPU port alone (the reference is Python and cannot travel to the
GPU box; see DESIGN.md).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

FLOP_PER_WINDOW = {(6, 3840): 121.6e6, (14, 3840): 131.9e6, (6, 7680): 242.8e6}   # SURVEY §8d (minimal count)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--channels", type=int, default=6)
    ap.add_argument("--seq-len", type=int, default=3840)
    ap.add_argument("--cpu-seconds", type=float, default=20.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-library-baseline", action="store_true", help="skip the stock PyTorch/cuDNN leg (reference model on the same GPU)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-subrecords", action="store_true",
                    help="train_step: skip the loso / preprocess / dp sub-records (BASELINE.json configs[2..4]) of the default line")
    ap.add_argument("--workload", default="train_step", choices=["train_step", "loso", "preprocess", "dp"],
                    help="train_step = headline metric (default); loso = 15-fold LOSO wall-clock; preprocess = resample+window")
    ap.add_argument("--epochs", type=int, default=100, help="loso: EPOCHS (reference main.py:62 uses 100, patience 20)")
    ap.add_argument("--dp-exchange", default="peer", choices=["peer", "nccl"],
                    help="dp: 'peer' = symmetric memory + our peer kernels (gradient all-reduce fused with Adam, CUDA graph); "
                         "'nccl' = torch.distributed all-reduces")
    ap.add_argument("--concurrent-folds", type=int, default=4, help="loso: folds interleaved per GPU on separate CUDA streams (1 = one after another)")
    ap.add_argument("--subjects", type=int, default=15, help="loso / preprocess: number of synthetic subjects")
    ap.add_argument("--minutes", type=float, default=100.0, help="loso / preprocess: recording length (100 = 4.2 M chest samples)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps of the train_step workload (--impl ours, the headline path; no other workload "
                         "takes it), write what the last of them returned (loss, logits, gradient, updated state_dict) as "
                         "DIR/<name>.npy; the inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.workload != "train_step" or args.impl != "ours"):
        ap.error("--dump-outputs applies to the train_step workload of --impl ours")
    return args


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the measured region (B200_PROFILING.md)."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.thread = index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            return
        def pump():
            for line in self.proc.stdout:
                self.rows.append(line.strip())
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        sm, smax, reasons = [], [], set()
        for r in self.rows:
            parts = [x.strip() for x in r.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                smax.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


class _ReferenceStep:
    """The reference's own training step -- ``CnnGruAttentionModel`` from the UNMODIFIED reference ``models.py``
    (``/root/reference`` or its byte-identical staging ``baseline/_ref``, oracle/build_ref.py), driven exactly as
    trainer.py:68-69,140-153 drives it: ``inputs.to(device)``, ``zero_grad``, forward, ``CrossEntropyLoss``,
    ``backward``, ``Adam(lr=1e-3, weight_decay=1e-4).step()``, ``loss.item()``.  ``device`` = "cpu" is the reference arm;
    ``device`` = "cuda" is the same stock PyTorch / cuDNN path on the B200 ("the library kernel to beat", SURVEY 8d-iii)."""

    def __init__(self, args, device):
        import torch
        from oracle import ref_harness
        models = ref_harness.load("models")
        torch.manual_seed(0)
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            self.model = models.CnnGruAttentionModel(in_channels=args.channels, num_classes=2).to(device)   # main.py:116, trainer.py:58
        self.model.train()
        self.opt = torch.optim.Adam(self.model.parameters(), lr=1e-3, weight_decay=1e-4)                  # trainer.py:68
        self.crit = torch.nn.CrossEntropyLoss().to(device)                                                # trainer.py:69
        self.device = device

    def __call__(self, x, y):
        x, y = x.to(self.device), y.to(self.device)                                                        # trainer.py:140-142
        self.opt.zero_grad()
        loss = self.crit(self.model(x), y)
        loss.backward()
        self.opt.step()
        return loss.item()                                                                                 # trainer.py:152


def cpu_reference_run(args, steps, warmup, budget_s=None):
    """Time the reference's CPU training step: the unmodified reference ``models.py`` when it is present (kind
    "reference"), else oracle/cpu_port.py (kind "port").  ``steps`` timed steps after ``warmup`` (the first included),
    or, with ``budget_s``, as many of them as fit in about that many seconds of CPU work."""
    import torch
    from oracle import ref_harness
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    if ref_harness.available():
        step = _ReferenceStep(args, "cpu")
        kind = "reference"
        what = (f"the unmodified reference models.py ({ref_harness.REFERENCE_ROOT}) driven as trainer.py:140-153 "
                f"(zero_grad, forward, CrossEntropyLoss, backward, Adam, loss.item())")
    else:
        from oracle import cpu_port
        p, bufs = cpu_port.make_state(C=args.channels, seed=0)
        step = cpu_port.CpuTrainStep(p, bufs)
        kind = "port"
        what = "oracle/cpu_port.py = the reference step through the same ATen CPU kernels (reference tree not staged)"
    g = torch.Generator().manual_seed(1)
    x = torch.randn(args.batch, args.channels, args.seq_len, generator=g)
    y = torch.randint(0, 2, (args.batch,), generator=g)
    t0 = time.perf_counter()
    step(x, y)
    first = time.perf_counter() - t0
    warm = max(0, warmup - 1 if budget_s is None else min(warmup - 1, int(0.25 * budget_s / max(first, 1e-3))))
    for _ in range(warm):
        step(x, y)
    n = steps if budget_s is None else max(1, min(steps, int(budget_s / max(first, 1e-3))))
    t0 = time.perf_counter()
    for _ in range(n):
        step(x, y)
    dt = time.perf_counter() - t0
    return {"value": args.batch * n / dt, "unit": "windows/s", "cores": threads, "kind": kind,
            "ms_per_step": 1e3 * dt / n, "timed_steps": n,
            "sample": f"{n} full training steps (B={args.batch}, C={args.channels}, T={args.seq_len}, dropout 0.5, Adam) of "
                      f"{what}, {threads} threads"}


def library_gpu_run(args, dev, steps=30, warmup=5):
    """SURVEY 8d-(iii): the UNMODIFIED reference model on the SAME B200 through stock PyTorch (cuDNN GRU / conv, ATen
    BatchNorm / pooling, torch.optim.Adam) -- "the library kernel to beat".  Same B / C / T, three precision settings:
    PyTorch's defaults (what the reference runs: trainer.py never enables AMP and sets no backend flag), strict fp32
    (TF32 off for matmul and cuDNN -- the arithmetic our kernels match) and TF32 allowed everywhere.  Device-timed with CUDA events, inputs resident in HBM
    (``value``) and with the reference's own per-step H2D copy + ``loss.item()`` (``e2e``)."""
    import torch
    from oracle import ref_harness
    if not ref_harness.available():
        return {"unavailable": "reference modules not staged under baseline/_ref"}
    B, C, T = args.batch, args.channels, args.seq_len
    gen = torch.Generator().manual_seed(7)
    hx = torch.randn(8, B, C, T, generator=gen).pin_memory()
    hy = torch.randint(0, 2, (8, B), generator=gen).pin_memory()
    dx, dy = hx.to(dev), hy.to(dev)
    out = {"unit": "windows/s", "kind": "reference models.py on cuda via stock PyTorch/cuDNN (unmodified)",
           "torch": torch.__version__, "cudnn": torch.backends.cudnn.version(), "steps": steps, "warmup": warmup}
    saved = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    try:
        for tag, tf32 in (("pytorch_default", None), ("fp32_strict", (False, False)), ("tf32_allowed", (True, True))):
            torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = tf32 if tf32 else saved
            step = _ReferenceStep(args, dev)

            def dev_step(i):                       # inputs already in HBM; no host read-back inside the loop
                step.opt.zero_grad()
                loss = step.crit(step.model(dx[i % 8]), dy[i % 8])
                loss.backward()
                step.opt.step()
                return loss
            for i in range(warmup):
                dev_step(i)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(steps):
                dev_step(i)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            t0 = time.perf_counter()
            for i in range(steps):
                step(hx[i % 8], hy[i % 8])         # trainer.py:140-153 verbatim: H2D, step, loss.item()
            torch.cuda.synchronize()
            e2e_ms = 1e3 * (time.perf_counter() - t0) / steps
            out[tag] = {"value": B / (ms * 1e-3), "ms_per_step": ms, "e2e_value": B / (e2e_ms * 1e-3), "e2e_ms_per_step": e2e_ms}
            del step
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = saved
    out["flags"] = {"pytorch_default": {"matmul.allow_tf32": saved[0], "cudnn.allow_tf32": saved[1]}}
    out["value"] = out["pytorch_default"]["value"]            # what the unmodified reference runs (trainer.py sets no flag)
    out["ms_per_step"] = out["pytorch_default"]["ms_per_step"]
    return out


def config_dict(args, n_gpus):
    return {"workload": "cnn_gru_attention single LOSO fold per GPU (BASELINE.json configs[1])",
            "batch": args.batch, "channels": args.channels, "seq_len": args.seq_len, "num_classes": 2,
            "hidden": 64, "gru_layers": 2, "dropout": 0.5, "optimizer": "Adam lr=1e-3 wd=1e-4",
            "global_batch": args.batch * n_gpus, "parallelism": f"fold-sharded x{n_gpus} (no collective)",
            "l2_policy": "device-resident input pool of 48 batches (283 MB > 126 MB L2) cycled; activations ~170 MB/step"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_run(args, args.steps, args.warmup)
    line = {"impl": "reference", "metric": "train windows/sec (fwd+bwd+Adam) CnnGruAttention", "value": r["value"],
            "unit": "windows/s", "n_gpus": args.gpus, "steps": r["timed_steps"], "requested_steps": args.steps,
            "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config_dict(args, args.gpus),
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    if not args.no_subrecords:
        try:
            line["loso"] = reference_loso_leg(args)
        except Exception as exc:                          # never take the reference line down
            line["loso"] = {"unavailable": f"{type(exc).__name__}: {exc}"}
    print(json.dumps(line), flush=True)


def run_ours(args):
    import torch
    import torch.distributed as dist
    from multimodalsignal_b200 import _ext
    from multimodalsignal_b200.models import CnnGruAttentionModel
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _ext.lib()

    B, Cc, T = args.batch, args.channels, args.seq_len
    torch.manual_seed(42 + rank)                          # per-fold seeding (SURVEY §7 hard part 5)
    model = CnnGruAttentionModel(Cc, 2, dropout=0.5).to(dev).train()
    opt = FlatAdam(model, lr=1e-3, weight_decay=1e-4)
    step = FusedTrainStep(model, opt, B, T, use_graph=not args.no_graph)

    NB = 48
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    pool_x = torch.randn(NB, B, Cc, T, device=dev, generator=gen)
    pool_y = torch.randint(0, 2, (NB, B), device=dev, generator=gen)
    pool_x[:, :, 0, :] += pool_y[:, :, None].float() * 0.5
    NH = 8
    host_x = torch.randn(NH, B, Cc, T).pin_memory()
    host_y = torch.randint(0, 2, (NH, B)).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    l0 = lib.mms_launch_count()
    step(pool_x[0], pool_y[0])                            # eager: counts the kernels of one step
    torch.cuda.synchronize()
    kernels_per_step = int(lib.mms_launch_count() - l0)
    for i in range(1, max(args.warmup, 3)):
        step(pool_x[i % NB], pool_y[i % NB])
    barrier()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()

    # ---- value: device-resident inputs -------------------------------------------------------
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for i in range(args.steps):
        step(pool_x[i % NB], pool_y[i % NB])
    ev1.record()
    barrier()
    ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    loss_after = step.last_loss()
    if args.dump_outputs:                                 # before the e2e loop below trains the same model further
        dump_outputs(Path(args.dump_outputs), step, model, f"rank{rank}_" if world > 1 else "")

    # ---- e2e: pinned host batch -> H2D -> step -> loss.item() every step ----------------------
    # warm-up of THIS path (copy stream, pinned loss ring, prefetch pipeline): the same loop, untimed
    step.prefetch(host_x[0], host_y[0])
    wt = None
    for i in range(max(args.warmup, 3)):
        step.prefetch(host_x[(i + 1) % NH], host_y[(i + 1) % NH])
        step.run_prefetched()
        nt = step.post_loss()
        if wt is not None:
            step.read_loss(wt)
        wt = nt
    step.run_prefetched()
    step.read_loss(wt)
    torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    sink = 0.0
    step.prefetch(host_x[0], host_y[0])                   # same look-ahead pipeline Trainer.train uses
    ticket = None
    for i in range(args.steps):
        if i + 1 < args.steps:
            step.prefetch(host_x[(i + 1) % NH], host_y[(i + 1) % NH])   # H2D of batch i+1 on the copy stream
        step.run_prefetched()
        nxt_ticket = step.post_loss()                     # async D2H of this step's loss (pinned ring)
        if ticket is not None:
            sink += step.read_loss(ticket)                # every step's loss is read on the host, one step late
        ticket = nxt_ticket
    sink += step.read_loss(ticket)
    e1.record()
    torch.cuda.synchronize()
    e2e_ms = torch.tensor([max(e0.elapsed_time(e1), 1e3 * (time.perf_counter() - t0))], device=dev)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_total = float(e2e_ms.item())

    # keep the sampler under the same load until it has a few samples
    if rank == 0:
        t_end = time.perf_counter() + 1.5
        while len(sampler.rows) < 5 and time.perf_counter() < t_end + 3.0:
            for i in range(50):
                step(pool_x[i % NB], pool_y[i % NB])
            torch.cuda.synchronize()
        clocks = sampler.stop()
    barrier()

    # ---- sub-records: BASELINE.json configs[2..4] in the same driver-run line (every rank takes part in the sharded legs) ----
    sub = {}
    if not args.no_subrecords and args.workload == "train_step":
        import copy
        largs = copy.copy(args)
        largs.subjects, largs.minutes, largs.epochs, largs.concurrent_folds = 15, 100.0, 100, 4
        try:
            sub["loso"], streams, mine = loso_measure(largs, world, rank, local, init_pg=False)
        except Exception as exc:                          # a sub-record must never take the headline down
            sub["loso"], streams, mine = {"unavailable": f"{type(exc).__name__}: {exc}"}, None, None
        if world > 1:
            dp = {}
            for exch in ("peer", "nccl"):
                try:
                    dp[exch] = dp_measure(args, world, rank, dev, 256, 14, 3840, 200, exch)
                except Exception as exc:
                    dp[exch] = {"unavailable": f"{type(exc).__name__}: {exc}"}
            sub["dp"] = dict(dp.get("peer", {}), nccl={k: dp["nccl"].get(k) for k in ("value", "ms_per_step", "unavailable") if k in dp["nccl"]})
        elif rank == 0:
            if streams is not None and not args.no_cpu_baseline:
                try:
                    sub["loso"]["fold_vs_reference"] = fold_parity_measure(largs, streams)
                    sub["loso"]["accuracy_delta_vs_reference"] = sub["loso"]["fold_vs_reference"].get("accuracy_delta_vs_reference")
                except Exception as exc:
                    sub["loso"]["fold_vs_reference"] = {"unavailable": f"{type(exc).__name__}: {exc}"}
            try:
                largs.steps = 3
                sub["preprocess"] = preprocess_measure(largs, mine)
            except Exception as exc:
                sub["preprocess"] = {"unavailable": f"{type(exc).__name__}: {exc}"}
            sub["dp"] = {"unavailable": "intra-fold data parallelism needs N > 1 (measured in the N = 2, 4, 8 lines)"}
        streams = mine = None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- live per-kernel times of the same step (eager, event-bracketed launches) -------------
    PROF_STEPS = 20
    lib.mms_set_side_streams(0)                           # serialised launches -> clean per-kernel durations
    lib.mms_profile_enable(1)
    for i in range(PROF_STEPS):
        step.load(pool_x[i % NB], pool_y[i % NB])
        step._enqueue()
    buf = (__import__("ctypes").c_char * 16384)()
    lib.mms_profile_report(buf, 16384)
    lib.mms_profile_enable(0)
    lib.mms_set_side_streams(1)
    kern = {}
    for line in buf.value.decode().strip().splitlines():
        name, cnt, tot = line.rsplit(" ", 2)
        kern[name] = {"launches_per_step": int(cnt) / PROF_STEPS, "ms_per_step": float(tot) / PROF_STEPS,
                      "avg_us": 1e3 * float(tot) / int(cnt)}
    kern_total = sum(k["ms_per_step"] for k in kern.values())
    top = max(kern, key=lambda k: kern[k]["ms_per_step"])

    pk = peaks()
    H, L, O = 64, model_seq_len(T), 32
    M = B * L
    # algorithmic FLOPs per step of the GEMM-shaped kernels (2 FLOP per MAC, minimal counts, SURVEY §8d):
    #   GRU kernels: recurrent mat-vec, layer 0 both directions (2L steps) + top layer forward (L) + its 1 reverse step
    #   tc_gemm_nt : gi0 [M x 6H x O], gi_top [M x 3H x 2H], dx_top [M x 2H x 3H], dseq [M x O x 6H]
    #   tc_gemm_tn : dW_ih / dW_hh of the top forward direction and of both layer-0 directions
    gru_flops = 2.0 * 3 * H * H * B * (2 * L + L + 1)
    flops_by_kernel = {
        "gru_fwd_v2_kernel": gru_flops, "gru_bwd_ring_kernel": gru_flops, "gru_fwd_kernel": gru_flops, "gru_bwd_kernel": gru_flops,
        "tc_gemm_nt_kernel": 2.0 * M * (6 * H * O + 3 * H * 2 * H + 2 * H * 3 * H + O * 6 * H),
        "tc_gemm_tn_batch_kernel": 2.0 * M * 3 * H * ((2 * H + H) + 2 * (O + H)),
        "tc_gemm_tn_kernel": 2.0 * M * 3 * H * ((2 * H + H) + 2 * (O + H)),
    }
    # weight-gradient kernels and weight transposes run on side streams, hidden behind the recurrences
    # algorithmic HBM bytes per step of the recurrence kernels (every operand row read or written exactly once):
    #   forward : read gi (3H) + write h (H) + write the stash (r, z, n, W_hn h + b_hn: 4H)         = 8H floats per (b, t, direction)
    #   backward: read stash (4H) + h_{t-1} (H) + upstream gradient (H) + write D (dr, dz, dn, dq: 4H) = 10H floats
    # over 2L direction-steps of layer 0 plus L + 1 of the top layer
    dir_steps = B * (2 * L + L + 1)
    bytes_by_kernel = {"gru_fwd_v2_kernel": 4.0 * 8 * H * dir_steps, "gru_bwd_ring_kernel": 4.0 * 10 * H * dir_steps,
                       "gru_fwd_kernel": 4.0 * 8 * H * dir_steps, "gru_bwd_kernel": 4.0 * 10 * H * dir_steps}
    overlapped = {"tc_gemm_tn_kernel", "tc_gemm_tn_batch_kernel", "gemm_tn_acc_kernel", "conv1d_wgrad_kernel", "transpose_pad_kernel", "transpose_pad_multi_kernel",
                  "wgrad_reduce_kernel", "conv2_w_relayout_kernel", "head_bwd_kernel", "gemm_nn_kernel", "dropout_rows_kernel", "gemm_nt_bias_kernel", "gemm_skinny_kernel"}
    critical = {k: v for k, v in kern.items() if k not in overlapped}
    top = max(critical, key=lambda k: critical[k]["ms_per_step"])
    # DRAM traffic of the SAME kernel (name as launched, template arguments ignored) from the ncu --set full capture of this
    # round's default step: profiles/r2_ncu_full_summary.json (tools/ncu_summary.py over gpurun_out/r2c6_default + r2c8_convbwd)
    traffic, traffic_src = None, None
    for summ in (ROOT / "profiles" / "r2_ncu_full_summary.json",):
        if summ.exists():
            recs = [r for k, v in json.loads(summ.read_text()).items() if k.split("<")[0] == top for r in v]
            if recs:
                traffic = sum(r["dram_read_bytes"] + r["dram_write_bytes"] for r in recs) / len(recs)
                traffic_src = (f"profiles/{summ.name}: ncu --set full of {top}, dram__bytes_read.sum + dram__bytes_write.sum, mean of its "
                               f"{len(recs)} launches in one step (cold L2: ncu flushes the caches between replays)")
    launches = kern[top]["launches_per_step"]
    flop_launch = flops_by_kernel[top] / launches if top in flops_by_kernel else None
    byte_launch = bytes_by_kernel[top] / launches if top in bytes_by_kernel else None
    t_launch = kern[top]["avg_us"] * 1e-6
    # which roof bounds the kernel: operational intensity against the ridge point of the measured peaks
    ridge = pk["bf16_tflops_sustained"] * 1e12 / (pk["hbm_gbs"] * 1e9)
    hbm_bound = byte_launch is not None and (flop_launch is None or flop_launch / byte_launch < ridge)
    roof = {"kernel": top, "avg_us": kern[top]["avg_us"], "launches_per_step": launches,
            "share_of_critical_path_kernel_time": kern[top]["ms_per_step"] / sum(v["ms_per_step"] for v in critical.values()),
            "selection": "largest per-step time among kernels on the step's critical path (side-stream kernels excluded)",
            "traffic": traffic, "traffic_source": traffic_src, "ns_per_time_step": 1e3 * kern[top]["avg_us"] / L if top.startswith("gru_") else None}
    if hbm_bound:
        roof.update({"bound": "hbm", "unit": "GB/s", "peak": pk["hbm_gbs"], "peak_source": f"{pk['source']} HBM copy bandwidth",
                     "achieved": byte_launch / t_launch / 1e9, "algorithmic_bytes_per_launch": byte_launch,
                     "operational_intensity_flop_per_byte": flop_launch / byte_launch if flop_launch else None,
                     "ridge_flop_per_byte": ridge})
        roof["frac"] = roof["achieved"] / roof["peak"]
        if flop_launch:
            roof["tensor_view"] = {"flop_per_launch": flop_launch, "achieved_tflops": flop_launch / t_launch / 1e12,
                                   "frac_of_bf16_sustained": flop_launch / t_launch / 1e12 / pk["bf16_tflops_sustained"]}
        roof["note"] = ("fp32 recurrence: ~10 FLOP per byte, far below the ridge, so HBM is the roof that bounds it; what it actually "
                        f"runs into is latency -- 240 serial time steps per launch, {1e3 * kern[top]['avg_us'] / L:.0f} ns per time step")
    elif flop_launch:
        roof.update({"bound": "tensor", "unit": "TFLOP/s", "peak": pk["bf16_tflops_sustained"],
                     "peak_source": f"{pk['source']} bf16 sustained (kernel timed inside a long step)",
                     "achieved": flop_launch / t_launch / 1e12, "flop_per_launch": flop_launch, "note": "3xTF32 tcgen05 GEMM"})
        roof["frac"] = roof["achieved"] / roof["peak"]
    else:
        roof.update({"bound": "hbm", "unit": "GB/s", "peak": pk["hbm_gbs"], "achieved": None, "frac": None})
    kernel_table = {k: {"ms_per_step": round(v["ms_per_step"], 5), "launches_per_step": v["launches_per_step"],
                        "avg_us": round(v["avg_us"], 2), "side_stream": k in overlapped,
                        "tflops": round(flops_by_kernel[k] / (v["ms_per_step"] * 1e-3) / 1e12, 3) if k in flops_by_kernel else None}
                    for k, v in kern.items()}

    value = world * B * args.steps / (ms_total * 1e-3)
    e2e_value = world * B * args.steps / (e2e_total * 1e-3)
    fpw = FLOP_PER_WINDOW.get((Cc, T))
    line = {
        "metric": "train windows/sec (fwd+bwd+Adam) CnnGruAttention",
        "value": value, "unit": "windows/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": config_dict(args, world),
        "e2e": {"value": e2e_value, "unit": "windows/s", "ms_per_step": e2e_total / args.steps,
                "h2d_bytes_per_step": B * Cc * T * 4 + B * 8, "d2h_bytes_per_step": 4},
        "gpu_launches": kernels_per_step * args.steps, "kernels_per_step": kernels_per_step,
        "cuda_graph": not args.no_graph, "clocks": clocks, "roofline": roof,
        "step_roofline": {"flop_per_window": fpw, "achieved_tflops": (value / world) * fpw / 1e12 if fpw else None,
                          "frac_of_bf16_sustained": (value / world) * fpw / 1e12 / pk["bf16_tflops_sustained"] if fpw else None},
        "kernels": kernel_table,
        "eager_kernel_ms_per_step": kern_total, "final_loss": loss_after,
    }
    line.update(sub)
    if world == 1 and not args.no_library_baseline:
        try:
            line["library_gpu_baseline"] = library_gpu_run(args, dev)
            lg = line["library_gpu_baseline"]
            if "value" in lg:
                lg["ours_over_library"] = value / lg["value"]
                lg["ours_over_library_e2e"] = e2e_value / lg["pytorch_default"]["e2e_value"]
        except Exception as exc:                          # the baseline leg must never take the bench line down
            line["library_gpu_baseline"] = {"unavailable": f"{type(exc).__name__}: {exc}"}
    if not args.no_cpu_baseline and world == 1:
        r = cpu_reference_run(args, steps=10 ** 6, warmup=2, budget_s=args.cpu_seconds)
        line["cpu_baseline"] = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, step, model, prefix=""):
    """What a caller of the fused training step holds after its last call: the loss, the logits, the flat gradient and
    every state_dict entry (updated parameters, BatchNorm statistics), as float32 (integers as float64).  Independent of
    T, and of B apart from the logits: about 1 MB at the default configuration."""
    import numpy as np
    out_dir.mkdir(parents=True, exist_ok=True)
    arrays = {"loss": step.loss, "logits": step.logits, "grads": step.opt.grads}
    arrays.update({f"state.{k}": v for k, v in model.state_dict().items()})
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        np.save(out_dir / f"{prefix}{name}.npy", a.astype(np.float32 if a.dtype.kind == "f" else np.float64))


def model_seq_len(T):
    l1 = (T + 6 - 7) // 2 + 1
    p1 = (l1 - 1) // 2 + 1
    l2 = (p1 + 4 - 5) // 2 + 1
    return (l2 - 1) // 2 + 1


NORTH_STAR_CHANNELS = ["chest_ECG", "chest_EDA", "chest_EMG", "chest_Resp", "wrist_BVP", "wrist_EDA"]   # README.md:85


def _synthetic_subjects(args, rank=0, world=1):
    """The synthetic recordings of the subjects rank ``rank`` owns (subject i belongs to rank i % world), generated on a
    small thread pool (numpy releases the GIL): (all subject ids, {sid: SyntheticSubject}, protocol)."""
    from concurrent.futures import ThreadPoolExecutor
    from multimodalsignal_b200 import synth
    sids = synth.ALL_SUBJECTS[:args.subjects]
    protocol = synth.FULL_PROTOCOL if args.minutes >= 80 else synth.SHORT_PROTOCOL
    mine = [sid for i, sid in enumerate(sids) if i % world == rank]
    with ThreadPoolExecutor(max(1, min(8, (os.cpu_count() or 1) // max(1, world)))) as ex:
        subs = list(ex.map(lambda sid: synth.make_subject(sid, synth.ALL_SUBJECTS.index(sid), minutes=args.minutes, protocol=protocol), mine))
    return sids, dict(zip(mine, subs)), protocol


def preprocess_measure(args, subjects=None):
    """BASELINE.json configs[3]: resample (700/64/32/4 Hz -> 64 Hz) + windowing of synthetic recordings, chest 8 +
    wrist 6 channels.  value = subjects/s with the raw recordings resident in HBM; e2e includes the H2D copy of
    the raw streams and the D2H copy of the float64 window array the reference saves (preprocess.py:217-222)."""
    import numpy as np
    import torch
    from multimodalsignal_b200 import _ext, preprocess as pp
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    lib = _ext.lib()
    if subjects is None:
        sids, subjects, _ = _synthetic_subjects(args)
    sids = list(subjects.keys())
    subs = [subjects[sid] for sid in sids]
    datas = [s.as_pickle_dict() for s in subs]
    protos = [pp.base_halving_quirk(s.sid, s.protocol) for s in subs]

    def on_device(i):
        chest = {k.decode(): v for k, v in datas[i][b"signal"][b"chest"].items()}
        wrist = {k.decode(): v for k, v in datas[i][b"signal"][b"wrist"].items()}
        dev = torch.device("cuda", torch.cuda.current_device())
        up = pp._UPLOADER                                                # pinned, threaded staging (what preprocess_subject uses)
        staged = up.groups([up._columns(chest, pp.CHEST_CHANNELS)] + [up._columns(wrist, [n]) for n in pp.WRIST_CHANNELS], dev)
        return staged[0], dict(zip(pp.WRIST_CHANNELS, staged[1:]))

    def process(rows, wr, proto, want_windows):
        streams = pp.resample_subject_rows(rows, wr, 64)                # what preprocess_subject does with the staged rows
        starts, labels, window = pp.window_plan(proto, 64)
        sub = pp.SubjectStreams("S", streams, starts, labels, window, pp.CHEST_CHANNEL_NAMES + pp.WRIST_CHANNEL_NAMES)
        return sub.windows_f64() if want_windows else sub, len(labels), window

    staged = [on_device(i) for i in range(len(subs))]
    torch.cuda.synchronize()
    for i in range(len(subs)):                                          # warm-up: every subject once (each has its own lengths -> its own
        process(*staged[i], protos[i], True)                            # workspace sizes in the caching allocator)
    torch.cuda.synchronize()
    sampler = ClockSampler(torch.cuda.current_device())
    sampler.start()
    time.sleep(0.4)                                                     # nvidia-smi's start-up (NVML initialisation) stalls launches: keep it out of
    l0 = lib.mms_launch_count()                                         # a region that is ~100 host-enqueued launches per subject
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = args.steps                                                   # 15 subjects per pass, ~26 ms per pass
    e0.record()
    nwin = 0
    for _ in range(reps):
        for i in range(len(subs)):
            w, n, window = process(*staged[i], protos[i], True)
            nwin += n
            del w
    e1.record()
    torch.cuda.synchronize()
    dev_s = e0.elapsed_time(e1) * 1e-3
    launches = int(lib.mms_launch_count() - l0)
    # e2e: host arrays in, host float64 windows out -- a three-stage software pipeline over the subjects: while subject i is
    # staged (pinned, threaded), copied up and resampled on the compute stream, the window array of subject i-1 travels back on
    # a copy stream into one of two pinned buffers (what run_preprocessing does with _NpyWriter, minus the file system)
    copy_stream = torch.cuda.Stream()
    out_elems = int(max(n for _, n, _ in [process(*staged[i], protos[i], False) for i in range(len(subs))]) * window * 14 * 1.05)
    pinned = [torch.empty(out_elems, dtype=torch.float64).pin_memory() for _ in range(2)]     # the caller's destination arrays
    pinned_free = [None, None]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    h2d = d2h = 0
    pending = None

    def drain(item):
        nonlocal d2h
        w, ev, slot = item
        if pinned[slot] is None or pinned[slot].numel() < w.numel():
            pinned[slot] = torch.empty(int(w.numel() * 1.25), dtype=torch.float64).pin_memory()
        if pinned_free[slot] is not None:
            pinned_free[slot].synchronize()                             # the host has consumed what this buffer held before
        copy_stream.wait_event(ev)
        with torch.cuda.stream(copy_stream):
            host = pinned[slot][:w.numel()].view(w.shape)
            host.copy_(w, non_blocking=True)                            # the float64 window array preprocess.py:218 saves
            w.record_stream(copy_stream)
            done = torch.cuda.Event()
            done.record(copy_stream)
        pinned_free[slot] = done
        d2h += w.numel() * 8

    for i in range(len(subs)):
        rows, wr = on_device(i)
        h2d += rows.numel() * 8 + sum(v.numel() * 8 for v in wr.values())
        w, n, window = process(rows, wr, protos[i], True)
        ev = torch.cuda.Event()
        ev.record()
        if pending is not None:
            drain(pending)
        pending = (w, ev, i & 1)
    drain(pending)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    clocks = sampler.stop()
    # algorithmic bytes (SURVEY §8d): read every source sample once as stored + write the windows
    src_bytes = sum(sum(np.asarray(v).size for v in d[b"signal"][b"chest"].values()) * 8 +
                    sum(np.asarray(v).size for v in d[b"signal"][b"wrist"].values()) * 8 for d in datas)
    win_bytes = (nwin // reps) * window * 14 * 8
    algo = src_bytes + win_bytes
    pk = peaks()
    # cpu baseline: the numpy oracle (== scipy.signal.resample arithmetic) on a bounded sample: one subject, chest only
    from oracle import preprocess_oracle as po      # cpu_baseline leg only
    t0 = time.perf_counter()
    po.preprocess_subject(subs[0].sid, subs[0].chest, subs[0].protocol, 64)
    cpu_s = time.perf_counter() - t0
    line = {"metric": "preprocess subjects/sec (resample 700/64/32/4 Hz -> 64 Hz + 60 s / 10 s windowing)",
            "value": len(subs) * reps / dev_s, "unit": "subjects/s", "n_gpus": 1, "steps": reps, "warmup": 2,
            "ms_per_step": 1e3 * dev_s / reps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": {"workload": "preprocess 15 synthetic subjects, chest 8 + wrist 6 channels (BASELINE.json configs[3])",
                                            "subjects": len(subs), "minutes": args.minutes, "windows_per_pass": nwin // reps},
            "e2e": {"value": len(subs) / e2e_s, "unit": "subjects/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": launches, "clocks": clocks,
            "roofline": {"kernel": "resample + window pipeline (fft_fast_fwd_kernel / fft_fast_inv_kernel dominate)", "bound": "hbm", "unit": "GB/s",
                         "achieved": algo * reps / dev_s / 1e9, "peak": pk["hbm_gbs"], "frac": algo * reps / dev_s / 1e9 / pk["hbm_gbs"],
                         "traffic": None, "algorithmic_bytes_per_pass": algo,
                         "note": "chirp-z: 12 register-resident passes over 9 * 2^19 complex doubles per PAIR of chest signals + 6 over 9 * 2^16 "
                                 "per signal (DESIGN section 5); algorithmic bytes count the source once and the windows once"},
            "cpu_baseline": {"value": 1.0 / cpu_s, "unit": "subjects/s", "cores": os.cpu_count(), "kind": "port",
                             "sample": "oracle/preprocess_oracle.py on 1 synthetic subject, chest channels only (8 FFT round trips "
                                       "of N = 4.2 M + window stacking); the reference's scipy path measured the same arithmetic"}}
    return line


def run_preprocess(args):
    print(json.dumps(preprocess_measure(args)), flush=True)


def _gru_bytes_per_window(T, H=64):
    """Algorithmic HBM bytes of the four recurrence launches per trained window (DESIGN.md section 3): forward 8 H floats and
    backward 10 H floats per (time step, direction), over 2 L direction-steps of layer 0 + L + 1 of the top layer."""
    L = model_seq_len(T)
    return 4.0 * (8 + 10) * H * (3 * L + 1)


def loso_measure(args, world, rank, local, init_pg=True):
    """BASELINE.json configs[2]: full 15-subject LOSO-CV (main.py:91-156 semantics: 100 epochs, patience 20, batch 64,
    Adam 1e-3 / 1e-4) with the folds sharded over the ranks.  value = wall-clock seconds (max over ranks) from
    raw synthetic recordings on the host to cv_summary.txt.  Returns (record on rank 0 / None elsewhere, streams, the synthetic subjects this rank generated)."""
    import tempfile
    import numpy as np
    import torch
    import torch.distributed as dist
    from multimodalsignal_b200 import _ext, main as mm, preprocess as pp
    torch.cuda.set_device(local)
    if world > 1 and init_pg and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = _ext.lib()
    sids, mine, protocol = _synthetic_subjects(args, rank, world)
    mm.ALL_SUBJECTS = list(sids)
    mm.CHANNELS_TO_USE = list(NORTH_STAR_CHANNELS)
    mm.EPOCHS = args.epochs
    # one-time process costs (library imports, CUDA context, kernel attributes) are not LOSO work: warm them
    import sklearn.metrics  # noqa: F401
    import sklearn.model_selection  # noqa: F401
    from multimodalsignal_b200.models import CnnGruAttentionModel
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    _m = CnnGruAttentionModel(len(NORTH_STAR_CHANNELS), 2).cuda().train()
    _st = FusedTrainStep(_m, FlatAdam(_m), mm.BATCH_SIZE, 3840)
    for _ in range(3):
        _st(torch.zeros(mm.BATCH_SIZE, len(NORTH_STAR_CHANNELS), 3840, device="cuda"), torch.zeros(mm.BATCH_SIZE, dtype=torch.int64, device="cuda"))
    del _st, _m
    # ... and the preprocessing kernels' modules (lazy loading), on a 9-minute recording: its staging buffers and workspaces are
    # a fraction of what the 100-minute recordings need, so allocating those stays inside the timed region
    from multimodalsignal_b200 import synth as _synth
    _w = _synth.make_subject("S2", 0, minutes=_synth.SHORT_MINUTES, protocol=_synth.SHORT_PROTOCOL)
    pp.preprocess_subject("S2", _w.as_pickle_dict(), pp.base_halving_quirk("S2", _w.protocol), 64, include_wrist=True).windows_f64()
    del _w
    torch.cuda.synchronize()
    if world > 1:        # NCCL builds its communicator lazily at the first collective: also a one-time process cost
        _w = torch.zeros(1 << 20, device="cuda")
        dist.broadcast(_w, src=0)
        dist.all_reduce(_w)
        dist.barrier()
        del _w
    l0 = lib.mms_launch_count()
    t0 = time.perf_counter()
    # every rank keeps all subjects resident (replicated, ~0.65 GB); the resampling itself is sharded over the ranks
    # and the streams are exchanged GPU-to-GPU (NCCL broadcast over NVLink)
    items = [(sid, (mine[sid].as_pickle_dict if sid in mine else (lambda: None)), pp.base_halving_quirk(sid, protocol)) for sid in sids]
    streams = pp.preprocess_subjects_sharded(items, 64, include_wrist=True)
    torch.cuda.synchronize()
    t_pre = time.perf_counter() - t0
    out_dir = Path(tempfile.mkdtemp(prefix="mms_loso_"))
    import contextlib
    import io
    fold_times = []

    def timed_fold(*a):
        tf = time.perf_counter()
        r = mm.run_fold(*a)
        torch.cuda.synchronize()
        r["seconds"] = time.perf_counter() - tf
        fold_times.append(r["seconds"])
        return r

    with contextlib.redirect_stdout(io.StringIO()):
        results = mm.run_simple_experiment(out_dir, None, pp.CHEST_CHANNEL_NAMES + pp.WRIST_CHANNEL_NAMES, subject_streams=streams,
                                           fold_fn=timed_fold if args.concurrent_folds <= 1 else None,
                                           concurrent_folds=args.concurrent_folds)
    torch.cuda.synchronize()
    total = torch.tensor([time.perf_counter() - t0], device="cuda")
    if world > 1:
        dist.all_reduce(total, op=dist.ReduceOp.MAX)
    launches = int(lib.mms_launch_count() - l0)
    if rank != 0:
        return None, streams, mine
    windows = sum(r["windows_trained"] for r in results)
    secs = float(total.item())
    pk = peaks()
    wps = windows / max(1e-9, secs - t_pre)
    gbs = wps * _gru_bytes_per_window(3840) / 1e9
    line = {"metric": "15-fold LOSO wall-clock (preprocess + train + evaluate)", "value": secs, "unit": "s",
            "n_gpus": world, "steps": len(results), "warmup": 0, "ms_per_step": 1e3 * secs / max(1, len(results)),
            "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "cnn_gru_attention full LOSO-CV, folds sharded over ranks (BASELINE.json configs[2])",
                       "subjects": len(sids), "channels": NORTH_STAR_CHANNELS, "epochs_max": args.epochs, "patience": mm.PATIENCE,
                       "batch": mm.BATCH_SIZE, "minutes": args.minutes, "concurrent_folds_per_gpu": args.concurrent_folds},
            "preprocess_s": t_pre, "windows_trained": windows, "train_windows_per_s": wps,
            "accuracy_mean": float(np.mean([r["accuracy"] for r in results])),
            "f1_mean": float(np.mean([r["f1_score"] for r in results])),
            "roofline": {"kernel": "gru_fwd_v2_kernel + gru_bwd_ring_kernel (the recurrences of every co-resident fold)", "bound": "hbm",
                         "unit": "GB/s", "achieved": gbs, "peak": pk["hbm_gbs"], "frac": gbs / pk["hbm_gbs"], "traffic": None,
                         "algorithmic_bytes_per_window": _gru_bytes_per_window(3840),
                         "note": "whole-job figure: windows trained per second of the train + evaluate phase x the recurrences' "
                                 "algorithmic bytes per window, all GPUs together"},
            "folds": [{k: r[k] for k in ("subject", "accuracy", "f1_score", "windows_trained", "seconds", "start_s", "end_s") if k in r} for r in results],
            "host_seconds_by_phase": {k: round(sum(r.get("timing", {}).get(k, 0.0) for r in results), 3)
                                      for k in ("train_enqueue", "train_wait", "evaluate", "bookkeeping")},
            "gpu_launches_rank0_uncaptured": launches,
            "summary_file": str(out_dir / "cv_summary.txt")}
    line["roofline"]["peak"] = pk["hbm_gbs"] * world
    line["roofline"]["frac"] = gbs / (pk["hbm_gbs"] * world)
    return line, streams, mine


def run_loso(args):
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    line, streams, _ = loso_measure(args, world, rank, local)
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            try:
                line["fold_vs_reference"] = fold_parity_measure(args, streams)
            except Exception as exc:
                line["fold_vs_reference"] = {"unavailable": f"{type(exc).__name__}: {exc}"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ---- matched accuracy: one LOSO fold through the UNMODIFIED reference Trainer (CPU) and through ours (B200) --------------
PARITY_FOLD = "S2"            # BASELINE.md 4.3: fold "test S2"
PARITY_EPOCHS = 2


def _write_reference_npy(streams, out_dir, channels):
    """The .npy files reference dataset.py:25-36 loads, for the channels in use only: {sid}_X.npy float64 [N, W, C],
    {sid}_y.npy, _channel_names.txt -- from the device-resident streams of our preprocessing (byte-identical to what the
    reference's run_preprocessing writes: tests/test_gpu_preprocess.py)."""
    import numpy as np
    out_dir.mkdir(parents=True, exist_ok=True)
    (out_dir / "_channel_names.txt").write_text("".join(f"{c}\n" for c in channels))
    for sid, sub in streams.items():
        if not len(sub.labels):
            continue
        idx = [sub.channel_names.index(c) for c in channels]
        w = sub.windows_f64(idx)                    # [N, W, len(channels)] float64 on the device
        np.save(out_dir / f"{sid}_X.npy", w.cpu().numpy())
        np.save(out_dir / f"{sid}_y.npy", np.asarray(sub.labels))
        del w


def reference_fold_run(data_dir, channels, sids, epochs=PARITY_EPOCHS, fold=PARITY_FOLD, dropout=0.0, threads=None):
    """Fold ``fold`` of reference main.py:98-125 -- the reference's own WesadDataset, DataLoader, CnnGruAttentionModel and
    Trainer, unmodified, on the host cores -- for ``epochs`` epochs.  dropout = 0 makes the run deterministic, so that ours
    (same initial weights, same batch order) must reproduce it to fp32 rounding.  Returns losses, accuracy, F1, seconds."""
    import contextlib
    import io
    import tempfile
    import warnings
    import numpy as np
    import torch
    from torch.utils.data import DataLoader
    from oracle import ref_harness
    from multimodalsignal_b200 import main as mm
    ds_mod, models, trainer_mod = ref_harness.load("dataset"), ref_harness.load("models"), ref_harness.load("trainer")
    torch.set_num_threads(threads or os.cpu_count() or 1)
    names = (Path(data_dir) / "_channel_names.txt").read_text().split()
    train_s, val_s = mm.fold_split(fold, list(sids))                      # main.py:102-103 (sklearn, seed 42)
    mk = lambda subs: ds_mod.WesadDataset(Path(data_dir), subs, channels, names, classification_mode="stress_binary")
    torch.manual_seed(42)
    np.random.seed(42)
    t_load = time.perf_counter()
    train_ds, val_ds, test_ds = mk(train_s), mk(val_s), mk([fold])
    t_load = time.perf_counter() - t_load
    tl = DataLoader(train_ds, batch_size=64, shuffle=True, num_workers=0)
    vl = DataLoader(val_ds, batch_size=64, shuffle=False, num_workers=0)
    te = DataLoader(test_ds, batch_size=64, shuffle=False, num_workers=0)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model = models.CnnGruAttentionModel(in_channels=len(channels), num_classes=2, cnn_out_channels=32, gru_hidden_size=64,
                                            gru_num_layers=2, dropout=dropout)
    init = {k: v.clone() for k, v in model.state_dict().items()}
    cfg = {'trainer': {'epochs': epochs, 'learning_rate': 1e-3, 'early_stopping': {'enabled': True, 'patience': 20, 'delta': 0},
                       'weight_decay': 1e-4}}
    tmp = Path(tempfile.mkdtemp(prefix="mms_ref_fold_"))
    dev_was = torch.cuda.is_available
    torch.cuda.is_available = lambda: False          # trainer.py:57 picks cuda when it can: this leg is the CPU path
    try:
        with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
            tr = trainer_mod.Trainer(model, tmp / "fold", cfg)
            t0 = time.perf_counter()
            tr.train(tl, vl)
            t_train = time.perf_counter() - t0
            test_loss, test_acc, test_f1 = tr.evaluate(te, is_test=True)
    finally:
        torch.cuda.is_available = dev_was
    log = (tmp / "fold" / "training_log.txt").read_text(encoding="utf-8")
    return {"fold": fold, "epochs": epochs, "dropout": dropout, "n_train": len(train_ds), "n_val": len(val_ds), "n_test": len(test_ds),
            "train_seconds": t_train, "dataset_seconds": t_load, "windows_per_s": epochs * len(train_ds) / t_train,
            "test_loss": float(test_loss), "test_accuracy": float(test_acc), "test_f1": float(test_f1), "log": log,
            "init": init, "train_subjects": train_s, "val_subjects": val_s, "cores": torch.get_num_threads()}


def reference_loso_leg(args, minutes=100.0):
    """The reference arm's LOSO figure (BASELINE.md 4.3): fold "test S2" of the 15-subject protocol for PARITY_EPOCHS epochs
    through the reference's own dataset.py / models.py / trainer.py on the host cores, on the same synthetic recordings as
    our arm (windows by the numpy restatement of preprocess.py: no GPU code on this path), and the extrapolation to 15 folds."""
    import copy
    import shutil
    import tempfile
    from concurrent.futures import ThreadPoolExecutor
    import numpy as np
    from oracle import preprocess_oracle as po, ref_harness
    if not ref_harness.available():
        return {"unavailable": "reference modules not staged under baseline/_ref"}
    largs = copy.copy(args)
    largs.subjects, largs.minutes = 15, minutes
    t0 = time.perf_counter()
    sids, subs, protocol = _synthetic_subjects(largs)
    root = Path(tempfile.mkdtemp(prefix="mms_ref_loso_"))
    data_dir = root / "data" / "all_raw"
    data_dir.mkdir(parents=True)
    (data_dir / "_channel_names.txt").write_text("".join(f"{c}\n" for c in NORTH_STAR_CHANNELS))
    wrist_fs = {"BVP": 64, "EDA": 4}

    def prep(sid):
        sub = subs[sid]
        res = {}
        for name in NORTH_STAR_CHANNELS:
            where, ch = name.split("_")
            if where == "chest":
                res[name] = po.resample_signal(sub.chest[ch], 700, 64)
        num = len(next(iter(res.values())))
        for name in NORTH_STAR_CHANNELS:
            where, ch = name.split("_")
            if where == "wrist":
                y = po.resample_signal(sub.wrist[ch], wrist_fs[ch], 64)
                if len(y) < num:
                    y = np.concatenate([y, np.repeat(y[-1:], num - len(y), axis=0)], axis=0)
                res[name] = y[:num]
        starts, labels, w = po.window_plan(po.apply_subject_quirk(sid, protocol), 64)
        X = np.stack([np.stack([res[c][a:a + w, 0] for c in NORTH_STAR_CHANNELS], axis=1) for a in starts]) if len(starts) else np.zeros((0, w, 6))
        np.save(data_dir / f"{sid}_X.npy", X)
        np.save(data_dir / f"{sid}_y.npy", np.asarray(labels))
        return len(labels)

    try:
        with ThreadPoolExecutor(max(1, min(8, os.cpu_count() or 1))) as ex:
            nwin = sum(ex.map(prep, sids))
        t_prep = time.perf_counter() - t0
        ref = reference_fold_run(data_dir, NORTH_STAR_CHANNELS, sids)
    finally:
        shutil.rmtree(root, ignore_errors=True)
    per_epoch = ref["train_seconds"] / PARITY_EPOCHS
    return {"metric": "LOSO fold wall-clock, reference Trainer on the host cores", "fold": PARITY_FOLD, "epochs": PARITY_EPOCHS, "dropout": 0.0,
            "cores": ref["cores"], "windows_total": nwin, "n_train": ref["n_train"], "n_val": ref["n_val"], "n_test": ref["n_test"],
            "preprocess_and_generate_s": t_prep, "train_seconds": ref["train_seconds"], "seconds_per_epoch": per_epoch,
            "windows_per_s": ref["windows_per_s"], "test_accuracy": ref["test_accuracy"], "test_f1": ref["test_f1"],
            "test_loss": ref["test_loss"], "epoch_losses": _log_losses(ref["log"]),
            "extrapolated_15_fold_s": 15 * 40 * per_epoch,
            "extrapolation": "15 folds x ~40 epochs (where early stopping ends the synthetic folds in our GPU run) x the measured seconds per epoch"}


def _log_losses(log):
    """(train loss, validation loss) per epoch from a training_log.txt of reference trainer.py:171-176 (ours writes the same lines)."""
    import re
    return [(float(a), float(b)) for a, b in re.findall(r"训练损失: ([0-9.eE+-]+).*?验证损失: ([0-9.eE+-]+)", log)]


def fold_parity_measure(args, streams):
    """north_star "matched accuracy against the reference": fold S2, 2 epochs, dropout 0 (deterministic), the SAME .npy files,
    initial weights and batch order through the reference Trainer on the host cores and through ours on the GPU."""
    import contextlib
    import io
    import shutil
    import tempfile
    import torch
    from torch.utils.data import DataLoader
    from oracle import ref_harness
    if not ref_harness.available():
        return {"unavailable": "reference modules not staged under baseline/_ref"}
    from multimodalsignal_b200 import main as mm
    from multimodalsignal_b200.dataset import WesadDataset
    from multimodalsignal_b200.models import CnnGruAttentionModel
    from multimodalsignal_b200.trainer import Trainer
    sids = list(streams.keys())
    root = Path(tempfile.mkdtemp(prefix="mms_parity_"))
    try:
        data_dir = root / "data" / "all_raw"
        _write_reference_npy(streams, data_dir, NORTH_STAR_CHANNELS)
        ref = reference_fold_run(data_dir, NORTH_STAR_CHANNELS, sids)
        # ours: the file path of run_fold_async (the reference's data flow), same seed -> same shuffle order, same initial weights
        torch.manual_seed(42)
        import numpy as np
        np.random.seed(42)
        names = (data_dir / "_channel_names.txt").read_text().split()
        mk = lambda subs: WesadDataset(data_dir, subs, NORTH_STAR_CHANNELS, names, classification_mode="stress_binary")
        train_ds, val_ds, test_ds = mk(ref["train_subjects"]), mk(ref["val_subjects"]), mk([PARITY_FOLD])
        tl = DataLoader(train_ds, batch_size=64, shuffle=True, num_workers=0, pin_memory=True)
        vl = DataLoader(val_ds, batch_size=64, shuffle=False, num_workers=0, pin_memory=True)
        te = DataLoader(test_ds, batch_size=64, shuffle=False, num_workers=0, pin_memory=True)
        model = CnnGruAttentionModel(in_channels=len(NORTH_STAR_CHANNELS), num_classes=2, cnn_out_channels=32, gru_hidden_size=64,
                                     gru_num_layers=2, dropout=0.0)
        same_init = all(torch.equal(v, ref["init"][k]) for k, v in model.state_dict().items())
        if not same_init:
            model.load_state_dict(ref["init"])
        cfg = {'trainer': {'epochs': PARITY_EPOCHS, 'learning_rate': 1e-3, 'early_stopping': {'enabled': True, 'patience': 20, 'delta': 0},
                           'weight_decay': 1e-4}}
        with contextlib.redirect_stdout(io.StringIO()):
            tr = Trainer(model, root / "fold_ours", cfg)
            t0 = time.perf_counter()
            tr.train(tl, vl)
            torch.cuda.synchronize()
            t_ours = time.perf_counter() - t0
            test_loss, test_acc, test_f1 = tr.evaluate(te, is_test=True)
        ours_losses = _log_losses((root / "fold_ours" / "training_log.txt").read_text(encoding="utf-8"))
        ref_losses = _log_losses(ref["log"])
        n = min(len(ours_losses), len(ref_losses))
        return {"fold": PARITY_FOLD, "epochs": PARITY_EPOCHS, "dropout": 0.0, "n_train": ref["n_train"], "n_val": ref["n_val"], "n_test": ref["n_test"],
                "same_initial_weights_from_seed": bool(same_init),
                "reference": {"kind": "unmodified reference dataset.py / models.py / trainer.py on the host cores", "cores": ref["cores"],
                              "train_seconds": ref["train_seconds"], "windows_per_s": ref["windows_per_s"], "test_loss": ref["test_loss"],
                              "test_accuracy": ref["test_accuracy"], "test_f1": ref["test_f1"], "epoch_losses": ref_losses},
                "ours": {"kind": "multimodalsignal_b200 Trainer + DataLoader on the same files (B200)", "train_seconds": t_ours,
                         "windows_per_s": PARITY_EPOCHS * ref["n_train"] / t_ours, "test_loss": float(test_loss), "test_accuracy": float(test_acc),
                         "test_f1": float(test_f1), "epoch_losses": ours_losses},
                "accuracy_delta_vs_reference": float(test_acc) - ref["test_accuracy"],
                "f1_delta_vs_reference": float(test_f1) - ref["test_f1"],
                "max_epoch_loss_delta": max([max(abs(o[0] - r[0]), abs(o[1] - r[1])) for o, r in zip(ours_losses[:n], ref_losses[:n])], default=None),
                "reference_extrapolation": {"fifteen_folds_s": 15 * ref["train_seconds"] / PARITY_EPOCHS * 40,
                                            "how": "15 folds x ~40 epochs (where early stopping ends the synthetic folds on the GPU run) x the "
                                                   "reference's measured seconds per epoch; BASELINE.md 4.3 allows the extrapolation to be stated"}}
    finally:
        shutil.rmtree(root, ignore_errors=True)


def dp_measure(args, world, rank, dev, B, Cc, T, steps, exchange):
    """BASELINE.json configs[4]: intra-fold data parallelism -- ONE fold, the global batch split over the ranks, SyncBN + one
    flat-gradient exchange per step (strong scaling).  The process group must exist.  Returns the record on every rank."""
    import torch
    import torch.distributed as dist
    from multimodalsignal_b200.models import CnnGruAttentionModel
    from multimodalsignal_b200.parallel import DataParallelTrainStep
    from multimodalsignal_b200.trainer import FlatAdam
    assert B % world == 0, "global batch must divide over the ranks"
    b = B // world
    torch.manual_seed(42)
    model = CnnGruAttentionModel(Cc, 2, dropout=0.5).to(dev).train()
    peer = "symm" if exchange == "peer" else None
    step = DataParallelTrainStep(model, FlatAdam(model, lr=1e-3, weight_decay=1e-4), b, B, T, rank=rank, peer=peer)
    gen = torch.Generator(device=dev).manual_seed(7 + rank)
    NB = 16
    px = torch.randn(NB, b, Cc, T, device=dev, generator=gen)
    py = torch.randint(0, 2, (NB, b), device=dev, generator=gen)
    for i in range(max(3, args.warmup if args.warmup < 20 else 20)):
        step(px[i % NB], py[i % NB])
    dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        step(px[i % NB], py[i % NB])
    e1.record()
    dist.barrier()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    loss = step.global_loss()
    del step
    return {"metric": "train windows/sec (fwd+bwd+Adam) CnnGruAttention, intra-fold data parallel", "value": B * steps / (ms.item() * 1e-3),
            "unit": "windows/s", "n_gpus": world, "steps": steps, "warmup": max(3, args.warmup if args.warmup < 20 else 20),
            "ms_per_step": ms.item() / steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "intra-fold data parallel (BASELINE.json configs[4])", "global_batch": B, "local_batch": b, "channels": Cc,
                       "seq_len": T, "parallelism": (f"dp{world}: SyncBN (4 x <=1 KB) + flat gradient (0.5 MB) exchanged by peer-memory kernels over NVLink, "
                                       "gradient all-reduce fused with Adam, one CUDA graph per rank") if peer else
                                      f"dp{world}: SyncBN (4 x <=1 KB all-reduce) + 1 flat gradient all-reduce (0.5 MB) per step (NCCL)",
                       "exchange": exchange, "cuda_graph": bool(peer)},
            "final_loss": loss}


def run_dp(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    line = dp_measure(args, world, rank, dev, args.batch, args.channels, args.seq_len, args.steps, args.dp_exchange)
    if rank == 0:
        print(json.dumps(line), flush=True)
    dist.destroy_process_group()


def main():
    args = parse()
    # stdout hygiene: the driver parses ONE JSON line from rank 0, but NCCL / libraries may print to fd 1
    # ("NCCL version ..."): keep a private copy of the real stdout for the JSON line and send everything
    # else to stderr.
    global print
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    import builtins

    def print(*a, **k):                      # noqa: A001 - only the JSON lines are printed by this file
        k.pop("flush", None)
        builtins.print(*a, file=real_stdout, flush=True, **k)

    if args.workload == "preprocess":
        run_preprocess(args)
    elif args.workload == "loso":
        run_loso(args)
    elif args.workload == "dp":
        run_dp(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
