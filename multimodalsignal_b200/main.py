"""Drop-in for the reference ``main.py`` (standard LOSO experiment, main.py:91-156) with the folds
sharded over the GPUs of one box.

Configuration constants, the sklearn fold split (``train_test_split(14 subjects, 0.2, seed 42)``),
the per-fold ``Trainer`` config and the ``cv_summary.txt`` format are the reference's.  What is new:

* ``python -m multimodalsignal_b200.main`` under ``torchrun --nproc-per-node N`` gives every rank
  the folds ``rank, rank + N, ...`` (LOSO folds are independent -- no collective on the data
  path); rank 0 gathers the 15 ``(accuracy, f1)`` pairs and writes the summary.
* seeding is per fold (``SEED + fold_index``) instead of once per run (main.py:71-72): a sharded
  run cannot reproduce a single global RNG stream consumed fold after fold (SURVEY §7 hard part 5).
  The sklearn split is deterministic per fold and is unchanged.
* the hierarchical experiment (main.py:159-247) is dead code upstream (SURVEY D7) and not provided.
"""
from __future__ import annotations

import os
import warnings
from datetime import datetime
from pathlib import Path

import numpy as np
import torch

warnings.filterwarnings("ignore", message="Initializing zero-element tensors is a no-op")

# --- reference configuration (main.py:20-67) -------------------------------------------------------
USE_HIERARCHICAL_CLASSIFICATION = False
RUN_NAME = 'simple_binary'
CLASSIFICATION_MODE = 'stress_binary'
NUM_CLASSES = 2
MODEL_TO_USE = 'cnn_gru_attention'            # 'cnn_gru' = the same stack without attention (SURVEY D3)
CHANNELS_TO_USE = ['chest_ECG', 'chest_EDA', 'chest_Resp']
MODEL_PARAMS = {
    'cnn_gru_attention': {'cnn_out_channels': 32, 'gru_hidden_size': 64, 'gru_num_layers': 2, 'dropout': 0.5},
    'cnn_gru': {'cnn_out_channels': 32, 'gru_hidden_size': 64, 'gru_num_layers': 2, 'dropout': 0.5},
}
PROCESSED_DATA_PATH = Path('./data')
EARLY_DATA_PATH = PROCESSED_DATA_PATH / 'chest_raw'
SEED = 42
NUM_WORKERS = 0
EPOCHS = 100
BATCH_SIZE = 64
LEARNING_RATE = 0.001
PATIENCE = 20
WEIGHTS_DECAY = 1e-4
USE_CLASS_WEIGHTS = False                     # class-weighted CrossEntropyLoss, 'balanced' weights (never enabled upstream, SURVEY D9)
ATTRIBUTION_STEPS = 0                         # > 0: integrated-gradients channel attribution of each fold's test set, this many steps
MC_DROPOUT_SAMPLES = 0                        # > 0: MC-dropout uncertainty of each fold's test set, this many samples per window
GRAD_CLIP_NORM = None                         # a number: clip the gradient to this total 2-norm before every Adam step (clip_grad_norm_)
ALL_SUBJECTS = [f"S{i}" for i in range(2, 18) if i != 12]
CONCURRENT_FOLDS = int(os.environ.get("MMS_CONCURRENT_FOLDS", "1"))     # folds interleaved per GPU (new; 1 = the reference's loop)


def fold_split(subject_to_test, all_subjects=None, seed=SEED):
    """reference main.py:102-103: 14 remaining subjects -> 11 train / 3 validation."""
    from sklearn.model_selection import train_test_split
    all_subjects = ALL_SUBJECTS if all_subjects is None else all_subjects
    train_val = [s for s in all_subjects if s != subject_to_test]
    train_subjects, val_subjects = train_test_split(train_val, test_size=0.2, random_state=seed)
    return train_subjects, val_subjects


def folds_for_rank(n_folds: int, rank: int, world: int):
    """Round-robin fold assignment: rank r trains folds r, r + world, ..."""
    return list(range(rank, n_folds, world))


def trainer_config():
    return {'trainer': {'epochs': EPOCHS, 'learning_rate': LEARNING_RATE,
                        'early_stopping': {'enabled': True, 'patience': PATIENCE, 'delta': 0},
                        'weight_decay': WEIGHTS_DECAY, 'use_class_weights': USE_CLASS_WEIGHTS,
                        'grad_clip_norm': GRAD_CLIP_NORM}}


def run_fold_async(fold_index, subject_to_test, run_output_dir, all_channel_names, subject_streams=None, stream=None,
                   quiet=False):
    """One LOSO fold (the body of the reference loop, main.py:98-125) as a generator that yields the CUDA events it
    waits for (see ``trainer.Trainer``), so several folds can be interleaved on one GPU.  The shuffling generator is
    private to the fold (``SEED + fold_index``), which makes a fold's batches independent of what runs beside it."""
    import contextlib
    from torch.utils.data import DataLoader
    from .dataset import DeviceBatchLoader, DeviceWesadDataset, WesadDataset
    from .models import CnnGruAttentionModel
    from .trainer import Trainer

    torch.manual_seed(SEED + fold_index)
    np.random.seed(SEED + fold_index)
    shuffle_gen = torch.Generator().manual_seed(SEED + fold_index)
    if not quiet:
        print(f"\n--- 处理折叠: 测试受试者 {subject_to_test} ---")
    fold_output_dir = Path(run_output_dir) / f'fold_test_on_{subject_to_test}'
    fold_output_dir.mkdir(parents=True, exist_ok=True)
    train_subjects, val_subjects = fold_split(subject_to_test)

    with (torch.cuda.stream(stream) if stream is not None else contextlib.nullcontext()):
        if subject_streams is not None:         # device-resident path (SURVEY §8f N1)
            mk = lambda subs: DeviceWesadDataset(subject_streams, subs, CHANNELS_TO_USE, classification_mode=CLASSIFICATION_MODE)
            train_ds, val_ds, test_ds = mk(train_subjects), mk(val_subjects), mk([subject_to_test])
            train_loader = DeviceBatchLoader(train_ds, BATCH_SIZE, shuffle=True, generator=shuffle_gen)
            val_loader = DeviceBatchLoader(val_ds, BATCH_SIZE)
            test_loader = DeviceBatchLoader(test_ds, BATCH_SIZE)
        else:                                   # file path, exactly the reference's data flow
            mk = lambda subs: WesadDataset(EARLY_DATA_PATH, subs, CHANNELS_TO_USE, all_channel_names,
                                           classification_mode=CLASSIFICATION_MODE)
            train_ds, val_ds, test_ds = mk(train_subjects), mk(val_subjects), mk([subject_to_test])
            train_loader = DataLoader(train_ds, batch_size=BATCH_SIZE, shuffle=True, num_workers=NUM_WORKERS, pin_memory=True,
                                      generator=shuffle_gen)
            val_loader = DataLoader(val_ds, batch_size=BATCH_SIZE, shuffle=False, num_workers=NUM_WORKERS, pin_memory=True)
            test_loader = DataLoader(test_ds, batch_size=BATCH_SIZE, shuffle=False, num_workers=NUM_WORKERS, pin_memory=True)
        model = CnnGruAttentionModel(in_channels=len(CHANNELS_TO_USE), num_classes=NUM_CLASSES,
                                     attention=(MODEL_TO_USE != 'cnn_gru'), **MODEL_PARAMS[MODEL_TO_USE])
    config = trainer_config()
    config['trainer']['quiet'] = quiet
    trainer = Trainer(model, fold_output_dir, config, stream=stream)
    yield from trainer.train_async(train_loader, val_loader)
    out = yield from trainer.evaluate_async(test_loader, want_lists=True)
    _, test_acc, test_f1 = trainer.finish_test(*out)
    result = {'subject': subject_to_test, 'accuracy': float(test_acc), 'f1_score': float(test_f1),
              'windows_trained': int(trainer.windows_trained), 'timing': dict(trainer.timing)}
    if ATTRIBUTION_STEPS > 0:
        att = trainer.channel_attribution(test_loader, steps=ATTRIBUTION_STEPS, channel_names=CHANNELS_TO_USE)
        result['channel_attribution'] = att.tolist()
    if MC_DROPOUT_SAMPLES > 0:
        result['uncertainty'] = trainer.mc_dropout_uncertainty(test_loader, samples=MC_DROPOUT_SAMPLES)
    return result


def run_fold(fold_index, subject_to_test, run_output_dir, all_channel_names, subject_streams=None):
    """One LOSO fold, blocking (the reference's loop body)."""
    from .trainer import drive
    return drive(run_fold_async(fold_index, subject_to_test, run_output_dir, all_channel_names, subject_streams))


def run_folds_interleaved(fold_indices, make_fold, concurrent_folds):
    """Drive up to ``concurrent_folds`` fold generators at once from this thread, each on its own CUDA stream.

    A single training step of this model keeps a B200 mostly idle (the GRU recurrences are latency-bound and occupy
    128 thread blocks of 4 warps), and LOSO folds share nothing, so co-resident folds overlap almost for free.
    ``make_fold(fold_index, stream)`` returns a generator that yields CUDA events; a fold is resumed as soon as the
    event it waits for has completed.  Returns the fold results in ``fold_indices`` order."""
    import time
    pending = list(fold_indices)
    results, active = {}, []
    t_begin = time.perf_counter()
    streams = [torch.cuda.Stream() for _ in range(max(1, concurrent_folds))]
    free = list(range(len(streams)))
    while pending or active:
        while pending and free:
            k = free.pop(0)
            idx = pending.pop(0)
            active.append([idx, k, make_fold(idx, streams[k]), None, time.perf_counter() - t_begin])
        progressed = False
        for slot in list(active):
            idx, k, gen, ev, started = slot
            if ev is not None and not ev.query():
                continue
            progressed = True
            try:
                slot[3] = next(gen)
            except StopIteration as done:
                results[idx] = done.value
                if isinstance(done.value, dict):
                    done.value['start_s'], done.value['end_s'] = started, time.perf_counter() - t_begin
                active.remove(slot)
                free.append(k)
        if not progressed:
            time.sleep(20e-6)
    return [results[i] for i in fold_indices]


def write_summary(run_output_dir, results):
    """reference main.py:128-156 (same file format)."""
    accs = [r['accuracy'] for r in results]
    f1s = [r['f1_score'] for r in results]
    summary_file = Path(run_output_dir) / 'cv_summary.txt'
    with open(summary_file, 'w', encoding='utf-8') as f:
        f.write("实验配置:\n")
        for key, val in (("MODEL_TO_USE", MODEL_TO_USE), ("RUN_NAME", RUN_NAME), ("SEED", SEED),
                         ("CHANNELS_TO_USE", CHANNELS_TO_USE), ("EPOCHS", EPOCHS), ("BATCH_SIZE", BATCH_SIZE),
                         ("LEARNING_RATE", LEARNING_RATE), ("NUM_WORKERS", NUM_WORKERS), ("PATIENCE", PATIENCE),
                         ("NUM_CLASSES", NUM_CLASSES), ("MODEL_PARAMS", MODEL_PARAMS)):
            f.write(f"{key}: {val}\n")
        f.write("\n每个折叠的详细结果:\n")
        for res in results:
            f.write(f"  - 测试 {res['subject']}: Accuracy = {res['accuracy']:.4f}, F1-score = {res['f1_score']:.4f}\n")
        f.write("\n最终平均性能:\n")
        f.write(f"平均准确率 (Accuracy): {np.mean(accs):.4f} ± {np.std(accs):.4f}\n")
        f.write(f"平均 F1 分数 (Weighted F1-score): {np.mean(f1s):.4f} ± {np.std(f1s):.4f}\n")
    print(f"交叉验证汇总结果已保存至: {summary_file}")
    print("\n--- 最终平均性能 ---")
    print(f"平均准确率 (Accuracy): {np.mean(accs):.4f} ± {np.std(accs):.4f}")
    print(f"平均 F1 分数 (Weighted F1-score): {np.mean(f1s):.4f} ± {np.std(f1s):.4f}")
    return summary_file


def write_attribution_summary(run_output_dir, results):
    """Mean +- std over the folds of each fold's ``Trainer.channel_attribution`` (channels x classes)."""
    att = np.array([r['channel_attribution'] for r in results], dtype=np.float64)       # [folds, nc, C]
    mean, std = att.mean(axis=0), att.std(axis=0)
    path = Path(run_output_dir) / 'attribution_summary.txt'
    with open(path, 'w', encoding='utf-8') as f:
        f.write(f"# integrated gradients, {ATTRIBUTION_STEPS} steps, zero baseline, target = predicted class; "
                f"{len(results)} folds\n")
        f.write("# per fold: mean over the test windows of each true class of |S_c| / sum_c' |S_c'|; here mean +- std over folds\n")
        f.write("channel" + "".join(f"\tclass_{k}" for k in range(att.shape[1])) + "\n")
        for c, name in enumerate(CHANNELS_TO_USE[:att.shape[2]]):
            f.write(name + "".join(f"\t{mean[k, c]:.4f} ± {std[k, c]:.4f}" for k in range(att.shape[1])) + "\n")
    return path


def write_uncertainty_summary(run_output_dir, results):
    """Mean +- std over the folds of each number of the folds' ``Trainer.mc_dropout_uncertainty``; a NaN (an AUROC of a
    fold without errors) is left out of its mean and counted."""
    keys = [k for k in results[0]['uncertainty'] if k not in ('windows', 'samples')]
    path = Path(run_output_dir) / 'uncertainty_summary.txt'
    with open(path, 'w', encoding='utf-8') as f:
        f.write(f"# MC dropout, {MC_DROPOUT_SAMPLES} samples per window; {len(results)} folds; mean +- std over the folds\n")
        for k in keys:
            v = np.array([r['uncertainty'][k] for r in results], dtype=np.float64)
            ok = v[~np.isnan(v)]
            line = f"{k}\t{ok.mean():.4f} ± {ok.std():.4f}" if ok.size else f"{k}\tnan"
            f.write(line + (f"\t({v.size - ok.size} folds NaN)" if ok.size < v.size else "") + "\n")
    return path


def gather_results(local_results, world):
    """Collect the per-fold results of every rank on all ranks, ordered by subject (ALL_SUBJECTS)."""
    if world > 1:
        import torch.distributed as dist
        bucket = [None] * world
        dist.all_gather_object(bucket, local_results)
        merged = [r for part in bucket for r in part]
    else:
        merged = list(local_results)
    order = {s: i for i, s in enumerate(ALL_SUBJECTS)}
    return sorted(merged, key=lambda r: order.get(r['subject'], len(order)))


def run_simple_experiment(run_output_dir, device, all_channel_names, subject_streams=None, fold_fn=None,
                          concurrent_folds=1):
    """Standard LOSO experiment; with torch.distributed initialised the folds are sharded over the ranks, and with
    ``concurrent_folds > 1`` each rank additionally interleaves that many of its folds on separate CUDA streams."""
    import torch.distributed as dist
    world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    rank = dist.get_rank() if world > 1 else 0
    print("\n" + "=" * 80)
    print(f"开始执行标准二分类实验 (模式: {CLASSIFICATION_MODE})")
    print("=" * 80)
    mine = folds_for_rank(len(ALL_SUBJECTS), rank, world)
    if concurrent_folds > 1 and fold_fn is None:
        if subject_streams is not None:        # normalise every subject once, before the fold streams start reading them
            from .dataset import normalise_gather
            for sub in subject_streams.values():
                if len(sub.labels):
                    normalise_gather(sub, CHANNELS_TO_USE)
        torch.cuda.synchronize()
        make = lambda i, st: run_fold_async(i, ALL_SUBJECTS[i], run_output_dir, all_channel_names, subject_streams, stream=st,
                                            quiet=True)
        local = run_folds_interleaved(mine, make, concurrent_folds)
        torch.cuda.synchronize()
    else:
        fold_fn = run_fold if fold_fn is None else fold_fn
        local = [fold_fn(i, ALL_SUBJECTS[i], run_output_dir, all_channel_names, subject_streams) for i in mine]
    results = gather_results(local, world)
    if rank == 0:
        print("\n\n====== 留一法交叉验证全部完成 ======")
        write_summary(run_output_dir, results)
        if ATTRIBUTION_STEPS > 0:
            write_attribution_summary(run_output_dir, results)
        if MC_DROPOUT_SAMPLES > 0:
            write_uncertainty_summary(run_output_dir, results)
    return results


def main():
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("multimodalsignal_b200.main needs a CUDA device (B200); there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.manual_seed(SEED)
    np.random.seed(SEED)
    stamp = [datetime.now().strftime('%Y%m%d_%H%M%S')]
    if world > 1:
        dist.broadcast_object_list(stamp, src=0)
    run_output_dir = Path('./output') / RUN_NAME / f'run_{stamp[0]}'
    run_output_dir.mkdir(parents=True, exist_ok=True)
    print(f"====== 运行结果将保存至: {run_output_dir} ======")
    device = torch.device("cuda", local_rank)
    print(f"====== 使用设备: {device} ======")
    with open(EARLY_DATA_PATH / '_channel_names.txt', 'r') as f:
        all_channel_names = [line.strip() for line in f]
    if USE_HIERARCHICAL_CLASSIFICATION:
        raise NotImplementedError("the hierarchical experiment is dead code upstream (SURVEY D7) and out of scope")
    run_simple_experiment(run_output_dir, device, all_channel_names, concurrent_folds=CONCURRENT_FOLDS)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
