"""Generate ``tests/golden/*`` by executing the UNMODIFIED reference modules.

TEST INFRASTRUCTURE ONLY.  Run in the authoring container (needs
``/root/reference``):  ``python -m oracle.make_golden``.  The outputs are committed;
the GPU box never runs this script.

Every fixture records the library versions it was produced with, because the
reference itself pins nothing at these boundaries (SURVEY §8c: "parity unpinned"
by the reference; the pin is these files).
"""
from __future__ import annotations

import json
import sys
import tempfile
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from oracle import golden_inputs as gi, ref_harness  # noqa: E402
from multimodalsignal_b200 import synth  # noqa: E402

GOLDEN = ROOT / "tests" / "golden"


def _versions():
    import scipy
    import sklearn
    import pandas
    return {"torch": torch.__version__, "numpy": np.__version__, "scipy": scipy.__version__,
            "sklearn": sklearn.__version__, "pandas": pandas.__version__}


# --------------------------------------------------------------------------- model
MODEL_CASES = {
    # name: (C, num_classes, B, T, model kwargs, adam steps)
    "c6_t640": (6, 2, 4, 640, {}, 3),
    "c3_t336_ternary": (3, 3, 3, 336, {}, 0),
    "c14_t3840": (14, 2, 2, 3840, {}, 0),
    "c8_h32_l1": (8, 2, 3, 320, {"gru_hidden_size": 32, "gru_num_layers": 1}, 2),
    # north-star window length with M = B*L = 1920 rows >= 1024: the tcgen05 NT / TN GEMMs of the product path
    # (model.cu TC_MIN_ROWS) are pinned to the reference itself, not only to the oracle
    "c6_t3840_b8": (6, 2, 8, 3840, {}, 2),
}


def _keep(out, name, a):
    """Output ``name`` in full or, when it is large, the fixed seeded subset of its elements (flat indices under
    ``idx/<key>``).  A gradient also keeps its largest magnitude: the scale of the tests' tolerance."""
    a = np.asarray(a)
    key = name.split("/", 1)[1]
    if name.startswith("grad/"):
        out[f"absmax/{name}"] = np.float32(np.abs(a).max() if a.size else 0.0)
    idx = gi.subset_indices(key, a.size)
    if idx is None:
        out[name] = a
    else:
        out[f"idx/{key}"] = idx
        out[name] = a.reshape(-1)[idx]


def pack_model_case(meta, x, y, sd, outputs):
    """A model fixture: the reference's outputs (gradients and post-Adam weights subset by ``_keep``) and the digests of
    the inputs it ran on, which tests/conftest.py rebuilds from the seeds (oracle/golden_inputs.py)."""
    digests = {"x": gi.digest(x), "y": gi.digest(y), **{f"sd/{k}": gi.digest(v) for k, v in sd.items()}}
    out = {}
    for k, v in outputs.items():
        if k.startswith(("grad/", "sd_adam/")):
            _keep(out, k, v)
        else:
            out[k] = v
    out["meta"] = np.frombuffer(json.dumps(dict(meta, inputs="model_case", input_sha256=digests)).encode(), dtype=np.uint8)
    return out


def make_model_case(name, C, nc, B, T, kwargs, adam_steps):
    ref_models = ref_harness.load("models")
    torch.manual_seed(1234 + C)
    torch.set_num_threads(1)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model = ref_models.CnnGruAttentionModel(in_channels=C, num_classes=nc, dropout=0.0, **kwargs)
    gi.perturb_batchnorm(model)
    x, y = gi.model_windows(C, nc, B, T)
    xt, yt = torch.from_numpy(x), torch.from_numpy(y)
    sd = {k: v.detach().numpy().copy() for k, v in model.state_dict().items()}
    out = {}

    model.train()
    crit = torch.nn.CrossEntropyLoss()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=1e-4)   # trainer.py:68
    opt.zero_grad()
    logits = model(xt)
    loss = crit(logits, yt)
    loss.backward()
    out["train_logits"] = logits.detach().numpy().copy()
    out["train_loss"] = np.float32(loss.item())
    for k, v in model.named_parameters():
        g = v.grad if v.grad is not None else torch.zeros_like(v)
        out[f"grad/{k}"] = g.detach().numpy().copy()
    for k, v in model.state_dict().items():
        if "running" in k or "num_batches" in k:
            out[f"sd_after_fwd/{k}"] = v.detach().numpy().copy()
    model.eval()
    with torch.no_grad():
        out["eval_logits"] = model(xt).numpy().copy()
    model.train()
    if adam_steps:
        losses = [loss.item()]
        opt.step()
        for _ in range(adam_steps - 1):
            opt.zero_grad()
            l2 = crit(model(xt), yt)
            l2.backward()
            opt.step()
            losses.append(l2.item())
        out["adam_losses"] = np.asarray(losses, dtype=np.float32)
        out["adam_steps"] = np.int64(adam_steps)
        for k, v in model.state_dict().items():
            out[f"sd_adam/{k}"] = v.detach().numpy().copy()
    meta = {"C": C, "num_classes": nc, "B": B, "T": T, "kwargs": kwargs, "versions": _versions(),
            "source": "reference models.py CnnGruAttentionModel, dropout=0.0, float32, CPU"}
    np.savez_compressed(GOLDEN / f"model_{name}.npz", **pack_model_case(meta, x, y, sd, out))
    print(f"model_{name}: loss={loss.item():.6f}")


# ----------------------------------------------------------------------- preprocess
def pack_resample_cases(meta, xs, ys):
    """The resample fixture: the reference's outputs in full, the digests of the inputs (rebuilt from their seed)."""
    out = {}
    for i, ((_, _, f0, f1), y) in enumerate(zip(gi.RESAMPLE_CASES, ys)):
        out[f"y{i}"] = y
        out[f"fs{i}"] = np.asarray([f0, f1], dtype=np.int64)
    out["n_cases"] = np.int64(len(ys))
    digests = {f"x{i}": gi.digest(x) for i, x in enumerate(xs)}
    out["meta"] = np.frombuffer(json.dumps(dict(meta, inputs="resample_cases", input_sha256=digests)).encode(), dtype=np.uint8)
    return out


def make_resample_cases():
    """reference ``preprocess.resample_signal`` on the short 1-D / 2-D arrays of ``golden_inputs.RESAMPLE_CASES``."""
    with tempfile.TemporaryDirectory() as tmp:
        pp = ref_harness.load("preprocess", scratch_dir=tmp)
    xs = gi.resample_signals()
    ys = [pp.resample_signal(x, f0, f1) for x, (_, _, f0, f1) in zip(xs, gi.RESAMPLE_CASES)]
    meta = {"versions": _versions(), "source": "reference preprocess.resample_signal"}
    np.savez_compressed(GOLDEN / "resample_cases.npz", **pack_resample_cases(meta, xs, ys))
    print("resample_cases:", len(xs))


def _run_reference_preprocessing(tmp: Path, fs: int, index_probe: bool):
    """``run_preprocessing()`` with PROCESS_TARGETS=['raw'] (the path main.py reads,
    SURVEY D6).  With ``index_probe`` the library resampler is swapped for
    ``arange(num)`` so the saved windows expose the reference's own start indices."""
    import os
    pp = ref_harness.load("preprocess", scratch_dir=str(tmp))
    pp.WESAD_ROOT = tmp / "WESAD"
    pp.OUTPUT_PATH = tmp / "data"
    pp.PROCESS_TARGETS = ["raw"]
    pp.RAW_FS = fs
    pp.RAW_PATH = pp.OUTPUT_PATH / f"chest_raw_{fs}{'_probe' if index_probe else ''}"
    pp.RAW_PATH.mkdir(parents=True, exist_ok=True)
    saved = pp.resample_signal
    if index_probe:
        def probe(signal_data, original_fs, target_fs):
            num = int(len(signal_data) * (target_fs / original_fs))
            col = np.arange(num, dtype=np.float64)
            return np.column_stack([col] * signal_data.shape[1]) if signal_data.ndim > 1 else col
        pp.resample_signal = probe
    try:
        old = os.getcwd()
        os.chdir(tmp)
        pp.run_preprocessing()
    finally:
        os.chdir(old)
        pp.resample_signal = saved
    return pp.RAW_PATH


def make_preprocess_goldens():
    out = {}
    with tempfile.TemporaryDirectory() as tmpd:
        tmp = Path(tmpd)
        # (1) index / label parity at FULL protocol size, all 15 subjects, 64 and 128 Hz.
        # Signals are 1 sample/column dummies of the right length: only len() matters to the probe.
        root = tmp / "WESAD"
        import pickle
        for idx, sid in enumerate(synth.ALL_SUBJECTS):
            n = int(700 * 60 * synth.FULL_MINUTES) + 137 * idx
            d = root / sid
            d.mkdir(parents=True, exist_ok=True)
            chest = {b"ACC": np.zeros((n, 3), dtype=np.int8), b"ECG": np.zeros((n, 1), dtype=np.int8),
                     b"EDA": np.zeros((n, 1), dtype=np.int8), b"EMG": np.zeros((n, 1), dtype=np.int8),
                     b"Resp": np.zeros((n, 1), dtype=np.int8), b"Temp": np.zeros((n, 1), dtype=np.int8)}
            with open(d / f"{sid}.pkl", "wb") as f:
                pickle.dump({b"signal": {b"chest": chest}}, f, protocol=4)
            (d / f"{sid}_quest.csv").write_text(synth.quest_csv_text(synth.FULL_PROTOCOL))
        for fs in (64, 128):
            path = _run_reference_preprocessing(tmp, fs, index_probe=True)
            for sid in synth.ALL_SUBJECTS:
                X = np.load(path / f"{sid}_X.npy")
                y = np.load(path / f"{sid}_y.npy")
                out[f"full/{fs}/{sid}/starts"] = X[:, 0, 7].astype(np.int64)
                out[f"full/{fs}/{sid}/labels"] = y.astype(np.int64)
                out[f"full/{fs}/{sid}/shape"] = np.asarray(X.shape, dtype=np.int64)
                assert np.all(X[:, 1, 0] == X[:, 0, 0] + 1)
            names = (path / "_channel_names.txt").read_text()
            out["channel_names"] = np.frombuffer(names.encode(), dtype=np.uint8)
        import shutil
        shutil.rmtree(root)
        shutil.rmtree(tmp / "data")

        # (2) value parity on the SHORT protocol with the real resampler, S2 (quirk) and S5.
        synth.write_wesad_tree(root, subjects=["S2", "S5"], minutes=synth.SHORT_MINUTES,
                               protocol=synth.SHORT_PROTOCOL, with_wrist=False)
        # run_preprocessing() iterates all 15 ids and skips missing pickles (preprocess.py:66-68,140-141)
        for fs in (64, 128):
            path = _run_reference_preprocessing(tmp, fs, index_probe=False)
            for sid in ("S2", "S5"):
                X = np.load(path / f"{sid}_X.npy")
                y = np.load(path / f"{sid}_y.npy")
                out[f"short/{fs}/{sid}/shape"] = np.asarray(X.shape, dtype=np.int64)
                out[f"short/{fs}/{sid}/labels"] = y.astype(np.int64)
                out[f"short/{fs}/{sid}/X_sub"] = X[:, ::61, :].copy()          # every 61st sample
                out[f"short/{fs}/{sid}/X_rowsum"] = X.sum(axis=1)
            # (3) dataset normalisation on those files (reference dataset.py)
            if fs == 64:
                ds_mod = ref_harness.load("dataset")
                all_names = (path / "_channel_names.txt").read_text().split()
                for mode in ("stress_binary", "ternary"):
                    chans = ["chest_ECG", "chest_EDA", "chest_EMG", "chest_Resp"]
                    ds = ds_mod.WesadDataset(path, ["S2", "S5", "S99"], chans, all_names, classification_mode=mode)
                    out[f"dataset/{mode}/labels"] = ds.labels.astype(np.int64)
                    out[f"dataset/{mode}/data_sub"] = ds.data[:, ::61, :].copy()
                    xi, yi = ds[3]
                    out[f"dataset/{mode}/item3_x_sub"] = xi.numpy()[:, ::61].copy()
                    out[f"dataset/{mode}/item3_y"] = np.int64(yi.item())
                    out[f"dataset/{mode}/len"] = np.int64(len(ds))
    out["meta"] = np.frombuffer(json.dumps({
        "versions": _versions(), "short_protocol": synth.SHORT_PROTOCOL, "short_minutes": synth.SHORT_MINUTES,
        "source": "reference preprocess.run_preprocessing (PROCESS_TARGETS=['raw']) and dataset.WesadDataset"
    }).encode(), dtype=np.uint8)
    np.savez_compressed(GOLDEN / "preprocess_golden.npz", **out)
    print("preprocess_golden written")


def make_fold_table():
    """reference main.py:102-103 -- sklearn ``train_test_split(14 subjects, 0.2, seed 42)``."""
    from sklearn.model_selection import train_test_split
    table = {}
    for s in synth.ALL_SUBJECTS:
        tv = [t for t in synth.ALL_SUBJECTS if t != s]
        tr, va = train_test_split(tv, test_size=0.2, random_state=42)
        table[s] = {"train": tr, "val": va}
    (GOLDEN / "fold_table.json").write_text(json.dumps({"versions": _versions(), "folds": table}, indent=1))
    print("fold_table written")


def main():
    GOLDEN.mkdir(parents=True, exist_ok=True)
    only = [a.split("=", 1)[1] for a in sys.argv if a.startswith("--model-case=")]
    for name, spec in MODEL_CASES.items():
        if not only or name in only:
            make_model_case(name, *spec)
    if only:
        return
    make_resample_cases()
    make_preprocess_goldens()
    make_fold_table()
    make_trainer_golden()


if __name__ == "__main__" and "--trainer-only" not in sys.argv:
    main()


# --------------------------------------------------------------------------- trainer
TRAINER_CASE = {"train": ["S3", "S4"], "val": ["S5"], "test": ["S2"], "channels": ["chest_ECG", "chest_EDA", "chest_Resp"],
                "batch_size": 8, "epochs": 2, "seed": 42}


def make_trainer_golden():
    """Two epochs of the UNMODIFIED reference Trainer (CPU, dropout = 0 so the run is deterministic)
    on short synthetic recordings preprocessed by the reference's own run_preprocessing()."""
    import io
    import contextlib
    from torch.utils.data import DataLoader
    case = TRAINER_CASE
    with tempfile.TemporaryDirectory() as tmpd:
        tmp = Path(tmpd)
        synth.write_wesad_tree(tmp / "WESAD", subjects=["S2", "S3", "S4", "S5"], minutes=synth.SHORT_MINUTES,
                               protocol=synth.SHORT_PROTOCOL, with_wrist=False)
        path = _run_reference_preprocessing(tmp, 64, index_probe=False)
        names = (path / "_channel_names.txt").read_text().split()
        ds_mod = ref_harness.load("dataset")
        models = ref_harness.load("models")
        trainer_mod = ref_harness.load("trainer")
        mk = lambda subs: ds_mod.WesadDataset(path, subs, case["channels"], names, classification_mode="stress_binary")
        torch.manual_seed(case["seed"])
        np.random.seed(case["seed"])
        torch.set_num_threads(1)
        train_ds, val_ds, test_ds = mk(case["train"]), mk(case["val"]), mk(case["test"])
        tl = DataLoader(train_ds, batch_size=case["batch_size"], shuffle=True, num_workers=0)
        vl = DataLoader(val_ds, batch_size=case["batch_size"], shuffle=False, num_workers=0)
        te = DataLoader(test_ds, batch_size=case["batch_size"], shuffle=False, num_workers=0)
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            model = models.CnnGruAttentionModel(in_channels=3, num_classes=2, dropout=0.0)
        cfg = {'trainer': {'epochs': case["epochs"], 'learning_rate': 1e-3,
                           'early_stopping': {'enabled': True, 'patience': 20, 'delta': 0}, 'weight_decay': 1e-4}}
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf), contextlib.redirect_stderr(io.StringIO()):
            tr = trainer_mod.Trainer(model, tmp / "fold", cfg)
            tr.train(tl, vl)
            test_loss, test_acc, test_f1 = tr.evaluate(te, is_test=True)
        log = (tmp / "fold" / "training_log.txt").read_text(encoding="utf-8")
        ckpt = torch.load(tmp / "fold" / "best_model.pt", weights_only=True)
        out = {"case": case, "versions": _versions(), "log": log,
               "n_train": len(train_ds), "n_val": len(val_ds), "n_test": len(test_ds),
               "test": {"loss": test_loss, "acc": test_acc, "f1": test_f1},
               "best_model_keys": list(ckpt.keys()),
               "best_model_shapes": {k: list(v.shape) for k, v in ckpt.items()},
               "final_fc3_bias": model.classifier[3].bias.detach().tolist(),
               "final_bn1_running_mean": model.cnn_encoder[1].running_mean.tolist()}
        (GOLDEN / "trainer_golden.json").write_text(json.dumps(out, indent=1, ensure_ascii=False))
    print("trainer_golden written:", out["test"])


if __name__ == "__main__" and "--trainer-only" in sys.argv:
    GOLDEN.mkdir(parents=True, exist_ok=True)
    make_trainer_golden()
