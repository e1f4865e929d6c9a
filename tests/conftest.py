"""pytest configuration: the ``gpu`` marker and shared fixtures.

``-m "not gpu"`` runs in the CPU-only authoring container (oracle vs golden, host
logic, C-ABI symbol checks); ``-m gpu`` runs on a B200 and compares the CUDA path,
called through the C-ABI, with the oracle.
"""
import json
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))
GOLDEN = ROOT / "tests" / "golden"


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_collection_modifyitems(config, items):
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def _golden_inputs(meta):
    """The inputs a fixture's reference run saw, rebuilt from their seeds (oracle/golden_inputs.py)."""
    from oracle import golden_inputs as gi
    if meta["inputs"] == "resample_cases":
        return {f"x{i}": x for i, x in enumerate(gi.resample_signals())}
    x, y = gi.model_windows(meta["C"], meta["num_classes"], meta["B"], meta["T"])
    sd = gi.model_state(meta["C"], meta["num_classes"], meta["kwargs"])
    return {"x": x, "y": y, **{f"sd/{k}": v for k, v in sd.items()}}


def load_golden(name):
    """A fixture as ``{entry: array}`` and its meta.  Inputs are not stored: they are rebuilt from their seeds and must
    match the SHA-256 digests the fixture keeps of the inputs the reference ran on."""
    from oracle import golden_inputs as gi
    with np.load(GOLDEN / name) as f:
        z = {k: f[k] for k in f.files}
    meta = json.loads(bytes(z["meta"]).decode()) if "meta" in z else {}
    if "input_sha256" in meta:
        z.update(_golden_inputs(meta))
        bad = [k for k, h in meta["input_sha256"].items() if k not in z or gi.digest(z[k]) != h]
        assert not bad, f"{name}: inputs rebuilt from the seeds differ from those the reference ran on: {bad}"
    return z, meta


def golden_state(z, prefix):
    import torch
    out = {}
    for k in z:
        if k.startswith(prefix + "/"):
            out[k[len(prefix) + 1:]] = torch.from_numpy(np.array(z[k]))
    return out


def golden_kept(z, name, got):
    """``got`` (the full array that output ``name`` of the fixture describes) and the fixture's values, both flat, at the
    elements the fixture keeps: all of them, or the fixed seeded subset ``idx/<key>`` of a large output."""
    idx = z.get("idx/" + name.split("/", 1)[1])
    got = np.asarray(got).reshape(-1)
    return (got if idx is None else got[idx]), z[name].reshape(-1)


MODEL_CASES = ["c6_t640", "c3_t336_ternary", "c14_t3840", "c8_h32_l1", "c6_t3840_b8"]
