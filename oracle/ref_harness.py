"""Import the UNMODIFIED reference modules (17LiQi/MultimodalSignal: models.py, dataset.py, ...).

Where they are looked for, first match wins: the directory named by ``MMS_REFERENCE_ROOT``; a copy of the
reference installed under ``oracle/_ref/`` (the tree itself or one directory down); the byte-identical staging
``baseline/_ref/`` made by ``oracle/build_ref.py``.  Both directories are git-ignored: no reference source enters
the history.  Without any of them ``available()`` is False and the reference legs of ``bench.py`` say so.

TEST INFRASTRUCTURE ONLY.  Used by ``oracle/make_golden.py`` to produce the
committed fixtures under ``tests/golden/`` and by ``bench.py --impl reference``
when the reference tree is present.

The reference imports three packages that are absent here and are not on the hot
path: ``matplotlib`` / ``seaborn`` (trainer.py:9-10, plotting only -- the plotting
call is already wrapped in try/except, trainer.py:250-273) and ``neurokit2``
(preprocess.py:9, feature branch only).  Empty stub modules are injected for
those names; nothing else is changed.
"""
from __future__ import annotations

import contextlib
import importlib
import os
import sys
import types
from pathlib import Path

_INSTALLED = Path(__file__).resolve().parent / "_ref"
_STAGED = Path(__file__).resolve().parents[1] / "baseline" / "_ref"     # oracle/build_ref.py


def _has_models(d: Path) -> bool:
    try:
        return (d / "models.py").is_file()
    except OSError:                  # a directory this user may not search counts as absent
        return False


def _find_root() -> Path:
    env = os.environ.get("MMS_REFERENCE_ROOT")
    if env:
        return Path(env)
    candidates = [_INSTALLED]
    if _INSTALLED.is_dir():
        candidates += sorted(d for d in _INSTALLED.iterdir() if d.is_dir())
    return next((d for d in candidates + [_STAGED] if _has_models(d)), _STAGED)


REFERENCE_ROOT = _find_root()
_STUBS = ("matplotlib", "matplotlib.pyplot", "seaborn", "neurokit2")


def available() -> bool:
    return _has_models(REFERENCE_ROOT)


def staged_ok() -> bool:
    """True when the files under ``baseline/_ref`` still hash to their manifest (i.e. are the unmodified reference)."""
    import hashlib
    import json
    man = _STAGED / "MANIFEST.json"
    if not man.exists():
        return False
    want = json.loads(man.read_text())["sha256"]
    return all((_STAGED / n).exists() and hashlib.sha256((_STAGED / n).read_bytes()).hexdigest() == h for n, h in want.items())


def _install_stubs():
    for name in _STUBS:
        if name not in sys.modules:
            try:
                importlib.import_module(name)
            except Exception:
                sys.modules[name] = types.ModuleType(name)
    mpl = sys.modules["matplotlib"]
    if not hasattr(mpl, "pyplot"):
        mpl.pyplot = sys.modules["matplotlib.pyplot"]


@contextlib.contextmanager
def _cwd(path):
    old = os.getcwd()
    os.chdir(path)
    try:
        yield
    finally:
        os.chdir(old)


def load(name: str, scratch_dir=None):
    """Import reference module ``name`` under the alias ``mms_ref_<name>`` so it can
    never shadow (or be shadowed by) this repo's modules of the same name.
    ``preprocess`` creates ``./data`` directories at import time (preprocess.py:14-15),
    so it is imported with ``scratch_dir`` as the working directory."""
    if not available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    _install_stubs()
    alias = f"mms_ref_{name}"
    if alias in sys.modules:
        return sys.modules[alias]
    # the reference modules import each other by bare name (main.py:9-11)
    saved = {k: sys.modules.get(k) for k in ("models", "dataset", "trainer", "preprocess", "main")}
    sys.path.insert(0, str(REFERENCE_ROOT))
    try:
        for k in saved:
            sys.modules.pop(k, None)
        with _cwd(scratch_dir or os.getcwd()):
            mod = importlib.import_module(name)
        sys.modules[alias] = mod
        return mod
    finally:
        sys.path.remove(str(REFERENCE_ROOT))
        for k, v in saved.items():
            sys.modules.pop(k, None)
            if v is not None:
                sys.modules[k] = v
