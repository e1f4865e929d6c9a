"""One LOSO fold end to end with gradient-norm clipping (main.GRAD_CLIP_NORM): synthetic recordings of a few subjects,
preprocessing on the device, main.run_fold, then the fold's training log, which holds one "Gradient norm before clipping"
line per epoch.

    python tools/grad_clip_fold.py [--max-norm 1.0] [--epochs 3] [--subjects 5] [--minutes 9] [--out DIR]
"""
import argparse
import sys
import tempfile
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--max-norm", type=float, default=1.0)
    ap.add_argument("--epochs", type=int, default=3)
    ap.add_argument("--subjects", type=int, default=5)
    ap.add_argument("--minutes", type=float, default=None)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("grad_clip_fold needs a CUDA device (B200)")
    from multimodalsignal_b200 import main as mm, preprocess as pp, synth
    sids = synth.ALL_SUBJECTS[:args.subjects]
    minutes = args.minutes or synth.SHORT_MINUTES
    subs = {sid: synth.make_subject(sid, synth.ALL_SUBJECTS.index(sid), minutes=minutes, protocol=synth.SHORT_PROTOCOL) for sid in sids}
    items = [(sid, subs[sid].as_pickle_dict, pp.base_halving_quirk(sid, synth.SHORT_PROTOCOL)) for sid in sids]
    streams = pp.preprocess_subjects_sharded(items, 64, include_wrist=True)
    mm.ALL_SUBJECTS = list(sids)
    mm.EPOCHS = args.epochs
    mm.GRAD_CLIP_NORM = args.max_norm
    out = Path(args.out) if args.out else Path(tempfile.mkdtemp(prefix="mms_clip_fold_"))
    res = mm.run_fold(0, sids[0], out, pp.CHEST_CHANNEL_NAMES + pp.WRIST_CHANNEL_NAMES, subject_streams=streams)
    logs = sorted(out.rglob("training_log.txt"))
    for p in logs:
        print(p.read_text(encoding="utf-8"))
    print({k: v for k, v in res.items() if isinstance(v, (int, float, str))})
    n = sum(l.startswith("Gradient norm before clipping") for p in logs for l in p.read_text(encoding="utf-8").splitlines())
    print(f"grad_clip_fold: {n} gradient-norm lines over {args.epochs} epochs")
    return 0 if n >= 1 else 1


if __name__ == "__main__":
    sys.exit(main())
