"""torchrun entry: real NCCL data-parallel steps (SyncBN + one flat gradient all-reduce) on WORLD_SIZE GPUs
must equal the single-device full-batch step.  Used by tests/test_gpu_parallel.py (needs >= 2 GPUs) and by hand:
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tools/dp_check.py
--peer: the symmetric-memory exchange with the peer kernels; --clip: gradient-norm clipping (FlatAdam max_grad_norm) on
every rank and on the reference step.
"""
import os
import sys
import warnings
from pathlib import Path

import numpy as np
import torch
import torch.distributed as dist

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))


def main():
    from conftest import golden_state, load_golden
    from multimodalsignal_b200.models import CnnGruAttentionModel
    from multimodalsignal_b200.parallel import DataParallelTrainStep
    from multimodalsignal_b200.trainer import FlatAdam, FusedTrainStep
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    z, meta = load_golden("model_c6_t640.npz")
    sd = golden_state(z, "sd")

    def model():
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            m = CnnGruAttentionModel(meta["C"], meta["num_classes"], dropout=0.0)
        m.load_state_dict(sd, strict=True)
        return m.cuda().train()

    x, y = torch.from_numpy(z["x"]).cuda(), torch.from_numpy(z["y"]).cuda()
    B, T = x.shape[0], x.shape[2]
    assert B % world == 0
    b = B // world
    m = model()
    peer = "symm" if "--peer" in sys.argv else None      # symmetric memory + the peer kernels instead of NCCL all-reduces
    clip = 0.05 if "--clip" in sys.argv else None        # well below the gradient norm of this batch: every step clips
    step = DataParallelTrainStep(m, FlatAdam(m, lr=1e-3, weight_decay=1e-4, max_grad_norm=clip), b, B, T, rank=rank, peer=peer)
    losses = []
    for _ in range(3 if peer is None else 5):      # peer mode: eager step, graph capture, replays
        step(x[rank * b:(rank + 1) * b], y[rank * b:(rank + 1) * b])
        losses.append(step.global_loss())
    ok = True
    if rank == 0:
        ref = model()
        ref_step = FusedTrainStep(ref, FlatAdam(ref, lr=1e-3, weight_decay=1e-4, max_grad_norm=clip), B, T, use_graph=False)
        ref_losses = []
        for _ in range(len(losses)):
            ref_step(x, y)
            ref_losses.append(ref_step.last_loss())
        np.testing.assert_allclose(losses, ref_losses, atol=2e-5)
        if clip is None:
            np.testing.assert_allclose(losses[:3], z["adam_losses"][:3], atol=1e-4)
        else:
            assert ref_step.opt.clip_coef.item() < 1.0 and step.opt.clip_coef.item() < 1.0
            np.testing.assert_allclose(step.opt.grad_norm.item(), ref_step.opt.grad_norm.item(), rtol=1e-4)
        ref_sd = ref.state_dict()
        for k, v in m.state_dict().items():
            if v.numel():
                np.testing.assert_allclose(v.float().cpu().numpy(), ref_sd[k].float().cpu().numpy(), atol=2e-5, err_msg=k)
        print(f"dp_check ok: world={world} losses={losses}")
    # every rank holds identical parameters after the step
    flat = m.flat_parameters().clone()
    dist.broadcast(flat, src=0)
    assert torch.equal(flat, m.flat_parameters()), "replicas diverged"
    dist.destroy_process_group()
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
