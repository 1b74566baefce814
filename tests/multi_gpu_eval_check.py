#!/usr/bin/env python
"""Multi-GPU check of SplatTrainer.evaluate (run under torchrun on >= 2 B200s; NOT collected by pytest):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tests/multi_gpu_eval_check.py

For comm = "exchange" and "nccl": after a few training steps (one view per rank), every rank evaluates its own C held-out
views.  Every rank must return the same rows, bit for bit, and they must equal, bit for bit, the rows of one trainer in
this process that holds the same Gaussians and evaluates all world * C views itself.  Prints one JSON line (rank 0)."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from qed_splatter_b200.metrics import METRIC_NAMES  # noqa: E402
from qed_splatter_b200.scenes import scene_s0  # noqa: E402
from qed_splatter_b200.trainer import SplatTrainer, TrainConfig  # noqa: E402

C_LOCAL = 5  # held-out views per rank: with two ranks, the one-process reference renders them in two chunks
STEPS = 4


def _bits(rows):
    return torch.stack([rows[n] for n in METRIC_NAMES], 1).contiguous().view(torch.int64)


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
    dev = torch.device("cuda", torch.cuda.current_device())
    dist.init_process_group("nccl", device_id=dev)
    bg = torch.tensor([0.2, 0.5, 0.8], device=dev)
    train = scene_s0(N=20000, C=world, size=128).to(dev)
    held = scene_s0(N=20000, C=world * C_LOCAL, size=128, seed=7).to(dev)
    out = {"world": world}
    for comm in ("exchange", "nccl"):
        p = (train.means, train.quats, torch.log(train.scales), torch.logit(train.opacities), train.sh)
        tr = SplatTrainer(*p, cfg=TrainConfig(comm=comm, sh_degree_interval=2), rank=rank, world_size=world)
        sl = slice(rank, rank + 1)
        for _ in range(STEPS):
            tr.step(train.viewmats[sl], train.Ks[sl], train.width, train.height, train.gt_rgb[sl], train.gt_depth[sl], bg, total_views=world)
        mine = slice(rank * C_LOCAL, (rank + 1) * C_LOCAL)
        rows = _bits(tr.evaluate(held.viewmats[mine], held.Ks[mine], held.width, held.height, held.gt_rgb[mine], held.gt_depth[mine], bg))
        gathered = [torch.empty_like(rows) for _ in range(world)]
        dist.all_gather(gathered, rows)
        assert all(torch.equal(g, rows) for g in gathered), f"{comm}: ranks disagree"
        # one process, the same Gaussians and step, all views
        a = tr.arena
        v = a.views(a.param)
        solo = SplatTrainer(v["means"].clone(), v["quats"].clone(), v["scales"].clone(), v["opacities"].clone(), v["sh"].clone(), cfg=tr.cfg)
        solo.step_count = tr.step_count
        ref = _bits(solo.evaluate(held.viewmats, held.Ks, held.width, held.height, held.gt_rgb, held.gt_depth, bg))
        assert torch.equal(ref, rows), f"{comm}: rows differ from one process evaluating every view"
        out[comm] = {"views": int(rows.shape[0]), "psnr_mean": float(rows.view(torch.float64)[:, 0].mean())}
    if rank == 0:
        print(json.dumps(out))
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
