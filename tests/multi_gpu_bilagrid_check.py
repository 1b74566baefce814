#!/usr/bin/env python
"""Multi-GPU check of the bilateral grid in SplatTrainer (run under torchrun on >= 2 B200s; NOT collected by pytest):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tests/multi_gpu_bilagrid_check.py

For comm = "exchange" (the per-view grid rows and ids summed by this library's all-reduce kernel) and "nccl":
1. N ranks x 1 view == 1 rank x N views: the dense grid gradient of the first step (TV + every view's row) equals the one
   of a single-process trainer fed all N views (float tolerance), and is bit-identical on every rank.
2. After 3 steps every replica holds bit-identical grids.
Prints one JSON line (rank 0)."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from qed_splatter_b200.scenes import scene_s0  # noqa: E402
from qed_splatter_b200.trainer import SplatTrainer, TrainConfig  # noqa: E402


def _trainer(s, dev, comm, world, rank, num_cameras):
    cfg = TrainConfig(use_bilateral_grid=True, bilateral_grid_lr=1e-2, bilateral_grid_warmup=0, stop_split_at=0, comm=comm)
    p = (s.means.to(dev), s.quats.to(dev), torch.log(s.scales).to(dev), torch.logit(s.opacities).to(dev), s.sh.to(dev))
    return SplatTrainer(*p, cfg=cfg, rank=rank, world_size=world, num_cameras=num_cameras)


def run(dev, rank, world, comm):
    s = scene_s0(N=20000, C=world, size=128)
    t = s.to(dev)
    bg = torch.tensor([0.2, 0.5, 0.8], device=dev)
    ids = torch.arange(world) * 2 + 1  # every other grid has no view
    sl = slice(rank, rank + 1)
    tr = _trainer(s, dev, comm, world, rank, 2 * world)
    grads = []
    for _ in range(3):
        tr.step(t.viewmats[sl], t.Ks[sl], s.width, s.height, t.gt_rgb[sl], t.gt_depth[sl], bg, total_views=world, camera_ids=ids[sl])
        grads.append(tr.bilagrid.grad.clone())
    single = _trainer(s, dev, "nccl", 1, 0, 2 * world)
    single.step(t.viewmats, t.Ks, s.width, s.height, t.gt_rgb, t.gt_depth, bg, camera_ids=ids)
    ref = single.bilagrid.grad
    err = float((grads[0] - ref).abs().max())
    scale = float(ref.abs().max())
    gathered = [torch.empty_like(tr.bilagrid.param) for _ in range(world)]
    dist.all_gather(gathered, tr.bilagrid.param)
    g0 = [torch.empty_like(grads[0]) for _ in range(world)]
    dist.all_gather(g0, grads[0])
    return dict(comm=tr.comm, grad_max_err=err, grad_scale=scale, grad_ok=err <= 1e-4 * scale,
                grad_bit_identical=all(torch.equal(g.view(torch.int32), g0[0].view(torch.int32)) for g in g0),
                grids_bit_identical=all(torch.equal(g.view(torch.int32), gathered[0].view(torch.int32)) for g in gathered))


def main():
    world, rank, local = int(os.environ["WORLD_SIZE"]), int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    res = dict(world=world, runs=[run(dev, rank, world, comm) for comm in ("exchange", "nccl")])
    ok = all(r["grad_ok"] and r["grad_bit_identical"] and r["grids_bit_identical"] for r in res["runs"])
    flag = torch.tensor([1.0 if ok else 0.0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    res["ok_all_ranks"] = bool(flag.item() == 1.0)
    if rank == 0:
        print(json.dumps(res))
    assert res["ok_all_ranks"], res
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
