#!/usr/bin/env python
"""Multi-GPU check of SplatTrainer's per-camera tables, the camera optimizer and the bilateral grid (run under torchrun on
>= 2 B200s; NOT collected by pytest):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tests/multi_gpu_trainer_check.py

For each table and comm = "exchange" (this library's NVLink path: the pose table gradient, or the per-view grid rows and
ids, summed by its all-reduce kernel) and "nccl":
1. N ranks x 1 view == 1 rank x N views: the table gradient of the first step (camera optimizer: data term + regulariser;
   grid: TV + every view's row) equals the one of a single-process trainer fed all N views (float tolerance), and is
   bit-identical on every rank.
2. After 3 steps every replica holds a bit-identical table.
Prints one JSON line (rank 0)."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from qed_splatter_b200.scenes import camera_to_worlds, scene_s0  # noqa: E402
from qed_splatter_b200.trainer import SplatTrainer, TrainConfig  # noqa: E402

TABLES = {
    "camera_opt": dict(camera_optimizer="SO3xR3", camera_opt_lr=1e-3, camera_opt_warmup=0),
    "bilagrid": dict(use_bilateral_grid=True, bilateral_grid_lr=1e-2, bilateral_grid_warmup=0),
}


def _trainer(s, dev, table, comm, world, rank, num_cameras):
    cfg = TrainConfig(**TABLES[table], stop_split_at=0, comm=comm)
    p = (s.means.to(dev), s.quats.to(dev), torch.log(s.scales).to(dev), torch.logit(s.opacities).to(dev), s.sh.to(dev))
    return SplatTrainer(*p, cfg=cfg, rank=rank, world_size=world, num_cameras=num_cameras)


def _grad_and_table(tr):
    if tr.camera_opt is not None:
        return tr.camera_opt.pose_grad, tr.pose_adjustment.contiguous()
    return tr.bilagrid.grad, tr.bilagrid.param


def run(dev, rank, world, table, comm):
    s = scene_s0(N=20000, C=world, size=128)
    t = s.to(dev)
    bg = torch.tensor([0.2, 0.5, 0.8], device=dev)
    c2w, ids = camera_to_worlds(s.viewmats).to(dev), torch.arange(world) * 2 + 1  # every other table row has no view

    def step(tr, sl, **kw):
        if table == "camera_opt":  # the views come as poses, adjusted by the table
            kw["camera_to_worlds"] = c2w[sl]
        viewmats = None if table == "camera_opt" else t.viewmats[sl]
        tr.step(viewmats, t.Ks[sl], s.width, s.height, t.gt_rgb[sl], t.gt_depth[sl], bg, camera_ids=ids[sl], **kw)

    sl = slice(rank, rank + 1)
    tr = _trainer(s, dev, table, comm, world, rank, 2 * world)
    grads = []
    for _ in range(3):
        step(tr, sl, total_views=world)
        grads.append(_grad_and_table(tr)[0].clone())
    single = _trainer(s, dev, table, "nccl", 1, 0, 2 * world)
    step(single, slice(0, world))
    ref = _grad_and_table(single)[0]
    err = float((grads[0] - ref).abs().max())
    scale = float(ref.abs().max())
    param = _grad_and_table(tr)[1]
    gathered = [torch.empty_like(param) for _ in range(world)]
    dist.all_gather(gathered, param)
    g0 = [torch.empty_like(grads[0]) for _ in range(world)]
    dist.all_gather(g0, grads[0].contiguous())
    return dict(table=table, comm=tr.comm, grad_max_err=err, grad_scale=scale, grad_ok=err <= 1e-4 * scale,
                grad_bit_identical=all(torch.equal(g.view(torch.int32), g0[0].view(torch.int32)) for g in g0),
                tables_bit_identical=all(torch.equal(g.view(torch.int32), gathered[0].view(torch.int32)) for g in gathered))


def main():
    world, rank, local = int(os.environ["WORLD_SIZE"]), int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    res = dict(world=world, runs=[run(dev, rank, world, table, comm) for table in TABLES for comm in ("exchange", "nccl")])
    ok = all(r["grad_ok"] and r["grad_bit_identical"] and r["tables_bit_identical"] for r in res["runs"])
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
