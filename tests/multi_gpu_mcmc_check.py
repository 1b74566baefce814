#!/usr/bin/env python
"""Multi-GPU check of SplatTrainer(strategy="mcmc") (run under torchrun on >= 2 B200s; NOT collected by pytest):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tests/multi_gpu_mcmc_check.py

For comm = "exchange" (this library's NVLink path) and "nccl":
1. N ranks x 1 view == 1 rank x N views: the Gaussian gradient of the first step (data term + the MCMC regularisers, added
   once after the sum) equals the one of a single-process trainer fed all N views (float tolerance).
2. After refine steps (relocation of dead Gaussians and growth) and noise steps, every replica holds the same N and
   bit-identical parameter, exp_avg and exp_avg_sq arenas: the draws derive from (seed, step) alone, no broadcast.
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


def _trainer(s, dev, comm, world, rank):
    o = s.opacities.clone()
    o[::17] = 0.002  # dead Gaussians for the first relocation
    cfg = TrainConfig(strategy="mcmc", max_gs_num=24000, warmup_length=1, refine_every=3, comm=comm)
    p = (s.means.to(dev), s.quats.to(dev), torch.log(s.scales).to(dev), torch.logit(o).to(dev), s.sh.to(dev))
    return SplatTrainer(*p, cfg=cfg, rank=rank, world_size=world)


def run(dev, rank, world, comm):
    s = scene_s0(N=20000, C=world, size=128)
    t = s.to(dev)
    bg = torch.tensor([0.2, 0.5, 0.8], device=dev)
    sl = slice(rank, rank + 1)
    tr = _trainer(s, dev, comm, world, rank)
    infos, grad0 = [], None
    for it in range(10):
        _, info = tr.step(t.viewmats[sl], t.Ks[sl], s.width, s.height, t.gt_rgb[sl], t.gt_depth[sl], bg, total_views=world)
        if it == 0:
            grad0 = tr.arena.grad.clone()
        if info is not None:
            infos.append(info)
    single = _trainer(s, dev, "nccl", 1, 0)
    single.step(t.viewmats, t.Ks, s.width, s.height, t.gt_rgb, t.gt_depth, bg)
    ref = single.arena.grad
    err = float((grad0 - ref).abs().max())
    scale = float(ref.abs().max())
    n = torch.tensor([float(tr.arena.N)], device=dev)
    ns = [torch.empty_like(n) for _ in range(world)]
    dist.all_gather(ns, n)
    same_n = all(float(x) == float(n) for x in ns)
    identical = same_n
    if same_n:
        for buf in (tr.arena.param, tr.arena.exp_avg, tr.arena.exp_avg_sq):
            got = [torch.empty_like(buf) for _ in range(world)]
            dist.all_gather(got, buf.contiguous())
            identical = identical and all(torch.equal(g.view(torch.int32), got[0].view(torch.int32)) for g in got)
    return dict(comm=tr.comm, N=tr.arena.N, refines=infos, grad_max_err=err, grad_scale=scale, grad_ok=err <= 1e-4 * scale, same_n=same_n,
                arenas_bit_identical=identical, grew=tr.arena.N > 20000, relocated=any(i["n_relocated"] > 0 for i in infos))


def main():
    world, rank, local = int(os.environ["WORLD_SIZE"]), int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    res = dict(world=world, runs=[run(dev, rank, world, comm) for comm in ("exchange", "nccl")])
    ok = all(r["grad_ok"] and r["arenas_bit_identical"] and r["grew"] and r["relocated"] for r in res["runs"])
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
