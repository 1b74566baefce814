#!/usr/bin/env python
"""Multi-GPU check of SplatTrainer.state_dict() / SplatTrainer.from_state_dict() (run under torchrun on >= 2 B200s; NOT
collected by pytest):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tests/multi_gpu_checkpoint_check.py

For comm = "exchange" and "nccl", strategy "default" with the camera optimizer, one view per rank:
1. Run A and control run A' go uninterrupted; run B saves in the middle of a refine interval (every rank's statistics in
   flight), writes the state with torch.save, reads it back and resumes at the same world size.  A, A' and B take the same
   refine decisions, B's replicas stay bit-identical, and B's state lies within the spread of A' around A
   (tests/test_gpu_checkpoint.py's rule).
2. The same checkpoint resumed by one process (rank 0, alone): the statistics of both ranks land on it summed (radii: max),
   and its first refine step after the resume takes the same decisions (the refine info) as the multi-rank run.
Prints one JSON line (rank 0)."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from qed_splatter_b200.scenes import camera_to_worlds, scene_s0  # noqa: E402
from qed_splatter_b200.trainer import SplatTrainer, TrainConfig  # noqa: E402
from test_checkpoint_cpu import _through_file  # noqa: E402
from test_gpu_checkpoint import spread_violations  # noqa: E402

STEPS, K = 10, 5  # refine at 3 and 9 (reset at 6): statistics of step 4 in flight at the save
CFG = dict(warmup_length=1, refine_every=3, reset_alpha_every=2, pause_refine_after_reset=3, sh_degree_interval=3, camera_optimizer="SO3xR3",
           camera_opt_warmup=0)


def _inputs(dev, world, rank):
    s = scene_s0(N=20000, C=world, size=128)
    t = s.to(dev)
    sl = slice(rank, rank + 1)
    c2w = camera_to_worlds(s.viewmats).to(dev)
    return s, (t.Ks[sl], s.width, s.height, t.gt_rgb[sl], t.gt_depth[sl], torch.tensor([0.2, 0.5, 0.8], device=dev)), c2w[sl], torch.tensor([rank])


def _step(tr, args, c2w, ids, world):
    return tr.step(None, *args, total_views=world, camera_to_worlds=c2w, camera_ids=ids)[1]


def _run(dev, world, rank, comm, save_at=None):
    s, args, c2w, ids = _inputs(dev, world, rank)
    o = s.opacities.clone()
    o[::17] = 0.002
    p = (s.means.to(dev), s.quats.to(dev), torch.log(s.scales).to(dev), torch.logit(o).to(dev), s.sh.to(dev))
    tr = SplatTrainer(*p, cfg=TrainConfig(comm=comm, **CFG), rank=rank, world_size=world, num_cameras=world)
    infos, saved = [], None
    for i in range(STEPS):
        if i == save_at:
            saved = _through_file(tr.state_dict())
            tr = SplatTrainer.from_state_dict(saved, rank=rank, world_size=world, process_group=dist.group.WORLD)
        infos.append(_step(tr, args, c2w, ids, world))
    return tr, infos, saved


def _identical(tr, world):
    ok = True
    for buf in (tr.arena.param, tr.arena.exp_avg, tr.arena.exp_avg_sq, tr.camera_opt.param):
        got = [torch.empty_like(buf) for _ in range(world)]
        dist.all_gather(got, buf.contiguous())
        ok = ok and all(torch.equal(g.view(torch.int32), got[0].view(torch.int32)) for g in got)
    return ok


def run(dev, rank, world, comm):
    A, infos_a, _ = _run(dev, world, rank, comm)
    A1, infos_a1, _ = _run(dev, world, rank, comm)
    B, infos_b, saved = _run(dev, world, rank, comm, save_at=K)
    sa, sa1, sb = A.state_dict(), A1.state_dict(), B.state_dict()
    bad = spread_violations(sa, [sa1], sb)
    res = dict(comm=B.comm, N=B.arena.N, same_decisions=infos_a == infos_a1 == infos_b, refines=[i for i in infos_b if i is not None],
               replicas_bit_identical=_identical(B, world), within_spread=not bad, violations=[list(map(str, v)) for v in bad[:4]],
               rows_differ=not torch.equal(saved["strategy_state"]["grad2d"][0], saved["strategy_state"]["grad2d"][1]))
    # the same checkpoint resumed by rank 0 alone, fed every view: its next refine takes the multi-rank run's decisions
    if rank == 0:
        s = scene_s0(N=20000, C=world, size=128)
        t = s.to(dev)
        one = SplatTrainer.from_state_dict(saved, world_size=1)
        rows = saved["strategy_state"]
        res["one_rank_sum"] = bool(torch.equal(one.state.count.cpu(), rows["count"].sum(0)) and torch.equal(one.state.radii.cpu(), rows["radii"].amax(0)))
        ids = torch.arange(world)
        one_infos = [one.step(None, t.Ks, s.width, s.height, t.gt_rgb, t.gt_depth, torch.tensor([0.2, 0.5, 0.8], device=dev),
                              camera_to_worlds=camera_to_worlds(s.viewmats).to(dev), camera_ids=ids)[1] for _ in range(K, STEPS)]
        first = next(i for i, x in enumerate(infos_b[K:]) if x is not None)
        res["one_rank_first_refine"] = one_infos[first]
        res["one_rank_same_first_refine"] = one_infos[first] == infos_b[K + first]
    return res


def main():
    world, rank, local = int(os.environ["WORLD_SIZE"]), int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    res = dict(world=world, runs=[run(dev, rank, world, comm) for comm in ("exchange", "nccl")])
    ok = all(r["same_decisions"] and r["replicas_bit_identical"] and r["within_spread"] and r["rows_differ"] for r in res["runs"])
    if rank == 0:
        ok = ok and all(r["one_rank_sum"] and r["one_rank_same_first_refine"] for r in res["runs"])
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
