#!/usr/bin/env python
"""Cost of splatfacto's MCMC strategy (TrainConfig(strategy="mcmc"), qed_splatter_b200/mcmc.py), with CUDA events.

    python benchmarks/mcmc_bench.py --out profiles/r07_mcmc.json
    torchrun --nproc-per-node 8 benchmarks/mcmc_bench.py --cases s3 --out profiles/r07_mcmc_s3_n8.json

  kernels     at N = 1M, 3M, 6M (5 % of the Gaussians dead): the per-step launches qed_mcmc_noise and qed_mcmc_reg, and the
              refine-step pieces: sample (5 % N draws: weights, int64 scan, Philox draws), relocate (the values pass with
              zeroed moments + the copies into the dead rows) and add (the values pass + qed_arena_gather to N + 5 %);
              median ms per call over alternating rounds.
  trainer     SplatTrainer.step on S1 (1M Gaussians, one 1920x1080 view) and S3 (6M, 1440x1080; under torchrun one view per
              rank, the trainer's default comm) with strategy "default" and "mcmc" (max_gs_num = N, so the add step is empty
              and N stays fixed), warmup_length 0 and refine_every 100, over steps 1 .. 2 * refine_every: every step timed
              with its own events.  Reported: the median of the ordinary steps, the refine steps, and the mean over the
              window (= the ordinary step + the refine cost amortised over refine_every steps).
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from pose_grad_bench import alternate, gpu_info  # noqa: E402
from qed_splatter_b200 import _lib, mcmc  # noqa: E402
from qed_splatter_b200._lib import ptr  # noqa: E402
from qed_splatter_b200.scenes import scene_s1, scene_s3  # noqa: E402
from qed_splatter_b200.trainer import GROUPS, GaussianArena, SplatTrainer, TrainConfig  # noqa: E402


def kernels_case(N, dev, rounds, reps):
    g = torch.Generator(device=dev).manual_seed(0)
    o = torch.rand(N, device=dev, generator=g) * 0.9 + 0.05
    o[::20] = 0.001  # 5 % dead
    a = GaussianArena(torch.randn(N, 3, device=dev, generator=g), torch.randn(N, 4, device=dev, generator=g),
                      torch.log(torch.rand(N, 3, device=dev, generator=g) * 0.05 + 0.001), torch.logit(o), torch.randn(N, 16, 3, device=dev, generator=g))
    st = mcmc.MCMCStrategy(dev, cap_max=2 * N)
    lib = st.lib
    dead, n_dead = st.dead_rows(a)
    n_new = mcmc.growth(N, 2 * N)
    draws, counts = st.draw(a, n_dead, 600, mcmc.STREAM_RELOCATE, True)
    add_draws, add_counts = st.draw(a, n_new, 600, mcmc.STREAM_ADD, False)
    starts = st._starts(a)
    ws = st._workspace(N)
    total = torch.empty(1, dtype=torch.int64, device=dev)
    out_d = torch.empty(n_dead, dtype=torch.int32, device=dev)
    out_c = torch.empty(N, dtype=torch.int32, device=dev)
    new_off, n = GaussianArena.layout(N + n_new)
    new_starts = torch.tensor([new_off[k][0] for k in GROUPS], dtype=torch.int64)
    new_p, new_m, new_v = (torch.empty(n, device=dev) for _ in range(3))
    src = torch.cat([torch.arange(N, dtype=torch.int32, device=dev), add_draws])
    fresh = torch.cat([torch.zeros(N, dtype=torch.uint8, device=dev), torch.ones(n_new, dtype=torch.uint8, device=dev)])
    op = a.view(a.param, "opacities")
    s = _lib.current_stream

    def sample():
        _lib.check(lib.qed_mcmc_sample(N, ptr(op), 0.005, 1, n_dead, 42, 600, 1, ptr(out_d), ptr(out_c), ptr(total), ptr(ws), ws.numel(), s()), "sample")

    def relocate():
        _lib.check(lib.qed_mcmc_relocate(N, ptr(counts), 0.005, 1, n_dead, ptr(draws), ptr(dead), ptr(a.param), ptr(a.exp_avg), ptr(a.exp_avg_sq),
                                         starts.data_ptr(), s()), "relocate")

    def add():
        _lib.check(lib.qed_mcmc_relocate(N, ptr(add_counts), 0.005, 0, 0, None, None, ptr(a.param), None, None, starts.data_ptr(), s()), "add")
        _lib.check(lib.qed_arena_gather(N + n_new, ptr(src), ptr(fresh), None, None, None, ptr(a.param), ptr(a.exp_avg), ptr(a.exp_avg_sq),
                                        starts.data_ptr(), ptr(new_p), ptr(new_m), ptr(new_v), new_starts.data_ptr(), s()), "gather")

    fns = dict(noise=lambda: st.inject_noise(a, 7, 1e-9), reg=lambda: st.regularize(a), sample=sample, relocate=relocate, add=add)
    alternate(fns, 2, 3)
    r = alternate(fns, rounds, reps)
    return dict(N=N, n_dead=n_dead, n_new=n_new, **{f"{k}_ms": v for k, v in r.items()})


def trainer_case(name, dev, rank, world, pg, steps_per_refine=100):
    if name == "s1":
        t = scene_s1().to(dev)
    else:
        t = scene_s3(view_offset=rank, total_views=world).to(dev) if world > 1 else scene_s3().to(dev)
    bg = torch.tensor([0.2, 0.5, 0.8], device=dev)
    N = t.means.shape[0]
    res = dict(scene=name, N=N, width=t.width, height=t.height, world=world, refine_every=steps_per_refine)
    for strategy in ("default", "mcmc"):
        cfg = TrainConfig(strategy=strategy, max_gs_num=N, warmup_length=0, refine_every=steps_per_refine, sh_degree_interval=1)
        tr = SplatTrainer(t.means.clone(), t.quats.clone(), torch.log(t.scales), torch.logit(t.opacities), t.sh.clone(), cfg=cfg, rank=rank,
                          world_size=world, process_group=pg)
        tr.step_count = 1  # steps 1 .. 2 * refine_every: two refine steps, none at step 0
        ev, kinds, infos = [], [], []
        for _ in range(2 * steps_per_refine):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            refine = tr.step_count % steps_per_refine == 0
            a.record()
            _, info = tr.step(t.viewmats, t.Ks, t.width, t.height, t.gt_rgb, t.gt_depth, bg)
            b.record()
            ev.append((a, b))
            kinds.append(refine)
            if info is not None:
                infos.append(info)
        torch.cuda.synchronize()
        ms = [a.elapsed_time(b) for a, b in ev]
        plain = sorted(m for m, k in zip(ms, kinds) if not k)
        ref = [m for m, k in zip(ms, kinds) if k]
        med = plain[len(plain) // 2]
        res[strategy] = dict(step_ms_median=med, refine_step_ms=ref, window_mean_ms=sum(ms) / len(ms),
                             refine_cost_amortised_ms=(sum(ref) / len(ref) - med) / steps_per_refine, N_end=tr.arena.N, refine_info=infos,
                             comm=tr.comm)
        del tr
        torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=11)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--cases", default="kernels,s1,s3")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    pg = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD
    cases = a.cases.split(",")
    res = dict(bench="mcmc", **gpu_info(), world=world, rounds=a.rounds, reps=a.reps)
    if "kernels" in cases and world == 1:
        res["kernels"] = [kernels_case(N, dev, a.rounds, a.reps) for N in (1_000_000, 3_000_000, 6_000_000)]
        torch.cuda.empty_cache()
    for name in ("s1", "s3"):
        if name in cases:
            res[f"trainer_{name}"] = trainer_case(name, dev, rank, world, pg)
    if rank == 0:
        print(json.dumps(res))
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "w") as f:
                f.write(json.dumps(res, indent=1) + "\n")
    if world > 1:
        import torch.distributed as dist

        dist.destroy_process_group()


if __name__ == "__main__":
    main()
