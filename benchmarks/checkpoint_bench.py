#!/usr/bin/env python
"""Cost of saving and resuming a run (SplatTrainer.state_dict / SplatTrainer.from_state_dict) against the step time.

    python benchmarks/checkpoint_bench.py --out profiles/r08_checkpoint.json

For S1 (1M Gaussians, one 1920x1080 view) and S3 (6M, one 1440x1080 view), each with the SO3xR3 camera optimizer and the
bilateral grid (default 16x16x8 shape) on at 1000 cameras, strategy "default", full SH:
  step_ms              median of `--steps` ordinary steps after a warm-up, CUDA events around each
  state_dict_s         state_dict() (device-to-host copies into fresh pageable CPU tensors), host clock between synchronises
  save_s / fsync_s     torch.save to a file in the local temporary directory, then flush + os.fsync of that file
  load_s               torch.load(weights_only=True) of that file (right after writing it, so mostly from the page cache)
  resume_first_step_s  from_state_dict + its first step(), host clock between synchronises (includes the host-to-device
                       copies, the trainer's allocations and the first step's buffer sizing)
  save_fraction_per_2000_steps = (state_dict_s + save_s + fsync_s) / (2000 * step_ms): the share of run time that saving
                       every 2000 steps (splatfacto's steps_per_save) costs
Each host-clock figure is the median of `--repeats` runs.
"""
import argparse
import json
import os
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from pose_grad_bench import gpu_info  # noqa: E402
from qed_splatter_b200.scenes import camera_to_worlds, scene_s1, scene_s3  # noqa: E402
from qed_splatter_b200.trainer import SplatTrainer, TrainConfig  # noqa: E402

NUM_CAMERAS = 1000


def _timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def _median(v):
    return sorted(v)[len(v) // 2]


def case(name, dev, steps, repeats, tmpdir):
    t = (scene_s1() if name == "s1" else scene_s3()).to(dev)
    bg = torch.tensor([0.2, 0.5, 0.8], device=dev)
    c2w = camera_to_worlds(t.viewmats.cpu()).to(dev)
    cfg = TrainConfig(camera_optimizer="SO3xR3", use_bilateral_grid=True, sh_degree_interval=1, camera_opt_warmup=0, bilateral_grid_warmup=0)
    tr = SplatTrainer(t.means.clone(), t.quats.clone(), torch.log(t.scales), torch.logit(t.opacities), t.sh.clone(), cfg=cfg,
                      num_cameras=NUM_CAMERAS)
    k = [0]

    def step(trainer):
        k[0] += 1
        ids = torch.tensor([k[0] % NUM_CAMERAS])
        return trainer.step(None, t.Ks, t.width, t.height, t.gt_rgb, t.gt_depth, bg, camera_to_worlds=c2w, camera_ids=ids)

    for _ in range(5):
        step(tr)
    ev = []
    for _ in range(steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        step(tr)
        b.record()
        ev.append((a, b))
    torch.cuda.synchronize()
    step_ms = _median([a.elapsed_time(b) for a, b in ev])

    path = os.path.join(tmpdir, f"{name}.pt")
    sd_s, save_s, fsync_s, load_s, resume_s, first_ms = [], [], [], [], [], []
    for _ in range(repeats):
        dt, state = _timed(tr.state_dict)
        sd_s.append(dt)
        with open(path, "wb") as f:
            t0 = time.perf_counter()
            torch.save(state, f)
            f.flush()
            t1 = time.perf_counter()
            os.fsync(f.fileno())
            t2 = time.perf_counter()
        save_s.append(t1 - t0)
        fsync_s.append(t2 - t1)
        nbytes = os.path.getsize(path)
        del state
        dt, loaded = _timed(lambda: torch.load(path, weights_only=True))
        load_s.append(dt)

        def resume():
            r = SplatTrainer.from_state_dict(loaded)
            step(r)
            return r

        dt, resumed = _timed(resume)
        resume_s.append(dt)
        del loaded
        # the resumed trainer's second step: back to the ordinary step time
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        step(resumed)
        b.record()
        b.synchronize()
        first_ms.append(a.elapsed_time(b))
        del resumed
        torch.cuda.empty_cache()
    os.remove(path)
    res = dict(scene=name, N=tr.arena.N, width=t.width, height=t.height, num_cameras=NUM_CAMERAS,
               bilateral_grid_shape=list(cfg.bilateral_grid_shape), checkpoint_bytes=nbytes, step_ms=step_ms,
               state_dict_s=_median(sd_s), save_s=_median(save_s), fsync_s=_median(fsync_s), load_s=_median(load_s),
               resume_first_step_s=_median(resume_s), resumed_second_step_ms=_median(first_ms),
               all=dict(state_dict_s=sd_s, save_s=save_s, fsync_s=fsync_s, load_s=load_s, resume_first_step_s=resume_s))
    save_total = res["state_dict_s"] + res["save_s"] + res["fsync_s"]
    res["save_total_s"] = save_total
    res["run_time_per_2000_steps_s"] = 2000 * step_ms / 1e3
    res["save_fraction_per_2000_steps"] = save_total / (2000 * step_ms / 1e3)
    del tr
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="s1,s3")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("checkpoint_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = dict(bench="checkpoint", **gpu_info(), steps=a.steps, repeats=a.repeats)
    with tempfile.TemporaryDirectory() as tmpdir:
        for name in a.cases.split(","):
            res[f"trainer_{name}"] = case(name, dev, a.steps, a.repeats, tmpdir)
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
