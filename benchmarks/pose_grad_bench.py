#!/usr/bin/env python
"""Cost of the camera pose gradient (v_viewmats): the default and the pose variants timed alternately in one process
with CUDA events.

    python benchmarks/pose_grad_bench.py --out profiles/r03_pose_grad.json

  project_bwd   qed_project_bwd vs qed_project_bwd_pose on the same packed gradient record (fused path, SH degree 3,
                RGB+ED) at S1 (1M Gaussians, one 1920x1080 view) and S0 (10k Gaussians, 8 views of 256x256); at S1 also
                the kernel variants of the test hook qed_debug_set_project_bwd_one, which split the extra cost of the pose
                kernel into occupancy (4 instead of 5 resident blocks) and the pose work itself
  fused_step    FusedSplatStep.step with pose_gradients False / True at S1
  autograd      get_viewmat -> rasterization -> depth_supervised_loss -> backward() without / with pose gradients at S1

Milliseconds per call: the median over rounds of (event time of `reps` back-to-back calls) / reps.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from qed_splatter_b200 import _lib, depth_supervised_loss, get_viewmat, ops, rasterization  # noqa: E402
from qed_splatter_b200._lib import ptr  # noqa: E402
from qed_splatter_b200.pipeline import FusedSplatStep  # noqa: E402
from qed_splatter_b200.scenes import scene_s0, scene_s1  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in out.split(","))
        return dict(device=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:  # the measurement stands without it, but say so
        return dict(device=torch.cuda.get_device_name(), power_limit=f"unknown ({e})")


def alternate(fns, rounds, reps):
    """fns: {name: callable}; each round times `reps` calls of every fn in turn -> {name: median ms per call}."""
    times = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                fn()
            b.record()
            b.synchronize()
            times[k].append(a.elapsed_time(b) / reps)
    return {k: sorted(v)[len(v) // 2] for k, v in times.items()}


def project_bwd_case(s, dev, rounds, reps, split=False):
    lib = _lib.load()
    t = {k: v.to(dev).contiguous() for k, v in dict(means=s.means, quats=s.quats, scales=s.scales, opacities=s.opacities, sh=s.sh,
                                                      viewmats=s.viewmats, Ks=s.Ks).items()}
    C, N, K = t["viewmats"].shape[0], t["means"].shape[0], t["sh"].shape[1]
    with torch.no_grad():
        radii, _, _, conics = ops.project_gaussians(t["means"], t["quats"], t["scales"], t["opacities"], t["sh"], t["viewmats"], t["Ks"], s.width,
                                                    s.height, sh_degree=3)[:4]
    packed = torch.randn(C * N, 12, device=dev, generator=torch.Generator(device=dev).manual_seed(0)) * 1e-3
    outs = [torch.empty(N, 3, device=dev), torch.empty(N, 4, device=dev), torch.empty(N, 3, device=dev), torch.empty(N, device=dev),
            torch.empty(N, K, 3, device=dev)]
    v_vm = torch.empty(C, 4, 4, device=dev)
    ws_bytes = lib.qed_project_bwd_pose_workspace_bytes(C, N)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    args = (C, N, ptr(t["means"]), ptr(t["quats"]), ptr(t["scales"]), ptr(t["opacities"]), 0, ptr(t["sh"]), K, 3, 0, ptr(t["viewmats"]), ptr(t["Ks"]),
            s.width, s.height, 0.3, 0, 3, 1, ptr(radii), ptr(conics), None, None, None, None, None, None, ptr(packed), *map(ptr, outs))

    def default():
        _lib.check(lib.qed_project_bwd(*args, _lib.current_stream()), "qed_project_bwd")

    def pose():
        _lib.check(lib.qed_project_bwd_pose(*args, ptr(v_vm), ptr(ws), ws_bytes, _lib.current_stream()), "qed_project_bwd_pose")

    fns = dict(default=default, pose=pose)
    if split:
        # the single-view kernel's variants through the test hook qed_debug_set_project_bwd_one (5 = the default):
        #   default_one6:    single-view kernel at 6 resident blocks (80 registers)
        #   default_generic: the multi-view kernel at 4 resident blocks (128 registers), no pose
        #   pose_generic:    the multi-view pose kernel at 4 resident blocks (warp reduction per view)
        # "pose" itself is the single-view pose kernel at 4 resident blocks (128 registers)
        def hooked(fn, one):
            def run():
                lib.qed_debug_set_project_bwd_one(one)
                fn()
                lib.qed_debug_set_project_bwd_one(5)
            return run
        fns.update(default_one6=hooked(default, 6), default_generic=hooked(default, 0), pose_generic=hooked(pose, 0))
    alternate(fns, 2, 3)  # warm-up
    r = alternate(fns, rounds, reps)
    out = dict(C=C, N=N, width=s.width, height=s.height, visible=int((radii > 0).sum()), default_ms=r["default"], pose_ms=r["pose"],
               extra_ms=r["pose"] - r["default"])
    if split:
        out["variants_ms"] = {k: v for k, v in r.items()}
    return out


def fused_step_case(s, dev, rounds, reps):
    t = s.to(dev)
    fs = FusedSplatStep(dev)
    bg = torch.tensor([0.2, 0.5, 0.8], device=dev)
    args = (t.means, t.quats, t.scales, t.opacities, t.sh, t.viewmats, t.Ks, t.width, t.height, 3, t.gt_rgb, t.gt_depth, bg)
    fns = dict(default=lambda: fs.step(*args), pose=lambda: fs.step(*args, pose_gradients=True))
    alternate(fns, 2, 3)
    r = alternate(fns, rounds, reps)
    return dict(default_ms=r["default"], pose_ms=r["pose"], extra_ms=r["pose"] - r["default"])


def autograd_case(s, dev, rounds, reps):
    t = s.to(dev)
    bg = torch.tensor([0.2, 0.5, 0.8], device=dev)
    leaves = [x.clone().requires_grad_(True) for x in (t.means, t.quats, t.scales, t.opacities, t.sh)]
    W, tr = t.viewmats[:, :3, :3], t.viewmats[:, :3, 3:]
    R = W.transpose(1, 2)
    c2w = torch.cat([R * torch.tensor([[[1.0, -1.0, -1.0]]], device=dev), -(R @ tr)], dim=-1).contiguous()

    def run(pose):
        pose_in = c2w.clone().requires_grad_(pose)
        vm = get_viewmat(pose_in, pose_gradients=pose)
        r, a, _ = rasterization(*leaves, vm, t.Ks, t.width, t.height, sh_degree=3, render_mode="RGB+ED", pose_gradients=pose)
        depth_supervised_loss(r, a, t.gt_rgb, t.gt_depth, bg)[0].backward()

    fns = dict(default=lambda: run(False), pose=lambda: run(True))
    alternate(fns, 2, 3)
    r = alternate(fns, rounds, reps)
    return dict(default_ms=r["default"], pose_ms=r["pose"], extra_ms=r["pose"] - r["default"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=15)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    s1, s0 = scene_s1(), scene_s0()
    res = dict(bench="pose_grad", **gpu_info(), rounds=a.rounds, reps=a.reps,
               project_bwd_s1=project_bwd_case(s1, dev, a.rounds, a.reps, split=True), project_bwd_s0=project_bwd_case(s0, dev, a.rounds, a.reps),
               fused_step_s1=fused_step_case(s1, dev, a.rounds, max(a.reps // 4, 1)), autograd_s1=autograd_case(s1, dev, a.rounds, max(a.reps // 4, 1)))
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
