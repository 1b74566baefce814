#!/usr/bin/env python
"""Cost of splatfacto's camera optimizer (SO3xR3 pose table) in SplatTrainer, timed alternately in one process with CUDA events.

    python benchmarks/camera_opt_bench.py --out profiles/r04_camera_opt.json

  trainer_s1     SplatTrainer.step at S1 (1M Gaussians, one 1920x1080 view, SH degree 3, no densification) with the camera
                 optimizer off and on (a 1000-camera table; camera ids handed over on the host, as a data loader does)
  table_kernels  the four launches the optimizer adds per step (apply, table backward, regulariser, table Adam), alone
  exchange_s1    the projection backward of the multi-GPU exchange without / with pose gradients at S1, one rank emulated on
                 one device (peer stores to a local buffer; the NVLink traffic of a real multi-GPU run is not included)

Milliseconds per call: the median over rounds of (event time of `reps` back-to-back calls) / reps.
"""
import argparse
import ctypes
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from pose_grad_bench import alternate, gpu_info  # noqa: E402
from qed_splatter_b200 import _lib, ops  # noqa: E402
from qed_splatter_b200._lib import ptr  # noqa: E402
from qed_splatter_b200.camera_opt import CameraPoseOptimizer  # noqa: E402
from qed_splatter_b200.scenes import camera_to_worlds, scene_s1  # noqa: E402
from qed_splatter_b200.trainer import SplatTrainer, TrainConfig  # noqa: E402

NUM_CAMERAS = 1000


def trainer_case(s, dev, rounds, reps):
    t = s.to(dev)
    bg = torch.tensor([0.2, 0.5, 0.8], device=dev)
    params = lambda: (t.means.clone(), t.quats.clone(), torch.log(t.scales), torch.logit(t.opacities), t.sh.clone())
    base = dict(stop_split_at=0, sh_degree_interval=1)  # no refine / opacity reset: every step does the same work
    off = SplatTrainer(*params(), cfg=TrainConfig(**base))
    on = SplatTrainer(*params(), cfg=TrainConfig(camera_optimizer="SO3xR3", camera_opt_warmup=0, **base), num_cameras=NUM_CAMERAS)
    c2w, ids = camera_to_worlds(t.viewmats), torch.tensor([17])
    vm = t.viewmats.contiguous()
    fns = dict(off=lambda: off.step(vm, t.Ks, t.width, t.height, t.gt_rgb, t.gt_depth, bg),
               on=lambda: on.step(None, t.Ks, t.width, t.height, t.gt_rgb, t.gt_depth, bg, camera_to_worlds=c2w, camera_ids=ids))
    alternate(fns, 2, 3)  # warm-up (reaches SH degree 3)
    r = alternate(fns, rounds, reps)
    return dict(off_ms=r["off"], on_ms=r["on"], extra_ms=r["on"] - r["off"], num_cameras=NUM_CAMERAS)


def table_kernels_case(dev, rounds, reps):
    cam = CameraPoseOptimizer(NUM_CAMERAS, dev)
    cam.pose_adjustment.normal_(0, 0.01)
    c2w = camera_to_worlds(scene_s1(N=10, targets=False).viewmats.to(dev))
    ids = torch.tensor([17], dtype=torch.int32, device=dev)
    v = torch.randn(1, 4, 4, device=dev)
    fns = dict(apply=lambda: cam._viewmats(c2w, ids), backward=lambda: cam._backward(v, ids, c2w), regularize=cam.regularize,
               adam=lambda: cam.step(2000))
    alternate(fns, 2, 3)
    r = alternate(fns, rounds, reps)
    return dict(num_cameras=NUM_CAMERAS, views=1, **{f"{k}_ms": x for k, x in r.items()})


def exchange_case(s, dev, rounds, reps):
    lib = _lib.load()
    t = {k: v.to(dev).contiguous() for k, v in dict(means=s.means, quats=s.quats, scales=s.scales, opacities=s.opacities, sh=s.sh,
                                                      viewmats=s.viewmats, Ks=s.Ks).items()}
    C, N, K = t["viewmats"].shape[0], t["means"].shape[0], t["sh"].shape[1]
    with torch.no_grad():
        radii, _, _, conics = ops.project_gaussians(t["means"], t["quats"], t["scales"], t["opacities"], t["sh"], t["viewmats"], t["Ks"], s.width,
                                                    s.height, sh_degree=3)[:4]
    packed = torch.randn(C * N, 12, device=dev, generator=torch.Generator(device=dev).manual_seed(0)) * 1e-3
    outs = [torch.empty(N, 3, device=dev), torch.empty(N, 4, device=dev), torch.empty(N, 3, device=dev), torch.empty(N, device=dev)]
    xch = torch.zeros((C * N + C) * 4, device=dev)
    peers = (ctypes.c_void_p * 1)(xch.data_ptr())
    v_vm = torch.empty(C, 4, 4, device=dev)
    ws_bytes = lib.qed_project_bwd_pose_workspace_bytes(C, N)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    args = (C, N, ptr(t["means"]), ptr(t["quats"]), ptr(t["scales"]), ptr(t["opacities"]), 0, ptr(t["sh"]), K, 3, ptr(t["viewmats"]), ptr(t["Ks"]),
            s.width, s.height, 0.3, 0, 1, ptr(radii), ptr(conics), None, ptr(packed), *map(ptr, outs), None, peers, 1, 0, C, 3.0)

    def default():
        _lib.check(lib.qed_project_bwd_exchange(*args, _lib.current_stream()), "qed_project_bwd_exchange")

    def pose():
        _lib.check(lib.qed_project_bwd_exchange_pose(*args, ptr(v_vm), ptr(ws), ws_bytes, _lib.current_stream()), "qed_project_bwd_exchange_pose")

    fns = dict(default=default, pose=pose)
    alternate(fns, 2, 3)
    r = alternate(fns, rounds, reps)
    return dict(C=C, N=N, world=1, default_ms=r["default"], pose_ms=r["pose"], extra_ms=r["pose"] - r["default"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=15)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    s1 = scene_s1()
    res = dict(bench="camera_opt", **gpu_info(), rounds=a.rounds, reps=a.reps,
               trainer_s1=trainer_case(s1, dev, a.rounds, max(a.reps // 4, 1)), table_kernels=table_kernels_case(dev, a.rounds, a.reps * 5),
               exchange_s1=exchange_case(s1, dev, a.rounds, a.reps))
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
