#!/usr/bin/env python
"""Cost of splatfacto's bilateral grid, timed alternately in one process with CUDA events.

    python benchmarks/bilagrid_bench.py --out profiles/r05_bilagrid.json

  loss_1080p     the loss stage alone on one 1920x1080 view (rgb_weight 0.8, SSIM 0.2, depth 0.2): qed_loss_fwd_bwd against
                 qed_loss_fwd_bwd_bilagrid with 1000 grids of the default 16x16x8 shape
  trainer_s1     SplatTrainer.step at S1 (1M Gaussians, one 1920x1080 view, SH degree 3, no densification) with the grid
                 off and on (1000 grids; camera ids handed over on the host, as a data loader does)
  grid_kernels   the per-step launches on the 1000 grids alone: TV (overwrites the dense gradient), accumulating one view's
                 row, and the dense Adam over all grids (qed_adam_arena, one group)

Milliseconds per call: the median over rounds of (event time of `reps` back-to-back calls) / reps.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from pose_grad_bench import alternate, gpu_info  # noqa: E402
from qed_splatter_b200 import _lib  # noqa: E402
from qed_splatter_b200._lib import ptr  # noqa: E402
from qed_splatter_b200.scenes import scene_s1  # noqa: E402
from qed_splatter_b200.trainer import SplatTrainer, TrainConfig  # noqa: E402

NUM_GRIDS = 1000
X, Y, L = 16, 16, 8


def identity_grids(dev):
    return torch.eye(3, 4, device=dev).reshape(1, 12, 1, 1, 1).repeat(NUM_GRIDS, 1, L, Y, X).contiguous()


def loss_case(dev, rounds, reps, W=1920, H=1080):
    lib = _lib.load()
    gen = torch.Generator(device=dev).manual_seed(0)
    render = torch.rand(1, H, W, 4, device=dev, generator=gen)
    alphas = torch.rand(1, H, W, 1, device=dev, generator=gen)
    gt_rgb = torch.rand(1, H, W, 3, device=dev, generator=gen)
    gt_depth = torch.rand(1, H, W, 1, device=dev, generator=gen) + 1
    bg = torch.tensor([0.2, 0.5, 0.8], device=dev)
    grids = identity_grids(dev) + 0.05 * torch.randn(NUM_GRIDS, 12, L, Y, X, device=dev, generator=gen)
    ids = torch.tensor([17], dtype=torch.int32, device=dev)
    stats = torch.zeros(8, dtype=torch.float64, device=dev)
    loss = torch.empty(3, device=dev)
    v_render, v_alphas = torch.empty_like(render), torch.empty_like(alphas)
    rows = torch.empty(1, 12, L, Y, X, device=dev)
    ws_off = torch.empty(lib.qed_loss_workspace_bytes(1, W, H, 0.2), dtype=torch.uint8, device=dev)
    ws_on = torch.empty(lib.qed_loss_bilagrid_workspace_bytes(1, W, H, 0.2), dtype=torch.uint8, device=dev)
    common = (1, W, H, ptr(render), ptr(alphas), ptr(gt_rgb), 0, ptr(gt_depth), 0, 1.0, None, 0, ptr(bg), 0.8, 0.2, 0.2, 1.0, ptr(stats), ptr(loss),
              ptr(v_render), ptr(v_alphas))

    def off():
        _lib.check(lib.qed_loss_fwd_bwd(*common, ptr(ws_off), ws_off.numel(), _lib.current_stream()), "qed_loss_fwd_bwd")

    def on():
        _lib.check(lib.qed_loss_fwd_bwd_bilagrid(*common, ptr(grids), ptr(ids), NUM_GRIDS, X, Y, L, ptr(rows), ptr(ws_on), ws_on.numel(),
                                                 _lib.current_stream()), "qed_loss_fwd_bwd_bilagrid")

    fns = dict(off=off, on=on)
    alternate(fns, 2, 3)
    r = alternate(fns, rounds, reps)
    return dict(width=W, height=H, ssim_lambda=0.2, num_grids=NUM_GRIDS, grid_shape_xyl=[X, Y, L], off_ms=r["off"], on_ms=r["on"],
                extra_ms=r["on"] - r["off"])


def trainer_case(dev, rounds, reps):
    t = scene_s1().to(dev)
    bg = torch.tensor([0.2, 0.5, 0.8], device=dev)
    params = lambda: (t.means.clone(), t.quats.clone(), torch.log(t.scales), torch.logit(t.opacities), t.sh.clone())  # noqa: E731
    base = dict(stop_split_at=0, sh_degree_interval=1)  # no refine / opacity reset: every step does the same work
    off = SplatTrainer(*params(), cfg=TrainConfig(**base))
    on = SplatTrainer(*params(), cfg=TrainConfig(use_bilateral_grid=True, bilateral_grid_warmup=0, **base), num_cameras=NUM_GRIDS)
    ids = torch.tensor([17])
    fns = dict(off=lambda: off.step(t.viewmats, t.Ks, t.width, t.height, t.gt_rgb, t.gt_depth, bg),
               on=lambda: on.step(t.viewmats, t.Ks, t.width, t.height, t.gt_rgb, t.gt_depth, bg, camera_ids=ids))
    alternate(fns, 2, 3)  # warm-up (reaches SH degree 3)
    r = alternate(fns, rounds, reps)
    return dict(num_grids=NUM_GRIDS, ssim_lambda=TrainConfig().ssim_lambda, off_ms=r["off"], on_ms=r["on"], extra_ms=r["on"] - r["off"])


def grid_kernels_case(dev, rounds, reps):
    lib = _lib.load()
    grids = identity_grids(dev) + 0.05 * torch.randn(NUM_GRIDS, 12, L, Y, X, device=dev)
    v = torch.empty_like(grids)
    partials = torch.empty(NUM_GRIDS, dtype=torch.float64, device=dev)
    tv = torch.empty(1, device=dev)
    rows = torch.randn(1, 12, L, Y, X, device=dev) * 1e-4
    ids = torch.tensor([17], dtype=torch.int32, device=dev)
    m, s = torch.zeros_like(grids), torch.zeros_like(grids)
    n = grids.numel()
    ends = torch.tensor([n], dtype=torch.int64, device=dev)
    lr = torch.tensor([2e-3], device=dev)
    st = _lib.current_stream

    fns = dict(
        tv=lambda: _lib.check(lib.qed_bilagrid_tv(NUM_GRIDS, X, Y, L, ptr(grids), 10.0, ptr(v), ptr(partials), ptr(tv), st()), "tv"),
        accumulate=lambda: _lib.check(lib.qed_bilagrid_accumulate(1, ptr(ids), ptr(rows), NUM_GRIDS, X, Y, L, ptr(v), st()), "accumulate"),
        adam=lambda: _lib.check(lib.qed_adam_arena(n, ptr(grids), ptr(v), ptr(m), ptr(s), 1, ptr(ends), ptr(lr), None, None, None, 0.9, 0.999, 1e-15,
                                                   2000, st()), "adam"))
    alternate(fns, 2, 3)
    r = alternate(fns, rounds, reps)
    return dict(num_grids=NUM_GRIDS, floats=n, **{f"{k}_ms": x for k, x in r.items()})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=15)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = dict(bench="bilagrid", **gpu_info(), rounds=a.rounds, reps=a.reps, loss_1080p=loss_case(dev, a.rounds, a.reps),
               trainer_s1=trainer_case(dev, a.rounds, max(a.reps // 4, 1)), grid_kernels=grid_kernels_case(dev, a.rounds, a.reps))
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
