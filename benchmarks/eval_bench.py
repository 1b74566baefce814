#!/usr/bin/env python
"""Cost of held-out evaluation: qed_eval_metrics alone, the same metrics as torch ops, and SplatTrainer.evaluate.

    python benchmarks/eval_bench.py --out profiles/r09_eval.json

  kernel        `qed_eval_metrics` on one 1920x1080 view per launch (uint8 RGB, raw uint16 depth), cycling over `--pool`
                distinct input sets (about 52 MB each, more than the 126 MB L2 together), CUDA events around `--launches`
                launches.  bytes_per_view = what the metrics must read (render 16 + alpha 4 + RGB 3 + depth 2 B/pixel); its
                rate over the kernel time is given as a fraction of the 7.7 TB/s HBM3e data-sheet bandwidth.
  torch         the same per-view metrics written as torch ops on the GPU: composite and clamp, mean squared error, SSIM
                by F.conv2d (separable 11-tap Gaussian, valid windows) and the depth metrics by boolean masks; same inputs.
  evaluate_*    SplatTrainer.evaluate on 64 held-out views at S1 (1M Gaussians, 1920x1080) and S3 (6M, 1440x1080), and at S1
                with num_downscales=2 (training steps at 1/4 resolution), host clock between synchronises, per view; against
                the median ordinary step() of the same trainer (one view).  Then `--rounds` windows of `--steps` steps of
                that trainer after the evaluation, alternating with a twin trainer that took the same steps and never
                evaluated: whatever an evaluation leaves behind that slows training shows as after_over_twin > 1.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from pose_grad_bench import gpu_info  # noqa: E402
from qed_splatter_b200 import _lib  # noqa: E402
from qed_splatter_b200.metrics import METRIC_NAMES  # noqa: E402
from qed_splatter_b200.scenes import scene_s1, scene_s3  # noqa: E402
from qed_splatter_b200.trainer import SplatTrainer, TrainConfig  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
W, H = 1920, 1080


def _inputs(dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    render = torch.rand(1, H, W, 4, device=dev, generator=g)
    render[..., 3] = 0.5 + 10.0 * render[..., 3]
    alphas = torch.rand(1, H, W, 1, device=dev, generator=g)
    alphas[alphas < 0.1] = 0.0
    gt_rgb = torch.randint(0, 256, (1, H, W, 3), device=dev, generator=g, dtype=torch.uint8)
    gt_depth = torch.randint(0, 20000, (1, H, W), device=dev, generator=g, dtype=torch.int32).to(torch.int16)
    return render, alphas, gt_rgb, gt_depth


def torch_metrics(render, alphas, gt_rgb, gt_depth, bg, depth_unit_scale=0.001, tol=0.1):
    """The per-view metrics as plain torch ops (what a user would otherwise write): -> [C, 11] float64."""
    rgb = torch.clamp(render[..., :3] + (1 - alphas) * bg, 0.0, 1.0)
    gt = gt_rgb.float() / 255.0
    depth = render[..., 3]
    fill = depth.flatten(1).amax(1).clamp_min(0)[:, None, None]
    depth = torch.where(alphas[..., 0] > 0, depth, fill).double()
    g32 = ((gt_depth.to(torch.int32) & 0xFFFF).double() * depth_unit_scale).float()  # compared with the tolerance in float32
    g = g32.double()
    mse = ((rgb.double() - gt.double()) ** 2).flatten(1).mean(1)
    X, Y = gt.permute(0, 3, 1, 2), rgb.permute(0, 3, 1, 2)
    c = torch.arange(11, dtype=torch.float64, device=render.device) - 5
    w = torch.exp(-(c ** 2) / (2 * 1.5 ** 2))
    w = (w / w.sum()).float()

    def filt(t):
        t = F.conv2d(t, w.view(1, 1, 11, 1).expand(3, 1, 11, 1), groups=3)
        return F.conv2d(t, w.view(1, 1, 1, 11).expand(3, 1, 1, 11), groups=3)

    mu1, mu2 = filt(X), filt(Y)
    s1, s2, s12 = filt(X * X) - mu1 * mu1, filt(Y * Y) - mu2 * mu2, filt(X * Y) - mu1 * mu2
    smap = ((2 * mu1 * mu2 + 1e-4) * (2 * s12 + 9e-4)) / ((mu1 * mu1 + mu2 * mu2 + 1e-4) * (s1 + s2 + 9e-4))
    ssim = smap.flatten(1).double().mean(1)
    rows = []
    for v in range(render.shape[0]):
        valid = torch.isfinite(g32[v]) & (g32[v] > tol)
        gv, dv = g[v][valid], depth[v][valid]
        t = torch.maximum(gv / dv, dv / gv)
        rows.append(torch.stack([torch.abs(gv - dv).div(gv).mean(), ((gv - dv) ** 2 / gv).mean(), ((gv - dv) ** 2).mean().sqrt(),
                                 ((gv.log() - dv.log()) ** 2).mean().sqrt(), (t < 1.25).double().mean(), (t < 1.25 ** 2).double().mean(),
                                 (t < 1.25 ** 3).double().mean(), valid.sum().double()]))
    return torch.cat([torch.stack([10 * torch.log10(1 / mse), ssim, mse], 1), torch.stack(rows)], 1)


def _events(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(n):
        fn(i)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n


def kernel_case(dev, pool, launches, rounds):
    sets = [_inputs(dev, 100 + i) for i in range(pool)]
    bg = torch.tensor([0.2, 0.5, 0.8], device=dev)
    out = torch.empty(1, len(METRIC_NAMES), dtype=torch.float64, device=dev)
    lib = _lib.load()
    ws_bytes = lib.qed_eval_metrics_workspace_bytes(1, W, H)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    stream = _lib.current_stream()
    ptr = _lib.ptr

    def kernel(i):
        r, a, rgb, dep = sets[i % pool]
        _lib.check(lib.qed_eval_metrics(1, W, H, ptr(r), ptr(a), ptr(rgb), 1, ptr(dep), 1, 0.001, ptr(bg), 0.1, ptr(out), ptr(ws), ws_bytes, stream),
                   "qed_eval_metrics")

    def torch_ops(i):
        r, a, rgb, dep = sets[i % pool]
        torch_metrics(r, a, rgb, dep, bg)

    for i in range(pool):  # warm-up of every shape; and the two agree
        kernel(i)
        t = torch_metrics(*sets[i], bg)
        torch.testing.assert_close(out, t, rtol=1e-4, atol=1e-4)
    ms = {"kernel": [], "torch": []}
    for _ in range(rounds):  # alternating
        ms["kernel"].append(_events(kernel, launches))
        ms["torch"].append(_events(torch_ops, max(launches // 20, pool)))
    med = {k: sorted(v)[len(v) // 2] for k, v in ms.items()}
    nbytes = W * H * (16 + 4 + 3 + 2)
    return dict(width=W, height=H, pool=pool, pool_bytes=pool * nbytes, launches=launches, rounds=rounds, bytes_per_view=nbytes,
                kernel_ms_per_view=med["kernel"], kernel_bytes_per_s=nbytes / (med["kernel"] / 1e3),
                kernel_fraction_of_hbm=nbytes / (med["kernel"] / 1e3) / HBM_BYTES_PER_S,
                torch_ms_per_view=med["torch"], torch_over_kernel=med["torch"] / med["kernel"], all_ms=ms)


def _step_ms(tr, step_args, steps):
    """Median of `steps` ordinary steps, CUDA events around each."""
    ev = []
    for _ in range(steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        tr.step(*step_args)
        b.record()
        ev.append((a, b))
    torch.cuda.synchronize()
    return sorted(a.elapsed_time(b) for a, b in ev)[steps // 2]


def evaluate_case(name, dev, views, steps, repeats, rounds):
    """`name` s1 / s3, or s1_ds: S1 under splatfacto's resolution schedule (num_downscales=2: training steps at 1/4
    resolution, the evaluation at full resolution)."""
    s1 = name.startswith("s1")
    held = (scene_s1(C=views) if s1 else scene_s3(C=views)).to(dev)
    train = (scene_s1(C=1, seed=7) if s1 else scene_s3(C=1, view_offset=3, total_views=views)).to(dev)
    bg = torch.tensor([0.2, 0.5, 0.8], device=dev)
    cfg = dict(sh_degree_interval=1, num_downscales=2 if name.endswith("_ds") else 0)
    # `tr` evaluates; `twin` takes the same steps and never evaluates
    tr, twin = (SplatTrainer(held.means.clone(), held.quats.clone(), torch.log(held.scales), torch.logit(held.opacities), held.sh.clone(),
                             cfg=TrainConfig(**cfg)) for _ in range(2))
    step_args = (train.viewmats, train.Ks, train.width, train.height, train.gt_rgb, train.gt_depth, bg)
    for _ in range(5):
        tr.step(*step_args)
        twin.step(*step_args)
    step_ms = _step_ms(tr, step_args, steps)
    _step_ms(twin, step_args, steps)  # same step count as `tr`
    args = (held.viewmats, held.Ks, held.width, held.height, held.gt_rgb, held.gt_depth, bg)
    tr.evaluate(*args)  # warm-up
    times = []
    for _ in range(repeats):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rows = tr.evaluate(*args)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    eval_s = sorted(times)[repeats // 2]
    # what an evaluation leaves behind for training: steps of `tr` after it against the twin's, alternating
    after, never = [], []
    for _ in range(rounds):
        after.append(_step_ms(tr, step_args, steps))
        never.append(_step_ms(twin, step_args, steps))
    med = lambda v: sorted(v)[len(v) // 2]  # noqa: E731
    res = dict(scene=name, N=tr.arena.N, width=held.width, height=held.height, views=views, sh_degree=tr.sh_degree_to_use(),
               train_downscale=tr.downscale_factor(), step_ms=step_ms, evaluate_s=eval_s, evaluate_ms_per_view=eval_s / views * 1e3,
               evaluate_view_over_step=eval_s / views * 1e3 / step_ms, psnr_mean=float(rows["psnr"].mean()), all_evaluate_s=times,
               step_ms_after_evaluate=med(after), step_ms_twin_never_evaluated=med(never), after_over_twin=med(after) / med(never),
               all_step_ms_after_evaluate=after, all_step_ms_twin=never)
    del tr, twin, held, train
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pool", type=int, default=8)
    ap.add_argument("--launches", type=int, default=400)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--cases", default="s1,s3,s1_ds")
    ap.add_argument("--views", type=int, default=64)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("eval_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    torch.backends.cudnn.allow_tf32 = False
    res = dict(bench="eval", **gpu_info(), hbm_bytes_per_s=HBM_BYTES_PER_S)
    res["kernel_1080p"] = kernel_case(dev, a.pool, a.launches, a.rounds)
    print(json.dumps(res["kernel_1080p"]), flush=True)
    for name in a.cases.split(","):
        if name:
            res[f"evaluate_{name}"] = evaluate_case(name, dev, a.views, a.steps, a.repeats, a.rounds)
            print(json.dumps(res[f"evaluate_{name}"]), flush=True)
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
