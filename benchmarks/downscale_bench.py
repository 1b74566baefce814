#!/usr/bin/env python
"""Cost of splatfacto's resolution schedule, timed alternately in one process with CUDA events.

    python benchmarks/downscale_bench.py --out profiles/r06_downscale.json

  pass_1080p     qed_downscale_ground_truth alone on one 1920x1080 view (uint8 RGB + raw uint16 depth + bool mask), d = 2
                 and 4.  Every call reads another of COPIES input sets (together larger than the 126 MB L2), so the
                 full-resolution reads come from HBM.  Bytes = 6 B read per full-resolution pixel + 20 / d^2 B written.
  torch_1080p    the torch formulation of the same reduction on the same inputs (TF32 off): `.float() / 255` + conv2d on
                 the image, the depth converted to float metres + conv2d, the mask `.float()` + conv2d.
  trainer_s1     SplatTrainer.step at S1 (1M Gaussians, one 1920x1080 view, SH degree 3, no densification, frozen) with
                 num_downscales=2 at one step of each phase (d = 4, 2, 1), against num_downscales=0 (d = 1).

Milliseconds per call: the median over rounds of (event time of `reps` back-to-back calls) / reps.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from pose_grad_bench import alternate, gpu_info  # noqa: E402
from qed_splatter_b200.data_side import downscale_ground_truth  # noqa: E402
from qed_splatter_b200.scenes import scene_s1  # noqa: E402
from qed_splatter_b200.trainer import SplatTrainer, TrainConfig  # noqa: E402

COPIES = 24  # 24 x 12.4 MB of 1080p inputs: more than the L2 holds
HBM_TBPS = 7.7  # data sheet, one B200 (not reached; the ratio below is against it)


def cached_inputs(dev, W=1920, H=1080, n=COPIES):
    g = torch.Generator(device=dev).manual_seed(0)
    return [(torch.randint(0, 256, (1, H, W, 3), dtype=torch.uint8, device=dev, generator=g),
             torch.randint(0, 20000, (1, H, W), dtype=torch.int32, device=dev, generator=g).to(torch.uint16),
             torch.rand(1, H, W, device=dev, generator=g) > 0.2) for _ in range(n)]


def pass_case(dev, rounds, reps, W=1920, H=1080):
    ins = cached_inputs(dev, W, H)
    res = {}
    for d in (2, 4):
        h, w = H // d, W // d
        out = (torch.empty(1, h, w, 3, device=dev), torch.empty(1, h, w, 1, device=dev), torch.empty(1, h, w, 1, device=dev))
        k = [0]

        def kernel():
            rgb, dep, mk = ins[k[0] % COPIES]
            k[0] += 1
            downscale_ground_truth(rgb, dep, mk, d, out=out)

        def torch_path():
            rgb, dep, mk = ins[k[0] % COPIES]
            k[0] += 1
            wt = (1.0 / (d * d)) * torch.ones((1, 1, d, d), dtype=torch.float32, device=dev)
            F.conv2d((rgb[0].float() / 255.0).permute(2, 0, 1)[:, None], wt, stride=d)
            F.conv2d((dep.to(torch.float64) * 0.001).to(torch.float32)[None], wt, stride=d)
            F.conv2d(mk.float()[None], wt, stride=d)

        fns = dict(kernel=kernel, torch=torch_path)
        alternate(fns, 2, 3)
        r = alternate(fns, rounds, reps)
        nbytes = W * H * 6 + h * w * 20
        res[f"d{d}"] = dict(kernel_ms=r["kernel"], torch_ms=r["torch"], bytes=nbytes, kernel_tbps=nbytes / r["kernel"] / 1e9,
                            kernel_share_of_datasheet_hbm=nbytes / r["kernel"] / 1e9 / HBM_TBPS)
    return dict(width=W, height=H, inputs="uint8 rgb, uint16 depth, bool mask", input_copies=COPIES, **res)


def trainer_case(dev, rounds, reps):
    t = scene_s1().to(dev)
    rgb = (t.gt_rgb * 255).round().to(torch.uint8)
    dep = (t.gt_depth[..., 0] * 1000).round().to(torch.int32).to(torch.uint16)
    bg = torch.tensor([0.2, 0.5, 0.8], device=dev)
    params = lambda: (t.means.clone(), t.quats.clone(), torch.log(t.scales), torch.logit(t.opacities), t.sh.clone())  # noqa: E731
    # no refine and no opacity reset inside the timed steps; SH degree 3 from the first step; learning rates 0, so Adam does
    # its full work but every arm renders the same Gaussians in every round
    frozen = dict(lr_means=1e-30, lr_means_final=1e-30, lr_quats=0.0, lr_scales=0.0, lr_opacities=0.0, lr_features_dc=0.0, lr_features_rest=0.0)
    base = dict(sh_degree_interval=1, refine_every=10 ** 9, resolution_schedule=3000, **frozen)
    sched = SplatTrainer(*params(), cfg=TrainConfig(num_downscales=2, **base))
    plain = SplatTrainer(*params(), cfg=TrainConfig(**base))

    def at(tr, step):
        def fn():
            tr.step_count = step  # hold the phase: every timed step renders at the same factor
            tr.step(t.viewmats, t.Ks, t.width, t.height, rgb, dep, bg)
        return fn

    fns = dict(d4=at(sched, 3), d2=at(sched, 3003), d1=at(sched, 6003), plain_d1=at(plain, 6003))
    alternate(fns, 2, 3)
    r = alternate(fns, rounds, reps)
    return dict(ssim_lambda=TrainConfig().ssim_lambda, gt="uint8 rgb, uint16 depth, full resolution",
                **{f"{k}_ms": v for k, v in r.items()})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=15)
    ap.add_argument("--reps", type=int, default=40)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    torch.backends.cudnn.allow_tf32 = False
    res = dict(bench="downscale", **gpu_info(), rounds=a.rounds, reps=a.reps, pass_1080p=pass_case(dev, a.rounds, a.reps),
               trainer_s1=trainer_case(dev, a.rounds, max(a.reps // 8, 1)))
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
