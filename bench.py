#!/usr/bin/env python
"""bench.py — the driver's measurement contract for the depth-supervised splat hot path.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W

Workload = BASELINE.json configs[1]: synthetic 1M-Gaussian scene, one 1920x1080 view per GPU,
RGB+ED forward + qed-splatter loss (RGB-L1 + masked depth-L1) + full backward to the six parameter
tensors.  A "step" is one pass of that hot path over one view per GPU; for N>1 the views are sharded over
the ranks against a replicated Gaussian set and the step ends with the NCCL all-reduce of the flat
gradient arena and of the densification statistics (weak scaling).

metric  = fwd+bwd RGB+depth Mpix/s (whole job: N*H*W*K / time, device-timed, max over ranks).
value   = fused C-ABI pipeline with everything resident in HBM.
e2e     = the same work through the reference-facing call: `rasterization()` (gsplat surface, torch autograd) followed by
          THE REFERENCE'S OWN LINES for the loss, written with torch ops exactly as qed_splatter/model.py:295-306 and
          :87-116 write them (+ the L1 line of splatfacto's parent loss), then `backward()`; the step's inputs (camera,
          ground-truth RGB as the uint8 image cache of config.py:37 + float depth) are copied from pinned host memory
          and the loss is read back every step.  The Gaussian parameters are model state and stay resident, as in
          the reference.  For N>1 the five parameter gradients go out as one coalesced NCCL group call (as DDP / FSDP
          issue them).
e2e_fused_loss = the same with the package's drop-in for those lines, `depth_supervised_loss()` (one autograd op).
train   = full trainer iterations/s (trainer.SplatTrainer: 0.8 L1 + 0.2 (1-SSIM) + 0.2 depth-L1, Adam, strategy
          statistics, pipelined gradient all-reduce) -- the second half of BASELINE.json's metric.
--impl reference = the CPU arm: the oracle (`oracle/`, a port — the reference's own arithmetic lives in the
          un-vendored gsplat and cannot be run here) on the host cores on a bounded sample of THE SAME workload (see
          cpu_sample_step); `cpu_baseline` in the GPU arm's line is the same sample, same code.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "fwd+bwd RGB+depth Mpix/s"
UNIT = "Mpix/s"
PARAM_FLOATS = 3 + 4 + 3 + 1 + 48  # means, quats, scales, opacity, SH(16x3) = 59 floats / Gaussian

# dram__bytes_read.sum + dram__bytes_write.sum per step and stage, from the committed `ncu --set full` capture of one
# step of this workload: profiles/r02_dram_bytes.json, written by benchmarks/ncu_dram_bytes.py from the .ncu-rep
# (profiles/README.md has the command).  Absent file / stage -> traffic null.
DRAM_BYTES_JSON = os.path.join(ROOT, "profiles", "r02_dram_bytes.json")


def load_ncu_traffic():
    try:
        d = json.load(open(DRAM_BYTES_JSON))
        return {k: float(v["dram_bytes"]) for k, v in d.get("stages", {}).items()}, d.get("workload")
    except Exception:
        return {}, None


# SURVEY.md §8(d) per-unit figures (D = 4 channels)
FLOP_PER_PAIR_FWD = 30.0
FLOP_PER_PAIR_BWD = 100.0
BYTES_PROJ_FWD_PER_GAUSS = 44.0
BYTES_PROJ_FWD_PER_VISIBLE = 192.0 + 100.0  # SH read + records written
BYTES_PROJ_BWD_PER_GAUSS = 44.0 + 4.0 + 236.0  # inputs + radii read, gradients written
BYTES_PROJ_BWD_PER_VISIBLE = 48.0 + 12.0 + 192.0  # packed grads + conic + SH read


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of the measured window (>= 1)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--gaussians", type=int, default=1_000_000)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--mode", default="RGB+ED", choices=["RGB+ED", "RGB+D"])
    ap.add_argument("--sort", default="two_level", choices=["two_level", "own", "cub"])
    ap.add_argument("--comm-chunks", type=int, default=1, help="Gaussian ranges of the projection backward whose SH gradients are all-reduced while the next range computes (N>1)")
    ap.add_argument("--comm", default="exchange", choices=["exchange", "nccl"],
                    help="N>1, how the gradient arena is summed over the ranks: this library's NVLink path (view-colour exchange + one "
                         "all-reduce kernel, comm.ViewShardedGradients) or torch.distributed / NCCL all-reduce (the library baseline)")
    ap.add_argument("--radix-onesweep", type=int, default=None, choices=[0, 1, 2],
                    help="A/B hook: 0 = three kernels per radix pass everywhere, 1 = look-back passes for sorts of <= 444 blocks (library default), 2 = everywhere")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-bucket", action="store_true", help="e2e, N>1: all-reduce one flat bucket of gradient views instead of a coalesced group call")
    ap.add_argument("--gt-float", action="store_true", help="e2e: ground-truth RGB as float32 instead of the uint8 image cache")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--repeats", type=int, default=5, help="extra timed windows of K steps after the measured one (spread: median / p10 / p90)")
    ap.add_argument("--no-multi-gpu-check", action="store_true", help="N>1: skip the N-rank == 1-rank gradient / replica-identity check")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last step of the measured window returned (loss, gradients, radii, render, alphas, strategy "
                         "statistics; a fixed seeded sample of Gaussians and pixels) as DIR/<name>.npy, for comparing two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl ours)")
    return args


# ------------------------------------------------------------------------------------------------
# --dump-outputs
# ------------------------------------------------------------------------------------------------
DUMP_GAUSSIANS = 1 << 16  # sampled Gaussians: 59 gradient floats + radii + 3 statistics each
DUMP_PIXELS = 1 << 18     # sampled pixels: render (4) + alpha
DUMP_MAX_BYTES = 64 << 20


def _dump_sample(n: int, k: int, seed: int):
    """Sorted indices of a fixed seeded sample of k of range(n) (all of them when n <= k)."""
    import torch

    if n <= k:
        return torch.arange(n)
    return torch.randperm(n, generator=torch.Generator().manual_seed(seed))[:k].sort().values


def collect_outputs(out, stats) -> dict:
    """Host copies (float32, float64 indices) of a fused step's StepOutput + the strategy statistics, sampled so that
    the whole dump stays under DUMP_MAX_BYTES.  Same arguments -> same inputs -> same sample."""
    import torch

    N = out.radii.shape[-1]
    gi = _dump_sample(N, DUMP_GAUSSIANS, seed=1)
    gd = gi.to(out.radii.device)
    res = {"loss": out.loss.float().cpu(), "gaussian_index": gi.double()}
    for k, g in out.grads.items():
        res["grad_" + k] = g.reshape(N, -1).index_select(0, gd).float().cpu()
    res["radii"] = out.radii.reshape(-1, N).index_select(1, gd).float().cpu()
    res["strategy_stats"] = stats.index_select(1, gd).float().cpu()  # grad2d, count, radii_max
    C, H, W = out.render.shape[:3]
    pi = _dump_sample(C * H * W, DUMP_PIXELS, seed=2)
    pd = pi.to(out.render.device)
    res["pixel_index"] = pi.double()
    res["render"] = out.render.reshape(C * H * W, -1).index_select(0, pd).float().cpu()
    res["alphas"] = out.alphas.reshape(C * H * W).index_select(0, pd).float().cpu()
    total = sum(t.numel() * t.element_size() for t in res.values())
    assert total <= DUMP_MAX_BYTES, f"output dump of {total} B exceeds {DUMP_MAX_BYTES} B"
    return res


def write_outputs(dump_dir: str, res: dict) -> None:
    import numpy as np

    os.makedirs(dump_dir, exist_ok=True)
    for k, t in res.items():
        np.save(os.path.join(dump_dir, k + ".npy"), t.numpy())


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock / power / throttle reasons sampled DURING the timed regions.  NVML from a thread (every 5 ms, so even a
    30 ms window holds several samples); `nvidia-smi -lms` as the fallback when pynvml is not importable."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    PERIOD_S = 0.005

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.thread = None
        self.lines = []
        self.samples = []  # (sm_mhz, power_w, reasons bitmask)
        self.sm_max = None
        self._stop = threading.Event()
        self.how = None

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.gpu]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else self.gpu
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons

            def loop():
                while not self._stop.is_set():
                    try:
                        self.samples.append((float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)),
                                             pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0, int(get_reasons(h))))
                    except Exception:
                        pass
                    time.sleep(self.PERIOD_S)

            self.thread = threading.Thread(target=loop, daemon=True)
            self.thread.start()
            self.how = "nvml"
            return
        except Exception:
            self.thread = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
            self.how = "nvidia-smi"
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    @staticmethod
    def _pct(v, q):
        return v[min(len(v) - 1, max(0, int(round(q * (len(v) - 1)))))] if v else None

    def stop(self):
        sm, power, reasons = [], [], set()
        if self.how == "nvml":
            self._stop.set()
            self.thread.join(timeout=1)
            # NVML bits: 0x8 hw_slowdown, 0x20 sw_thermal, 0x40 hw_thermal, 0x4 sw_power_cap
            for f, pw, r in self.samples:
                sm.append(f)
                power.append(pw)
                for bit, name in ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap")):
                    if r & bit:
                        reasons.add(name)
            mx = self.sm_max
        elif self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
            mx = None
            for ln in self.lines:
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    mx = float(f[2])
                    power.append(float(f[3]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        else:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"], "samples": 0}
        sm.sort()
        return {"sm_mhz": self._pct(sm, 0.5), "sm_mhz_p10": self._pct(sm, 0.1), "sm_mhz_p90": self._pct(sm, 0.9), "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(power) if power else None, "sampler": self.how}


# ------------------------------------------------------------------------------------------------
# CPU arm (oracle) on a bounded sample of the workload
# ------------------------------------------------------------------------------------------------
CPU_TILE_STRIDE = 8  # every 8th tile column x every 8th tile row = 1/64 of the tiles, spread over the whole image


def workload_name(args) -> str:
    return (f"S1 (BASELINE.json configs[1]): {args.gaussians} Gaussians (SH degree 3), one {args.width}x{args.height} view per GPU, "
            f"{args.mode} forward + RGB-L1/depth-L1 loss + backward to means/quats/scales/opacities/SH")


def bench_config(args, world: int) -> dict:
    """The `config` object: names the workload; identical in the GPU arm and in `--impl reference`."""
    return {
        "workload": workload_name(args),
        "parallelism": f"view-sharded x{world}, replicated Gaussians, gradient arena ({PARAM_FLOATS * 4} B/Gaussian) summed over the ranks every step "
                       "(densification accumulators are all-reduced when a refine step consumes them, not per step)",
        "cache": "inputs larger than L2 (236 MB parameters + ~0.3 GB intermediates per step vs 126 MB L2); no explicit flush",
        "sort": args.sort,
    }


class CpuSample:
    """The CPU arm's bounded sample of the SAME workload (full Gaussian count, full resolution, same camera):
    projection + SH and the tile intersection (incl. the 64-bit key sort) run on everything, forward and backward;
    compositing + loss forward / backward run on a systematic 1/64 sample of the 16x16 tiles (every 8th tile row and
    column, spread over the whole image, so the sample sees the image's mean splat density).  One step's time for the
    whole image is then   t = t_project+SH(fwd+bwd) + t_intersect + (t_composite(fwd+bwd) + t_loss) / sampled_fraction,
    every term measured in that step; Mpix/s = W * H / t."""

    def __init__(self, args):
        import torch

        from qed_splatter_b200.scenes import scene_s1

        self.W, self.H = args.width, args.height
        self.mode = args.mode
        self.s = scene_s1(N=args.gaussians, width=self.W, height=self.H)
        self.tw, self.th = (self.W + 15) // 16, (self.H + 15) // 16
        keep = torch.zeros(self.th, self.tw, dtype=torch.bool)
        keep[CPU_TILE_STRIDE // 2 - 1::CPU_TILE_STRIDE, CPU_TILE_STRIDE // 2 - 1::CPU_TILE_STRIDE] = True
        self.keep = keep.flatten()
        self.picks = torch.nonzero(self.keep).flatten().tolist()
        self.pix = keep.repeat_interleave(16, 0).repeat_interleave(16, 1)[:self.H, :self.W][None, :, :, None].float()
        self.frac = float(self.pix.sum()) / (self.W * self.H)
        self.desc = (f"same workload ({args.gaussians} Gaussians, {self.W}x{self.H}, {args.mode}, float32): projection+SH and tile "
                     f"intersection/sort fwd+bwd over everything; compositing+loss fwd+bwd on a systematic sample of {len(self.picks)} of "
                     f"{self.tw * self.th} tiles ({self.frac:.4f} of the pixels), that part scaled by 1/{self.frac:.4f}")

    def step(self):
        import torch

        import oracle

        s, W, H, tw, th = self.s, self.W, self.H, self.tw, self.th
        leaves = {k: getattr(s, k).clone().requires_grad_(True) for k in ("means", "quats", "scales", "opacities", "sh")}
        t = [time.perf_counter()]
        radii, means2d, depths, conics, _ = oracle.fully_fused_projection(leaves["means"], leaves["quats"], leaves["scales"], s.viewmats, s.Ks, W, H)
        dirs = leaves["means"][None] - oracle.torch_impl.camera_positions(s.viewmats)[:, None, :]
        cols = torch.clamp_min(oracle.spherical_harmonics(3, dirs, leaves["sh"][None], masks=radii > 0) + 0.5, 0.0)
        cols = torch.cat([cols, depths[..., None]], -1)
        opac = leaves["opacities"][None]
        t.append(time.perf_counter())  # 1: project + SH forward
        _, ids, flat = oracle.isect_tiles(means2d, radii, depths, 16, tw, th)
        offs = oracle.isect_offset_encode(ids, 1, tw, th)
        t.append(time.perf_counter())  # 2: intersection
        b = torch.cat([offs.flatten().long(), torch.tensor([flat.numel()])])
        lens = torch.where(self.keep, b[1:] - b[:-1], torch.zeros(1, dtype=torch.long))
        off_sub = (torch.cumsum(lens, 0) - lens).reshape(1, th, tw).to(torch.int32)
        flat_sub = torch.cat([flat[b[i]:b[i + 1]] for i in self.picks]) if self.picks else flat[:0]
        render, alpha, _ = oracle.rasterize_to_pixels(means2d, conics, cols, opac, W, H, 16, off_sub, flat_sub)
        if self.mode == "RGB+ED":
            render = torch.cat([render[..., :3], render[..., 3:] / alpha.clamp(min=1e-10)], -1)
        rgb, d = oracle.composite_and_fill(render, alpha, torch.tensor([0.1, 0.2, 0.3]))
        loss = 0.8 * ((rgb - s.gt_rgb).abs() * self.pix).sum() / (self.pix.sum() * 3) + oracle.depth_l1_loss(d, s.gt_depth, 0.2, mask=self.pix)
        t.append(time.perf_counter())  # 3: composite + loss forward (sampled tiles)
        g = torch.autograd.grad(loss, [means2d, conics, cols, leaves["opacities"]], allow_unused=True)
        t.append(time.perf_counter())  # 4: composite + loss backward (sampled tiles)
        torch.autograd.backward([means2d, conics, cols], [g[0], g[1], g[2]])
        t.append(time.perf_counter())  # 5: project + SH backward
        d_ = [b_ - a_ for a_, b_ in zip(t[:-1], t[1:])]
        whole = d_[0] + d_[1] + d_[4] + (d_[2] + d_[3]) / self.frac
        return whole, sum(d_), float(loss)


def run_cpu_baseline(args, steps: int, warmup: int):
    import torch

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sample = CpuSample(args)
    for _ in range(warmup):
        sample.step()
    whole, spent = [], 0.0
    for _ in range(max(steps, 1)):
        w, t, _ = sample.step()
        whole.append(w)
        spent += t
    whole.sort()
    dt = sum(whole) / len(whole)
    mpix = args.width * args.height / dt / 1e6
    return {"value": mpix, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample.desc, "ms_per_step": dt * 1e3,
            "cpu_seconds_spent": spent, "steps": len(whole)}


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb = run_cpu_baseline(args, steps=max(args.steps, 1), warmup=max(args.warmup, 0))
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": bench_config(args, max(args.gpus, 1)),
        "note": "CPU arm: the oracle port (gsplat's reference rasterizer restated in torch) on the host cores; ms_per_step is the time of one "
                "whole-image step derived from the bounded sample described in cpu_baseline.sample",
        "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# N > 1: the view-sharded step equals the single-rank step (SURVEY.md section 8e "Check"); never inside a timed region
# ------------------------------------------------------------------------------------------------
def run_multi_gpu_check(torch, dist, dev, rank, world, with_exchange=True):
    """1. N ranks x 1 view, gradients summed over the ranks  ==  1 rank x N views (the whole batch in one process).
    2. 3 trainer steps (render, loss, backward, gradient reduction, Adam): every replica holds bit-identical parameters,
       and they equal (to float tolerance: the reduction order differs) a single-process trainer fed all N views."""
    from qed_splatter_b200.pipeline import FusedSplatStep
    from qed_splatter_b200.scenes import scene_s0
    from qed_splatter_b200.trainer import SplatTrainer, TrainConfig

    s = scene_s0(N=20000, C=world, size=160).to(dev)
    bg = torch.tensor([0.2, 0.3, 0.4], device=dev)
    sl = slice(rank, rank + 1)
    mine = dict(viewmats=s.viewmats[sl].contiguous(), Ks=s.Ks[sl].contiguous(), gt_rgb=s.gt_rgb[sl].contiguous(), gt_depth=s.gt_depth[sl].contiguous())
    fs = FusedSplatStep(dev)
    whole = fs.step(s.means, s.quats, s.scales, s.opacities, s.sh, s.viewmats, s.Ks, s.width, s.height, 3, s.gt_rgb, s.gt_depth, bg)
    ref = {k: v.clone() for k, v in whole.grads.items()}
    part = fs.step(s.means, s.quats, s.scales, s.opacities, s.sh, mine["viewmats"], mine["Ks"], s.width, s.height, 3, mine["gt_rgb"],
                   mine["gt_depth"], bg, grad_scale=1.0 / world)
    res = {"scene": f"S0-style: 20000 Gaussians, {world} views 160x160, one view per rank", "gradients": {}}
    ok = True
    for k, v in part.grads.items():
        g = v.clone()
        dist.all_reduce(g)
        d = (g - ref[k]).abs()
        scale = float(ref[k].abs().mean()) + 1e-20
        frac = float((d > 1e-4 * ref[k].abs() + 1e-5 * scale).float().mean())
        res["gradients"][k] = {"max_abs_diff_over_mean_abs": float(d.max()) / scale, "frac_outside_rtol1e-4": frac}
        ok = ok and frac < 1e-3 and float(d.max()) / scale < 1e-2
    # the same through this library's NVLink path (view-colour exchange + all-reduce kernel)
    from qed_splatter_b200.comm import ViewShardedGradients

    if not with_exchange:
        return _multi_gpu_check_trainer(torch, dist, dev, rank, world, s, mine, bg, res, ok, "nccl")
    xg = ViewShardedGradients(s.N, 1, dev)
    res["comm_path"] = xg.arena.path
    for rep in range(2):  # twice: both exchange buffers, stale records of the previous step present
        fs.step(s.means, s.quats, s.scales, s.opacities, s.sh, mine["viewmats"], mine["Ks"], s.width, s.height, 3, mine["gt_rgb"],
                mine["gt_depth"], bg, grad_scale=1.0 / world, exchange=xg)
    res["gradients_exchange"] = {}
    for k, g in xg.views().items():
        d = (g - ref[k]).abs()
        scale = float(ref[k].abs().mean()) + 1e-20
        frac = float((d > 1e-4 * ref[k].abs() + 1e-5 * scale).float().mean())
        res["gradients_exchange"][k] = {"max_abs_diff_over_mean_abs": float(d.max()) / scale, "frac_outside_rtol1e-4": frac}
        ok = ok and frac < 1e-3 and float(d.max()) / scale < 1e-2
    chk = torch.stack([xg.grad.double().sum(), xg.grad.view(torch.int32).sum().double()])
    allc = [torch.empty_like(chk) for _ in range(world)]
    dist.all_gather(allc, chk)
    res["exchange_arena_bit_identical_on_all_ranks"] = all(torch.equal(allc[0], c_) for c_ in allc)
    ok = ok and res["exchange_arena_bit_identical_on_all_ranks"]
    return _multi_gpu_check_trainer(torch, dist, dev, rank, world, s, mine, bg, res, ok, "auto")


def _multi_gpu_check_trainer(torch, dist, dev, rank, world, s, mine, bg, res, ok, comm):
    from qed_splatter_b200.trainer import SplatTrainer, TrainConfig

    identical, vs_single = True, None
    log_s, logit_o = torch.log(s.scales), torch.logit(s.opacities)
    tr = SplatTrainer(s.means.clone(), s.quats.clone(), log_s.clone(), logit_o.clone(), s.sh.clone(), cfg=TrainConfig(comm=comm), rank=rank, world_size=world, backend="cuda")
    tr.step_count = 3000
    for _ in range(3):
        tr.step(mine["viewmats"], mine["Ks"], s.width, s.height, mine["gt_rgb"], mine["gt_depth"], bg, total_views=world)
    gathered = [torch.empty_like(tr.arena.param) for _ in range(world)]
    dist.all_gather(gathered, tr.arena.param)
    for r in range(1, world):
        identical = identical and torch.equal(gathered[0], gathered[r])
    single = SplatTrainer(s.means.clone(), s.quats.clone(), log_s.clone(), logit_o.clone(), s.sh.clone(), cfg=TrainConfig(), rank=0, world_size=1, backend="cuda")
    single.step_count = 3000
    for _ in range(3):
        single.step(s.viewmats, s.Ks, s.width, s.height, s.gt_rgb, s.gt_depth, bg, total_views=world)
    d = (single.arena.param - tr.arena.param).abs()
    upd = (single.arena.param - torch.cat([t.reshape(-1) for t in (s.means, s.quats, log_s, logit_o, s.sh)])[:single.arena.param.numel()]).abs() \
        if single.arena.param.numel() == sum(t.numel() for t in (s.means, s.quats, log_s, logit_o, s.sh)) else None
    vs_single = {"max_abs_param_diff": float(d.max()), "frac_above_1e-5": float((d > 1e-5).float().mean()),
                 "mean_abs_update": float(upd.mean()) if upd is not None else None}
    ok = ok and identical and vs_single["frac_above_1e-5"] < 1e-2
    res["trainer_comm"] = tr.comm
    res.update({"replicas_bit_identical_after_3_steps": bool(identical), "vs_single_process_trainer": vs_single, "ok": bool(ok), "world": world})
    flag = torch.tensor([1.0 if ok else 0.0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    res["ok_all_ranks"] = bool(flag.item() > 0)
    return res


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def main_ours(args):
    import torch
    import torch.distributed as dist

    from qed_splatter_b200 import _lib, depth_supervised_loss, ops, rasterization
    from qed_splatter_b200.pipeline import FusedSplatStep
    from qed_splatter_b200.scenes import scene_s1

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    if args.radix_onesweep is not None:
        lib.qed_debug_set_radix_onesweep(args.radix_onesweep)
    K, W_ = args.steps, max(args.warmup, 3)
    width, height, N = args.width, args.height, args.gaussians

    # replicated Gaussians (same seed everywhere), one view per rank
    scene = scene_s1(N=N, width=width, height=height, C=max(world, 1))
    sl = slice(rank, rank + 1)
    means, quats, scales, opac, sh = (t.to(dev) for t in (scene.means, scene.quats, scene.scales, scene.opacities, scene.sh))
    viewmats, Ks = scene.viewmats[sl].contiguous().to(dev), scene.Ks[sl].contiguous().to(dev)
    gt_rgb_h = scene.gt_rgb[sl].contiguous().pin_memory()
    gt_depth_h = scene.gt_depth[sl].contiguous().pin_memory()
    vm_h, K_h = scene.viewmats[sl].contiguous().pin_memory(), scene.Ks[sl].contiguous().pin_memory()
    gt_rgb, gt_depth = gt_rgb_h.to(dev), gt_depth_h.to(dev)
    bg = torch.tensor([0.1, 0.2, 0.3], device=dev)
    del scene

    fs = FusedSplatStep(dev, sort_impl=args.sort)
    arena = torch.zeros(PARAM_FLOATS * N, device=dev)  # flat gradient arena: one all-reduce
    o = 0
    views = {}
    for name, shape in (("means", (N, 3)), ("quats", (N, 4)), ("scales", (N, 3)), ("opacities", (N,)), ("sh", (N, 16, 3))):
        n = 1
        for s_ in shape:
            n *= s_
        views[name] = arena[o:o + n].view(*shape)
        o += n
    stats = torch.zeros(3, N, device=dev)  # grad2d, count, radii_max (DefaultStrategy state)

    n_chunks = args.comm_chunks if world > 1 else 1
    sh_begin = 11 * N  # arena = [means 3N | quats 4N | scales 3N | opacities N | sh 48N]
    pending = []

    def on_chunk(k, n0, n1):
        # the SH block is 81 % of the gradient bytes: reduce each finished Gaussian range while the projection
        # backward of the next range is still running (NCCL runs on its own stream)
        pending.append(dist.all_reduce(arena[sh_begin + 48 * n0: sh_begin + 48 * n1], async_op=True))

    xg, comm_fallback = None, None
    if world > 1 and args.comm == "exchange":
        from qed_splatter_b200.comm import ViewShardedGradients

        try:  # symmetric memory (peer mappings / NVSwitch multicast) must be available on this box -- on every rank
            xg = ViewShardedGradients(N, 1, dev)
        except Exception as e:  # noqa: BLE001
            comm_fallback = f"{type(e).__name__}: {e}"[:300]
        ok_all = torch.tensor([0.0 if xg is None else 1.0], device=dev)
        dist.all_reduce(ok_all, op=dist.ReduceOp.MIN)
        if float(ok_all.item()) < 1.0:
            xg, comm_fallback = None, comm_fallback or "symmetric memory unavailable on another rank"
        else:
            del arena
            arena, views = xg.grad, xg.views()

    def step():
        if xg is not None:
            # the step ends (in stream order) with the gradient arena summed over all ranks on every rank: per-view colour
            # gradients exchanged by the projection backward, one all-reduce kernel, local rebuild of the SH gradient
            out = fs.step(means, quats, scales, opac, sh, viewmats, Ks, width, height, 3, gt_rgb, gt_depth, bg, render_mode=args.mode,
                          grad_scale=1.0 / world, exchange=xg)
            _lib.check(lib.qed_strategy_update(1, N, _lib.ptr(out.packed_grads), 1, _lib.ptr(out.radii), width, height, world, _lib.ptr(stats[0]),
                                               _lib.ptr(stats[1]), _lib.ptr(stats[2]), _lib.current_stream()), "qed_strategy_update")
            return out
        out = fs.step(means, quats, scales, opac, sh, viewmats, Ks, width, height, 3, gt_rgb, gt_depth, bg, render_mode=args.mode,
                      grad_scale=1.0 / world, grad_out=views, n_chunks=n_chunks, on_chunk=on_chunk if world > 1 else None)
        _lib.check(lib.qed_strategy_update(1, N, _lib.ptr(out.packed_grads), 1, _lib.ptr(out.radii), width, height, world, _lib.ptr(stats[0]),
                                           _lib.ptr(stats[1]), _lib.ptr(stats[2]), _lib.current_stream()), "qed_strategy_update")
        if world > 1:
            # gradients every step (SH ranges already in flight, then the 11 small floats per Gaussian); the
            # densification accumulators are reduced only when a refine step consumes them (SUM / MAX are
            # associative), exactly as trainer.SplatTrainer does
            pending.append(dist.all_reduce(arena[:sh_begin], async_op=True))
            for w in pending:
                w.wait()
            pending.clear()
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_window(fn, steps):
        """`steps` calls of fn bracketed by barrier + synchronize on both sides, device-timed, max over ranks -> ms."""
        barrier()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        t_ = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t_, op=dist.ReduceOp.MAX)
        return float(t_.item())

    def pct(v, q):
        v = sorted(v)
        return v[min(len(v) - 1, max(0, int(round(q * (len(v) - 1)))))]

    def spread(windows_ms, steps):
        per = [w / steps for w in windows_ms]
        return {"windows": len(per), "steps_per_window": steps, "ms_per_step_median": pct(per, 0.5), "ms_per_step_p10": pct(per, 0.1),
                "ms_per_step_p90": pct(per, 0.9), "ms_per_step_min": min(per), "ms_per_step_max": max(per)}

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(W_):
        out = step()
    barrier()
    last = {}

    def measured_step():
        last["out"] = step()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # THE measurement (contract): exactly K steps, one window
    ms_total = timed_window(measured_step, K)
    dumped = collect_outputs(last["out"], stats) if args.dump_outputs and rank == 0 else None
    ms_per_step = ms_total / K
    value = world * width * height / (ms_per_step * 1e-3) / 1e6
    # R more windows of K steps: run-to-run spread (median / p10 / p90), and enough wall time for >= 10 clock samples
    windows = [ms_total] + [timed_window(step, K) for _ in range(args.repeats)]
    clocks = sampler.stop() if rank == 0 else None
    repeats = spread(windows, K)

    # ---- stage timing (same inputs, CUDA events between the stages on the launching stream) ----
    stage_ms = {}
    for _ in range(K):
        fs.marks = []
        out = step()
        torch.cuda.synchronize()
        m = fs.marks
        for (_, a), (name, b) in zip(m[:-1], m[1:]):
            stage_ms[name] = stage_ms.get(name, 0.0) + a.elapsed_time(b) / K
    fs.marks = None
    n_visible = int((out.radii > 0).sum())
    M = int(fs._buf["tiles"][:N].sum())  # gsplat's bounding-box intersection count (one local view)
    n_exact = fs.n_isects_exact()        # entries of the exact tile lists the step actually builds, sorts and composites
    loss = [float(x) for x in out.loss.tolist()]

    # ---- pair counters for the compositing roofline (instrumented launches, outside any timed region) ----
    counters = fs.count_pairs()
    launches_per_step = fs.launches_per_step + ((n_chunks - 1) if (world > 1 and xg is None) else 0)  # this library's kernels only (chunked: extra project_bwd launches)
    if xg is not None:
        launches_per_step += 2  # + the all-reduce kernel and the SH-gradient rebuild
    comm_info = None
    if world > 1:
        comm_info = {"impl": "exchange" if xg is not None else "nccl", "path": xg.arena.path if xg is not None else "torch.distributed all_reduce",
                     "bytes_all_reduced_per_rank": (xg.offsets["sh"][0] * 4) if xg is not None else PARAM_FLOATS * N * 4,
                     "bytes_exchanged_per_rank": (n_visible * 16) if xg is not None else 0, "fallback_reason": comm_fallback}

    # ---- second half of the metric: train iters/s (full qed-splatter step through trainer.SplatTrainer: render,
    # 0.8 L1 + 0.2 (1-SSIM) + 0.2 depth-L1, backward, gradient all-reduce pipelined with Adam, strategy statistics) ----
    train = None
    if not args.no_train:
        from qed_splatter_b200.trainer import SplatTrainer, TrainConfig

        tcfg = TrainConfig(render_mode="RGB+D" if args.mode == "RGB+D" else "RGB+ED", refine_every=10 ** 9)
        tr = SplatTrainer(means.clone(), quats.clone(), torch.log(scales), torch.logit(opac.clamp(1e-4, 1 - 1e-4)), sh.clone(), cfg=tcfg,
                          rank=rank, world_size=world, backend="cuda")
        tr.step_count = 3000  # SH degree 3, no opacity reset inside the timed window
        for _ in range(W_):
            tr.step(viewmats, Ks, width, height, gt_rgb, gt_depth, bg, total_views=world)
        tw_ = [timed_window(lambda: tr.step(viewmats, Ks, width, height, gt_rgb, gt_depth, bg, total_views=world), K) for _ in range(1 + min(args.repeats, 2))]
        tms = tw_[0] / K
        train = {"train_iters_per_s": 1e3 / tms, "repeats": spread(tw_, K), "ms_per_step": tms, "views_per_s": world * 1e3 / tms,
                 "loss": "0.8 L1 + 0.2 (1-SSIM) + 0.2 depth-L1", "optimizer": "fused Adam over the 59-float/Gaussian arena",
                 "comm_chunks": tcfg.comm_chunks if world > 1 else 1}
        del tr
        torch.cuda.empty_cache()

    # ---- e2e through the public API with host buffers ----
    e2e = e2e_fused_loss = None
    if not args.no_e2e:
        params = [t.clone().requires_grad_(True) for t in (means, quats, scales, opac, sh)]
        # N > 1: the five parameter gradients are reduced as ONE coalesced NCCL group call (what DDP / FSDP do), no
        # flattening copies; `--e2e-bucket` uses a flat bucket of gradient views (gradient_as_bucket_view) instead
        grad_bucket, grad_views = None, None
        if world > 1 and args.e2e_bucket:
            grad_bucket = torch.zeros(sum(p_.numel() for p_ in params), device=dev)
            grad_views, o_ = [], 0
            for p_ in params:
                grad_views.append(grad_bucket[o_:o_ + p_.numel()].view_as(p_))
                o_ += p_.numel()
        # the step's inputs come from pinned host memory on a copy stream (what a data loader does): the camera first (the
        # render needs it), the ground truth once the render is launched; the loss waits on the copy event, so the H2D of the
        # ground truth overlaps projection/sort/compositing
        copy_stream = torch.cuda.Stream()
        vm_d, K_d = torch.empty_like(viewmats), torch.empty_like(Ks)
        # ground-truth RGB travels as the reference's data side holds it: the uint8 image cache (config.py:37
        # cache_images_type="uint8"); depth_supervised_loss converts it in-kernel (--torch-loss: torch .float() / 255)
        e2e_rgb_h = gt_rgb_h if args.gt_float else (gt_rgb_h * 255.0).round().clamp(0, 255).to(torch.uint8).contiguous().pin_memory()
        rgb_d, depth_d = torch.empty(e2e_rgb_h.shape, dtype=e2e_rgb_h.dtype, device=dev), torch.empty_like(gt_depth)
        cam_ready, gt_ready = torch.cuda.Event(), torch.cuda.Event()

        def e2e_step(reference_lines: bool):
            copy_stream.wait_stream(torch.cuda.current_stream())  # previous step is done with the buffers
            with torch.cuda.stream(copy_stream):
                vm_d.copy_(vm_h, non_blocking=True)
                K_d.copy_(K_h, non_blocking=True)
                cam_ready.record(copy_stream)
            torch.cuda.current_stream().wait_event(cam_ready)
            vm, Kc, rgb_gt, d_gt = vm_d, K_d, rgb_d, depth_d
            if grad_bucket is None:
                for p_ in params:
                    p_.grad = None
            else:
                grad_bucket.zero_()
                for p_, g_ in zip(params, grad_views):
                    p_.grad = g_  # autograd accumulates in place
            render, alpha, info = rasterization(params[0], params[1], params[2], params[3], params[4], vm, Kc, width, height,
                                                tile_size=16, packed=False, near_plane=0.01, far_plane=1e10, render_mode=args.mode,
                                                sh_degree=3, sparse_grad=False, absgrad=True, rasterize_mode="classic")
            info["means2d"].retain_grad()
            # the ground truth is only needed by the loss: its copies are queued (copy stream) once the render is launched and
            # run under the projection / intersection / compositing kernels
            with torch.cuda.stream(copy_stream):
                rgb_d.copy_(e2e_rgb_h, non_blocking=True)
                depth_d.copy_(gt_depth_h, non_blocking=True)
                gt_ready.record(copy_stream)
            torch.cuda.current_stream().wait_event(gt_ready)
            if reference_lines:
                rgb_gt = rgb_gt.float() / 255.0 if rgb_gt.dtype == torch.uint8 else rgb_gt  # splatfacto get_gt_img
                # qed_splatter/model.py:295-297, 304-306 as written
                rgb = render[:, ..., :3] + (1 - alpha) * bg
                rgb = torch.clamp(rgb, 0.0, 1.0)
                depth_im = render[:, ..., 3:4]
                depth_im = torch.where(alpha > 0, depth_im, depth_im.detach().max())
                # qed_splatter/model.py:101-116 as written (boolean-index gathers and the numel() test included)
                valid_mask = torch.isfinite(depth_im) & torch.isfinite(d_gt) & (d_gt > 0.0)
                valid_depth_out = depth_im[valid_mask]
                valid_depth_batch = d_gt[valid_mask]
                if valid_depth_out.numel() > 0:
                    l_d = torch.abs(valid_depth_out - valid_depth_batch).mean()
                else:
                    l_d = torch.tensor(0.0, device=depth_im.device)
                l_rgb = 0.8 * torch.abs(rgb_gt - rgb).mean()  # the L1 line of splatfacto's parent loss (model.py:83-85)
                loss_t = (l_rgb + 0.2 * l_d) / world
            else:
                # the same lines through the package's drop-in for them (losses.depth_supervised_loss)
                loss_t = depth_supervised_loss(render, alpha, rgb_gt, d_gt, bg, rgb_weight=0.8, depth_lambda=0.2)[0] / world
            loss_t.backward()
            if world > 1:
                if grad_bucket is not None:
                    dist.all_reduce(grad_bucket)
                else:
                    with dist._coalescing_manager(device=dev):
                        for p_ in params:
                            dist.all_reduce(p_.grad)
            return float(loss_t.item())  # D2H read of the step's result

        h2d = vm_h.numel() * 4 + K_h.numel() * 4 + e2e_rgb_h.numel() * e2e_rgb_h.element_size() + gt_depth_h.numel() * 4
        last = {}

        def run_e2e(reference_lines: bool):
            def one():
                last["loss"] = e2e_step(reference_lines)

            for _ in range(W_):
                one()
            wins = [timed_window(one, K) for _ in range(1 + min(args.repeats, 2))]
            ms_ = wins[0] / K
            return {"value": world * width * height / (ms_ * 1e-3) / 1e6, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_, "loss": last["loss"], "repeats": spread(wins, K),
                    "api": "qed_splatter_b200.rasterization (gsplat surface) + " +
                           ("the reference's own loss lines in torch (qed_splatter/model.py:295-306, 101-116 + splatfacto's L1 line)"
                            if reference_lines else "qed_splatter_b200.depth_supervised_loss (model.py:295-306, 73-118 as one autograd op)") +
                           " + backward(); inputs from pinned host memory, loss read back, every step"}

        e2e = run_e2e(True)               # headline: the model's own lines on top of the drop-in call
        e2e_fused_loss = run_e2e(False)   # with the package's fused drop-in for those lines
        del params
        torch.cuda.empty_cache()

    # ---- N > 1: N ranks x 1 view == 1 rank x N views, replicas identical (outside every timed region) ----
    multi_gpu_check = None
    if world > 1 and not args.no_multi_gpu_check:
        multi_gpu_check = run_multi_gpu_check(torch, dist, dev, rank, world, with_exchange=xg is not None)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        hbm_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
        traffic, traffic_workload = load_ncu_traffic()
        if traffic_workload is not None and traffic_workload != workload_name(args):
            traffic = {}  # the capture belongs to another workload
        fp32_peak = 148 * 128 * 2 * sm_mhz * 1e6 / 1e12  # TFLOP/s at the SM clock seen during the timed region

        def fp32_roof(name, pairs, evaluated, flop_per_pair):
            # algorithmic work = (pixel, Gaussian) pairs that pass the alpha test and are composited / differentiated:
            # independent of how well an implementation culls; pairs_evaluated (>= pairs) is what this one touched
            t_ms = stage_ms.get(name)
            if not t_ms or not pairs:
                return None
            ach = pairs * flop_per_pair / (t_ms * 1e-3) / 1e12
            return {"kernel": name, "bound": "fp32", "achieved": ach, "peak": fp32_peak, "unit": "TFLOP/s", "frac": ach / fp32_peak,
                    "traffic": traffic.get(name), "ms": t_ms, "pairs_composited": pairs, "pairs_evaluated": evaluated,
                    "flop_per_pair": flop_per_pair,
                    "peak_source": f"derived: 148 SM x 128 lanes x 2 FLOP x {sm_mhz:.0f} MHz (median SM clock sampled during the timed region)"}

        def hbm_roof(name, bytes_):
            t_ms = stage_ms.get(name)
            if not t_ms:
                return None
            ach = bytes_ / (t_ms * 1e-3) / 1e9
            tr_ = traffic.get(name)
            return {"kernel": name, "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                    "traffic": tr_, "traffic_over_algorithmic": (tr_ / bytes_) if tr_ else None, "ms": t_ms, "algorithmic_bytes": bytes_,
                    "peak_source": hbm_src}

        tile_bits = (((width + 15) // 16) * ((height + 15) // 16)).bit_length()
        tile_passes = (tile_bits + 7) // 8
        # two-level intersection build (DESIGN.md §5): algorithmic bytes
        #   prepare: flags scan (4 r + 8 w + 8 r per (c,n)), compaction (8 w), 4 radix passes over the visible entries
        #            (4 r upsweep + 8 r + 8 w downsweep each), gather scan (4 + 4 r, 8 w)
        #   fill   : emit 8 w per isect, tile_passes radix passes (20 B each), ranges pass (4 r key + 4 r flat)
        bytes_prepare = N * 20.0 + n_visible * (8.0 + 4 * 20.0 + 16.0)
        bytes_fill = M * (8.0 + tile_passes * 20.0 + 8.0)
        stages = [
            fp32_roof("raster_bwd", counters.get("bwd_pairs_contributing"), counters.get("bwd_pairs_evaluated"), FLOP_PER_PAIR_BWD),
            fp32_roof("raster_fwd", counters.get("fwd_pairs_contributing"), counters.get("fwd_pairs_evaluated"), FLOP_PER_PAIR_FWD),
            hbm_roof("project_fwd", N * BYTES_PROJ_FWD_PER_GAUSS + n_visible * BYTES_PROJ_FWD_PER_VISIBLE),
            hbm_roof("project_bwd", N * BYTES_PROJ_BWD_PER_GAUSS + n_visible * BYTES_PROJ_BWD_PER_VISIBLE),
            hbm_roof("isect_prepare", bytes_prepare),
            hbm_roof("isect_fill", bytes_fill),
            hbm_roof("loss", width * height * (24.0 + 68.0)),
            # the reference formulation (gsplat: 64-bit keys, full radix sort), only present with --sort own|cub
            hbm_roof("sort", M * (((32 + tile_bits + 1 + 7) // 8) * 24.0 + 8.0)),
            hbm_roof("emit", M * 12.0),
        ]
        stages = [s for s in stages if s]
        dominant = max(stages, key=lambda s: s["ms"]) if stages else None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W_, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": bench_config(args, world),
            "workload_stats": {"n_visible": n_visible, "n_isects": M, "n_isects_exact": n_exact, "loss": loss,
                               "mean_gaussians_composited_per_pixel": counters.get("fwd_pairs_contributing", 0) / float(width * height),
                               "intermediates_mb_per_step": (N * 150 + M * 24) / 1e6},
            "repeats": repeats,
            "clocks": clocks,
            "e2e": e2e,
            "e2e_fused_loss": e2e_fused_loss,
            "train": train,
            "multi_gpu_check": multi_gpu_check,
            "comm": comm_info,
            "traffic_source": "profiles/r02_dram_bytes.json (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum, per step and stage)" if traffic else None,
            "gpu_launches": launches_per_step * K,
            "gpu_launches_per_step": launches_per_step,
            "roofline": dominant,
            "stages": stages,
            "stage_ms": stage_ms,
            "pair_counters": counters,
        }
        if world == 1 and not args.no_cpu_baseline:
            cb = run_cpu_baseline(args, steps=8, warmup=1)  # ~15 s of CPU work; the same sample and code as `--impl reference`
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "cpu_seconds_spent", "steps")}
        else:
            line["cpu_baseline"] = None
        if dumped is not None:
            write_outputs(args.dump_outputs, dumped)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        main_reference(a)
    else:
        main_ours(a)
