"""-m gpu: the bilateral grid in FusedSplatStep and SplatTrainer -- a frozen grid trains like the trainer without it, the
grids recover a per-camera colour change with the Gaussians frozen, and the exchange path (symmetric row buffer, its
all-reduce, the rebuild when the views per rank change) matches the plain trainer."""
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import bilagrid_oracle as bo
from helpers import scene_args
from qed_splatter_b200 import depth_supervised_loss, rasterization
from qed_splatter_b200.pipeline import FusedSplatStep
from qed_splatter_b200.scenes import scene_s0
from qed_splatter_b200.trainer import GROUPS, SplatTrainer, TrainConfig

pytestmark = pytest.mark.gpu
FROZEN = dict(lr_means=1e-30, lr_means_final=1e-30, lr_quats=0.0, lr_scales=0.0, lr_opacities=0.0, lr_features_dc=0.0, lr_features_rest=0.0)


def _gaussian_args(s, dev):
    return (s.means.to(dev), s.quats.to(dev), torch.log(s.scales).to(dev), torch.logit(s.opacities).to(dev), s.sh.to(dev))


@pytest.mark.parametrize("n_chunks", [1, 3])
def test_fused_step_grid_rows_match_depth_supervised_loss(cuda, n_chunks):
    """The grid in the fused step's loss stage gives the loss and grid rows of depth_supervised_loss on the same render."""
    s = scene_s0(N=3000, C=2, size=96).to(cuda)
    bg = torch.tensor([0.3, 0.1, 0.6], device=cuda)
    grids = (bo.identity_grids(3) + 0.1 * torch.randn(3, 12, 8, 16, 16, generator=torch.Generator().manual_seed(2))).to(cuda)
    ids = torch.tensor([2, 2], dtype=torch.int32, device=cuda)
    rows = torch.empty(2, 12, 8, 16, 16, device=cuda)
    fs = FusedSplatStep(cuda)
    out = fs.step(s.means, s.quats, s.scales, s.opacities, s.sh, s.viewmats, s.Ks, s.width, s.height, 3, s.gt_rgb, s.gt_depth, bg,
                  render_mode="RGB+D", ssim_lambda=0.2, n_chunks=n_chunks, bilateral_grid=(grids, ids, rows))
    g = grids.clone().requires_grad_(True)
    tot, _, _ = depth_supervised_loss(out.render.clone(), out.alphas.clone(), s.gt_rgb, s.gt_depth, bg, ssim_lambda=0.2, bilateral_grids=g,
                                      grid_ids=ids)
    tot.backward()
    assert float(out.loss[0]) == pytest.approx(float(tot), rel=1e-6)
    assert torch.equal(rows[0] + rows[1], g.grad[2]) and float(g.grad[:2].abs().max()) == 0.0


def test_frozen_grid_trains_like_grid_off(cuda):
    """Grid on with lr 0: identity grids, so the loss and Gaussian gradients equal the grid-off trainer's within the
    tolerance of the camera optimizer's frozen-table test (1e-6 of the largest value: the compositor's backward and the loss
    statistics use atomics; trilinear weights need not sum to exactly 1)."""
    s = scene_s0(N=6000, C=2, size=96)
    bg = torch.tensor([0.3, 0.3, 0.3], device=cuda)
    t = s.to(cuda)
    base = dict(stop_split_at=0, sh_degree_interval=1, ssim_lambda=0.2)
    off = SplatTrainer(*_gaussian_args(s, cuda), cfg=TrainConfig(**base))
    on = SplatTrainer(*_gaussian_args(s, cuda), cfg=TrainConfig(use_bilateral_grid=True, bilateral_grid_lr=0.0, **base), num_cameras=3)
    ids = torch.tensor([2, 0])
    for it in range(3):
        l_off, _ = off.step(t.viewmats, t.Ks, t.width, t.height, t.gt_rgb, t.gt_depth, bg)
        l_on, _ = on.step(t.viewmats, t.Ks, t.width, t.height, t.gt_rgb, t.gt_depth, bg, camera_ids=ids)
        if it == 0:  # identical parameters: identical renders, equal losses and gradients
            assert torch.equal(on._fused._fwd["render"].view(torch.int32), off._fused._fwd["render"].view(torch.int32))
            assert torch.allclose(l_on, l_off, rtol=1e-6, atol=1e-7)
            for g in GROUPS:
                a, b = off.arena.view(off.arena.grad, g), on.arena.view(on.arena.grad, g)
                assert float((a - b).abs().max()) <= 1e-6 * float(a.abs().max()), g
    assert torch.equal(on.bilateral_grids, bo.identity_grids(3).to(cuda)) and float(on.bilagrid.grad.abs().max()) > 0
    assert float(on.bilagrid_tv_loss) == 0.0
    with pytest.raises(ValueError, match="camera_ids"):
        on.step(t.viewmats, t.Ks, t.width, t.height, t.gt_rgb, t.gt_depth, bg)
    with pytest.raises(ValueError, match="camera_ids"):
        on.step(t.viewmats, t.Ks, t.width, t.height, t.gt_rgb, t.gt_depth, bg, camera_ids=torch.tensor([3, 0]))
    with pytest.raises(ValueError):  # both features off: camera_ids is still refused
        off.step(t.viewmats, t.Ks, t.width, t.height, t.gt_rgb, t.gt_depth, bg, camera_ids=ids)


def test_trainer_recovers_a_per_camera_colour_change(cuda):
    """Ground truth rendered by the library, then a known affine colour change per camera (gains 0.8-1.2, offsets +-0.05).
    SplatTrainer with the grid on and the Gaussians' learning rates at 0 trains the grids with their own Adam group (lr 2e-3,
    no warm-up).  The RGB L1 has to fall by a large factor; on a B200 it went from L1_FIRST to L1_LAST in 400 steps."""
    C, size = 4, 128
    s = scene_s0(N=4000, C=C, size=size)
    t = s.to(cuda)
    bg = torch.zeros(3, device=cuda)
    with torch.no_grad():
        render, alpha, _ = rasterization(**scene_args(s, cuda), width=size, height=size, sh_degree=3, render_mode="RGB+ED")
        clean = torch.clamp(render[..., :3] + (1 - alpha) * bg, 0, 1)
        gen = torch.Generator().manual_seed(11)
        gain = (0.8 + 0.4 * torch.rand(C, 1, 1, 3, generator=gen)).to(cuda)
        off = (0.1 * torch.rand(C, 1, 1, 3, generator=gen) - 0.05).to(cuda)
        gt_rgb = (clean * gain + off).contiguous()
    cfg = TrainConfig(use_bilateral_grid=True, bilateral_grid_warmup=0, bilateral_grid_lr_final=2e-3, depth_lambda=0.0, ssim_lambda=0.0,
                      stop_split_at=0, sh_degree_interval=1, render_mode="RGB+ED", **FROZEN)
    tr = SplatTrainer(*_gaussian_args(s, cuda), cfg=cfg, num_cameras=C)
    ids = torch.arange(C)
    l1 = []
    for _ in range(400):
        loss, _ = tr.step(t.viewmats, t.Ks, size, size, gt_rgb, t.gt_depth, bg, camera_ids=ids)
        l1.append(float(loss[1]))
    print("bilagrid recovery", dict(l1_first=l1[0], l1_last=l1[-1]))
    assert l1[-1] < l1[0] / 4, (l1[0], l1[-1])


def _exchange_worker(rank, port, out):
    """One process, an NCCL group of one: a trainer forced onto the exchange path next to the plain single-GPU trainer."""
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=dev)
    res = {}
    try:
        s = scene_s0(N=6000, C=2, size=96)
        cfg = dict(stop_split_at=0, use_bilateral_grid=True, bilateral_grid_warmup=0, bilateral_grid_lr=1e-2, **FROZEN)
        xt = SplatTrainer(*_gaussian_args(s, dev), cfg=TrainConfig(comm="exchange", **cfg), num_cameras=4)
        xt.comm = "exchange"  # world 1 picks no collective; one rank runs the multi-GPU code path unchanged
        ref = SplatTrainer(*_gaussian_args(s, dev), cfg=TrainConfig(**cfg), num_cameras=4)
        bg = torch.tensor([0.2, 0.5, 0.8], device=dev)
        t = s.to(dev)
        ids = torch.tensor([3, 1])
        res.update(grad_err=[], grad_scale=[], exchanges=[])
        for v in (slice(0, 1), slice(0, 1), slice(0, 2), slice(0, 2)):  # 1 -> 2 views per rank: new symmetric buffers
            for tr in (xt, ref):
                tr.step(t.viewmats[v], t.Ks[v], s.width, s.height, t.gt_rgb[v], t.gt_depth[v], bg, camera_ids=ids[v])
            res["grad_err"].append(float((xt.bilagrid.grad - ref.bilagrid.grad).abs().max()))
            res["grad_scale"].append(float(ref.bilagrid.grad.abs().max()))
            res["exchanges"].append(id(xt._xg))
        res["comm"] = xt.comm
        res["grid_err"] = float((xt.bilateral_grids - ref.bilateral_grids).abs().max())
        res["grid_moved"] = float((ref.bilateral_grids - bo.identity_grids(4).to(dev)).abs().max())
        res["tv"] = [float(xt.bilagrid_tv_loss), float(ref.bilagrid_tv_loss)]
    except RuntimeError as e:  # no symmetric memory on this machine
        res["error"] = str(e)
    torch.save(res, out)
    dist.destroy_process_group()


def test_trainer_exchange_path_on_one_gpu(cuda, tmp_path):
    out = str(tmp_path / "xchg.pt")
    mp.spawn(_exchange_worker, args=(29500 + (os.getpid() + 17) % 2000, out), nprocs=1, join=True)
    r = torch.load(out)
    if "error" in r and "symmetric memory" in r["error"]:
        pytest.skip(r["error"])
    assert "error" not in r, r
    assert r["comm"] == "exchange", r
    assert r["exchanges"][0] == r["exchanges"][1] != r["exchanges"][2] == r["exchanges"][3], r  # rebuilt once
    for err, scale in zip(r["grad_err"], r["grad_scale"]):
        assert scale > 0 and err <= 1e-4 * scale, r
    assert r["grid_moved"] > 0 and r["grid_err"] <= 1e-3 * r["grid_moved"], r
    assert r["tv"][0] == pytest.approx(r["tv"][1], rel=1e-4) and r["tv"][0] > 0
