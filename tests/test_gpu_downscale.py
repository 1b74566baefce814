"""-m gpu: splatfacto's resolution schedule -- the ground-truth pass (qed_downscale_ground_truth) against its oracle and
torch's conv2d, depth_supervised_loss(gt_downscale=) against the same loss on the oracle's ground truth and against the
oracle's reference step at down=2, FusedSplatStep across resolution changes, and SplatTrainer(num_downscales=...) against a
twin trainer fed the rescaled camera and the downscaled ground truth by hand (one GPU, and the exchange path)."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn.functional as F

import downscale_oracle as do
import reference_model as rm
from helpers import assert_close_frac
from qed_splatter_b200 import _lib, depth_supervised_loss, rasterization
from qed_splatter_b200.data_side import downscale_ground_truth
from qed_splatter_b200.pipeline import FusedSplatStep
from qed_splatter_b200.scenes import scene_s0
from qed_splatter_b200.trainer import GROUPS, SplatTrainer, TrainConfig, rescaled_camera

pytestmark = pytest.mark.gpu
COMBOS = [("u8", "u16", "bool"), ("u8", "u16", None), ("f32", "f32", "u8"), ("u8", "f32", "f32"), ("f32", "u16", "bool")]


def _cached_gt(s, seed=5):
    """The scene's ground truth as nerfstudio caches it: uint8 image, raw uint16 depth (mm), bool mask, full resolution."""
    rgb = (s.gt_rgb * 255).round().to(torch.uint8)
    dep = torch.from_numpy((s.gt_depth[..., 0].numpy() * 1000).round().astype(np.uint16))
    mask = torch.rand(s.gt_rgb.shape[:3], generator=torch.Generator().manual_seed(seed)) > 0.2
    return rgb, dep, mask


@pytest.mark.parametrize("d", [2, 4])
@pytest.mark.parametrize("C,W,H", [(1, 1920, 1080), (3, 1920, 1080), (3, 250, 190)])
@pytest.mark.parametrize("combo", COMBOS)
def test_kernel_is_the_oracle_bit_for_bit(cuda, d, C, W, H, combo):
    gt_rgb, gt_depth, mask = do.make_inputs(C, H, W, *combo, seed=C + d)
    want = do.downscale_ground_truth(gt_rgb, gt_depth, mask, d)
    got = downscale_ground_truth(gt_rgb.to(cuda), gt_depth.to(cuda), None if mask is None else mask.to(cuda), d)
    assert got[0].shape == (C, H // d, W // d, 3) and got[1].shape == (C, H // d, W // d, 1)
    for g, w in zip(got, want):
        if w is None:
            assert g is None
            continue
        g = g.cpu()
        nan = torch.isnan(w)
        # NaN at the same places (the device writes its canonical NaN, the CPU keeps the input's payload), all else bit for bit
        assert torch.equal(torch.isnan(g), nan) and torch.equal(g[~nan].view(torch.int32), w[~nan].view(torch.int32))


@pytest.mark.parametrize("d", [2, 4, 8])
def test_kernel_against_torch_cuda_conv2d(cuda, d):
    """torch's CUDA conv2d (TF32 off: with it on, the reference's own values are TF32-rounded) on the same float image,
    and torch's CUDA `image.float() / 255.0` (splatfacto get_gt_img) bit for bit at factor 1."""
    gt_rgb, gt_depth, mask = do.make_inputs(2, 1080, 1920, "u8", "u16", "bool", seed=d)
    rgb, dep, mk = gt_rgb.to(cuda), gt_depth.to(cuda), mask.to(cuda)
    got = downscale_ground_truth(rgb, dep, mk, d)
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        w = (1.0 / (d * d)) * torch.ones((1, 1, d, d), dtype=torch.float32, device=cuda)
        for c in range(2):
            ref_rgb = F.conv2d((rgb[c].float() / 255.0).permute(2, 0, 1)[:, None], w, stride=d).squeeze(1).permute(1, 2, 0)
            ref_dep = F.conv2d(do.to_float(dep[c].cpu(), "depth").to(cuda)[None, None], w, stride=d)[0].permute(1, 2, 0)
            ref_mk = F.conv2d(mk[c].float()[None, None], w, stride=d)[0].permute(1, 2, 0)
            # d^2 terms summed in another order: the bound grows with the block
            assert do.ulp_distance(got[0][c], ref_rgb) <= max(4, d)
            assert do.ulp_distance(got[1][c], ref_dep) <= max(4, d)
            assert do.ulp_distance(got[2][c], ref_mk) <= max(4, d)
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    one = downscale_ground_truth(rgb, dep, mk, 1)
    assert torch.equal(one[0], rgb.float() / 255.0) and torch.equal(one[2][..., 0], mk.float())


def test_bad_arguments(cuda):
    rgb, dep, mk = (t.to(cuda) for t in do.make_inputs(1, 20, 30, "u8", "u16", "bool"))
    for d in (0, 21):
        with pytest.raises(ValueError):
            downscale_ground_truth(rgb, dep, mk, d)
    with pytest.raises(ValueError):
        downscale_ground_truth(rgb, dep[:, :10], mk, 2)
    with pytest.raises(RuntimeError):
        downscale_ground_truth(rgb.cpu(), dep, mk, 2)
    lib = _lib.load()
    out = torch.empty(10 * 15 * 3, device=cuda)
    p = _lib.ptr
    assert lib.qed_downscale_ground_truth(1, 30, 20, 0, p(rgb), 1, p(dep), 1, 0.001, None, 0, p(out), p(out), None, None) == -1
    assert lib.qed_downscale_ground_truth(1, 30, 20, 2, None, 1, p(dep), 1, 0.001, None, 0, p(out), p(out), None, None) == -1
    assert lib.qed_downscale_ground_truth(1, 30, 20, 2, p(rgb), 1, p(dep), 1, 0.001, p(mk), 1, p(out), p(out), None, None) == -1
    assert lib.qed_downscale_ground_truth(1, 30, 20, 31, p(rgb), 1, p(dep), 1, 0.001, None, 0, p(out), p(out), None, None) == -1


@pytest.mark.parametrize("d", [2, 4])
@pytest.mark.parametrize("ssim,with_mask,grid", [(0.0, False, False), (0.2, True, False), (0.2, True, True), (0.0, False, True)])
def test_loss_on_full_resolution_gt_is_the_loss_on_downscaled_gt(cuda, d, ssim, with_mask, grid):
    C, H, W = 2, 190, 250
    gt_rgb, gt_depth, mask = do.make_inputs(C, H, W, "u8", "u16", "bool" if with_mask else None, seed=d)
    h, w = H // d, W // d
    g = torch.Generator().manual_seed(3)
    render = torch.rand(C, h, w, 4, generator=g).to(cuda)
    render[..., 3] *= 20
    alphas = torch.rand(C, h, w, 1, generator=g).to(cuda)
    bg = torch.tensor([0.2, 0.4, 0.6], device=cuda)
    small = [None if t is None else t.to(cuda) for t in do.downscale_ground_truth(gt_rgb, gt_depth, mask, d)]
    kw = dict(ssim_lambda=ssim)
    grids = None
    if grid:
        import bilagrid_oracle as bo

        grids = (bo.identity_grids(3) + 0.05 * torch.randn(3, 12, 8, 16, 16, generator=g)).to(cuda)
        kw["grid_ids"] = torch.tensor([2, 0], dtype=torch.int32, device=cuda)
    res = []
    for args, extra in (((gt_rgb.to(cuda), gt_depth.to(cuda), None if mask is None else mask.to(cuda)), dict(gt_downscale=d)),
                        ((small[0], small[1], small[2]), {})):
        r, a = render.clone().requires_grad_(True), alphas.clone().requires_grad_(True)
        gr = None if grids is None else grids.clone().requires_grad_(True)
        tot, l_rgb, l_dep = depth_supervised_loss(r, a, args[0], args[1], bg, mask=args[2], bilateral_grids=gr, **kw, **extra)
        tot.backward()
        res.append([tot.detach(), l_rgb, l_dep, r.grad, a.grad] + ([] if gr is None else [gr.grad]))
    for x, y in zip(*res):
        assert torch.equal(x, y)
    with pytest.raises(ValueError):  # render not at H // d x W // d
        depth_supervised_loss(render[:, :-1], alphas[:, :-1], gt_rgb.to(cuda), gt_depth.to(cuda), bg, gt_downscale=d)


def _leaves(s, cuda):
    lv = dict(means=s.means, scales=torch.log(s.scales), quats=s.quats * 1.7, features_dc=s.sh[:, 0, :], features_rest=s.sh[:, 1:, :],
              opacities=torch.logit(s.opacities)[:, None])
    return {k: v.clone().to(cuda).requires_grad_(True) for k, v in lv.items()}


def test_reference_step_at_half_resolution(cuda):
    """rasterization() at the rescaled camera + depth_supervised_loss(gt_downscale=2) on the uint8 image against
    tests/reference_model.oracle_reference_step(down=2) (pinned to the reference's lines by the CPU test)."""
    s = scene_s0(N=1500, C=2, size=96)
    cam = 1
    rgb_u8, dep_u16, mask = _cached_gt(s)
    s.gt_rgb = rgb_u8
    s.gt_depth = do.to_float(dep_u16, "depth")[..., None]
    bg = torch.tensor([0.1, 0.5, 0.9])
    c2w = rm.c2w_from_viewmat(s.viewmats[cam:cam + 1])
    ref_out, ref_loss, ref_leaves = rm.oracle_reference_step(s, cam, c2w, bg, step=3000, mask=mask[cam][..., None], down=2)
    sum(ref_loss.values()).backward()

    lv = _leaves(s, cuda)
    Ks, w, h = rescaled_camera(s.Ks[cam:cam + 1].to(cuda), s.width, s.height, 2)
    colors = torch.cat((lv["features_dc"][:, None, :], lv["features_rest"]), dim=1)
    render, alpha, _ = rasterization(means=lv["means"], quats=lv["quats"] / lv["quats"].norm(dim=-1, keepdim=True), scales=torch.exp(lv["scales"]),
                                     opacities=torch.sigmoid(lv["opacities"]).squeeze(-1), colors=colors, viewmats=ref_out["viewmat"].to(cuda), Ks=Ks,
                                     width=w, height=h, render_mode="RGB+D", sh_degree=3, absgrad=True)
    tot, l_rgb, l_dep = depth_supervised_loss(render, alpha, rgb_u8[cam:cam + 1].to(cuda), dep_u16[cam:cam + 1].to(cuda), bg.to(cuda), rgb_weight=0.8,
                                              depth_lambda=0.2, ssim_lambda=0.2, mask=mask[cam:cam + 1].to(cuda), gt_downscale=2)
    assert float(l_rgb) == pytest.approx(float(ref_loss["main_loss"]), rel=2e-4, abs=1e-6)
    assert float(l_dep) == pytest.approx(float(ref_loss["depth_loss"]), rel=2e-4, abs=1e-6)
    tot.backward()
    for k, ref in ref_leaves.items():
        assert_close_frac(lv[k].grad, ref.grad, 1e-3, 1e-3 * float(ref.grad.abs().mean() + 1e-12), 5e-3, f"v_{k}")


@pytest.mark.parametrize("C,n_chunks", [(2, 1), (1, 3)])
def test_fused_step_across_resolution_changes(cuda, C, n_chunks):
    """One FusedSplatStep driven through d = 4 -> 2 -> 1 -> 4 matches a fresh object at each size (the growing lists of
    the larger renders overflow the reused object's capacity and repeat)."""
    s = scene_s0(N=20000, C=C, size=192)
    t = s.to(cuda)
    rgb, dep, mask = (x.to(cuda) for x in _cached_gt(s))
    bg = torch.tensor([0.3, 0.2, 0.1], device=cuda)
    args = (t.means, t.quats, torch.log(t.scales), torch.logit(t.opacities), t.sh, t.viewmats)
    reused = FusedSplatStep(cuda)
    for d in (4, 2, 1, 4):
        Ks, w, h = rescaled_camera(t.Ks, s.width, s.height, d)
        outs = []
        for fs in (reused, FusedSplatStep(cuda)):
            o = fs.step(*args, Ks, w, h, 3, rgb, dep, bg, render_mode="RGB+D", ssim_lambda=0.2, activations=3, mask=mask, n_chunks=n_chunks,
                        gt_downscale=d)
            outs.append(dict(loss=o.loss.clone(), render=o.render.clone(), **{k: v.clone() for k, v in o.grads.items()}))
        a, b = outs
        assert a["render"].shape == (C, h, w, 4)
        assert torch.equal(a["render"], b["render"])
        assert torch.allclose(a["loss"], b["loss"], rtol=1e-6, atol=0), d
        # the compositor's backward sums with atomics: on a B200 two orders differed by up to 1.5e-6 of the largest
        # scales gradient at 192x192
        for k in ("means", "quats", "scales", "opacities", "sh"):
            assert float((a[k] - b[k]).abs().max()) <= 1e-5 * float(b[k].abs().max()), (d, k)
    assert reused.overflow_repeats >= 1


def _gaussian_args(s, dev):
    return (s.means.to(dev), s.quats.to(dev), torch.log(s.scales).to(dev), torch.logit(s.opacities).to(dev), s.sh.to(dev))


def _twin_kwargs(t, cuda, rgb, dep, mask, d, cam_opt, grid):
    """Step arguments of the schedule trainer (full resolution) and of its twin (rescaled camera, downscaled ground truth)."""
    Ks, w, h = rescaled_camera(t.Ks, t.width, t.height, d)
    small = [x.to(cuda) for x in (do.downscale_ground_truth(rgb, dep, mask, d) if d > 1 else (rgb, dep, mask))]
    kw = {}
    if cam_opt:
        kw.update(camera_to_worlds=rm.c2w_from_viewmat(t.viewmats.cpu()).to(cuda), camera_ids=torch.tensor([1, 0]))
    elif grid:
        kw.update(camera_ids=torch.tensor([1, 0]))
    vm = None if cam_opt else t.viewmats
    full = ((vm, t.Ks, t.width, t.height, rgb.to(cuda), dep.to(cuda)), dict(mask=mask.to(cuda), **kw))
    twin = ((vm, Ks, w, h, small[0], small[1]), dict(mask=small[2], **kw))
    return full, twin


@pytest.mark.parametrize("cam_opt,grid", [(False, False), (True, True)])
def test_trainer_schedule_equals_hand_fed_twin(cuda, cam_opt, grid):
    s = scene_s0(N=6000, C=2, size=128)
    t = s.to(cuda)
    rgb, dep, mask = _cached_gt(s)
    bg = torch.tensor([0.3, 0.3, 0.3], device=cuda)
    extra = dict(sh_degree_interval=1)
    if cam_opt:
        extra.update(camera_optimizer="SO3xR3", camera_opt_warmup=0)
    if grid:
        extra.update(use_bilateral_grid=True, bilateral_grid_warmup=0)
    sched = SplatTrainer(*_gaussian_args(s, cuda), cfg=TrainConfig(num_downscales=2, resolution_schedule=2, **extra), num_cameras=2)
    twin = SplatTrainer(*_gaussian_args(s, cuda), cfg=TrainConfig(**extra), num_cameras=2)
    factors = []
    for it in range(8):
        d = sched.downscale_factor()
        factors.append(d)
        full, small = _twin_kwargs(t, cuda, rgb, dep, mask, d, cam_opt, grid)
        l_s, _ = sched.step(*full[0], bg, **full[1])
        l_t, _ = twin.step(*small[0], bg, **small[1])
        assert sched._fused._fwd["render"].shape[1:3] == (128 // d, 128 // d)
        assert torch.allclose(l_s, l_t, rtol=1e-6, atol=1e-9), (it, d)
        for g in GROUPS:
            a, b = sched.arena.view(sched.arena.param, g), twin.arena.view(twin.arena.param, g)
            assert float((a - b).abs().max()) <= 1e-6 * float(b.abs().max()), (it, g)
        for name in ("grad2d", "count", "radii"):
            a, b = getattr(sched.state, name), getattr(twin.state, name)
            assert float((a - b).abs().max()) <= 1e-6 * float(b.abs().max()) + 1e-30, (it, name)
        if cam_opt:
            assert float((sched.pose_adjustment - twin.pose_adjustment).abs().max()) <= 1e-6 * float(twin.pose_adjustment.abs().max()) + 1e-12
        if grid:
            assert float((sched.bilateral_grids - twin.bilateral_grids).abs().max()) <= 1e-6
    assert factors == [4, 4, 2, 2, 1, 1, 1, 1]


def _exchange_worker(rank, port, out):
    """An NCCL group of one: a schedule trainer on the exchange path next to the plain one, across a schedule boundary."""
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=dev)
    res = {}
    try:
        s = scene_s0(N=6000, C=2, size=96)
        t = s.to(dev)
        rgb, dep, mask = (x.to(dev) for x in _cached_gt(s))
        cfg = dict(num_downscales=1, resolution_schedule=2, sh_degree_interval=1)
        xt = SplatTrainer(*_gaussian_args(s, dev), cfg=TrainConfig(comm="exchange", **cfg))
        xt.comm = "exchange"  # world 1 picks no collective; one rank runs the multi-GPU code path unchanged
        ref = SplatTrainer(*_gaussian_args(s, dev), cfg=TrainConfig(**cfg))
        bg = torch.tensor([0.2, 0.5, 0.8], device=dev)
        res.update(loss_err=[], exchanges=[], sizes=[])
        p0 = ref.arena.param.clone()
        for _ in range(5):  # d = 2, 2, 1, 1, 1
            ls = [tr.step(t.viewmats, t.Ks, s.width, s.height, rgb, dep, bg, mask=mask)[0] for tr in (xt, ref)]
            res["loss_err"].append(float((ls[0] - ls[1]).abs().max() / ls[1].abs().max()))
            res["exchanges"].append(id(xt._xg))
            res["sizes"].append(tuple(xt._fused._fwd["render"].shape[1:3]))
        res["comm"] = xt.comm
        res["param_err"] = float((xt.arena.param - ref.arena.param).abs().max())
        res["param_moved"] = float((ref.arena.param - p0).abs().max())
    except RuntimeError as e:  # no symmetric memory on this machine
        res["error"] = str(e)
    torch.save(res, out)
    dist.destroy_process_group()


def test_trainer_exchange_path_across_a_schedule_boundary(cuda, tmp_path):
    out = str(tmp_path / "xchg.pt")
    mp.spawn(_exchange_worker, args=(29500 + (os.getpid() + 41) % 2000, out), nprocs=1, join=True)
    r = torch.load(out)
    if "error" in r and "symmetric memory" in r["error"]:
        pytest.skip(r["error"])
    assert "error" not in r, r
    assert r["comm"] == "exchange", r
    assert r["sizes"] == [(48, 48), (48, 48), (96, 96), (96, 96), (96, 96)], r
    assert len(set(r["exchanges"])) == 1, r  # the exchange buffers survive the resolution change
    assert max(r["loss_err"]) <= 1e-5, r
    assert r["param_moved"] > 0 and r["param_err"] <= 1e-3 * r["param_moved"], r
