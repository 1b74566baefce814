"""GPU: the CUDA path against outputs of the REFERENCE'S OWN CODE.

1. `test_cuda_paths_match_reference_model_fixture`: tests/golden/ref_model_*.npz hold what the unmodified
   qed_splatter/model.py (QEDSplatterModel.get_outputs + get_loss_dict + backward, model.py:73-118, 199-321) produced
   (scripts/make_golden_reference_model.py; rasterization = the CPU oracle).
   Both product paths must reproduce them on the B200: the gsplat-surface `rasterization()` + `depth_supervised_loss()`
   and the fused `FusedSplatStep.step()` (folded activations, fused loss, `mask`); the get_viewmat kernel must
   reproduce the viewmat model.py built.
2. `test_unmodified_reference_model_runs_on_the_cuda_shim`: when the reference package is available
   (see tests/reference_model.py) the UNMODIFIED model.py itself runs on the GPU with
   `from gsplat.rendering import rasterization` resolved to the product's shim, and must give the same outputs, loss dict
   and parameter gradients -- with and without batch["mask"], and `info["means2d"]` must behave as gsplat's strategy
   expects (.grad after retain_grad(), .absgrad)."""
import os

import numpy as np
import pytest
import torch

import reference_model as rm
from helpers import assert_close_frac
from qed_splatter_b200 import depth_supervised_loss, rasterization
from qed_splatter_b200.pipeline import FusedSplatStep
from qed_splatter_b200.scenes import scene_s0

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
CASES = ["ref_model_plain", "ref_model_mask", "ref_model_boolmask_sh1"]
PARAMS = ("means", "scales", "quats", "features_dc", "features_rest", "opacities")


def _load(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    s = scene_s0(N=int(z["scene_N"]), C=int(z["scene_C"]), size=int(z["scene_size"]), seed=int(z["scene_seed"]))
    kind = str(z["mask_kind"])
    mask = None
    if kind != "None":
        m = torch.rand(s.height, s.width, 1, generator=torch.Generator().manual_seed(5)) > 0.3
        mask = m.float() if kind == "float" else m
    return z, s, int(z["cam"]), int(z["step"]), mask


def _check_grads(got, z, what):
    for k in PARAMS:
        ref = torch.from_numpy(z["grad_" + k])
        g = got[k].reshape(ref.shape)
        assert_close_frac(g, ref, 1e-3, 1e-3 * float(ref.abs().mean() + 1e-12), 5e-3, f"{what} v_{k}")


@pytest.mark.parametrize("name", CASES)
def test_cuda_paths_match_reference_model_fixture(cuda, name):
    z, s, cam, step, mask = _load(name)
    deg = min(step // 1000, 3)
    bg = torch.from_numpy(z["background"]).to(cuda)
    viewmat = torch.from_numpy(z["viewmat"]).to(cuda)
    K = s.Ks[cam:cam + 1].to(cuda)
    gt_rgb, gt_depth = s.gt_rgb[cam:cam + 1].to(cuda), s.gt_depth[cam:cam + 1].to(cuda)
    mk = mask[None].to(cuda) if mask is not None else None
    ref_total = float(z["main_loss"]) + float(z["depth_loss"])

    # (a) gsplat surface + the loss drop-in, parameters in splatfacto's stored form with torch activations (model.py:269-271)
    leaves = dict(means=s.means, scales=torch.log(s.scales), quats=s.quats * 1.7, features_dc=s.sh[:, 0, :], features_rest=s.sh[:, 1:, :],
                  opacities=torch.logit(s.opacities)[:, None])
    leaves = {k: v.clone().to(cuda).requires_grad_(True) for k, v in leaves.items()}
    colors = torch.cat((leaves["features_dc"][:, None, :], leaves["features_rest"]), dim=1)
    render, alpha, info = rasterization(
        means=leaves["means"], quats=leaves["quats"] / leaves["quats"].norm(dim=-1, keepdim=True), scales=torch.exp(leaves["scales"]),
        opacities=torch.sigmoid(leaves["opacities"]).squeeze(-1), colors=colors, viewmats=viewmat, Ks=K, width=s.width, height=s.height,
        tile_size=16, packed=False, near_plane=0.01, far_plane=1e10, render_mode="RGB+D", sh_degree=deg, sparse_grad=False, absgrad=True,
        rasterize_mode="classic")
    assert torch.equal(info["radii"][0].cpu(), torch.from_numpy(z["radii"]))
    rgb = torch.clamp(render[..., :3] + (1 - alpha) * bg, 0.0, 1.0)
    depth = torch.where(alpha > 0, render[..., 3:4], render[..., 3:4].detach().max())
    assert_close_frac(rgb[0], torch.from_numpy(z["rgb"]), 1e-4, 1e-4, 2e-3, "rgb")
    assert_close_frac(depth[0], torch.from_numpy(z["depth"]), 1e-4, 1e-4, 2e-3, "depth")
    assert_close_frac(alpha[0], torch.from_numpy(z["accumulation"]), 1e-4, 1e-4, 2e-3, "accumulation")
    total, l_rgb, l_depth = depth_supervised_loss(render, alpha, gt_rgb, gt_depth, bg, rgb_weight=0.8, depth_lambda=0.2, ssim_lambda=0.2, mask=mk)
    assert float(l_rgb) == pytest.approx(float(z["main_loss"]), rel=2e-4, abs=1e-6)
    assert float(l_depth) == pytest.approx(float(z["depth_loss"]), rel=2e-4, abs=1e-6)
    total.backward()
    _check_grads({k: v.grad for k, v in leaves.items()}, z, "rasterization+depth_supervised_loss")

    # (b) fused step: stored parameters straight in (activations folded), loss + mask fused
    fs = FusedSplatStep(cuda)
    # (the projection normalises the quaternion itself, so the stored, un-normalised parameter goes straight in and
    # the gradient comes back with respect to it -- what the trainer does)
    out = fs.step(s.means.to(cuda), (s.quats * 1.7).to(cuda), torch.log(s.scales).to(cuda), torch.logit(s.opacities).to(cuda),
                  s.sh.to(cuda), viewmat, K, s.width, s.height, deg, gt_rgb, gt_depth, bg, render_mode="RGB+D", rgb_weight=0.8, depth_lambda=0.2,
                  ssim_lambda=0.2, activations=3, mask=mk)
    assert float(out.loss[0]) == pytest.approx(ref_total, rel=2e-4, abs=1e-6)
    g = out.grads
    fused = dict(means=g["means"], scales=g["scales"], quats=g["quats"], features_dc=g["sh"][:, 0, :], features_rest=g["sh"][:, 1:, :],
                 opacities=g["opacities"][:, None])
    _check_grads(fused, z, "FusedSplatStep")


@pytest.mark.parametrize("name", CASES)
def test_get_viewmat_kernel_matches_reference_model_fixture(cuda, name):
    """The one-launch get_viewmat kernel on the model's camera against the viewmat the reference's own function built
    (model.py:22-38, stored in the fixture): rotation block and last row exact, translation to 1 ulp of the sum."""
    from qed_splatter_b200 import get_viewmat

    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    ref_vm = torch.from_numpy(z["viewmat"])
    got_vm = get_viewmat(torch.from_numpy(z["c2w"]).to(cuda)).cpu()
    assert torch.equal(got_vm[:, :3, :3], ref_vm[:, :3, :3]) and torch.equal(got_vm[:, 3], ref_vm[:, 3])
    torch.testing.assert_close(got_vm, ref_vm, rtol=0, atol=2e-6)


@pytest.mark.skipif(rm.reference_root() is None, reason="reference package not available (see tests/reference_model.py)")
@pytest.mark.parametrize("name", CASES)
def test_unmodified_reference_model_runs_on_the_cuda_shim(cuda, name):
    z, s, cam, step, mask = _load(name)
    with rm.reference_modules("cuda") as mod:
        assert mod.rasterization.__module__ == "qed_splatter_b200.rendering"  # model.py:7 resolved to the product
        model = rm.build_model(mod, s, cuda, step=step)
        model.train()
        camera = rm.make_camera(s, cam, cuda)
        out = model.get_outputs(camera)  # qed_splatter/model.py:199-321, unmodified
        batch = {"image": s.gt_rgb[cam].to(cuda), "depth_image": s.gt_depth[cam].to(cuda)}
        if mask is not None:
            batch["mask"] = mask.to(cuda)
        loss = model.get_loss_dict(out, batch)  # model.py:73-118 + the stand-in parent's splatfacto RGB loss
        sum(loss.values()).backward()
        assert torch.equal(model.radii.cpu(), torch.from_numpy(z["radii"]))
        for k in ("rgb", "depth", "accumulation"):
            assert_close_frac(out[k], torch.from_numpy(z[k]), 1e-4, 1e-4, 2e-3, k)
        assert float(loss["main_loss"]) == pytest.approx(float(z["main_loss"]), rel=2e-4, abs=1e-6)
        assert float(loss["depth_loss"]) == pytest.approx(float(z["depth_loss"]), rel=2e-4, abs=1e-6)
        _check_grads({k: model.gauss_params[k].grad for k in PARAMS}, z, "QEDSplatterModel")
        # what gsplat's DefaultStrategy reads from self.info (model.py:289-292)
        xys = model.info["means2d"]
        assert xys.grad is not None and xys.grad.shape == (1, s.N, 2)
        assert hasattr(xys, "absgrad") and xys.absgrad.shape == (1, s.N, 2)
        assert bool((xys.absgrad >= xys.grad.abs() - 1e-12).all())
        assert model.info["width"] == s.width and model.info["n_cameras"] == 1


@pytest.mark.skipif(rm.reference_root() is None, reason="reference package not available (see tests/reference_model.py)")
def test_reference_model_with_get_viewmat_rebound_to_the_kernel(cuda):
    """Row a1: `qed_splatter.model.get_viewmat = qed_splatter_b200.get_viewmat` (INTEGRATION.md 2b) -- the unmodified model
    then builds its viewmat (model.py:246) with the one-launch kernel; the kernel must agree with the reference's own
    function on the model's camera to the last bits that matter (rotation block exact, translation to 1 ulp of the sum)
    and the step must reproduce the fixture."""
    from qed_splatter_b200 import get_viewmat

    z, s, cam, step, mask = _load("ref_model_plain")
    with rm.reference_modules("cuda") as mod:
        model = rm.build_model(mod, s, cuda, step=step)
        model.train()
        camera = rm.make_camera(s, cam, cuda)
        ref_vm = mod.get_viewmat(camera.camera_to_worlds)  # the reference's own lines on the GPU
        got_vm = get_viewmat(camera.camera_to_worlds)
        assert torch.equal(got_vm[:, :3, :3], ref_vm[:, :3, :3]) and torch.equal(got_vm[:, 3], ref_vm[:, 3])
        torch.testing.assert_close(got_vm, ref_vm, rtol=0, atol=2e-6)
        mod.get_viewmat = get_viewmat
        out = model.get_outputs(camera)
        loss = model.get_loss_dict(out, {"image": s.gt_rgb[cam].to(cuda), "depth_image": s.gt_depth[cam].to(cuda)})
        for k in ("rgb", "depth", "accumulation"):
            assert_close_frac(out[k], torch.from_numpy(z[k]), 1e-4, 1e-4, 2e-3, k)
        assert float(loss["depth_loss"]) == pytest.approx(float(z["depth_loss"]), rel=2e-4, abs=1e-6)
