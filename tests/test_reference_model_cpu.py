"""CPU: the reference's OWN lines (qed_splatter/model.py, unmodified) pin the oracle's call-site restatements.

`QEDSplatterModel.get_outputs` + `get_loss_dict` are executed from the reference package with `gsplat` resolved to the
CPU oracle's rasterization; the result must equal the oracle-only formulation of the same step
(oracle.get_viewmat <- model.py:22-38, composite_and_fill <- :295-306, depth_l1_loss(mask) <- :87-116), i.e. these
restatements are pinned by reference-held code, with and without `batch["mask"]`.  Those tests skip when no reference
package is available (tests/reference_model.py); the stored outputs of the same step of the reference
(tests/golden/ref_model_*.npz, scripts/make_golden_reference_model.py) pin the restatement without it."""
import os

import numpy as np
import pytest
import torch

from qed_splatter_b200.scenes import scene_s0
import reference_model as rm

needs_reference = pytest.mark.skipif(rm.reference_root() is None, reason="reference package not available (see tests/reference_model.py)")
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _batch(s, cam, mask):
    b = {"image": s.gt_rgb[cam], "depth_image": s.gt_depth[cam]}
    if mask is not None:
        b["mask"] = mask
    return b


@needs_reference
@pytest.mark.parametrize("mask_kind,down", [(None, 1), ("float", 1), ("bool", 1), (None, 2)])
def test_reference_model_lines_equal_oracle_restatement(mask_kind, down):
    s = scene_s0(N=1500, C=2, size=48)
    cam = 1
    g = torch.Generator().manual_seed(5)
    mask = None
    if mask_kind is not None:
        mask = (torch.rand(s.height, s.width, 1, generator=g) > 0.3)
        mask = mask.float() if mask_kind == "float" else mask
    num_downscales = {1: 0, 2: 1}[down]
    with rm.reference_modules("oracle") as mod:
        assert mod.rasterization.__module__.startswith("oracle")
        model = rm.build_model(mod, s, "cpu", step=3000 if down == 1 else 2000, num_downscales=num_downscales)
        model.train()
        camera = rm.make_camera(s, cam, "cpu")
        assert torch.equal(mod.get_viewmat(camera.camera_to_worlds), __import__("oracle").get_viewmat(camera.camera_to_worlds))
        out = model.get_outputs(camera)
        loss = model.get_loss_dict(out, _batch(s, cam, mask))
        total = sum(loss.values())
        total.backward()
        bg = model._get_background_color()
        got_grads = {k: model.gauss_params[k].grad.clone() for k in model.gauss_params}
        c2w = camera.camera_to_worlds
    ref_out, ref_loss, leaves = rm.oracle_reference_step(s, cam, c2w, bg, step=model.step, mask=mask, down=down)
    sum(ref_loss.values()).backward()
    for k in ("rgb", "depth", "accumulation"):
        assert torch.equal(out[k].detach(), ref_out[k].detach()), k
    assert set(loss) == {"main_loss", "scale_reg", "depth_loss"}
    for k in ("main_loss", "depth_loss"):
        torch.testing.assert_close(loss[k].detach(), ref_loss[k].detach(), rtol=1e-6, atol=1e-7)
    for k, gref in leaves.items():
        torch.testing.assert_close(got_grads[k], gref.grad, rtol=1e-5, atol=1e-9, msg=lambda m: f"{k}: {m}")


@pytest.mark.parametrize("name", ["ref_model_plain", "ref_model_mask", "ref_model_boolmask_sh1"])
def test_oracle_restatement_matches_reference_model_fixture(name):
    """The oracle-only formulation of the step reproduces what the unmodified model.py computed (stored fixture):
    viewmat (model.py:22-38, also the data side's pinned float32 restatement), radii, outputs, loss terms, gradients."""
    import oracle
    from oracle import pointcloud as opc

    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    s = scene_s0(N=int(z["scene_N"]), C=int(z["scene_C"]), size=int(z["scene_size"]), seed=int(z["scene_seed"]))
    cam, step, kind = int(z["cam"]), int(z["step"]), str(z["mask_kind"])
    mask = None
    if kind != "None":
        mask = torch.rand(s.height, s.width, 1, generator=torch.Generator().manual_seed(5)) > 0.3
        mask = mask.float() if kind == "float" else mask
    c2w = torch.from_numpy(z["c2w"])
    assert torch.equal(c2w, rm.c2w_from_viewmat(s.viewmats[cam:cam + 1]))
    assert torch.equal(oracle.get_viewmat(c2w), torch.from_numpy(z["viewmat"]))
    assert np.array_equal(opc.get_viewmat_pinned(z["c2w"]), z["viewmat"])
    out, loss, leaves = rm.oracle_reference_step(s, cam, c2w, torch.from_numpy(z["background"]), step=step, mask=mask)
    sum(loss.values()).backward()
    assert torch.equal(out["info"]["radii"][0], torch.from_numpy(z["radii"]))
    for k in ("rgb", "depth", "accumulation"):
        assert torch.equal(out[k].detach(), torch.from_numpy(z[k])), k
    for k in ("main_loss", "depth_loss"):
        assert float(loss[k]) == float(z[k]), k
    for k, v in leaves.items():
        assert torch.equal(v.grad, torch.from_numpy(z["grad_" + k])), f"grad {k}"


@needs_reference
def test_reference_model_eval_path_and_empty_depth_mask():
    """Eval render (model.py:213-214, 256-257, 313-314) and the all-invalid depth branch (model.py:111-114)."""
    s = scene_s0(N=800, C=1, size=40)
    with rm.reference_modules("oracle") as mod:
        model = rm.build_model(mod, s, "cpu")
        model.eval()
        camera = rm.make_camera(s, 0, "cpu")
        with torch.no_grad():
            out = model.get_outputs(camera)
        assert out["rgb"].shape == (40, 40, 3) and out["depth"].shape == (40, 40, 1) and out["background"].shape == (40, 40, 3)
        batch = {"image": s.gt_rgb[0], "depth_image": torch.zeros_like(s.gt_depth[0])}
        loss = model.get_loss_dict(out, batch)
        assert float(loss["depth_loss"]) == 0.0
    import oracle

    assert float(oracle.depth_l1_loss(out["depth"], torch.zeros_like(s.gt_depth[0]))) == 0.0
