"""CPU: splatfacto's resolution schedule -- the oracle of the ground-truth pass against splatfacto's `_downscale_if_required`
(the stand-in's CPU conv2d), the schedule of SplatTrainer.downscale_factor and the render camera of a downscaled step
against nerfstudio's `rescale_output_resolution` (the stand-in's)."""
import pytest
import torch

import downscale_oracle as do
from qed_splatter_b200.data_side import downscaled_size
from qed_splatter_b200.trainer import SplatTrainer, TrainConfig, rescaled_camera


@pytest.mark.parametrize("d", [2, 4, 8])
@pytest.mark.parametrize("size", [(64, 48), (83, 61)])  # (W, H); the second is divisible by none of the factors
@pytest.mark.parametrize("rgb,depth,mask", [("u8", "u16", "bool"), ("f32", "f32", "u8"), ("u8", "f32", "f32"), ("f32", "u16", None)])
def test_oracle_matches_splatfacto_downscale(d, size, rgb, depth, mask):
    W, H = size
    C = 2
    gt_rgb, gt_depth, m = do.make_inputs(C, H, W, rgb, depth, mask, seed=d)
    o_rgb, o_dep, o_mk = do.downscale_ground_truth(gt_rgb, gt_depth, m, d)
    assert o_rgb.shape == (C, H // d, W // d, 3) and o_dep.shape == (C, H // d, W // d, 1)
    for c in range(C):
        # the same float image on both sides: the filter is compared here, the u8 conversion below
        ref_rgb = do.stub_downscale(do.to_float(gt_rgb[c], "rgb"), d)
        assert do.ulp_distance(o_rgb[c], ref_rgb) <= 2
        ref_dep = do.stub_downscale(do.to_float(gt_depth[c], "depth")[..., None], d)
        assert do.ulp_distance(o_dep[c], ref_dep) <= 2
        if m is not None:
            ref_mk = do.stub_downscale(m[c][..., None], d)  # bool / uint8 masks: conv2d on image.float()
            assert do.ulp_distance(o_mk[c], ref_mk) <= 2
    if depth == "f32":
        assert bool(torch.isnan(o_dep).any())  # NaN propagates to its block
    assert bool((o_dep == 0).sum() < o_dep.numel())


def test_u8_conversion_is_get_gt_img():
    """u8 * (1/255) is what torch's CUDA `image.float() / 255.0` computes (GtImage, tests/test_gpu_downscale.py checks it
    bit for bit on the device); the CPU's true division is within 1 ulp of it."""
    x = torch.arange(256, dtype=torch.uint8)
    assert do.ulp_distance(do.to_float(x, "rgb"), x.float() / 255.0) <= 1


def _trainer_at(step, **cfg):
    t = SplatTrainer.__new__(SplatTrainer)  # the schedule needs no Gaussians
    t.cfg, t.step_count = TrainConfig(**cfg), step
    return t


def test_schedule():
    got = [_trainer_at(s, num_downscales=2, resolution_schedule=3000).downscale_factor() for s in (0, 2999, 3000, 5999, 6000, 30000)]
    assert got == [4, 4, 2, 2, 1, 1]
    assert all(_trainer_at(s).downscale_factor() == 1 for s in (0, 1, 2999, 3000, 100000))
    assert [_trainer_at(s, num_downscales=1, resolution_schedule=2).downscale_factor() for s in range(4)] == [2, 2, 1, 1]
    assert TrainConfig().num_downscales == 0 and TrainConfig().resolution_schedule == 3000


@pytest.mark.parametrize("bad", [dict(num_downscales=-1), dict(resolution_schedule=0), dict(resolution_schedule=-5)])
def test_bad_schedule_config_raises(bad):
    with pytest.raises(ValueError):
        TrainConfig(**bad)
    cfg = TrainConfig()
    for k, v in bad.items():
        setattr(cfg, k, v)
    with pytest.raises(ValueError):
        cfg.validate()


@pytest.mark.parametrize("d", [2, 4, 8])
def test_render_camera_matches_rescale_output_resolution(d):
    Cameras = do.stub_cameras()
    W, H = 1920, 1080
    fx, fy, cx, cy = 1234.567, 1187.25, 961.3, 539.77
    cam = Cameras(torch.zeros(1, 3, 4), fx, fy, cx, cy, W, H)
    K = cam.get_intrinsics_matrices()
    cam.rescale_output_resolution(1.0 / d)
    Ks, w, h = rescaled_camera(K, W, H, d)
    assert torch.equal(Ks, cam.get_intrinsics_matrices())  # powers of two: exact
    assert torch.equal(Ks[:, :2], K[:, :2] / d) and torch.equal(Ks[:, 2], K[:, 2])
    assert (w, h) == (int(cam.width), int(cam.height)) == downscaled_size(W, H, d)
    assert (w, h) == {2: (960, 540), 4: (480, 270), 8: (240, 135)}[d]
    assert torch.equal(K, Cameras(torch.zeros(1, 3, 4), fx, fy, cx, cy, W, H).get_intrinsics_matrices())  # input not modified
    assert rescaled_camera(K, W, H, 1)[1:] == (W, H)


def test_render_camera_size_mismatch_raises():
    K = torch.eye(3)[None]
    with pytest.raises(ValueError, match=r"721x540.*720x540"):  # floor(1441 / 2 + 0.5) = 721, 1441 // 2 = 720
        rescaled_camera(K, 1441, 1080, 2)
    with pytest.raises(ValueError):
        downscaled_size(3, 100, 4)
    with pytest.raises(ValueError):
        downscaled_size(64, 64, 0)
