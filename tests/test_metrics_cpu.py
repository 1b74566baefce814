"""CPU: the float64 restatement of the held-out metrics, summarize(), argument checks and the exported surface."""
import math
import re
from pathlib import Path

import numpy as np
import pytest
import torch

import metrics_oracle as mo

ROOT = Path(__file__).resolve().parents[1]


def _views(C=2, H=16, W=20, seed=0):
    g = torch.Generator().manual_seed(seed)
    render = torch.rand(C, H, W, 4, generator=g)
    render[..., 3] = 0.5 + 4.0 * render[..., 3]
    alphas = torch.rand(C, H, W, 1, generator=g)
    return render, alphas, torch.rand(C, H, W, 3, generator=g), 0.5 + 4.0 * torch.rand(C, H, W, 1, generator=g), torch.tensor([0.1, 0.4, 0.7])


def test_oracle_identical_images_give_infinite_psnr_and_unit_ssim():
    render, _, _, gt_depth, bg = _views()
    alphas = torch.ones(2, 16, 20, 1)
    m = mo.image_metrics(render, alphas, render[..., :3].clone(), render[..., 3:].clone(), bg)
    assert np.all(np.isposinf(m[:, 0])) and np.all(m[:, 2] == 0.0)
    np.testing.assert_allclose(m[:, 1], 1.0, rtol=0, atol=1e-12)
    # prediction == ground truth depth: zero errors, every ratio 1
    np.testing.assert_array_equal(m[:, 3:7], 0.0)
    np.testing.assert_array_equal(m[:, 7:10], 1.0)
    np.testing.assert_array_equal(m[:, 10], 16 * 20)


def test_oracle_depth_metrics_by_hand():
    g = np.array([[1.0, 2.0, 4.0, 0.05],
                  [np.nan, 1.0, 2.0, np.inf],
                  [0.0, -1.0, 1.0, 1.0],
                  [3.0, 3.0, 3.0, 3.0]], np.float32)
    d = np.array([[1.0, 1.0, 4.0, 9.0],
                  [9.0, 1.2, 3.0, 9.0],
                  [9.0, 9.0, 1.5, 2.0],
                  [3.0, 3.0, 3.0, 3.0]], np.float32)
    # valid (finite and > 0.1): (0,0) (0,1) (0,2) (1,1) (1,2) (2,2) (2,3) and the last row
    pairs = [(1, 1), (2, 1), (4, 4), (1, 1.2000000476837158), (2, 3), (1, 1.5), (1, 2), (3, 3), (3, 3), (3, 3), (3, 3)]
    gg = np.array([p[0] for p in pairs], np.float64)
    dd = np.array([p[1] for p in pairs], np.float64)
    n = len(pairs)
    t = np.maximum(gg / dd, dd / gg)
    want = [np.sum(np.abs(gg - dd) / gg) / n, np.sum((gg - dd) ** 2 / gg) / n, math.sqrt(np.sum((gg - dd) ** 2) / n),
            math.sqrt(np.sum((np.log(gg) - np.log(dd)) ** 2) / n), np.sum(t < 1.25) / n, np.sum(t < 1.5625) / n, np.sum(t < 1.953125) / n, n]
    # by hand: ratios 1, 2, 1, 1.2, 1.5, 1.5, 2, 1, 1, 1, 1 -> a1 = 7/11, a2 = a3 = 9/11 (2 is not < 1.953125)
    assert want[4:7] == [7 / 11, 9 / 11, 9 / 11]
    np.testing.assert_allclose(mo.depth_metrics(d, g, 0.1), want, rtol=1e-15)
    # the tolerance moves the cut: > 2.5 keeps (0,2) and the last row only
    np.testing.assert_array_equal(mo.depth_metrics(d, g, 2.5)[[0, 4, 7]], [0.0, 1.0, 5])


def test_oracle_no_valid_depth_is_nan_and_zero_prediction_propagates():
    g = np.zeros((4, 4), np.float32)
    g[0, 0] = np.nan
    m = mo.depth_metrics(np.ones((4, 4), np.float32), g, 0.1)
    assert np.all(np.isnan(m[:7])) and m[7] == 0
    g = np.full((4, 4), 2.0, np.float32)
    d = np.full((4, 4), 2.0, np.float32)
    d[0, 0] = 0.0
    m = mo.depth_metrics(d, g, 0.1)
    assert math.isinf(m[3]) and m[4] == 15 / 16 and m[7] == 16  # rmse_log = inf, the zero pixel fails every threshold


def test_summarize_averages_views_and_depth_views_only():
    from qed_splatter_b200.metrics import METRIC_NAMES, summarize

    rows = torch.tensor([[20.0, 0.5, 0.01, 0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 100.0],
                         [30.0, 0.7, 0.001] + [float("nan")] * 7 + [0.0],
                         [40.0, 0.9, 0.0001, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8, 0.9, 50.0]], dtype=torch.float64)
    s = summarize({name: rows[:, k] for k, name in enumerate(METRIC_NAMES)})
    assert s["psnr"] == pytest.approx(30.0) and s["ssim"] == pytest.approx(0.7) and s["rgb_mse"] == pytest.approx(0.0111 / 3)
    for k, name in enumerate(METRIC_NAMES[3:10], start=3):
        assert s[name] == pytest.approx((float(rows[0, k]) + float(rows[2, k])) / 2), name
    assert s["n_views"] == 3 and s["n_views_depth"] == 2
    none = summarize({name: rows[1:2, k] for k, name in enumerate(METRIC_NAMES)})
    assert none["n_views_depth"] == 0 and math.isnan(none["abs_rel"]) and none["psnr"] == 30.0


def test_argument_validation():
    from qed_splatter_b200 import image_metrics

    render, alphas, gt_rgb, gt_depth, bg = _views()
    with pytest.raises(RuntimeError, match="CUDA"):
        image_metrics(render, alphas, gt_rgb, gt_depth, bg)
    with pytest.raises(ValueError, match="4-channel"):
        image_metrics(render[..., :3].contiguous(), alphas, gt_rgb, gt_depth, bg)
    with pytest.raises(ValueError, match="shapes"):
        image_metrics(render, alphas, gt_rgb[:1], gt_depth, bg)
    with pytest.raises(ValueError, match="shapes"):
        image_metrics(render, alphas, gt_rgb, gt_depth[:, :8], bg)
    with pytest.raises(ValueError, match="shapes"):  # the right element count in the wrong layout
        image_metrics(render, alphas.transpose(1, 2), gt_rgb, gt_depth, bg)
    with pytest.raises(ValueError, match="shapes"):
        image_metrics(render, alphas, gt_rgb, gt_depth.transpose(1, 2), bg)
    with pytest.raises(ValueError, match="shapes"):
        image_metrics(render, alphas, gt_rgb, gt_depth.reshape(2, -1), bg)
    with pytest.raises(ValueError, match="gt_rgb"):
        image_metrics(render, alphas, gt_rgb.double(), gt_depth, bg)
    with pytest.raises(ValueError, match="gt_depth"):
        image_metrics(render, alphas, gt_rgb, gt_depth.to(torch.int32), bg)
    with pytest.raises(ValueError, match="render"):
        image_metrics(render.half(), alphas, gt_rgb, gt_depth, bg)
    with pytest.raises(ValueError, match="> 10"):
        image_metrics(render[:, :10], alphas[:, :10], gt_rgb[:, :10], gt_depth[:, :10], bg)


def test_trainer_evaluate_needs_the_cuda_backend():
    from qed_splatter_b200.trainer import SplatTrainer

    N = 10
    tr = SplatTrainer(torch.zeros(N, 3), torch.tensor([[1.0, 0, 0, 0]]).repeat(N, 1), torch.zeros(N, 3), torch.zeros(N), torch.zeros(N, 16, 3),
                      backend="torch")
    render, alphas, gt_rgb, gt_depth, bg = _views(C=1)
    with pytest.raises(RuntimeError, match="CUDA"):
        tr.evaluate(torch.eye(4)[None], torch.eye(3)[None], 20, 16, gt_rgb, gt_depth, bg)


def test_exported_surface_and_abi():
    import qed_splatter_b200
    from qed_splatter_b200 import _lib, metrics

    assert qed_splatter_b200.image_metrics is metrics.image_metrics and qed_splatter_b200.summarize is metrics.summarize
    header = (ROOT / "include" / "qed_splat.h").read_text()
    assert int(re.search(r"#define QED_EVAL_METRICS (\d+)", header).group(1)) == len(metrics.METRIC_NAMES) == len(mo.NAMES)
    assert metrics.METRIC_NAMES == mo.NAMES
    assert "qed_eval_metrics" in _lib.SIGNATURES and "qed_eval_metrics_workspace_bytes" in _lib.SIGNATURES
    lib = _lib.load()
    # host-side answers, no device touched
    assert lib.qed_eval_metrics_workspace_bytes(1, 10, 100) == 0 and lib.qed_eval_metrics_workspace_bytes(0, 100, 100) == 0
    tiles = -(-1910 // 32) * -(-1070 // 32)
    assert lib.qed_eval_metrics_workspace_bytes(2, 1920, 1080) == 256 + 2 * 3 * tiles * 10 * 8
    assert lib.qed_eval_metrics(0, 64, 64, None, None, None, 0, None, 0, 0.001, None, 0.1, None, None, 0, None) == -1
    assert lib.qed_eval_metrics(1, 64, 64, None, None, None, 0, None, 0, 0.001, None, 0.1, None, None, 0, None) == -1
