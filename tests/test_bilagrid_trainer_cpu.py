"""CPU: the host logic of the bilateral grid in SplatTrainer (torch backend) -- schedule, table Adam against torch.optim.Adam,
row accumulation with repeated ids, TV, configuration checks, and the world-2 gloo path whose grids stay bit-identical and
equal one rank fed both views."""
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import bilagrid_oracle as bo
from qed_splatter_b200.bilateral_grid import BilateralGridOptimizer
from qed_splatter_b200.trainer import SplatTrainer, TrainConfig

SHAPE = (4, 3, 5)  # (X, Y, L): small grids keep the CPU tests fast


def _gaussians(N, seed=0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(N, 3, generator=g), torch.randn(N, 4, generator=g), torch.log(torch.rand(N, 3, generator=g) * 0.05 + 0.001),
            torch.logit(torch.rand(N, generator=g) * 0.9 + 0.05), torch.randn(N, 16, 3, generator=g))


def _rows(n, seed=5):
    X, Y, L = SHAPE
    return torch.randn(n, 12, L, Y, X, generator=torch.Generator().manual_seed(seed)) * 1e-3


def test_schedule_endpoints_and_defaults():
    cfg = TrainConfig(use_bilateral_grid=True)
    assert (cfg.bilateral_grid_shape, cfg.bilateral_grid_lr, cfg.bilateral_grid_lr_final, cfg.bilateral_grid_warmup,
            cfg.bilateral_grid_tv_weight) == ((16, 16, 8), 2e-3, 1e-4, 1000, 10.0)
    bg = BilateralGridOptimizer(3, "cpu", backend="torch")
    assert bg.lr_at(0) == 0.0
    assert bg.lr_at(500) == pytest.approx(2e-3 * 2 ** -0.5)
    assert bg.lr_at(1000) == pytest.approx(2e-3)
    assert bg.lr_at(30000) == pytest.approx(1e-4) and bg.lr_at(40000) == pytest.approx(1e-4)
    assert torch.equal(bg.grids, bo.identity_grids(3))


def test_table_adam_matches_torch_optim():
    bg = BilateralGridOptimizer(2, "cpu", shape=SHAPE, lr=1e-2, lr_final=1e-2, warmup_steps=0, backend="torch")
    ref = bo.identity_grids(2, *SHAPE).requires_grad_(True)
    opt = torch.optim.Adam([ref], lr=1e-2, eps=1e-15)
    for it in range(4):
        g = _rows(2, seed=it)
        bg.grids_grad.copy_(g)
        bg.step(it)
        ref.grad = g.clone()
        opt.step()
    assert torch.allclose(bg.grids, ref.detach(), rtol=1e-6, atol=1e-7)


def test_tv_and_accumulate_with_repeated_ids():
    bg = BilateralGridOptimizer(3, "cpu", shape=SHAPE, tv_weight=10.0, backend="torch")
    bg.grids.add_(torch.randn(bg.grids.shape, generator=torch.Generator().manual_seed(1)) * 0.1)
    g = bg.grids.clone().requires_grad_(True)
    tv = bo.total_variation(g, 10.0)
    tv.backward()
    assert float(bg.regularize()) == pytest.approx(float(tv), rel=1e-6)
    assert torch.allclose(bg.grids_grad, g.grad, rtol=1e-5, atol=1e-9)
    rows = _rows(3)
    bg.accumulate(torch.tensor([1, 1, 2], dtype=torch.int32), rows)
    assert torch.equal(bg.grids_grad[0], g.grad[0])
    assert torch.equal(bg.grids_grad[1], g.grad[1] + rows[0] + rows[1])
    assert torch.equal(bg.grids_grad[2], g.grad[2] + rows[2])


def test_config_and_trainer_arguments():
    for shape in ((1, 16, 8), (16, 16, 17), (16, 16), (16.0, 16, 8)):
        with pytest.raises(ValueError):
            TrainConfig(use_bilateral_grid=True, bilateral_grid_shape=shape)
    with pytest.raises(ValueError):
        TrainConfig(use_bilateral_grid=True, bilateral_grid_lr_final=0.0)
    TrainConfig(bilateral_grid_shape=(1, 1, 1))  # not checked while the grid is off
    with pytest.raises(ValueError, match="num_cameras"):
        SplatTrainer(*_gaussians(8), cfg=TrainConfig(use_bilateral_grid=True), backend="torch")
    tr = SplatTrainer(*_gaussians(8), cfg=TrainConfig(use_bilateral_grid=True, bilateral_grid_shape=SHAPE), backend="torch", num_cameras=3)
    assert tr.bilateral_grids.shape == (3, 12, 5, 3, 4) and tr.bilagrid_tv_loss.shape == (1,)
    with pytest.raises(ValueError, match="camera_ids"):
        tr.bilagrid_update(_rows(1), torch.tensor([3]))  # outside [0, num_cameras)
    off = SplatTrainer(*_gaussians(8), backend="torch")
    assert off.bilateral_grids is None and off.bilagrid_tv_loss is None


def _cfg():
    return TrainConfig(use_bilateral_grid=True, bilateral_grid_shape=SHAPE, bilateral_grid_warmup=0, bilateral_grid_lr=1e-2)


def _gloo_worker(rank, world, port, tmp):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    tr = SplatTrainer(*_gaussians(16), cfg=_cfg(), rank=rank, world_size=world, backend="torch", num_cameras=3)
    rows, ids = _rows(2), torch.tensor([2, 0])
    grads = []
    for it in range(3):
        sl = slice(rank, rank + 1)  # rank r holds view r
        tr.bilagrid_update(rows[sl] * (it + 1), ids[sl])
        grads.append(tr.bilagrid.grad.clone())
        tr.step_count += 1
    torch.save({"grids": tr.bilateral_grids.clone(), "grads": grads, "tv": tr.bilagrid_tv_loss.clone()}, os.path.join(tmp, f"r{rank}.pt"))
    dist.barrier()
    dist.destroy_process_group()


def test_gloo_world2_grids_identical_and_equal_single_rank(tmp_path):
    world, port = 2, 29500 + (os.getpid() + 13) % 2000
    mp.spawn(_gloo_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    r0, r1 = (torch.load(tmp_path / f"r{r}.pt") for r in range(world))
    assert torch.equal(r0["grids"], r1["grids"]) and torch.equal(r0["tv"], r1["tv"])
    assert all(torch.equal(a, b) for a, b in zip(r0["grads"], r1["grads"]))
    single = SplatTrainer(*_gaussians(16), cfg=_cfg(), backend="torch", num_cameras=3)
    rows, ids = _rows(2), torch.tensor([2, 0])
    for it in range(3):
        single.bilagrid_update(rows * (it + 1), ids)
        assert torch.equal(single.bilagrid.grad, r0["grads"][it]), it  # the same rows in the same order
        single.step_count += 1
    assert torch.equal(single.bilateral_grids, r0["grids"])
    assert float((single.bilateral_grids[1] - bo.identity_grids(1, *SHAPE)[0]).abs().max()) == 0.0  # no view, identity: TV 0
