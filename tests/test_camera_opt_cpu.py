"""CPU: splatfacto's SO3xR3 camera optimizer -- the float64 reference restatement (tests/camera_opt_oracle.py) against finite
differences through exp map -> compose -> get_viewmat -> render, the identity at a zero table and the clamp, the regulariser,
the lr schedule, the table Adam against torch.optim.Adam, and the world-2 gloo path of the trainer (torch backend)."""
import math
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import camera_opt_oracle as co
import oracle
from qed_splatter_b200 import camera_opt
from qed_splatter_b200.camera_opt import CameraPoseOptimizer, check_camera_ids
from qed_splatter_b200.scenes import camera_to_worlds
from qed_splatter_b200.trainer import SplatTrainer, TrainConfig
from test_oracle import _tiny
from test_pose_grad_cpu import _fd_check


def _adj(n, scale, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(n, 6, generator=g, dtype=torch.float64) * scale).contiguous()


@pytest.mark.parametrize("rot_scale", [0.02, 1e-3])  # |omega| above and below the 1e-2 clamp of theta
def test_pose_table_autograd_vs_finite_differences(rot_scale):
    s, a = _tiny(N=8, C=2, size=24, seed=5)
    c2w = camera_to_worlds(a["viewmats"])
    ids = torch.tensor([1, 1])  # both views share a table row; row 0 gets no gradient
    g = torch.Generator().manual_seed(9)
    adj = _adj(3, 1.0, 2) * torch.tensor([0.01] * 3 + [rot_scale] * 3, dtype=torch.float64)
    r0, al0, _ = oracle.rasterization(**a, width=s.width, height=s.height, sh_degree=3, render_mode="RGB+ED")
    wr = torch.randn(r0.shape, generator=g, dtype=torch.float64)
    wa = torch.randn(al0.shape, generator=g, dtype=torch.float64)

    def f(x):
        r, al, _ = oracle.rasterization(**{**a, "viewmats": co.viewmats(c2w, ids, x)}, width=s.width, height=s.height, sh_degree=3,
                                        render_mode="RGB+ED")
        return (r * wr).sum() + (al * wa).sum() + co.regularizer(x)

    grad = _fd_check(f, adj, g, eps=1e-7)
    assert float(grad[1].abs().max()) > 0


def test_zero_table_is_identity_and_clamp():
    c2w = camera_to_worlds(_tiny(N=4, C=3)[1]["viewmats"])
    ids = torch.tensor([0, 2, 1])
    zero = torch.zeros(3, 6, dtype=torch.float64)
    assert torch.equal(co.exp_map(zero), torch.eye(3, dtype=torch.float64).expand(3, 3, 3))
    assert torch.equal(co.adjusted_c2w(c2w, ids, zero), c2w)
    assert torch.equal(camera_opt.exp_map_so3xr3(zero)[:, :, :3], co.exp_map(zero))
    # at zero theta is clamped to 0.01: dR / d omega_m = sin(0.01) / 0.01 [e_m]x (the K^2 term is quadratic)
    J = torch.autograd.functional.jacobian(lambda x: co.exp_map(x[None])[0], torch.zeros(6, dtype=torch.float64))
    fac = math.sin(0.01) / 0.01
    for m in range(3):
        e = torch.zeros(3, dtype=torch.float64)
        e[m] = 1.0
        skew = torch.tensor([[0, -e[2], e[1]], [e[2], 0, -e[0]], [-e[1], e[0], 0]], dtype=torch.float64)
        assert torch.allclose(J[:, :, 3 + m], fac * skew, atol=1e-15)
        assert torch.equal(J[:, :, m], torch.zeros(3, 3, dtype=torch.float64))
    # below the clamp theta is constant: R = I + A K + B K^2 with A, B at theta = 0.01
    w = torch.tensor([0.003, -0.004, 0.002], dtype=torch.float64)
    adj = torch.cat([torch.zeros(3, dtype=torch.float64), w])[None]
    K = torch.tensor([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]], dtype=torch.float64)
    R = torch.eye(3, dtype=torch.float64) + fac * K + (1 - math.cos(0.01)) / 1e-4 * K @ K
    assert torch.allclose(co.exp_map(adj)[0], R, atol=1e-16)
    # the torch backend and the restatement agree
    adj = _adj(3, 0.05, 4)
    assert torch.allclose(camera_opt.viewmats_torch(c2w, ids, adj), co.viewmats(c2w, ids, adj), atol=1e-14)


def test_regularizer_gradient():
    adj = _adj(5, 0.1, 6)
    adj[2, :3] = 0.0  # zero norms: gradient 0, as in torch
    adj[4, 3:] = 0.0
    cam = CameraPoseOptimizer(5, "cpu", backend="torch")
    cam.pose_adjustment.copy_(adj.float())
    ref_adj = cam.pose_adjustment.detach().double().requires_grad_(True)
    ref = co.regularizer(ref_adj)
    ref.backward()
    val = cam.regularize()
    assert float(val) == pytest.approx(float(ref.detach()), rel=1e-6)
    assert torch.allclose(cam.pose_grad.double(), ref_adj.grad, rtol=1e-6, atol=1e-12)
    assert torch.equal(cam.pose_grad[2, :3], torch.zeros(3)) and torch.equal(cam.pose_grad[4, 3:], torch.zeros(3))
    assert float(cam.pose_grad[2, 3:].abs().sum()) > 0


def test_schedule_endpoints():
    cfg = TrainConfig()
    assert (cfg.camera_opt_lr, cfg.camera_opt_lr_final, cfg.camera_opt_warmup) == (1e-4, 5e-7, 1000)
    lr = lambda t: camera_opt.lr_at(t, cfg.camera_opt_lr, cfg.camera_opt_lr_final, cfg.camera_opt_warmup, cfg.max_steps)
    assert lr(0) == 0.0 and lr(500) == pytest.approx(1e-4 * math.sin(math.pi / 4))
    assert lr(1000) == pytest.approx(1e-4) and lr(30000) == pytest.approx(5e-7) and lr(40000) == pytest.approx(5e-7)
    assert lr(15500) == pytest.approx(math.sqrt(1e-4 * 5e-7))
    assert camera_opt.lr_at(10, 0.0, 5e-7, 0, 100) == 0.0


def test_config_and_trainer_arguments():
    with pytest.raises(ValueError):
        TrainConfig(camera_optimizer="SE3")
    cfg = TrainConfig()
    cfg.camera_optimizer = "off_by_one"
    with pytest.raises(ValueError):
        SplatTrainer(*_gaussians(8), cfg=cfg, backend="torch")
    with pytest.raises(ValueError):
        SplatTrainer(*_gaussians(8), cfg=TrainConfig(camera_optimizer="SO3xR3"), backend="torch")  # num_cameras missing
    tr = SplatTrainer(*_gaussians(8), cfg=TrainConfig(camera_optimizer="SO3xR3"), backend="torch", num_cameras=3)
    assert tr.pose_adjustment.shape == (3, 6) and float(tr.pose_adjustment.abs().sum()) == 0.0
    assert SplatTrainer(*_gaussians(8), backend="torch").pose_adjustment is None
    with pytest.raises(ValueError):
        check_camera_ids(torch.tensor([0, 3]), 2, 3, torch.device("cpu"))
    with pytest.raises(ValueError):
        check_camera_ids(torch.tensor([-1, 0]), 2, 3, torch.device("cpu"))
    with pytest.raises(ValueError):
        check_camera_ids(torch.tensor([0]), 2, 3, torch.device("cpu"))
    with pytest.raises(TypeError):
        check_camera_ids(torch.tensor([0.0, 1.0]), 2, 3, torch.device("cpu"))


def test_table_adam_matches_torch_optim():
    cam = CameraPoseOptimizer(4, "cpu", lr=1e-3, lr_final=1e-5, warmup_steps=3, max_steps=10, backend="torch")
    ref = torch.zeros(4, 6, requires_grad=True)
    opt = torch.optim.Adam([ref], lr=1.0, eps=1e-15)
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lambda t: cam.lr_at(t))
    g = torch.Generator().manual_seed(1)
    for t in range(8):
        grad = torch.randn(4, 6, generator=g) * 1e-2
        grad[t % 4] = 0.0  # a row without a view this step still moves by momentum
        cam.grad.zero_()
        cam.pose_grad.copy_(grad)
        ref.grad = grad.clone()
        opt.step()
        sched.step()
        cam.step(t)
        assert torch.allclose(cam.pose_adjustment, ref.detach(), rtol=1e-5, atol=1e-9), t
    assert float(cam.pose_adjustment.abs().min()) > 0


def _gaussians(N, seed=0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(N, 3, generator=g), torch.randn(N, 4, generator=g), torch.log(torch.rand(N, 3, generator=g) * 0.05 + 0.001),
            torch.logit(torch.rand(N, generator=g) * 0.9 + 0.05), torch.randn(N, 16, 3, generator=g))


def _views(seed=11):
    """Two views on cameras 2 and 0 of a 3-camera table, with stand-in viewmat gradients of a loss averaged over both."""
    g = torch.Generator().manual_seed(seed)
    c2w = camera_to_worlds(_tiny(N=4, C=2)[1]["viewmats"]).float()
    v = torch.randn(2, 4, 4, generator=g) * 0.5
    v[:, 3] = 0.0
    return c2w, torch.tensor([2, 0]), v


def _gloo_worker(rank, world, port, tmp):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    c2w, ids, v = _views()
    tr = SplatTrainer(*_gaussians(16), cfg=TrainConfig(camera_optimizer="SO3xR3", camera_opt_warmup=0, camera_opt_lr=1e-3), rank=rank,
                      world_size=world, backend="torch", num_cameras=3)
    grads = []
    for it in range(3):
        sl = slice(rank, rank + 1)  # rank r holds view r; its v_viewmats already carry 1 / total_views
        tr.camera_opt_update(v[sl] * (it + 1), ids[sl], c2w[sl])
        grads.append(tr.camera_opt.grad.clone())
        tr.step_count += 1
    torch.save({"table": tr.pose_adjustment.clone(), "grads": grads, "reg": tr.camera_opt_loss.clone()}, os.path.join(tmp, f"r{rank}.pt"))
    dist.barrier()
    dist.destroy_process_group()


def test_gloo_world2_pose_tables_identical_and_equal_single_rank(tmp_path):
    world, port = 2, 29500 + (os.getpid() + 7) % 2000
    mp.spawn(_gloo_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    r0, r1 = (torch.load(tmp_path / f"r{r}.pt") for r in range(world))
    assert torch.equal(r0["table"], r1["table"]) and torch.equal(r0["reg"], r1["reg"])
    assert all(torch.equal(a, b) for a, b in zip(r0["grads"], r1["grads"]))
    c2w, ids, v = _views()
    single = SplatTrainer(*_gaussians(16), cfg=TrainConfig(camera_optimizer="SO3xR3", camera_opt_warmup=0, camera_opt_lr=1e-3), backend="torch",
                          num_cameras=3)
    for it in range(3):
        single.camera_opt_update(v * (it + 1), ids, c2w)
        assert torch.allclose(single.camera_opt.grad, r0["grads"][it], rtol=1e-6, atol=1e-9), it
        single.step_count += 1
    assert torch.allclose(single.pose_adjustment, r0["table"], rtol=1e-5, atol=1e-9)
    # camera 1 has no view and a zero row: the regulariser's gradient is zero there too, so Adam leaves it at zero
    assert torch.equal(single.pose_adjustment[1], torch.zeros(6)) and float(single.pose_adjustment[[0, 2]].abs().min()) > 0
