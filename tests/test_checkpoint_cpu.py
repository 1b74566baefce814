"""CPU: SplatTrainer.state_dict() / SplatTrainer.from_state_dict() on the trainer's host logic (torch backend) -- a run saved,
written with torch.save, read with torch.load(weights_only=True) and resumed continues bit for bit like the uninterrupted
run (DefaultStrategy across grow / split / prune and an opacity reset, MCMC across relocation and growth, the camera
optimizer and the bilateral grid across a resolution change); the gloo world-size-2 path saves every rank's statistics
and restores them row by row, and states move between world sizes 1 and 2; state_dict() changes nothing and returns
tensors that own their storage; layout changes and malformed states raise ValueError; the Gaussians build splatfacto's
model."""
import copy
import dataclasses
import io
import os
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from qed_splatter_b200.trainer import GROUPS, SPLATFACTO_SHAPES, SplatTrainer, TrainConfig

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W, H = 64, 48
GRID = (4, 3, 5)  # (X, Y, L): small grids keep the tests fast
NUM_CAMERAS = 3

# refine at steps 3, 9, 15 (paused after the opacity resets at 0, 6, 12); a scene scale that makes ~20 % of the Gaussians
# "small" (duplicated when hot); screen-size pruning from step 7 on
DEFAULT = dict(warmup_length=2, refine_every=3, reset_alpha_every=2, pause_refine_after_reset=3, scene_scale=3.0)
# relocate + add at steps 3, 6, 9, 12; opacities clamped to min_opacity by a relocation are dead at the next one
MCMC = dict(strategy="mcmc", max_gs_num=90, warmup_length=1, refine_every=3, cull_alpha_thresh=0.2)
# the two tables, warm-ups short enough to move them, 1/2 resolution for steps 0-3 and full resolution from step 4
TABLES = dict(DEFAULT, warmup_length=1, camera_optimizer="SO3xR3", camera_opt_warmup=2, use_bilateral_grid=True, bilateral_grid_shape=GRID,
              bilateral_grid_warmup=2, num_downscales=1, resolution_schedule=4)


def _params(N=64, seed=0):
    g = torch.Generator().manual_seed(seed)
    means = torch.randn(N, 3, generator=g)
    quats = torch.randn(N, 4, generator=g)
    log_scales = torch.log(torch.rand(N, 3, generator=g) * 0.05 + 0.001)
    logit_op = torch.logit(torch.rand(N, generator=g) * 0.9 + 0.05)
    logit_op[::11] = -8.0  # pruned by DefaultStrategy, dead for MCMC
    sh = torch.randn(N, 16, 3, generator=g)
    return means, quats, log_scales, logit_op, sh


def _trainer(cfg, rank=0, world=1):
    return SplatTrainer(*_params(), cfg=TrainConfig(**cfg), rank=rank, world_size=world, backend="torch", num_cameras=NUM_CAMERAS)


def host_step(tr, rank=0):
    """One step of SplatTrainer.step's host logic on synthetic inputs seeded from (rank, step): the Gaussian gradients, the
    statistics at the step's render size, the camera and grid tables, the sum over the ranks and Adam, refine."""
    g = torch.Generator().manual_seed(1000 * tr.step_count + rank)
    a = tr.arena
    for name in GROUPS:
        v = a.view(a.grad, name)
        v.copy_(torch.randn(v.shape, generator=g) * 1e-3 / tr.world)
    if tr.mcmc is None:
        d = tr.downscale_factor()
        absgrad = torch.rand(1, a.N, 2, generator=g) ** 4 * 4e-5
        radii = torch.randint(0, 4, (1, a.N), generator=g, dtype=torch.int32)
        radii[torch.rand(1, a.N, generator=g) < 0.02] = 12  # split, and from step 7 on pruned as too large on screen
        tr.accumulate_stats(absgrad, radii, W // d, H // d, packed=False, n_cameras=tr.world)
    ids = torch.randint(0, NUM_CAMERAS, (1,), generator=g)
    if tr.camera_opt is not None:
        c2w = torch.eye(4)[None, :3].clone()
        c2w[0, :, 3] = torch.tensor([0.1, -0.2, 3.0])
        tr.camera_opt_update(torch.randn(1, 4, 4, generator=g) * 1e-2, ids, c2w)
    if tr.bilagrid is not None:
        X, Y, L = GRID
        tr.bilagrid_update(torch.randn(1, 12, L, Y, X, generator=g) * 1e-3, ids)
    tr._gaussian_update(False, False, [])
    info = tr.maybe_refine(tr.step_count)
    tr.step_count += 1
    return info


def _through_file(state):
    buf = io.BytesIO()
    torch.save(state, buf)
    buf.seek(0)
    return torch.load(buf, weights_only=True)


def _tensors(state, prefix=""):
    """{dotted key: tensor} of every tensor in a state dict."""
    out = {}
    for k, v in state.items():
        if isinstance(v, dict):
            out.update(_tensors(v, f"{prefix}{k}."))
        elif isinstance(v, torch.Tensor):
            out[prefix + k] = v
    return out


def _bits(t):
    return t.contiguous().view(torch.int32) if t.dtype == torch.float32 else t


def assert_states_equal(a, b):
    ta, tb = _tensors(a), _tensors(b)
    assert ta.keys() == tb.keys()
    for k in ta:
        assert ta[k].dtype == tb[k].dtype and ta[k].shape == tb[k].shape, k
        assert torch.equal(_bits(ta[k]), _bits(tb[k])), k
    plain = {k: v for k, v in a.items() if not isinstance(v, (dict, torch.Tensor))}
    assert plain == {k: v for k, v in b.items() if not isinstance(v, (dict, torch.Tensor))}
    assert a["config"] == b["config"]


def _resume(tr, rank=0, world=1):
    return SplatTrainer.from_state_dict(_through_file(tr.state_dict()), rank=rank, world_size=world, backend="torch")


@pytest.mark.parametrize("name,cfg,K", [("default", DEFAULT, 7), ("mcmc", MCMC, 5), ("tables", TABLES, 3)])
def test_resume_is_bitwise_the_uninterrupted_run(name, cfg, K):
    a = _trainer(cfg)
    infos_a = [host_step(a) for _ in range(2 * K)]
    b = _trainer(cfg)
    infos_b = [host_step(b) for _ in range(K)]
    b = _resume(b)
    assert b.step_count == K
    infos_b += [host_step(b) for _ in range(K)]
    assert infos_a == infos_b
    assert_states_equal(a.state_dict(), b.state_dict())
    after = [i for i in infos_a[K:] if i is not None]
    assert after, "the window after the resume must hold a refine step"
    if name == "default":
        i = after[0]
        assert i["n_dupli"] > 0 and i["n_split"] > 0 and i["n_prune"] > 0, infos_a
        assert any(s % 6 == 0 for s in range(K, 2 * K))  # an opacity reset after the resume
        assert float(a.state.count.sum()) > 0  # statistics in flight at the end as well
    if name == "mcmc":
        assert any(i["n_relocated"] > 0 for i in after) and any(i["n_added"] > 0 for i in after), infos_a
        assert a.arena.N > 64
    if name == "tables":
        assert b.downscale_factor() == 1 and _trainer(cfg).downscale_factor() == 2  # crossed the resolution change
        assert float(a.pose_adjustment.abs().max()) > 0 and float((a.bilateral_grids[0, 0, 0] - 1).abs().max()) > 0
        assert after[0]["n"] != 64


def test_state_dict_changes_nothing_and_owns_its_storage():
    cfg = TABLES
    live, twin = _trainer(cfg), _trainer(cfg)
    for _ in range(5):
        host_step(live)
        host_step(twin)

    def snapshot(tr):
        s = {f"arena.{k}": getattr(tr.arena, k).clone() for k in ("param", "grad", "exp_avg", "exp_avg_sq")}
        s.update({f"state.{k}": getattr(tr.state, k).clone() for k in ("grad2d", "count", "radii")})
        for t in ("camera_opt", "bilagrid"):
            s.update({f"{t}.{k}": getattr(getattr(tr, t), k).clone() for k in ("param", "grad", "exp_avg", "exp_avg_sq")})
        return s, (tr.step_count, tr.arena.N, dataclasses.asdict(tr.cfg))

    before = snapshot(live)
    state = live.state_dict()
    after = snapshot(live)
    assert before[1] == after[1]
    for k in before[0]:
        assert torch.equal(_bits(before[0][k]), _bits(after[0][k])), k
    for k, t in _tensors(state).items():
        assert t.device.type == "cpu" and t.is_contiguous() and t.storage_offset() == 0, k
        assert t.untyped_storage().nbytes() == t.numel() * t.element_size(), k  # not a view into a larger buffer
    for v in state.values():  # plain values only: weights_only loading rejects class instances
        assert isinstance(v, (int, dict))
    host_step(live)
    host_step(twin)
    assert_states_equal(live.state_dict(), twin.state_dict())


def test_state_keys_and_shapes():
    tr = _trainer(TABLES)
    for _ in range(2):
        host_step(tr)
    s = tr.state_dict()
    N = tr.arena.N
    assert s["format_version"] == 1 and s["step"] == 2 and s["num_cameras"] == NUM_CAMERAS and s["world_size"] == 1
    assert s["config"] == dataclasses.asdict(tr.cfg)
    for key in ("gauss_params", "exp_avg", "exp_avg_sq"):
        assert {k: tuple(v.shape) for k, v in s[key].items()} == {k: (N, *v) for k, v in SPLATFACTO_SHAPES.items()}
    assert {k: tuple(v.shape) for k, v in s["strategy_state"].items()} == {k: (1, N) for k in ("grad2d", "count", "radii")}
    assert {k: tuple(v.shape) for k, v in s["camera_optimizer"].items()} == {k: (NUM_CAMERAS, 6) for k in ("pose_adjustment", "exp_avg", "exp_avg_sq")}
    X, Y, L = GRID
    assert {k: tuple(v.shape) for k, v in s["bil_grids"].items()} == {k: (NUM_CAMERAS, 12, L, Y, X) for k in ("grids", "exp_avg", "exp_avg_sq")}
    sh = tr.arena.view(tr.arena.param, "sh")
    assert torch.equal(s["gauss_params"]["features_dc"], sh[:, 0]) and torch.equal(s["gauss_params"]["features_rest"], sh[:, 1:])
    assert torch.equal(s["gauss_params"]["opacities"][:, 0], tr.arena.view(tr.arena.param, "opacities"))
    m = _trainer(MCMC).state_dict()
    assert "strategy_state" not in m and "camera_optimizer" not in m and "bil_grids" not in m


def test_splatfacto_model_takes_the_gaussians():
    tr = _trainer(DEFAULT)
    for _ in range(4):  # a refine step (3) changed N
        host_step(tr)
    assert tr.arena.N != 64
    state = _through_file(tr.state_dict())
    stubs = os.path.join(ROOT, "tests", "stubs")
    sys.path.insert(0, stubs)
    try:
        from nerfstudio.models.splatfacto import SplatfactoModel, SplatfactoModelConfig

        model = SplatfactoModel(SplatfactoModelConfig(), gauss_params=state["gauss_params"])
    finally:
        sys.path.remove(stubs)
        for k in [k for k in sys.modules if k == "nerfstudio" or k.startswith("nerfstudio.")]:
            del sys.modules[k]
    assert model.num_points == tr.arena.N
    for k, v in tr.arena.splatfacto_views(tr.arena.param).items():
        assert torch.equal(model.gauss_params[k].detach(), v), k


def test_validation():
    tr = _trainer(TABLES)
    host_step(tr)
    s = tr.state_dict()
    ok = SplatTrainer.from_state_dict(s, TrainConfig(**dict(TABLES, max_steps=5000, lr_means=1e-3, comm="nccl")), backend="torch")
    assert ok.cfg.max_steps == 5000 and ok.step_count == 1
    for field, value in (("strategy", "mcmc"), ("camera_optimizer", "off"), ("use_bilateral_grid", False), ("bilateral_grid_shape", (4, 4, 4))):
        with pytest.raises(ValueError, match=field):
            SplatTrainer.from_state_dict(s, TrainConfig(**dict(TABLES, **{field: value})), backend="torch")
    for version in (0, 2, None):
        with pytest.raises(ValueError, match="format_version"):
            SplatTrainer.from_state_dict(dict(s, format_version=version), backend="torch")
    N = tr.arena.N
    bad_shapes = [("gauss_params", "quats", (N - 1, 4)), ("exp_avg", "features_rest", (N, 16, 3)), ("exp_avg_sq", "opacities", (N,)),
                  ("strategy_state", "count", (2, N)), ("camera_optimizer", "exp_avg", (NUM_CAMERAS + 1, 6)),
                  ("bil_grids", "grids", (NUM_CAMERAS, 12, 5, 3, 3))]
    for key, k, shape in bad_shapes:
        bad = copy.deepcopy(s)
        bad[key][k] = torch.zeros(shape)
        with pytest.raises(ValueError, match=f"{key}\\['{k}'\\]"):
            SplatTrainer.from_state_dict(bad, backend="torch")
    bad = copy.deepcopy(s)
    bad["num_cameras"] = NUM_CAMERAS + 1  # the tables disagree with it
    with pytest.raises(ValueError, match="camera_optimizer"):
        SplatTrainer.from_state_dict(bad, backend="torch")
    m = _trainer(MCMC)
    host_step(m)
    ms = m.state_dict()
    with pytest.raises(ValueError, match="max_gs_num"):
        SplatTrainer.from_state_dict(ms, TrainConfig(**dict(MCMC, max_gs_num=m.arena.N - 1)), backend="torch")
    SplatTrainer.from_state_dict(ms, TrainConfig(**dict(MCMC, max_gs_num=m.arena.N)), backend="torch")


# -- gloo, world size 2 ------------------------------------------------------------------------------
K2 = 7  # DEFAULT: statistics of steps 4-6 in flight at the save, refine at 9


def _gloo_worker(rank, world, port, tmp):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    a = _trainer(DEFAULT, rank, world)
    infos_a = [host_step(a, rank) for _ in range(2 * K2)]
    b = _trainer(DEFAULT, rank, world)
    infos_b = [host_step(b, rank) for _ in range(K2)]
    mid = b.state_dict()
    b = SplatTrainer.from_state_dict(_through_file(mid), rank=rank, world_size=world, backend="torch")
    infos_b += [host_step(b, rank) for _ in range(K2)]
    # a world-size-1 state opened by two ranks
    one = SplatTrainer.from_state_dict(torch.load(os.path.join(tmp, "w1.pt"), weights_only=True), rank=rank, world_size=world, backend="torch")
    torch.save({"mid": mid, "a": a.state_dict(), "b": b.state_dict(), "infos_a": infos_a, "infos_b": infos_b,
                "from_w1": {k: getattr(one.state, k).clone() for k in ("grad2d", "count", "radii")}}, os.path.join(tmp, f"r{rank}.pt"))
    dist.barrier()
    dist.destroy_process_group()


def test_gloo_world2_resume_and_other_world_sizes(tmp_path):
    single = _trainer(DEFAULT)
    for _ in range(K2):
        host_step(single)
    w1 = single.state_dict()
    torch.save(w1, tmp_path / "w1.pt")
    world, port = 2, 29500 + (os.getpid() + 517) % 2000
    mp.spawn(_gloo_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    r0, r1 = (torch.load(tmp_path / f"r{r}.pt", weights_only=True) for r in range(world))
    # the ranks' statistics differ and both rows are saved, identically on every rank
    mid = r0["mid"]
    assert mid["world_size"] == 2
    assert_states_equal(mid, r1["mid"])
    for k in ("grad2d", "count", "radii"):
        assert mid["strategy_state"][k].shape[0] == 2 and not torch.equal(mid["strategy_state"][k][0], mid["strategy_state"][k][1]), k
    # resumed at world size 2: bit for bit the uninterrupted run, replicas bit-identical
    for r in (r0, r1):
        assert r["infos_a"] == r["infos_b"] and any(i is not None and i["n"] != 64 for i in r["infos_a"][K2:])
        assert_states_equal(r["a"], r["b"])
    assert_states_equal(r0["b"], r1["b"])
    # the world-2 state at world size 1: rank 0 holds SUM / SUM / MAX of the rows
    tr = SplatTrainer.from_state_dict(mid, backend="torch")
    rows = mid["strategy_state"]
    assert torch.equal(tr.state.grad2d, rows["grad2d"][0] + rows["grad2d"][1])
    assert torch.equal(tr.state.count, rows["count"][0] + rows["count"][1])
    assert torch.equal(tr.state.radii, torch.maximum(rows["radii"][0], rows["radii"][1]))
    # the world-1 state at world size 2: rank 0 holds everything, rank 1 zeros
    for k in ("grad2d", "count", "radii"):
        assert torch.equal(r0["from_w1"][k], w1["strategy_state"][k][0]) and float(w1["strategy_state"][k].abs().sum()) > 0, k
        assert float(r1["from_w1"][k].abs().sum()) == 0.0 and r1["from_w1"][k].numel() == w1["strategy_state"][k].shape[1], k
