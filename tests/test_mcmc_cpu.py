"""CPU: splatfacto's MCMC strategy (qed_splatter_b200/mcmc.py, impl="torch") against tests/mcmc_oracle.py -- the relocation
arithmetic, the schedule, the growth sequence, relocate / add on given draws, noise and regularisers -- the config checks, the
numpy Philox restatement, and a gloo world-size-2 trainer whose replicas stay bit-identical through refine and noise steps."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import mcmc_oracle as mo
from qed_splatter_b200 import mcmc
from qed_splatter_b200.trainer import GROUPS, GaussianArena, SplatTrainer, TrainConfig


def _params(N, seed=0, op_lo=0.05, op_hi=0.95):
    g = torch.Generator().manual_seed(seed)
    means = torch.randn(N, 3, generator=g)
    quats = torch.randn(N, 4, generator=g)
    log_scales = torch.log(torch.rand(N, 3, generator=g) * 0.05 + 0.001)
    logit_op = torch.logit(torch.rand(N, generator=g) * (op_hi - op_lo) + op_lo)
    sh = torch.randn(N, 16, 3, generator=g)
    return means, quats, log_scales, logit_op, sh


def _np(arena, buf):
    return {g: arena.view(buf, g).double().numpy().copy() for g in GROUPS}


@pytest.mark.parametrize("n", range(1, 52))
def test_identity_matches_double_loop(n):
    B = mo.binoms()
    for o in (1e-6, 0.01, 0.5, 0.9, 1 - 6e-8):  # x = o' of an opacity up to float32's 1 - 2^-24
        x = 1.0 - (1.0 - o) ** (1.0 / n)
        loop = sum(B[i - 1, k] * (-1.0) ** k / np.sqrt(k + 1.0) * x ** (k + 1) for i in range(1, n + 1) for k in range(i))
        assert mo.denominator_identity(x, n) == pytest.approx(loop, rel=1e-11)
        t = mcmc.relocation_denominator(torch.tensor([x], dtype=torch.float64), torch.tensor([n]))
        assert float(t) == pytest.approx(loop, rel=1e-11)


def test_relocation_values():
    o = np.array([0.01, 0.2, 0.5, 0.9, 0.999, 1 - 1e-7])
    for n in (1, 2, 5, 51):
        o_new, s_new = mo.compute_relocation(o, np.ones((o.size, 3)), np.full(o.size, n))
        assert np.allclose(1 - (1 - o_new) ** n, o, rtol=1e-12)  # n copies at o' composite to the old opacity
        if n == 1:  # ratio 1 is the identity
            assert np.allclose(o_new, o, rtol=1e-15) and np.allclose(s_new, 1.0, rtol=1e-12)
        # the float32 path against the loop on the same float32 opacities
        o32 = o.astype(np.float32)
        t_o, t_s = mcmc.relocation_values(torch.tensor(o32), torch.ones(o.size, 3), torch.full((o.size,), n), 0.005)
        r_o, r_s = mo.compute_relocation(o32, np.ones((o.size, 3)), np.full(o.size, n))
        assert np.allclose(t_o.numpy(), np.clip(r_o.astype(np.float32), 0.005, 1 - mo.FLT_EPS), rtol=1e-6)
        assert np.allclose(t_s.numpy(), r_s, rtol=1e-6)
    # ratios above 51 are clamped (gsplat's n_max)
    a = mcmc.relocation_values(torch.tensor([0.5]), torch.ones(1, 3), torch.tensor([51]), 0.005)
    b = mcmc.relocation_values(torch.tensor([0.5]), torch.ones(1, 3), torch.tensor([80]), 0.005)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_config_validation():
    assert TrainConfig().strategy == "default"
    c = TrainConfig(strategy="mcmc")
    assert (c.max_gs_num, c.noise_lr, c.mcmc_opacity_reg, c.mcmc_scale_reg) == (1_000_000, 5e5, 0.01, 0.01)
    for bad in (dict(strategy="abc"), dict(strategy="mcmc", max_gs_num=0), dict(noise_lr=-1.0), dict(mcmc_opacity_reg=-0.1),
                dict(mcmc_scale_reg=-1e-3), dict(strategy="mcmc", cull_alpha_thresh=0.0)):
        with pytest.raises(ValueError):
            TrainConfig(**bad)
    c = TrainConfig()
    c.strategy = "nope"
    with pytest.raises(ValueError):
        SplatTrainer(*_params(8), cfg=c, backend="torch")


def test_refine_schedule_and_noise_every_step():
    cfg = TrainConfig(strategy="mcmc", max_gs_num=64)
    tr = SplatTrainer(*_params(40, 1), cfg=cfg, backend="torch")
    steps = (0, 100, 500, 501, 600, 700, 650, 14900, 15000, 15100, 20000)
    fired, moved = [], []
    for s in steps:
        before = tr.arena.view(tr.arena.param, "means").clone()
        info = tr.maybe_refine(s)
        fired.append(info is not None)
        moved.append(not torch.equal(before, tr.arena.view(tr.arena.param, "means")[:before.shape[0]]))
    assert fired == [False, False, False, False, True, True, False, True, False, False, False]
    assert all(moved)  # position noise on every step, also after stop_split_at
    assert [mcmc.is_refine_step(s, 500, 15000, 100) for s in steps] == fired


def test_growth_sequence_and_cap():
    seq, N = [], 100
    while True:
        n = mcmc.growth(N, 200)
        if not n:
            break
        N += n
        seq.append(N)
    assert seq == [105, 110, 115, 120, 126, 132, 138, 144, 151, 158, 165, 173, 181, 190, 199, 200]
    assert mcmc.growth(200, 200) == 0 and mcmc.growth(250, 200) == 0 and mcmc.growth(19, 10**6) == 0
    assert mcmc.growth(10**6 - 10, 10**6) == 10


def test_relocate_and_add_on_given_draws_match_the_oracle():
    N = 50
    p = _params(N, 2)
    logit_op = p[3]
    logit_op[[3, 7, 11, 20, 42]] = -8.0  # dead: sigmoid < 0.005 by a wide margin
    a = GaussianArena(*p)
    g = torch.Generator().manual_seed(5)
    a.exp_avg.copy_(torch.rand(a.exp_avg.shape, generator=g))
    a.exp_avg_sq.copy_(torch.rand(a.exp_avg_sq.shape, generator=g))
    P, M, V = _np(a, a.param), _np(a, a.exp_avg), _np(a, a.exp_avg_sq)
    strat = mcmc.MCMCStrategy("cpu", cap_max=10**6, impl="torch")
    dead, n_dead = strat.dead_rows(a)
    assert dead.tolist() == [3, 7, 11, 20, 42] and n_dead == 5
    draws = torch.tensor([9, 9, 30, 9, 1], dtype=torch.int32)  # ratio 4 for row 9
    strat.relocate(a, draws, dead)
    mo.relocate(P, M, V, draws.numpy(), dead.numpy(), 0.005)
    for name in GROUPS:
        assert np.allclose(a.view(a.param, name).double().numpy(), P[name], rtol=2e-6, atol=1e-6), name
        assert np.array_equal(a.view(a.exp_avg, name).double().numpy(), M[name]), name
        assert np.array_equal(a.view(a.exp_avg_sq, name).double().numpy(), V[name]), name
    add = torch.tensor([0, 5, 5, 49], dtype=torch.int32)
    strat.add(a, add)
    P2, M2, V2 = mo.sample_add(P, M, V, add.numpy(), 0.005)
    assert a.N == N + 4
    for name in GROUPS:
        assert np.allclose(a.view(a.param, name).double().numpy(), P2[name], rtol=2e-6, atol=1e-6), name
        assert np.array_equal(a.view(a.exp_avg, name).double().numpy(), M2[name]), name
    # draws exclude the dead rows during relocate, and come back as (draws, bincount)
    d, c = strat.draw(a, 200, step=600, stream=mcmc.STREAM_RELOCATE, zero_dead=True)
    assert d.numel() == 200 and torch.equal(c, torch.bincount(d.long(), minlength=a.N).to(torch.int32))
    dead_now = strat.dead_rows(a)[0]
    assert not bool(torch.isin(d, dead_now).any())


def test_noise_and_regularizers_match_the_oracle():
    N = 30
    p = _params(N, 3)
    a = GaussianArena(*p)
    P = _np(a, a.param)
    n = torch.randn(N, 3, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    pv = a.views(a.param)
    mcmc.apply_noise_torch(pv["means"], pv["quats"], pv["scales"], pv["opacities"], n.float(), 1e-4 * 5e5)
    mo.inject_noise(P, n.numpy(), 1e-4 * 5e5)
    assert np.allclose(pv["means"].double().numpy(), P["means"], rtol=1e-5, atol=1e-6)
    strat = mcmc.MCMCStrategy("cpu", impl="torch", opacity_reg=0.01, scale_reg=0.02)
    loss = strat.regularize(a)
    lo, ls, go, gs = mo.regularizers(P["opacities"], P["scales"], 0.01, 0.02)
    assert float(loss[0]) == pytest.approx(lo, rel=1e-6) and float(loss[1]) == pytest.approx(ls, rel=1e-6)
    assert np.allclose(a.view(a.grad, "opacities").double().numpy(), go, rtol=1e-5)
    assert np.allclose(a.view(a.grad, "scales").double().numpy(), gs, rtol=1e-5)


def test_philox_known_answers_and_sampler():
    # Random123 known-answer vectors of philox4x32-10
    out = mo.philox4x32_10(0, 0, 0, 0, 0)
    assert [int(x) for x in out] == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    out = mo.philox4x32_10(0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFFFFFFFFFF)
    assert [int(x) for x in out] == [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]
    o = np.array([0.5, 0.002, 0.9, 1e-30, 0.3])
    logit = np.log(o / (1 - o)).astype(np.float32)  # row 3: weight 0
    d, total = mo.sample(logit, 20000, seed=42, step=7, stream_id=1, zero_dead=True)
    assert total == int(sum(mo.weights(logit, 0.005, True)))
    cnt = np.bincount(d, minlength=5)
    assert cnt[1] == 0 and cnt[3] == 0  # dead / zero weight never drawn
    assert abs(cnt[2] / cnt.sum() - 0.9 / 1.7) < 0.02
    z = mo.normals(20000, 42, 3)
    assert abs(z.mean()) < 0.02 and abs(z.std() - 1) < 0.02


def _worker(rank, world, port, tmp):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    cfg = TrainConfig(strategy="mcmc", max_gs_num=80, warmup_length=1, refine_every=2)
    p = _params(64, 7)
    p[3][::9] = -8.0  # some dead Gaussians
    tr = SplatTrainer(*p, cfg=cfg, rank=rank, world_size=world, backend="torch")
    g = torch.Generator().manual_seed(100 + rank)  # every rank sees different views -> different gradients
    infos = []
    for it in range(7):
        tr.arena.grad.copy_(torch.randn(tr.arena.grad.shape, generator=g) * 1e-3 / world)
        tr._all_reduce(tr.arena.grad)
        tr._mcmc_regularize()
        tr.optimizer_step()
        infos.append(tr.maybe_refine(tr.step_count))
        tr.step_count += 1
    torch.save({"param": tr.arena.param, "m": tr.arena.exp_avg, "v": tr.arena.exp_avg_sq, "N": tr.arena.N, "infos": infos,
                "reg": tr.mcmc_reg_loss.clone()}, os.path.join(tmp, f"r{rank}.pt"))
    dist.barrier()
    dist.destroy_process_group()


def test_gloo_world2_mcmc_replicas_stay_identical(tmp_path):
    world, port = 2, 29500 + (os.getpid() + 711) % 2000
    mp.spawn(_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    r0, r1 = (torch.load(tmp_path / f"r{r}.pt") for r in range(world))
    assert r0["infos"] == r1["infos"] and r0["N"] == r1["N"] == 73  # 64 -> 67 -> 70 -> 73
    refines = [i for i in r0["infos"] if i is not None]
    assert len(refines) == 3 and refines[0]["n_relocated"] > 0 and refines[0]["n_added"] == 3
    for k in ("param", "m", "v", "reg"):
        assert torch.equal(r0[k], r1[k]), k
