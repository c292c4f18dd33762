"""
GPU tests of the MPPI planner (sg_plan_sample / sg_plan_update, VecScenarioEnv.planner / MPPIPlanner): sampling and
the update against the numpy restatement (tests/plan_oracle.py), the planner's rollouts against BranchRollout.run,
the receding horizon across auto-resets, an env left untouched, determinism, no host synchronisation or
allocation, a scene where planning avoids a collision, and the argument checks.  Vehicle scenes take the lean
vehicle kernel, the reference's test scenes the general kernel.
"""
import numpy as np
import pytest
import torch

from scenario_gym_b200 import (BoundingBox, CatalogEntry, Entity, MPPIPlanner, ObsSpec, PolicyAgent, Scenario,
                               Trajectory, VecScenarioEnv, Vehicle, synthetic)
from scenario_gym_b200.env import branch_scatter_index

from plan_oracle import sample, update
from test_branches_gpu import assert_states_equal, policy, state_of, xosc_scenarios

pytestmark = pytest.mark.gpu
OBS = ObsSpec(k_neighbours=4, lookahead=(1.0, 2.0))


def vehicle_env(seed=0, N=6, M=12, T=60, half_extent=25.0, **kw):
    """Vehicle-only scenes, every vehicle a PolicyAgent; scenario n has M - 2 (n % 3) vehicles, so rows are padded."""
    cfg = synthetic.vehicles_config(seed=seed, N=N, M=M, T=T, half_extent=half_extent)
    rows = synthetic.two_knot_rows(cfg).reshape(cfg.N, cfg.M, 2, 7)
    ce = CatalogEntry(None, "car1", "car", "Vehicle", BoundingBox(*synthetic.CAR1_BOX))
    scs = [Scenario([Vehicle(ce, trajectory=Trajectory(rows[n, m]), ref="ego" if m == 0 else f"entity_{m}")
                     for m in range(cfg.M - 2 * (n % 3))]) for n in range(cfg.N)]
    return VecScenarioEnv(scs, create_agent=lambda s, e: PolicyAgent(e), timestep=cfg.dt, obs=OBS, **kw)


def make_env(which):
    if which == "vehicles":
        env = vehicle_env()
        assert (env._slots_host < 0).any()
    else:
        env = VecScenarioEnv(xosc_scenarios(), obs=OBS, terminal_conditions=["max_length", "collision"])
    return env


def warm(env, steps=3):
    o, _ = env.reset()
    for _ in range(steps):
        o, *_ = env.step(policy(o))
    return o


def gather(env, flat, B, H):
    """The flat branch table [B][H][2][N*M] (+1) gathered back to [N, B, H, A, 2] (padding: the trailing element)."""
    idx = torch.from_numpy(branch_scatter_index(env._slots_host, env._engine.M, B, H)).to(flat.device)
    return flat[idx].view(env.N, B, H, env.A, 2)


# ---------------------------------------------------------------------------------------------- sampling
@pytest.mark.parametrize("which", ["vehicles", "xosc"])
def test_sample_against_restatement(which):
    env = make_env(which)
    warm(env)
    B, H, seed, k, sigma = 5, 7, 11, 3, (1.3, 0.2)
    pl = env.planner(B=B, H=H, sigma=sigma, seed=seed)
    br, eng, N, A = pl.branches, env._engine, env.N, env.A
    g = torch.Generator(device="cuda").manual_seed(1)
    mu0 = torch.randn((N, H, A, 2), generator=g, device="cuda", dtype=torch.float64)
    reset = torch.zeros(N, dtype=torch.uint8, device="cuda")
    reset[1::3] = 1
    slots = env._slots_host
    real = slots >= 0
    idx = branch_scatter_index(slots, eng.M, B, H).reshape(N, B, H, A, 2)
    written = torch.zeros(br._flat[torch.float32].numel(), dtype=torch.bool, device="cuda")
    written[torch.from_numpy(idx.transpose(0, 3, 1, 2, 4)[real].reshape(-1)).cuda()] = True
    sent = 123.25  # every entry sg_plan_sample does not write keeps it
    for dt, npdt in ((torch.float32, np.float32), (torch.float64, np.float64)):
        flat = br._flat[dt]
        for sig in (sigma, (0.0, 0.0)):
            flat.fill_(sent)
            mu = mu0.clone()
            eng.plan_sample(env._spec, B, H, seed, k, sig, mu, reset, flat)
            want_mu, want = sample(mu0.cpu().numpy(), reset.cpu().numpy(), slots, B, H, seed, k, sig, npdt)
            _, exact = sample(mu0.cpu().numpy(), reset.cpu().numpy(), slots, B, H, seed, k, sig, np.float64)
            got = gather(env, flat, B, H).cpu().numpy()
            assert np.array_equal(mu.cpu().numpy().transpose(0, 2, 1, 3)[real], want_mu.transpose(0, 2, 1, 3)[real])
            g_r, w_r = got.transpose(0, 3, 1, 2, 4)[real], want.transpose(0, 3, 1, 2, 4)[real]
            x_r = exact.transpose(0, 3, 1, 2, 4)[real]
            assert np.array_equal(g_r[:, 0], w_r[:, 0])  # branch 0 is the mean, exactly
            bad = g_r != w_r
            if bad.any():
                # device log / sincos are within a few ulp of libm.  fp32 table: one ulp, only where the fp64 value
                # lies next to a rounding boundary.  fp64 table: a few ulp of mu and sigma * z (an ulp of the noise
                # term can exceed an ulp of the sum where they cancel)
                gb, wb, xb = g_r[bad].astype(np.float64), w_r[bad].astype(np.float64), x_r[bad]
                if dt == torch.float32:
                    assert (np.abs(gb - wb) <= np.spacing(np.abs(w_r[bad])).astype(np.float64)).all()
                    assert (np.abs(xb - 0.5 * (gb + wb)) <= 1e-12 * np.abs(xb)).all()
                    assert bad.mean() < 1e-3, bad.mean()
                else:
                    m = np.broadcast_to(want_mu.transpose(0, 2, 1, 3)[real][:, None], g_r.shape)[bad]
                    assert (np.abs(gb - wb) <= 1e-14 * (np.abs(m) + np.abs(wb - m))).all()
            if sig == (0.0, 0.0):
                assert np.array_equal(g_r, np.broadcast_to(g_r[:, :1], g_r.shape))  # B copies of the mean
            assert (flat[~written] == sent).all()  # non-agent and padding entries untouched


# ---------------------------------------------------------------------------------------------- rollouts
@pytest.mark.parametrize("which", ["vehicles", "xosc"])
def test_rollouts_equal_branch_run(which):
    env = make_env(which)
    warm(env, 4)
    B, H = 6, 9
    pl = env.planner(B=B, H=H, sigma=(2.0, 0.3), seed=4)
    pl.plan()
    got = {k: v.clone() for k, v in pl.branches._out.items()}
    acts = gather(env, pl._table, B, H).contiguous()
    res = env.branches(B, H).run(acts)
    for k in ("reward", "terms", "terminated", "truncated", "ticks", "agent_mask"):
        assert torch.equal(res[k], got[k]), k


# ---------------------------------------------------------------------------------------------- update
@pytest.mark.parametrize("which", ["vehicles", "xosc"])
def test_update_against_restatement(which):
    env = make_env(which)
    warm(env, 2)
    B, H, lam = 8, 6, 0.5
    pl = env.planner(B=B, H=H, sigma=(2.0, 0.4), temperature=lam, seed=2)
    br, eng, N, A = pl.branches, env._engine, env.N, env.A
    g = torch.Generator(device="cuda").manual_seed(3)
    mu = torch.randn((N, H, A, 2), generator=g, device="cuda", dtype=torch.float64)
    eng.plan_sample(env._spec, B, H, 2, 0, (2.0, 0.4), mu, None, pl._table)
    br._roll(pl._tables)
    R = br._out["reward"].cpu().numpy()
    tab = gather(env, pl._table, B, H).cpu().numpy()
    new, action, shifted, best, rbest = update(mu.cpu().numpy(), tab, R, lam)
    real = env._slots_host >= 0

    def rows(x):  # the real agents' rows of [N, H, A, 2] / [N, A, ...]
        x = x.cpu().numpy() if isinstance(x, torch.Tensor) else x
        return x.transpose(0, 2, 1, 3)[real] if x.ndim == 4 else x[real]

    def close(a, b):
        np.testing.assert_allclose(rows(a), rows(b), rtol=1e-12, atol=1e-12)

    out = torch.full_like(mu, 7.0)
    act = torch.full((N, A, 2), 7.0, device="cuda")
    bb = torch.full((N, A), -7, dtype=torch.int32, device="cuda")
    rb = torch.full((N, A), 7.0, device="cuda")
    eng.plan_update(env._spec, B, H, lam, br._reward, pl._table, mu, out, False, None, bb, rb)
    close(out, new)
    assert np.array_equal(rows(bb), rows(best)) and np.array_equal(rows(rb), rows(rbest))
    assert (out.cpu().numpy().transpose(0, 2, 1, 3)[~real] == 7.0).all()  # padding agents are left alone
    refined = out.clone()
    eng.plan_update(env._spec, B, H, lam, br._reward, pl._table, mu, out, True, act, bb, rb)
    close(out, shifted)
    assert (rows(out)[:, -1] == 0).all()
    assert np.array_equal(rows(act), rows(refined[:, 0].float()))  # the first action of the refined mean
    assert (act.cpu().numpy()[~real] == 7.0).all()


# ---------------------------------------------------------------------------------------------- receding horizon
def test_receding_horizon_and_resets():
    env = vehicle_env(seed=5, N=8, M=8, T=12, half_extent=30.0)  # short episodes: auto-resets within 40 steps
    B, H, sigma, seed = 4, 5, (1.5, 0.2), 9
    pl = env.planner(B=B, H=H, sigma=sigma, temperature=2.0, seed=seed)
    env.reset()
    real = env._slots_host >= 0
    prev = torch.zeros(env.N, H, env.A, 2, dtype=torch.float64, device="cuda")
    seen = env._episode.clone()
    n_reset = n_kept = 0
    for step in range(40):
        reset = (env._episode != seen).cpu().numpy()
        seen = env._episode.clone()
        k = pl._k
        a, info = pl.plan()
        mu_start, tab = sample(prev.cpu().numpy(), reset, env._slots_host, B, H, seed, k, sigma,
                               np.float32 if pl._table.dtype == torch.float32 else np.float64)
        got = gather(env, pl._table, B, H).cpu().numpy()
        # branch 0 is the start mean: the last step's refined mean shifted one tick, zero after a reset
        assert np.array_equal(got[:, 0].transpose(0, 2, 1, 3)[real], tab[:, 0].transpose(0, 2, 1, 3)[real]), step
        new, action, shifted, _, _ = update(mu_start, got, info["reward"].cpu().numpy(), 2.0)
        np.testing.assert_allclose(info["mean"].cpu().numpy().transpose(0, 2, 1, 3)[real],
                                   shifted.transpose(0, 2, 1, 3)[real], rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(a.cpu().numpy()[real], action[real], rtol=1e-6, atol=1e-7)
        n_reset += int(reset.sum())
        n_kept += int((~reset).sum()) if step else 0
        prev = info["mean"].clone()
        env.step(a)
    assert n_reset > 0 and n_kept > 0
    # env.reset() restarts every mean, even where the episode counters stay 0
    env.reset()
    pl.plan()
    got = gather(env, pl._table, B, H)[:, 0].cpu().numpy()
    assert (got.transpose(0, 2, 1, 3)[real] == 0).all()


# ---------------------------------------------------------------------------------------------- isolation
def test_env_untouched_and_twin_step():
    env, twin = vehicle_env(seed=6), vehicle_env(seed=6)
    o, _ = env.reset()
    twin.reset()
    pl = env.planner(B=4, H=8, sigma=(1.0, 0.1), iterations=2, seed=1)
    for step in range(6):
        before = state_of(env._engine)
        snap = {k: t.clone() for k, t in env._snap.items()}
        obs, ep = env._obs.clone(), env._episode.clone()
        a, _ = pl.plan()
        assert_states_equal(before, state_of(env._engine), "env state")
        assert_states_equal(snap, env._snap, "env snapshot")
        assert torch.equal(obs, env._obs) and torch.equal(ep, env._episode)
        a = a.clone()
        o, rew, te, tr, info = env.step(a)
        o2, rew2, te2, tr2, info2 = twin.step(a)
        assert torch.equal(o, o2) and torch.equal(rew, rew2) and torch.equal(te, te2) and torch.equal(tr, tr2), step


# ---------------------------------------------------------------------------------------------- determinism
def test_determinism():
    envs = [vehicle_env(seed=7) for _ in range(3)]
    pls = [e.planner(B=6, H=10, sigma=(1.0, 0.2), iterations=2, seed=s) for e, s in zip(envs, (3, 3, 4))]
    for e in envs:
        e.reset()
    for step in range(4):
        acts = [p.plan()[0].clone() for p in pls]
        assert torch.equal(acts[0], acts[1]), step
        assert not torch.equal(acts[0], acts[2]), step
        for e, a in zip(envs, acts):
            e.step(a)


# ---------------------------------------------------------------------------------------------- no host round trips
def test_no_sync_and_no_allocation():
    env = vehicle_env(seed=8, N=16, M=8)
    env.reset()
    pls = [env.planner(B=3, H=5, iterations=1), env.planner(B=4, H=6, iterations=3, seed=5)]
    for p in pls:
        p.plan()
    torch.cuda.synchronize()
    mem = torch.cuda.memory_allocated()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for _ in range(3):
            for p in pls:
                p.plan()
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    assert torch.cuda.memory_allocated() == mem


# ---------------------------------------------------------------------------------------------- it plans
def collision_course_env():
    """The ego drives at 6 m/s towards a stopped vehicle 20 m ahead (15 m between the boxes): under zero actions it
    reaches it after 2.5 s, 25 ticks of 0.1 s."""
    ce = CatalogEntry("car", "car", "car", "car", BoundingBox(2.0, 5.0, 0.0, 0.0))
    ego, stopped = Entity(ce, ref="ego"), Entity(ce, ref="entity_1")
    ego.trajectory = Trajectory(np.array([[0.0, 0, 0], [10, 60, 0]]), fields=["t", "x", "y"])
    stopped.trajectory = Trajectory(np.array([[0.0, 20, 0], [10, 20, 0]]), fields=["t", "x", "y"])
    return VecScenarioEnv([Scenario([ego, stopped])], timestep=0.1)


def test_planner_avoids_a_collision():
    T = 60
    env = collision_course_env()
    env.reset()
    hit = False
    for _ in range(T):
        _, _, _, _, info = env.step(torch.zeros(1, 1, 2, device="cuda"))
        hit |= bool(info["terms"][0, 0, 1].item() > 0)
    assert hit, "the scene must collide under zero actions"
    env = collision_course_env()
    pl = env.planner(B=64, H=30, sigma=(1.0, 0.1), temperature=1.0, iterations=2, seed=0)
    env.reset()
    for step in range(T):
        a, _ = pl.plan()
        _, _, _, _, info = env.step(a)
        assert info["terms"][0, 0, 1].item() == 0, f"collision at step {step}"


# ---------------------------------------------------------------------------------------------- argument checks
def test_argument_checks():
    env = vehicle_env(seed=9, N=4, M=6)
    env.reset()
    bad = [dict(B=1), dict(B=0), dict(H=0), dict(iterations=0), dict(sigma=(-1.0, 0.1)),
           dict(sigma=(float("nan"), 0.1)), dict(sigma=(1.0,)), dict(temperature=0.0), dict(temperature=-1.0),
           dict(temperature=float("inf"))]
    for kw in bad:
        with pytest.raises(ValueError):
            env.planner(**{"B": 4, "H": 3, **kw})
    pl = env.planner(B=4, H=3)
    assert isinstance(pl, MPPIPlanner)
    eng, mu = env._engine, pl._mean[0]
    with pytest.raises(RuntimeError, match="sigma"):
        eng.plan_sample(env._spec, 4, 3, 0, 0, (float("inf"), 0.0), mu, None, pl._table)
    with pytest.raises(RuntimeError, match="lambda"):
        eng.plan_update(env._spec, 4, 3, 0.0, pl.branches._reward, pl._table, mu, pl._mean[1], False, None,
                        pl._best_branch, pl._best_reward)
    with pytest.raises(RuntimeError, match="overlap"):
        eng.plan_update(env._spec, 4, 3, 1.0, pl.branches._reward, pl._table, mu, mu, False, None,
                        pl._best_branch, pl._best_reward)
    with pytest.raises(RuntimeError, match="horizon"):
        eng.plan_sample(env._spec, 4, 0, 0, 0, (1.0, 0.0), mu, None, pl._table)
