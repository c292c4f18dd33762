"""
GPU tests of the randomised episode starts (sg_reset_scenarios_init, include/sg_b200.h; VecScenarioEnv(reset_spec),
env.reset(seed, start_time)): nothing drawn equals the masked reset, a start time equals the scene packed with
t0 := that time (and stays equal over 30 ticks), the device against the plain-C oracle on perturbed resets, the
distribution of the draws, seeded reproducibility, no host synchronisation, the vehicle fast path's promise kept
by the windows, branch rollouts from a perturbed state, and the argument checks.
"""
import dataclasses
import math

import numpy as np
import pytest
import torch
from scipy import stats

from oracle import golden_cases
from scenario_gym_b200 import (BoundingBox, CatalogEntry, ObsSpec, PolicyAgent, ResetSpec, Scenario, Trajectory,
                               VecScenarioEnv, Vehicle, abi, synthetic)
from scenario_gym_b200.engine import Engine
from scenario_gym_b200.packing import ScenarioSpec, SlotSpec, pack_scenarios

from helpers import all_xosc_specs
from reset_oracle import ResetOracleEngine, reset_init

pytestmark = pytest.mark.gpu
SKIP = ("coll_mask", "events", "trace_pose", "trace_present", "trace_t")
OBS = ObsSpec(k_neighbours=4, lookahead=(1.0, 2.0))
SIGMA = (0.6, 0.25, 0.04, 1.2)


def state_of(eng):
    return {name: eng.get(name).copy() for name, _, _ in abi.STATE_FIELDS if name not in SKIP}


def assert_states_equal(a, b, what=""):
    for k in a:
        assert np.array_equal(a[k], b[k], equal_nan=True), (what, k)


def dev_init(t_start=None, start_window=None, counter=None, perturb=None, sigma=(0.0,) * 4, seed=0):
    """(SgResetInit over device copies of the given host arrays, the tensors to keep alive)."""
    keep = {}
    r = abi.SgResetInit()
    for name, a, dt in (("t_start", t_start, np.float64), ("start_window", start_window, np.float64),
                        ("counter", counter, np.int64), ("perturb", perturb, np.uint8)):
        if a is not None:
            keep[name] = torch.from_numpy(np.ascontiguousarray(a, dt)).cuda()
            setattr(r, name, keep[name].data_ptr())
    for k, v in enumerate(sigma):
        r.sigma[k] = float(v)
    r.seed = int(seed)
    return r, keep


def rss_scene():
    cfg = golden_cases.rss_cfg()
    p = abi.default_params()
    p.timestep, p.features = cfg.dt, p.features | abi.FEAT_RSS
    return synthetic.pack_synthetic(cfg), p, cfg.actions


def xosc_scene():
    return pack_scenarios([s for _, s, _, _ in all_xosc_specs("xosc")]), abi.default_params(), None


def vehicle_scenarios(cfg):
    rows = synthetic.two_knot_rows(cfg).reshape(cfg.N, cfg.M, 2, 7)
    ce = CatalogEntry(None, "car1", "car", "Vehicle", BoundingBox(*synthetic.CAR1_BOX))
    return [Scenario([Vehicle(ce, trajectory=Trajectory(rows[n, m]), ref="ego" if m == 0 else f"entity_{m}")
                      for m in range(cfg.M)]) for n in range(cfg.N)]


def vehicle_env(cfg, **kw):
    return VecScenarioEnv(vehicle_scenarios(cfg), create_agent=lambda s, e: PolicyAgent(e), timestep=cfg.dt,
                          obs=kw.pop("obs", OBS), **kw)


def policy(obs):
    tx, ty = obs[..., 4], obs[..., 5]
    return torch.stack([(torch.sqrt(tx * tx + ty * ty) - obs[..., 0]).clamp(-5.0, 5.0),
                        torch.atan2(ty, tx).clamp(-0.7, 0.7)], -1)


# ---------------------------------------------------------------------------------------------- 1
@pytest.mark.parametrize("which", ["vehicles", "general"])
def test_nothing_drawn_is_the_masked_reset(which):
    scene, p, actions = rss_scene() if which == "vehicles" else xosc_scene()
    a, b = Engine(scene, p), Engine(scene, p)
    for e in (a, b):
        e.reset()
        e.rollout(20, actions=actions)
    mask = torch.from_numpy((np.arange(scene.N) % 3 != 1).astype(np.uint8)).cuda()
    a.reset(mask=mask)
    init, _keep = dev_init(start_window=np.zeros(scene.N), counter=np.arange(scene.N) * 3,
                           perturb=np.ones(scene.N * scene.M), seed=11)
    b.reset(mask=mask, init=init)
    assert_states_equal(state_of(a), state_of(b), which)


def test_env_with_default_spec_equals_env_without():
    cfg = synthetic.vehicles_config(seed=2, N=16, M=8, T=30, half_extent=20.0)
    e0, e1 = vehicle_env(cfg), vehicle_env(cfg, reset_spec=ResetSpec())
    o0, _ = e0.reset()
    o1, _ = e1.reset()
    assert torch.equal(o0, o1)
    finished = 0
    for k in range(50):
        a = policy(o0)
        o0, r0, te0, tr0, _ = e0.step(a)
        o1, r1, te1, tr1, _ = e1.step(a)
        assert torch.equal(o0, o1) and torch.equal(r0, r1), k
        assert torch.equal(te0, te1) and torch.equal(tr0, tr1), k
        finished += int((te0 | tr0).sum())
    assert finished > 0


# ---------------------------------------------------------------------------------------------- 2
def _start_equals_t0(scene, p, actions, seed):
    rng = np.random.default_rng(seed)
    win = abi.start_windows(scene, bool(p.persist), 1.0)
    start = scene.t0 + np.round(rng.uniform(0.0, 1.0, scene.N) * win, 3)
    moved = dataclasses.replace(scene, t0=start)
    a, b = Engine(scene, p), Engine(moved, abi.SgParams.from_buffer_copy(p))
    assert a._sc.kind_mask == b._sc.kind_mask
    init, _keep = dev_init(t_start=start, counter=np.zeros(scene.N))
    a.reset(init=init)
    a.tensor("event_count").zero_()
    b.reset()
    assert_states_equal(state_of(a), state_of(b), "reset")
    assert (start > scene.t0).any()
    a.rollout(30, actions=actions)
    b.rollout(30, actions=actions)
    assert_states_equal(state_of(a), state_of(b), "30 ticks")


def _random_table(scene, T, seed):
    g = np.random.default_rng(seed)
    return g.uniform([-3.0, -0.5], [3.0, 0.5], (T, scene.N * scene.M, 2)).transpose(0, 2, 1).copy()


def test_start_time_equals_packed_t0_lean_vehicles():
    scene, p, _ = rss_scene()
    _start_equals_t0(scene, p, _random_table(scene, 30, 1), 1)


def test_start_time_equals_packed_t0_sorted_sweep():
    cfg = synthetic.vehicles_config(seed=7, N=3, M=192, T=60, half_extent=40.0)
    scene = synthetic.pack_synthetic(cfg)
    p = abi.default_params()
    p.timestep = cfg.dt
    _start_equals_t0(scene, p, _random_table(scene, 30, 2), 2)


def test_start_time_equals_packed_t0_general_road():
    cfg = golden_cases.veh_cfg()
    net = golden_cases.road_network(golden_cases.ROAD_VEH_GEOMETRY)
    scs = vehicle_scenarios(cfg)
    for sc in scs:
        sc.road_network = net
    env = VecScenarioEnv(scs, create_agent=lambda s, e: PolicyAgent(e) if e is s.ego else None, timestep=cfg.dt,
                         terminal_conditions=["max_length", "ego_off_road"], obs=ObsSpec(road=True))
    eng = env._engine
    assert eng.params.terminal & abi.TERM_EGO_OFF_ROAD and eng.scene.n_networks > 0
    _start_equals_t0(eng.scene, eng.params, _random_table(eng.scene, 30, 3), 3)


# ---------------------------------------------------------------------------------------------- 3
def _close(a, b, tol=1e-12):
    a, b = np.asarray(a, float), np.asarray(b, float)
    same = (a == b) | (np.isnan(a) & np.isnan(b))
    return np.all(same | (np.abs(a - b) <= tol * np.maximum(1.0, np.abs(b))))


@pytest.mark.parametrize("which", ["vehicles", "general"])
def test_perturbed_reset_against_oracle(which):
    scene, p, _ = rss_scene() if which == "vehicles" else xosc_scene()
    N, M = scene.N, scene.M
    rng = np.random.default_rng(5)
    win = abi.start_windows(scene, False, 1.0)
    mask = np.ones(N, np.uint8)
    mask[N // 2] = 0
    perturb = (rng.random(N * M) < 0.7).astype(np.uint8)
    counter = rng.integers(0, 2**33, N)
    args = dict(start_window=win, counter=counter, perturb=perturb, sigma=SIGMA, seed=2**63 + 9)
    dev, ora = Engine(scene, p), ResetOracleEngine(scene, p)
    dev.reset()
    ora.reset()
    plain = dev.get("pose").copy()
    di, _dk = dev_init(**args)
    oi, _ok = reset_init(**args)
    dev.reset(mask=torch.from_numpy(mask).cuda(), init=di)
    ora.reset_init(mask, oi)
    got, want = state_of(dev), state_of(ora)
    assert (got["pose"][0] != plain[0]).any() and (got["t"] != scene.t0).any()
    for k in want:
        if want[k].dtype.kind == "f":
            assert _close(got[k], want[k]), k
        else:
            assert np.array_equal(got[k], want[k]), k


# ---------------------------------------------------------------------------------------------- 4
def test_draw_distributions():
    Nn, T = 4096, 10.0
    ts = np.linspace(0.0, T, 101)
    slots = []
    for m in range(4):
        r = np.zeros((len(ts), 7))
        r[:, 0], r[:, 1], r[:, 2], r[:, 4] = ts, 5.0 * ts, 20.0 * m, 0.3
        r[:, 1], r[:, 2] = 5.0 * ts * math.cos(0.3), 20.0 * m + 5.0 * ts * math.sin(0.3)
        slots.append(SlotSpec(abi.KIND_VEHICLE, r))
    scene = pack_scenarios([ScenarioSpec(list(slots)) for _ in range(Nn)])
    p = abi.default_params()
    win = abi.start_windows(scene, False, 1.0)
    assert np.allclose(win, T - 1.0)
    base, pert = Engine(scene, p), Engine(scene, p)
    common = dict(start_window=win, counter=np.full(Nn, 3), seed=1234)
    bi, _bk = dev_init(**common)
    pi, _pk = dev_init(perturb=np.ones(Nn * 4), sigma=SIGMA, **common)
    base.reset(init=bi)
    pert.reset(init=pi)
    t = base.get("t")
    assert np.array_equal(t, pert.get("t"))
    u = (t - scene.t0) / win
    assert stats.kstest(u, "uniform").pvalue > 1e-3
    b, q = state_of(base), state_of(pert)
    h = b["pose"][3]
    dx, dy = q["pose"][0] - b["pose"][0], q["pose"][1] - b["pose"][1]
    z = {"lon": (np.cos(h) * dx + np.sin(h) * dy) / SIGMA[0], "lat": (-np.sin(h) * dx + np.cos(h) * dy) / SIGMA[1],
         "heading": (q["pose"][3] - h) / SIGMA[2], "speed": (q["speed"] - b["speed"]) / SIGMA[3]}
    n = Nn * 4
    assert (b["speed"] > 4.9).all()  # (5 m/s: max(0, .) never clips at 1.2 m/s std)
    for k, v in z.items():
        assert abs(v.mean()) < 5.0 / math.sqrt(n), k
        assert abs(v.std() - 1.0) < 0.03, k
        assert stats.kstest(v, "norm").pvalue > 1e-3, k
    # the velocity turns with the heading and has the new speed
    assert np.allclose(np.arctan2(q["vel"][1], q["vel"][0]), q["pose"][3], atol=1e-9)
    assert np.allclose(np.hypot(q["vel"][0], q["vel"][1]), q["speed"], rtol=1e-12)


# ---------------------------------------------------------------------------------------------- 5
def _episodes(env, steps, seed=None):
    o, _ = env.reset(seed=seed)
    out = [o.clone()]
    for _ in range(steps):
        o, r, te, tr, _ = env.step(policy(o))
        out += [o.clone(), r.clone(), te.clone(), tr.clone()]
    return out


def test_seeded_reproducibility():
    cfg = synthetic.vehicles_config(seed=2, N=16, M=8, T=30, half_extent=20.0)
    spec = ResetSpec(start_offset=0.5, min_remaining=0.5, lon=0.5, lat=0.2, heading=0.05, speed=1.0, seed=7)
    e0, e1 = vehicle_env(cfg, reset_spec=spec), vehicle_env(cfg, reset_spec=spec)
    a, b = _episodes(e0, 70), _episodes(e1, 70)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    assert int(e0._episode.sum()) > 0
    # only finished scenarios advanced their draw counter (one draw per episode)
    assert torch.equal(e0._counter, e0._episode + 1)
    e2 = vehicle_env(cfg, reset_spec=dataclasses.replace(spec, seed=8))
    assert not torch.equal(_episodes(e2, 0)[0], a[0])
    # reset(seed=s) replays a seed's sequence
    assert all(torch.equal(x, y) for x, y in zip(_episodes(e2, 70, seed=7), a))
    assert all(torch.equal(x, y) for x, y in zip(_episodes(e0, 70, seed=7), a))


# ---------------------------------------------------------------------------------------------- 6
def test_no_host_synchronisation_with_a_spec():
    cfg = synthetic.vehicles_config(seed=2, N=16, M=8, T=30, half_extent=20.0)
    env = vehicle_env(cfg, reset_spec=ResetSpec(start_offset=1.0, lon=0.3, heading=0.02, speed=0.5))
    st = torch.full((env.N,), 0.25, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        o, _ = env.reset()
        for _ in range(40):
            o, *_ = env.step(policy(o))
        o, _ = env.reset(seed=3, start_time=st)
        o, *_ = env.step(policy(o))
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    assert torch.isfinite(o).all()


# ---------------------------------------------------------------------------------------------- 7
def test_windows_keep_the_vehicle_fast_path_promise():
    cfg = synthetic.vehicles_config(seed=3, N=32, M=16, T=40, half_extent=25.0)
    env = vehicle_env(cfg, reset_spec=ResetSpec(start_offset=100.0, min_remaining=0.2))
    eng = env._engine
    assert eng._sc.kind_mask == 1 << abi.KIND_VEHICLE  # (the vehicle fast path)
    veh = torch.from_numpy((eng.scene.kind.reshape(-1) == abi.KIND_VEHICLE)).cuda()
    assert (env.start_window > 0).all()
    for s in range(5):
        env.reset(seed=s)
        assert bool(eng.tensor("present")[veh].all()), s
        assert bool((eng.tensor("t") > torch.from_numpy(eng.scene.t0).cuda()).any())
    env.reset(start_time=torch.full((env.N,), 1e9, dtype=torch.float64, device="cuda"))
    assert bool(eng.tensor("present")[veh].all())
    assert torch.equal(eng.tensor("t"), torch.from_numpy(eng.scene.t0).cuda() + env.start_window)


# ---------------------------------------------------------------------------------------------- 8
def test_branch_h1_from_a_perturbed_state_equals_env_step():
    cfg = synthetic.vehicles_config(seed=4, N=8, M=64, T=40, half_extent=30.0)
    env = vehicle_env(cfg, terminal_conditions=["max_length", "ego_collision"],
                      reset_spec=ResetSpec(start_offset=0.5, lon=0.4, lat=0.2, heading=0.03, speed=1.0, seed=1))
    br = env.branches(1, 1, final_obs=True)
    o, _ = env.reset()
    finished = 0
    for k in range(cfg.T + 2):
        a = policy(o)
        got = {key: v[:, 0].clone() for key, v in br.run(a[:, None, None]).items()}
        o, rew, te, tr, info = env.step(a)
        assert torch.equal(got["reward"], rew) and torch.equal(got["final_obs"], info["final_obs"]), k
        assert torch.equal(got["terminated"], te) and torch.equal(got["truncated"], tr), k
        finished += int((te | tr).sum())
    assert finished > 0


# ---------------------------------------------------------------------------------------------- checks
def test_argument_checks():
    cfg = synthetic.vehicles_config(seed=2, N=4, M=4, T=20, half_extent=20.0)
    env = vehicle_env(cfg, reset_spec=ResetSpec())
    for bad in (torch.zeros(env.N, dtype=torch.float32, device="cuda"), torch.zeros(env.N + 1, dtype=torch.float64,
                device="cuda"), torch.zeros(env.N, dtype=torch.float64), [0.0] * env.N):
        with pytest.raises(ValueError, match="start_time"):
            env.reset(start_time=bad)
    with pytest.raises(ValueError, match="seed"):
        env.reset(seed=1.5)
    with pytest.raises(ValueError, match="reset_spec"):
        vehicle_env(cfg, reset_spec={"lon": 1.0})
    # NaN / negative start times are clamped on the device
    env.reset(start_time=torch.tensor([math.nan, -3.0, math.inf, 0.1], dtype=torch.float64, device="cuda"))
    t0 = torch.from_numpy(env._engine.scene.t0).cuda()
    w = env.start_window
    assert torch.equal(env._engine.tensor("t"), t0 + torch.stack([w[0] * 0, w[1] * 0, w[2], torch.minimum(
        w[3], torch.tensor(0.1, dtype=torch.float64, device="cuda"))]))
    eng = env._engine
    init, _keep = dev_init(counter=np.zeros(env.N), sigma=(0.0, -1.0, 0.0, 0.0))
    with pytest.raises(RuntimeError, match="sigma"):
        eng.reset(init=init)
    init, _keep = dev_init(sigma=(0.0, 0.0, 0.0, 0.0))
    with pytest.raises(RuntimeError, match="counter"):
        eng.reset(init=init)
