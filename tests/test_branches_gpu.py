"""
GPU tests of branched look-ahead rollouts (sg_fork_state, Engine.sharing_scene / fork_into,
VecScenarioEnv.branches): H = 1 against env.step, the fused horizon against one-tick stepping on three kernel
families, the oracle, the env left untouched, independent branches, branches finishing inside the horizon, no
host synchronisation or allocation, the argument checks and sg_fork_state itself.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import golden_cases
from oracle.env_runner import OracleEnvEngine
from scenario_gym_b200 import (BoundingBox, CatalogEntry, Entity, ObsSpec, Pedestrian, PolicyAgent, RSSDistances,
                               Scenario, Trajectory, VecScenarioEnv, Vehicle, abi, synthetic)
from scenario_gym_b200.engine import Engine

from helpers import golden, manifest, sub

pytestmark = pytest.mark.gpu
F32 = dict(rtol=2e-6, atol=2e-5)
SKIP = ("events", "trace_pose", "trace_present", "trace_t")
OBS = ObsSpec(k_neighbours=4, lookahead=(1.0, 2.0))


def vehicle_scenarios(cfg):
    rows = synthetic.two_knot_rows(cfg).reshape(cfg.N, cfg.M, 2, 7)
    ce = CatalogEntry(None, "car1", "car", "Vehicle", BoundingBox(*synthetic.CAR1_BOX))
    return [Scenario([Vehicle(ce, trajectory=Trajectory(rows[n, m]), ref="ego" if m == 0 else f"entity_{m}")
                      for m in range(cfg.M)]) for n in range(cfg.N)]


def vehicle_env(cfg, **kw):
    return VecScenarioEnv(vehicle_scenarios(cfg), create_agent=lambda s, e: PolicyAgent(e), timestep=cfg.dt,
                          obs=kw.pop("obs", OBS), **kw)


def xosc_scenarios(names=None):
    g, man = golden("xosc"), manifest()["xosc"]
    cls = {abi.ETYPE_VEHICLE: (Vehicle, "Vehicle"), abi.ETYPE_PEDESTRIAN: (Pedestrian, "Pedestrian")}
    out = []
    for name in sorted(man):
        if names is not None and not any(name.startswith(p) for p in names):
            continue
        inp = sub(g, f"xosc/{name}/in")
        ents = []
        for i in range(int(inp["n_entities"])):
            Cl, ctype = cls.get(int(inp["etype"][i]), (Entity, "MiscObject"))
            ce = CatalogEntry(None, "entry", None, ctype, BoundingBox(*[float(v) for v in inp["box"][i]]))
            ents.append(Cl(ce, trajectory=Trajectory(inp[f"traj{i}"]), ref=man[name]["refs"][i]))
        out.append(Scenario(ents))
    return out


def policy(obs):
    tx, ty = obs[..., 4], obs[..., 5]
    return torch.stack([(torch.sqrt(tx * tx + ty * ty) - obs[..., 0]).clamp(-5.0, 5.0),
                        torch.atan2(ty, tx).clamp(-0.7, 0.7)], -1)


def random_actions(env, B, H, seed, dtype=torch.float32):
    g = torch.Generator(device="cuda").manual_seed(seed)
    a = torch.rand((env.N, B, H, env.A, 2), generator=g, device="cuda", dtype=torch.float64)
    return (a * torch.tensor([8.0, 1.2], device="cuda", dtype=torch.float64)
            - torch.tensor([4.0, 0.6], device="cuda", dtype=torch.float64)).to(dtype)


def state_of(eng):
    return {name: eng.tensor(name).clone() for name, _, _ in abi.STATE_FIELDS if name not in SKIP}


def assert_states_equal(a, b, what=""):
    for k in a:
        assert torch.equal(a[k], b[k]), (what, k)


def step_actions_table(env, a):
    """env.step's one-tick table for actions [N, A, 2] (the env's own scatter, independent of the branches')."""
    buf = torch.zeros(1, 2, env.N * env._engine.M, dtype=a.dtype, device="cuda")
    buf[0].index_copy_(1, env._dst, a.reshape(env.N * env.A, 2).index_select(0, env._src).t())
    return buf


# ---------------------------------------------------------------------------------------------- 1
@pytest.mark.parametrize("which", ["vehicles", "xosc"])
def test_h1_equals_env_step(which):
    """B = 1, H = 1, final_obs: the branch scores bit for bit what the next env.step scores, over whole
    episodes (terminated / truncated included); xosc takes the general kernel and has pedestrians."""
    if which == "vehicles":
        cfg = synthetic.vehicles_config(seed=4, N=8, M=64, T=40, half_extent=30.0)
        env = vehicle_env(cfg, terminal_conditions=["max_length", "ego_collision"])
        steps = cfg.T + 2
    else:
        env = VecScenarioEnv(xosc_scenarios(), obs=OBS, terminal_conditions=["max_length", "collision"])
        assert (env._engine.scene.etype == abi.ETYPE_PEDESTRIAN).any()
        steps = 150
    br = env.branches(1, 1, final_obs=True)
    o, _ = env.reset()
    finished = 0
    for k in range(steps):
        a = policy(o)
        res = br.run(a[:, None, None])
        got = {key: v[:, 0].clone() for key, v in res.items()}
        o, rew, te, tr, info = env.step(a)
        assert torch.equal(got["reward"], rew), k
        assert torch.equal(got["terms"], info["terms"]), k
        assert torch.equal(got["terminated"], te) and torch.equal(got["truncated"], tr), k
        assert torch.equal(got["final_obs"], info["final_obs"]), k
        assert torch.equal(got["ticks"], torch.ones_like(got["ticks"])), k
        finished += int((te | tr).sum().item())
    assert finished > 0


# ---------------------------------------------------------------------------------------------- 2
def _fused_vs_single(env, B, H, warm, seed):
    o, _ = env.reset()
    for _ in range(warm):
        o, *_ = env.step(policy(o))
    acts = random_actions(env, B, H, seed, torch.float64)
    br = env.branches(B, H)
    br.run(acts)
    src = env._engine
    spare = Engine.sharing_scene(src)
    for b in range(B):
        src.fork_into([spare])
        for h in range(H):
            spare.rollout(1, actions=step_actions_table(env, acts[:, b, h]))
        assert_states_equal(state_of(spare), state_of(br.engines[b]), f"branch {b}")
    return br


def test_fused_horizon_equals_single_ticks_lean_vehicles():
    cfg = synthetic.vehicles_config(seed=6, N=16, M=64, T=60, half_extent=25.0)
    _fused_vs_single(vehicle_env(cfg), B=3, H=12, warm=5, seed=1)


def test_fused_horizon_equals_single_ticks_sorted_sweep():
    cfg = synthetic.vehicles_config(seed=7, N=3, M=192, T=40, half_extent=40.0)
    _fused_vs_single(vehicle_env(cfg), B=2, H=9, warm=3, seed=2)


def test_fused_horizon_equals_single_ticks_general_road():
    cfg = golden_cases.veh_cfg()
    net = golden_cases.road_network(golden_cases.ROAD_VEH_GEOMETRY)
    scs = vehicle_scenarios(cfg)
    for sc in scs:
        sc.road_network = net
    env = VecScenarioEnv(scs, create_agent=lambda s, e: PolicyAgent(e) if e is s.ego else None, timestep=cfg.dt,
                         terminal_conditions=["max_length", "ego_off_road"], obs=ObsSpec(road=True))
    assert env._engine.params.terminal & abi.TERM_EGO_OFF_ROAD  # (the general kernel)
    _fused_vs_single(env, B=3, H=15, warm=4, seed=3)


# ---------------------------------------------------------------------------------------------- 3
def test_branches_against_oracle():
    cfg = synthetic.vehicles_config(seed=8, N=6, M=16, T=60, half_extent=12.0)
    env = vehicle_env(cfg, terminal_conditions=["max_length", "collision"], state_callbacks=[RSSDistances()])
    o, _ = env.reset()
    for _ in range(6):
        o, *_ = env.step(policy(o))
    B, H = 4, 20
    acts = random_actions(env, B, H, 4, torch.float64)
    br = env.branches(B, H)
    res = {k: v.cpu().numpy() for k, v in br.run(acts).items()}
    src = env._engine
    slots = env._slots_host
    seen_coll = 0
    for b in range(B):
        cpu = OracleEnvEngine(src.scene, src.params)
        for name, _, _ in abi.STATE_FIELDS:
            if name not in SKIP + ("coll_mask",):
                cpu.state[name][...] = src.get(name).reshape(cpu.state[name].shape)
        cpu.state["event_count"][...] = 0
        cpu.env_spec(slots, OBS.k_neighbours, OBS.radius, OBS.lookahead, False,
                     weights=[env.reward_weights[t] for t in abi.ENV_TERMS])
        for k, t in env._snap.items():
            cpu.env[k][...] = t.cpu().numpy()
        table = torch.stack([step_actions_table(env, acts[:, b, h])[0] for h in range(H)]).cpu().numpy()
        t0 = cpu.state["tick"].copy()
        cpu.rollout(H, actions=table)
        rew, terms, te, tr = cpu.env_reward()
        assert np.array_equal(te, res["terminated"][:, b]) and np.array_equal(tr, res["truncated"][:, b]), b
        assert np.array_equal(cpu.state["tick"] - t0, res["ticks"][:, b]), b
        assert np.array_equal(terms[..., [1, 2, 4]], res["terms"][:, b][..., [1, 2, 4]]), b
        np.testing.assert_allclose(res["terms"][:, b], terms, **F32)
        np.testing.assert_allclose(res["reward"][:, b], rew, **F32)
        seen_coll += int(terms[..., 1].sum())
    assert seen_coll > 0


# ---------------------------------------------------------------------------------------------- 4
def test_env_untouched_and_twin_step():
    cfg = synthetic.vehicles_config(seed=9, N=8, M=32, T=50, half_extent=20.0)
    env, twin = vehicle_env(cfg, obs=ObsSpec(k_neighbours=4, lookahead=(1.0,), lidar_rays=16)), None
    twin = vehicle_env(cfg, obs=ObsSpec(k_neighbours=4, lookahead=(1.0,), lidar_rays=16))
    o, _ = env.reset()
    o2, _ = twin.reset()
    for _ in range(4):
        a = policy(o)
        o, *_ = env.step(a)
        o2, *_ = twin.step(a)
    br = env.branches(5, 10, final_obs=True)
    before = state_of(env._engine)
    snap = {k: t.clone() for k, t in env._snap.items()}
    obs, ep = env._obs.clone(), env._episode.clone()
    for s in range(3):
        br.run(random_actions(env, 5, 10, 10 + s))
    assert_states_equal(before, state_of(env._engine), "env state")
    assert_states_equal(snap, env._snap, "env snapshot")
    assert torch.equal(obs, env._obs) and torch.equal(ep, env._episode)
    for _ in range(3):
        a = policy(o)
        o, rew, te, tr, info = env.step(a)
        o2, rew2, te2, tr2, info2 = twin.step(a)
        assert torch.equal(o, o2) and torch.equal(rew, rew2) and torch.equal(te, te2) and torch.equal(tr, tr2)


# ---------------------------------------------------------------------------------------------- 5
def test_branches_are_independent():
    cfg = synthetic.vehicles_config(seed=10, N=6, M=24, T=50, half_extent=14.0)
    env = vehicle_env(cfg, terminal_conditions=["max_length", "collision"])
    o, _ = env.reset()
    o, *_ = env.step(policy(o))
    B, H = 4, 16
    one = random_actions(env, 1, H, 20)
    same = env.branches(B, H, final_obs=True).run(one.expand(-1, B, -1, -1, -1).contiguous())
    for b in range(1, B):
        for k, v in same.items():
            assert torch.equal(v[:, b], v[:, 0]), (k, b)
    acts = random_actions(env, B, H, 21)
    many = {k: v.clone() for k, v in env.branches(B, H, final_obs=True).run(acts).items()}
    single = env.branches(1, H, final_obs=True)
    for b in range(B):
        res = single.run(acts[:, b:b + 1].contiguous())
        for k, v in res.items():
            assert torch.equal(v[:, 0], many[k][:, b]), (k, b)


# ---------------------------------------------------------------------------------------------- 6
def test_finishing_inside_the_horizon():
    ce = CatalogEntry("car", "car", "car", "car", BoundingBox(2.0, 5.0, 0.0, 0.0))
    ego, hazard = Entity(ce, ref="ego"), Entity(ce, ref="entity_1")
    ego.trajectory = Trajectory(np.array([[0.0, 0, 0], [10, 20, 0]]), fields=["t", "x", "y"])
    hazard.trajectory = Trajectory(np.array([[0.0, 40, 0], [10, 20, 0]]), fields=["t", "x", "y"])
    env = VecScenarioEnv([Scenario([ego, hazard])], terminal_conditions=["max_length", "ego_collision"])
    env.reset()
    H = 400
    res = env.branches(2, H).run(torch.zeros(1, 2, H, 1, 2, device="cuda"))
    assert res["terminated"].all().item() and not res["truncated"].any().item()
    assert (res["terms"][0, :, 0, 1] == 1.0).all().item()
    assert (res["ticks"] < H).all().item() and (res["ticks"] > 0).all().item()
    # a scenario shorter than the horizon: truncated at its length
    short = Entity(ce, ref="ego")
    short.trajectory = Trajectory(np.array([[0.0, 0, 0], [1.0, 5, 0]]), fields=["t", "x", "y"])
    env2 = VecScenarioEnv([Scenario([short])])
    env2.reset()
    res = env2.branches(1, 90).run(torch.zeros(1, 1, 90, 1, 2, device="cuda", dtype=torch.float64))
    assert res["truncated"].item() and not res["terminated"].item()
    assert 0 < res["ticks"].item() < 90


# ---------------------------------------------------------------------------------------------- 7
def test_no_sync_and_no_allocation():
    cfg = synthetic.vehicles_config(seed=2, N=16, M=8, T=30, half_extent=20.0)
    env = vehicle_env(cfg)
    o, _ = env.reset()
    br, br_obs = env.branches(3, 5), env.branches(2, 4, final_obs=True)
    a32, a64 = random_actions(env, 3, 5, 1), random_actions(env, 2, 4, 2, torch.float64)
    br.run(a32)
    br_obs.run(a64)
    torch.cuda.synchronize()
    mem = torch.cuda.memory_allocated()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for _ in range(3):
            br.run(a32)
            br_obs.run(a64)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    assert torch.cuda.memory_allocated() == mem


# ---------------------------------------------------------------------------------------------- 8
def test_argument_checks():
    cfg = synthetic.vehicles_config(seed=3, N=4, M=8, T=20, half_extent=20.0)
    env = vehicle_env(cfg)
    env.reset()
    for B, H in ((0, 3), (2, 0), (-1, 1)):
        with pytest.raises(ValueError):
            env.branches(B, H)
    br = env.branches(2, 3)
    good = torch.zeros(env.N, 2, 3, env.A, 2, device="cuda")
    for bad in (torch.zeros(env.N, 3, 3, env.A, 2, device="cuda"), good[..., :1], good.to(torch.float16),
                good.to(torch.int32), good.cpu(), np.zeros((env.N, 2, 3, env.A, 2))):
        with pytest.raises(ValueError):
            br.run(bad)
    br.run(good)
    src = env._engine
    traced = Engine(src.scene, src.params, trace_cap=4)
    with pytest.raises(RuntimeError, match="trace"):
        src.fork_into([traced])
    other = Engine(synthetic.pack_synthetic(synthetic.vehicles_config(seed=3, N=4, M=9, T=20)), src.params)
    with pytest.raises(ValueError):
        src.fork_into([other])
    with pytest.raises(ValueError):
        src.fork_into([src])
    with pytest.raises(ValueError):
        src.fork_into([Engine.sharing_scene(src)], spec=env._spec)


# ---------------------------------------------------------------------------------------------- 9
def same_bytes(a, b):
    """Bit-equality (the scribbled buffers hold NaN patterns, which torch.equal calls unequal)."""
    return torch.equal(a.reshape(-1).view(torch.uint8), b.reshape(-1).view(torch.uint8))


def _scribble(eng, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    for t in eng._state_t.values():
        t.reshape(-1).view(torch.uint8).copy_(torch.randint(0, 256, (t.numel() * t.element_size(),), generator=g,
                                                device="cuda", dtype=torch.uint8))


@pytest.mark.parametrize("coll_matrix", [False, True])
@pytest.mark.parametrize("with_spec", [False, True])
def test_fork_state_direct(coll_matrix, with_spec):
    cfg = golden_cases.veh_cfg()
    p = abi.default_params()
    p.timestep, p.features = cfg.dt, p.features | abi.FEAT_RSS | (abi.FEAT_COLL_MATRIX if coll_matrix else 0)
    src = Engine(synthetic.pack_synthetic(cfg), p, coll_matrix=coll_matrix)
    src.reset()
    src.rollout(17, actions=cfg.actions)
    N, M, A = src.N, src.M, 5
    dsts = [Engine.sharing_scene(src, event_cap=64) for _ in range(3)]
    for k, d in enumerate(dsts):
        _scribble(d, k)
    spec = dst_specs = None
    keep = []
    if with_spec:
        def mk(seed):
            g = torch.Generator(device="cuda").manual_seed(seed)
            bufs = {"agent_slot": torch.zeros(N * A, dtype=torch.int32, device="cuda"),
                    "snap_dist": torch.randn(N * A, generator=g, device="cuda", dtype=torch.float64),
                    "snap_collided": torch.randint(0, 2, (N * A,), generator=g, device="cuda", dtype=torch.uint8),
                    "snap_pair_ticks": torch.randint(0, 99, (N,), generator=g, device="cuda", dtype=torch.int64),
                    "snap_rss": torch.randint(0, 4, (N,), generator=g, device="cuda", dtype=torch.uint8)}
            e = abi.SgEnvSpec()
            e.n_agents = A
            for k2, t in bufs.items():
                setattr(e, k2, t.data_ptr())
            keep.append(bufs)
            return e, bufs
        spec, sbuf = mk(100)
        dst_specs = [mk(101 + k)[0] for k in range(3)]
    before = [{k: t.clone() for k, t in d._state_t.items()} for d in dsts]
    src.fork_into(dsts, spec=spec, specs=dst_specs)
    torch.cuda.synchronize()
    for k, d in enumerate(dsts):
        for name, _, _ in abi.STATE_FIELDS:
            got = d.tensor(name)
            if name == "event_count":
                assert got.item() == 0
            elif name in SKIP or (name == "coll_mask" and not coll_matrix):
                assert same_bytes(got, before[k][name]), name  # not copied: left as it was
            else:
                assert same_bytes(got, src.tensor(name)), (k, name)
        if with_spec:
            for name in ("snap_dist", "snap_collided", "snap_pair_ticks", "snap_rss"):
                assert torch.equal(keep[1 + k][name], sbuf[name]), (k, name)
    # a destination continues exactly as the source
    src.rollout(9, actions=cfg.actions[17:])
    dsts[1].rollout(9, actions=cfg.actions[17:])
    for name, _, _ in abi.STATE_FIELDS:
        if name not in SKIP + ("event_count",) and (coll_matrix or name != "coll_mask"):
            assert torch.equal(dsts[1].tensor(name), src.tensor(name)), name


def test_fork_state_scenario_window():
    """A window (plane_stride / scenario_base) forks scenarios [2, 5) of a batch into the same rows of another."""
    cfg = golden_cases.veh_cfg()
    p = abi.default_params()
    p.timestep = cfg.dt
    src = Engine(synthetic.pack_synthetic(cfg), p)
    src.reset()
    src.rollout(11, actions=cfg.actions)
    dst = Engine.sharing_scene(src)
    _scribble(dst, 7)
    before = {k: t.clone() for k, t in dst._state_t.items()}
    N, M, n0, n1 = src.N, src.M, 2, 5
    sc = abi.SgScene.from_buffer_copy(src._sc)
    sc.n_scenarios, sc.plane_stride, sc.scenario_base = n1 - n0, N * M, n0

    def window(eng):
        st = abi.SgState.from_buffer_copy(eng._fork_view())
        for name, dtype, shape in abi.STATE_FIELDS:
            if name in SKIP or name in ("event_count", "coll_mask"):
                continue
            t = eng.tensor(name)
            per = M if "NM" in shape else (t.numel() // N if shape[0] == "N" else 0)
            setattr(st, name, t.data_ptr() + n0 * per * t.element_size())
        return st

    s, d = window(src), window(dst)
    arr = (C.POINTER(abi.SgState) * 1)(C.pointer(d))
    rc = src.lib["fork_state"](C.byref(sc), C.byref(s), arr, 1, None, None, src.dev_index, src._stream())
    assert rc == 0, src.lib["last_error"]().decode()
    torch.cuda.synchronize()
    for name, dtype, shape in abi.STATE_FIELDS:
        if name in SKIP or name in ("event_count", "coll_mask"):
            continue
        got, want, old = dst.tensor(name), src.tensor(name), before[name]
        if "NM" in shape:
            g, w, o = (x.reshape(-1, N, M) for x in (got, want, old))
        else:
            g, w, o = (x.reshape(N, -1) for x in (got, want, old))
            g, w, o = (x.unsqueeze(0) for x in (g, w, o))
        assert same_bytes(g[:, n0:n1].contiguous(), w[:, n0:n1].contiguous()), name
        assert same_bytes(g[:, :n0].contiguous(), o[:, :n0].contiguous()), name
        assert same_bytes(g[:, n1:].contiguous(), o[:, n1:].contiguous()), name
    assert dst.tensor("event_count").item() == 0
