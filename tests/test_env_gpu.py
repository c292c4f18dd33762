"""
GPU tests of the closed-loop environment (VecScenarioEnv; sg_env_observe / sg_env_reward /
sg_reset_scenarios): reference parity through the env, closed loops replayed through the fused rollout and
the oracle, device observations and rewards against the oracle, termination, auto-reset, the masked reset,
the absence of host synchronisation and the argument checks.
"""
import numpy as np
import pytest
import torch

from oracle import golden_cases
from oracle.env_runner import OracleEnvEngine
from oracle.runner import OracleEngine
from scenario_gym_b200 import (ActionTableAgent, BoundingBox, CatalogEntry, CollisionMetric, EgoAvgSpeed,
                               EgoDistanceTravelled, EgoMaxSpeed, Entity, Metric, ObsSpec, Pedestrian,
                               PolicyAgent, ScenarioGym, Scenario, Trajectory, VecScenarioEnv, Vehicle, abi,
                               synthetic)
from scenario_gym_b200.engine import Engine
from scenario_gym_b200.packing import pack_scenarios

from helpers import all_xosc_specs, golden, manifest, sub

pytestmark = pytest.mark.gpu
TOL = 1e-9
F32 = dict(rtol=2e-6, atol=2e-5)
FINAL_KEYS = ("ego_avg_speed", "ego_max_speed", "ego_distance_travelled")


def close(a, b, tol=TOL):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return np.all(np.abs(a - b) <= tol * np.maximum(1.0, np.abs(b)))


def vehicle_scenario(cfg, n):
    rows = synthetic.two_knot_rows(cfg).reshape(cfg.N, cfg.M, 2, 7)
    ce = CatalogEntry(None, "car1", "car", "Vehicle", BoundingBox(*synthetic.CAR1_BOX))
    return Scenario([Vehicle(ce, trajectory=Trajectory(rows[n, m]), ref="ego" if m == 0 else f"entity_{m}")
                     for m in range(cfg.M)])


def golden_scenarios(names=None):
    g, man = golden("xosc"), manifest()["xosc"]
    out = []
    for name in sorted(man):
        if names is not None and not any(name.startswith(p) for p in names):
            continue
        inp = sub(g, f"xosc/{name}/in")
        cls = {abi.ETYPE_VEHICLE: (Vehicle, "Vehicle"), abi.ETYPE_PEDESTRIAN: (Pedestrian, "Pedestrian")}
        ents = []
        for i in range(int(inp["n_entities"])):
            C, ctype = cls.get(int(inp["etype"][i]), (Entity, "MiscObject"))
            ce = CatalogEntry(None, "entry", None, ctype, BoundingBox(*[float(v) for v in inp["box"][i]]))
            ents.append(C(ce, trajectory=Trajectory(inp[f"traj{i}"]), ref=man[name]["refs"][i]))
        out.append((name, Scenario(ents), sub(g, f"xosc/{name}/out")))
    return out


def steer_to_target(obs):
    """A deterministic policy of the observation only: steer toward the first lookahead point, speed up to
    reach it in a second."""
    tx, ty = obs[..., 4], obs[..., 5]
    steer = torch.atan2(ty, tx).clamp(-0.7, 0.7)
    accel = (torch.sqrt(tx * tx + ty * ty) - obs[..., 0]).clamp(-5.0, 5.0)
    return torch.stack([accel, steer], -1)


def std_metrics():
    return [EgoAvgSpeed(), EgoMaxSpeed(), EgoDistanceTravelled(), CollisionMetric()]


# ---------------------------------------------------------------------------------------------- 1
def test_reference_parity_through_env():
    """Every vehicle a PolicyAgent fed the golden action table by episode step == the reference's golden
    record, and == the ActionTableAgent fused rollout of the same scene bit for bit."""
    cfg = golden_cases.veh_cfg()
    acts = cfg.actions.reshape(cfg.T, 2, cfg.N, cfg.M)
    g = golden("veh_rss")
    scs = [vehicle_scenario(cfg, n) for n in range(cfg.N)]
    env = VecScenarioEnv(scs, create_agent=lambda s, e: PolicyAgent(e), timestep=cfg.dt)
    assert env.A == cfg.M and [e.ref for e in env.agent_entities(0)][:2] == ["ego", "entity_1"]
    table = torch.from_numpy(np.ascontiguousarray(acts.transpose(0, 2, 3, 1))).cuda()  # [T, N, M, 2]
    rows = torch.arange(cfg.N, device="cuda")
    obs, info = env.reset()
    finals, ticks = None, None
    for k in range(cfg.T + 1):
        obs, rew, te, tr, info = env.step(table[info["episode_step"].long().clamp(max=cfg.T - 1), rows])
        done = (te | tr).cpu().numpy()
        if done.any():
            assert done.all(), "the scenes all end at the same tick"
            finals = {k2: v.cpu().numpy().copy() for k2, v in info["final"].items()}
            break
    assert finals is not None and not te.any()
    fused = ScenarioGym(timestep=cfg.dt, metrics=std_metrics())
    fused.set_scenarios(scs, create_agent=lambda s, e: ActionTableAgent(e, acts[:, :, scs.index(s), s.entities.index(e)]))
    fused.rollout()
    arr = fused.get_metric_arrays()
    for key in FINAL_KEYS:
        assert np.array_equal(finals[key], arr[key]), key
    assert np.array_equal(finals["tick"], fused._engine.get("tick"))
    assert np.array_equal(finals["t"], fused._engine.get("t"))
    assert np.array_equal(finals["first_coll_tick"], fused._engine.get("first_coll_tick"))
    for n in range(cfg.N):
        out = sub(g, f"veh/{n}/out")
        assert finals["t"][n] == float(out["t_end"])
        assert close(finals["ego_avg_speed"][n], out["ego_avg_speed"])
        assert close(finals["ego_distance_travelled"][n], out["ego_distance_travelled"])


# ---------------------------------------------------------------------------------------------- 2
def _closed_loop(scs, steps_cap=2000, obs=None):
    """Run the steer-to-target policy until every scenario finished once; returns (actions [T, N, A, 2],
    first-episode ticks, finals at the finishing step)."""
    env = VecScenarioEnv([s for _, s, _ in scs], obs=obs or ObsSpec(k_neighbours=4, lookahead=(1.0, 2.0)),
                         state_callbacks=None)
    o, info = env.reset()
    rec, finals, ticks = [], {}, {}
    for _ in range(steps_cap):
        a = steer_to_target(o)
        rec.append(a.clone())
        o, rew, te, tr, info = env.step(a)
        done = (te | tr).cpu().numpy()
        for n in np.nonzero(done)[0]:
            if n not in finals:
                finals[n] = {k: v[n].item() for k, v in info["final"].items()}
        if len(finals) == len(scs):
            break
    return env, torch.stack(rec).cpu().numpy(), finals


def test_closed_loop_replays_through_rollout_and_oracle():
    scs = golden_scenarios()
    env, rec, finals = _closed_loop(scs)
    N = len(scs)
    tables = [rec[: finals[n]["tick"], n, 0, :].astype(np.float64) for n in range(N)]
    gym = ScenarioGym(metrics=std_metrics())
    gym.set_scenarios([s for _, s, _ in scs],
                      create_agent=lambda s, e: ActionTableAgent(e, tables[[x for _, x, _ in scs].index(s)])
                      if e is s.ego else None)
    gym.rollout()
    arr = gym.get_metric_arrays()
    ticks = gym._engine.get("tick")
    for n in range(N):
        assert ticks[n] == finals[n]["tick"], n
        for key in FINAL_KEYS:
            assert arr[key][n] == finals[n][key], (n, key)
    cpu = OracleEngine(gym._engine.scene, gym._params)
    cpu.reset()
    cpu.rollout(-1, actions=gym._action_table_host)
    assert np.array_equal(cpu.get("tick"), ticks)
    for key, f in (("ego_avg_speed", "ego_avg_speed"), ("ego_max_speed", "ego_max_speed"),
                   ("ego_distance_travelled", "ego_dist")):
        assert close(cpu.get(f), [finals[n][key] for n in range(N)]), key
    assert np.array_equal(cpu.get("first_coll_tick"), [finals[n]["first_coll_tick"] for n in range(N)])


# ---------------------------------------------------------------------------------------------- 3
def _device_spec(eng, slots, K, radius, look, road, weights=(1.0, -10.0, -1.0, 0.1, -1.0)):
    N, A = slots.shape
    buf = {"agent_slot": torch.from_numpy(slots).cuda(), "snap_dist": torch.zeros(N * A, dtype=torch.float64).cuda(),
           "snap_collided": torch.zeros(N * A, dtype=torch.uint8).cuda(),
           "snap_pair_ticks": torch.zeros(N, dtype=torch.int64).cuda(), "snap_rss": torch.zeros(N, dtype=torch.uint8).cuda()}
    e = abi.SgEnvSpec()
    e.n_agents, e.k_neighbours, e.radius, e.n_lookahead, e.road = A, K, radius, len(look), int(road)
    for k, v in enumerate(look):
        e.lookahead[k] = v
    for k, v in enumerate(weights):
        e.weights[k] = v
    for k, t in buf.items():
        setattr(e, k, t.data_ptr())
    return e, buf


def _observe_against_oracle(scene, p, actions, slots, K, radius, look, road, ticks):
    gpu, cpu = Engine(scene, p), OracleEnvEngine(scene, p)
    N, A = slots.shape
    F = abi.env_n_features(K, len(look), road)
    e, keep = _device_spec(gpu, slots, K, radius, look, road)
    cpu.env_spec(slots, K, radius, look, road, weights=(1.0, -10.0, -1.0, 0.1, -1.0))
    obs, am = torch.zeros(N, A, F, device="cuda"), torch.zeros(N, A, dtype=torch.uint8, device="cuda")
    rew, terms = torch.zeros(N, A, device="cuda"), torch.zeros(N, A, 5, device="cuda")
    te, tr = torch.zeros(N, dtype=torch.uint8, device="cuda"), torch.zeros(N, dtype=torch.uint8, device="cuda")
    gpu.reset()
    done_ticks = 0
    for k in range(max(ticks) + 1):
        if k in ticks:
            for name, _, _ in abi.STATE_FIELDS:  # observe the device's own state on both sides
                if name not in ("events", "trace_pose", "trace_present", "trace_t", "coll_mask"):
                    cpu.state[name][...] = gpu.get(name).reshape(cpu.state[name].shape)
            gpu.env_observe(e, obs, am)
            want, want_am = cpu.env_observe()
            assert np.array_equal(am.cpu().numpy(), want_am)
            got = obs.cpu().numpy()
            nb = got[..., 4 + 3 * len(look):4 + 3 * len(look) + 10 * K].reshape(N, A, K, 10)
            wnb = want[..., 4 + 3 * len(look):4 + 3 * len(look) + 10 * K].reshape(N, A, K, 10)
            assert np.array_equal(nb[..., 6:], wnb[..., 6:]), "neighbour identities (box, type, valid)"
            np.testing.assert_allclose(got, want, **F32)
            gpu.rollout(1, actions=None if actions is None else actions[k:k + 1])
            for name, _, _ in abi.STATE_FIELDS:
                if name not in ("events", "trace_pose", "trace_present", "trace_t", "coll_mask"):
                    cpu.state[name][...] = gpu.get(name).reshape(cpu.state[name].shape)
            gpu.env_reward(e, rew, terms, te, tr)
            w_rew, w_terms, w_te, w_tr = cpu.env_reward()
            np.testing.assert_allclose(terms.cpu().numpy(), w_terms, **F32)
            np.testing.assert_allclose(rew.cpu().numpy(), w_rew, **F32)
            assert np.array_equal(te.cpu().numpy(), w_te) and np.array_equal(tr.cpu().numpy(), w_tr)
            done_ticks += 1
        else:
            gpu.rollout(1, actions=None if actions is None else actions[k:k + 1])
    assert done_ticks == len(ticks)


def test_observe_and_reward_against_oracle_vehicles():
    cfg = synthetic.vehicles_config(seed=5, N=8, M=64, T=40, half_extent=30.0)
    p = abi.default_params()
    p.timestep = cfg.dt
    slots = np.tile(np.arange(64, dtype=np.int32), (cfg.N, 1))
    _observe_against_oracle(synthetic.pack_synthetic(cfg), p, cfg.actions, slots, 8, 12.0, (0.5, 1.0, 3.0),
                            False, (0, 7, 23, 39))


def test_observe_and_reward_against_oracle_xosc():
    specs = all_xosc_specs("xosc")
    scene = pack_scenarios([s for _, s, _, _ in specs])
    p = abi.default_params()
    slots = np.tile(np.arange(3, dtype=np.int32), (scene.N, 1))
    slots[:, 1:] = np.where(np.arange(2)[None, :] + 1 < np.array([len(o) for _, _, o, _ in specs])[:, None],
                            slots[:, 1:], -1)
    assert (scene.etype == abi.ETYPE_PEDESTRIAN).any()
    _observe_against_oracle(scene, p, None, slots, 6, 0.0, (1.0, 4.0), False, (0, 30, 200))


def test_observe_and_reward_against_oracle_road():
    cfg = golden_cases.veh_cfg()
    scene = synthetic.pack_synthetic(cfg, road_network=golden_cases.road_network(golden_cases.ROAD_VEH_GEOMETRY))
    p = abi.default_params()
    p.timestep, p.terminal = cfg.dt, abi.TERM_MAX_LENGTH | abi.TERM_EGO_OFF_ROAD
    slots = np.tile(np.arange(cfg.M, dtype=np.int32), (cfg.N, 1))
    _observe_against_oracle(scene, p, cfg.actions, slots, 3, 0.0, (1.0,), True, (0, 10, 40))


# ---------------------------------------------------------------------------------------------- 4
def test_termination_head_on_ego_collision():
    ce = CatalogEntry("car", "car", "car", "car", BoundingBox(2.0, 5.0, 0.0, 0.0))
    ego, hazard = Entity(ce, ref="ego"), Entity(ce, ref="entity_1")
    ego.trajectory = Trajectory(np.array([[0.0, 0, 0], [10, 20, 0]]), fields=["t", "x", "y"])
    hazard.trajectory = Trajectory(np.array([[0.0, 40, 0], [10, 20, 0]]), fields=["t", "x", "y"])
    env = VecScenarioEnv([Scenario([ego, hazard])], terminal_conditions=["max_length", "ego_collision"])
    env.reset()
    zero = torch.zeros(1, 1, 2, device="cuda")
    hits = 0
    for k in range(400):
        _, rew, te, tr, info = env.step(zero)
        hits += int(info["terms"][0, 0, 1].item())
        if te.item() or tr.item():
            break
    assert te.item() and not tr.item() and hits == 1
    assert info["final"]["first_coll_tick"][0].item() == info["final"]["tick"][0].item()


def test_termination_off_road_and_max_length():
    cfg = golden_cases.veh_cfg()
    net = golden_cases.road_network(golden_cases.ROAD_VEH_GEOMETRY)
    scs = []
    for n in range(cfg.N):
        sc = vehicle_scenario(cfg, n)
        sc.road_network = net
        scs.append(sc)
    env = VecScenarioEnv(scs, timestep=cfg.dt, terminal_conditions=["max_length", "ego_off_road"],
                         obs=ObsSpec(road=True))
    o, _ = env.reset()
    seen_te = seen_tr = 0
    finished = np.zeros(cfg.N, bool)
    for k in range(cfg.T + 2):
        o, rew, te, tr, info = env.step(steer_to_target(o) * 0.0 + torch.tensor([3.0, 0.3], device="cuda"))
        te_, tr_ = te.cpu().numpy(), tr.cpu().numpy()
        fresh = ~finished & (te_ | tr_)
        seen_te += int(te_[fresh].sum())
        seen_tr += int(tr_[fresh].sum())
        off = info["terms"][:, 0, 2].cpu().numpy()
        assert np.all(off[te_ & fresh] == 1.0), "ego_off_road ends with the ego off the road"
        finished |= te_ | tr_
        if finished.all():
            break
    assert seen_te > 0
    env2 = VecScenarioEnv([s for _, s, _ in golden_scenarios(["a2281876"])])
    o, _ = env2.reset()
    for k in range(400):
        o, rew, te, tr, info = env2.step(steer_to_target(o))
        if te.item() or tr.item():
            break
    assert tr.item() and not te.item() and info["final"]["tick"][0].item() == k + 1


# ---------------------------------------------------------------------------------------------- 5
def test_auto_reset_episodes_repeat():
    scs = golden_scenarios(["a2281876", "a5e43fe4", "fbb6b5ca", "1518e754"])
    env = VecScenarioEnv([s for _, s, _ in scs], obs=ObsSpec(k_neighbours=4, lookahead=(1.0,)))
    N = env.N
    o, info = env.reset()
    obs_log, final_obs, finals, eps = [o.clone()], [], [], []
    for _ in range(2000):
        o, rew, te, tr, info = env.step(steer_to_target(o))
        obs_log.append(o.clone())
        final_obs.append(info["final_obs"].clone())
        finals.append({k: v.clone() for k, v in info["final"].items()})
        eps.append(info["episode"].clone())
        if (info["episode"] >= 2).all().item():
            break
    eps = torch.stack(eps).cpu().numpy()
    obs_log = torch.stack(obs_log).cpu().numpy()
    final_obs = torch.stack(final_obs).cpu().numpy()
    assert (eps[-1] >= 2).all()
    for n in range(N):
        ends = np.nonzero(np.diff(np.concatenate([[0], eps[:, n]])))[0]  # steps at which episodes ended
        L1, L2 = ends[0] + 1, ends[1] - ends[0]
        assert L1 == L2, "episodes of one scenario under a deterministic policy have one length"
        # obs_log[k] is the observation after k steps; episode 2 starts at obs_log[L1]
        assert np.array_equal(obs_log[:L1, n], obs_log[L1:2 * L1, n]), n
        assert np.array_equal(final_obs[ends[0], n], final_obs[ends[1], n])
        # without a reset, final_obs is the observation itself
        assert np.array_equal(final_obs[ends[0] - 1, n], obs_log[ends[0], n])
        for k in finals[0]:
            assert finals[ends[0]][k][n].item() == finals[ends[1]][k][n].item(), (n, k)
    # the longest scenario never finishes while the others reset around it: == a run with it alone
    longest = int(np.argmax([np.nonzero(eps[:, n])[0][0] for n in range(N)]))
    alone = VecScenarioEnv([scs[longest][1]], obs=ObsSpec(k_neighbours=4, lookahead=(1.0,)))
    o, _ = alone.reset()
    first_end = int(np.nonzero(eps[:, longest])[0][0])
    for k in range(first_end):
        assert np.array_equal(o[0].cpu().numpy(), obs_log[k, longest]), k
        o, *_ = alone.step(steer_to_target(o))


# ---------------------------------------------------------------------------------------------- 6
def _scenario_view(name, a, n, M):
    spec = dict((f, s) for f, _, s in abi.STATE_FIELDS)[name]
    if "NM" in spec:
        return a[..., n * M:(n + 1) * M]
    if spec[0] == "N":
        return a[n]
    return None


@pytest.mark.parametrize("which", ["vehicles", "general"])
def test_reset_scenarios_on_device(which):
    if which == "vehicles":
        cfg = golden_cases.rss_cfg()
        scene, actions = synthetic.pack_synthetic(cfg), cfg.actions
        p = abi.default_params()
        p.timestep, p.features = cfg.dt, p.features | abi.FEAT_RSS
        ticks = 25
    else:
        scene, actions = pack_scenarios([s for _, s, _, _ in all_xosc_specs("xosc")]), None
        p, ticks = abi.default_params(), 100
    eng, ref = Engine(scene, p), Engine(scene, p)
    ref.reset()
    eng.reset()
    eng.rollout(ticks, actions=actions)
    before = {name: eng.get(name).copy() for name, _, _ in abi.STATE_FIELDS}
    mask = (np.arange(scene.N) % 3 == 1).astype(np.uint8)
    eng.reset(mask=torch.from_numpy(mask).cuda())
    assert eng.get("event_count")[0] == before["event_count"][0]
    for name, _, _ in abi.STATE_FIELDS:
        if name == "coll_mask":  # (not allocated without the pair matrix)
            continue
        got_all, ref_all = eng.get(name), ref.get(name)
        for n in range(scene.N):
            got = _scenario_view(name, got_all, n, scene.M)
            if got is None:
                continue
            want = _scenario_view(name, ref_all if mask[n] else before[name], n, scene.M)
            assert np.array_equal(got, want, equal_nan=True), (which, name, n)


# ---------------------------------------------------------------------------------------------- 7
def test_no_host_synchronisation():
    cfg = synthetic.vehicles_config(seed=2, N=16, M=8, T=30, half_extent=20.0)
    env = VecScenarioEnv([vehicle_scenario(cfg, n) for n in range(cfg.N)],
                         create_agent=lambda s, e: PolicyAgent(e), timestep=cfg.dt)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        o, info = env.reset()
        for _ in range(10):
            o, rew, te, tr, info = env.step(steer_to_target(o))
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    assert torch.isfinite(o).all()


# ---------------------------------------------------------------------------------------------- 8
def test_argument_checks():
    scs = [s for _, s, _ in golden_scenarios(["a2281876"])]
    env = VecScenarioEnv(scs)
    env.reset()
    good = torch.zeros(1, 1, 2, device="cuda")
    for bad in (torch.zeros(1, 2, 2, device="cuda"), good.to(torch.float16), good.to(torch.int32), good.cpu(),
                np.zeros((1, 1, 2))):
        with pytest.raises(ValueError):
            env.step(bad)
    env.step(good.double())

    class Watch(Metric):
        def _reset(self, state):
            pass

        def _step(self, state):
            pass

        def get_state(self):
            return None

    from scenario_gym_b200 import Agent, EgoLocalizationSensor, StateCallback, VehicleController

    class HostPolicy(Agent):
        def __init__(self, entity):
            super().__init__(entity, VehicleController(entity), EgoLocalizationSensor(entity))

    with pytest.raises(NotImplementedError):
        VecScenarioEnv(scs, create_agent=lambda s, e: HostPolicy(e) if e is s.ego else None)
    with pytest.raises(NotImplementedError):
        VecScenarioEnv(scs, state_callbacks=[StateCallback()])
    with pytest.raises(NotImplementedError):
        VecScenarioEnv(scs, terminal_conditions=["max_length", lambda st: False])
    with pytest.raises(NotImplementedError):
        VecScenarioEnv(scs, record=True)
    gym = ScenarioGym(metrics=[Watch()])
    gym.set_scenarios(scs, create_agent=lambda s, e: PolicyAgent(e) if e is s.ego else None)
    with pytest.raises(RuntimeError, match="VecScenarioEnv"):
        gym.rollout()
    with pytest.raises(RuntimeError, match="VecScenarioEnv"):
        gym.step()
