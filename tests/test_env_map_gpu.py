"""
GPU tests of the map block of sg_env_observe (sg_env_map_kernel): the device against the brute-force oracle
(tests/map_oracle.c) on vehicle scenes over a town, the crafted exact cases bit for bit, agents on cell
boundaries, a long edge spanning many cells, several networks in one batch, and the block through VecScenarioEnv
(the other blocks unchanged, auto-reset and final_obs, no host synchronisation, branches, argument checks).
"""
import dataclasses
import math

import numpy as np
import pytest
import torch

from scenario_gym_b200 import (BoundingBox, CatalogEntry, ObsSpec, PolicyAgent, Scenario, Trajectory,
                               VecScenarioEnv, Vehicle, abi, synthetic)
from scenario_gym_b200.engine import Engine
from scenario_gym_b200.packing import pack_road_networks
from scenario_gym_b200.road_network import PolygonArea, Road, RoadNetwork

from map_oracle import MapOracleEngine
from test_env_map_cpu import RN_FIELDS, crafted_network, crafted_state

pytestmark = pytest.mark.gpu
F32 = dict(rtol=2e-6, atol=2e-5)
SKIP = ("events", "trace_pose", "trace_present", "trace_t", "coll_mask")


def _device_spec(scene, slots, Km, radius, table, K=2, look=(1.0,)):
    N, A = slots.shape
    buf = {"agent_slot": torch.from_numpy(slots).cuda(), "snap_dist": torch.zeros(N * A, dtype=torch.float64).cuda(),
           "snap_collided": torch.zeros(N * A, dtype=torch.uint8).cuda(),
           "snap_pair_ticks": torch.zeros(N, dtype=torch.int64).cuda(), "snap_rss": torch.zeros(N, dtype=torch.uint8).cuda()}
    for k in abi.MAP_FIELDS:
        a = table[k] if table[k].size else np.zeros((1,) + table[k].shape[1:], table[k].dtype)
        buf[k] = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    e = abi.SgEnvSpec()
    e.n_agents, e.k_neighbours, e.radius, e.n_lookahead = A, K, 0.0, len(look)
    for k, v in enumerate(look):
        e.lookahead[k] = v
    for k, t in buf.items():
        setattr(e, k, t.data_ptr())
    e.map_edges, e.map_radius, e.map_networks = Km, radius, scene.n_networks
    return e, buf


def _copy_state(gpu, cpu):
    for name, _, _ in abi.STATE_FIELDS:
        if name not in SKIP:
            cpu.state[name][...] = gpu.get(name).reshape(cpu.state[name].shape)


def _check_map(got, want, Km):
    """Device vs oracle map blocks [..., 10 Km]: flag and valid columns equal, coordinates within fp32 rounding
    (the device's sincos against libm's cos / sin)."""
    g, w = got.reshape(-1, Km, 10), want.reshape(-1, Km, 10)
    assert np.array_equal(g[..., 6:], w[..., 6:])
    np.testing.assert_allclose(g[..., :6], w[..., :6], **F32)
    return int(w[..., 9].sum())


def _map_against_oracle(scene, p, actions, slots, Km, radius, ticks, cell=None):
    gpu, cpu = Engine(scene, p), MapOracleEngine(scene, p)
    N, A = slots.shape
    table = abi.map_table(scene.rn_poly_off, scene.rn_edge_off, scene.rn_edges, radius, cell=cell)
    e, keep = _device_spec(scene, slots, Km, radius, table)
    _, F = cpu.env_spec(slots, 2, 0.0, (1.0,), map_edges=Km, map_radius=radius, table=table)
    obs, am = torch.zeros(N, A, F, device="cuda"), torch.zeros(N, A, dtype=torch.uint8, device="cuda")
    gpu.reset()
    found = 0
    for k in range(max(ticks) + 1):
        if k in ticks:
            _copy_state(gpu, cpu)
            gpu.env_observe(e, obs, am)
            want, want_am = cpu.env_observe()
            got = obs.cpu().numpy()
            assert np.array_equal(am.cpu().numpy(), want_am)
            F0 = F - 10 * Km
            np.testing.assert_allclose(got[..., :F0], want[..., :F0], **F32)
            found += _check_map(got[..., F0:], want[..., F0:], Km)
        if k < max(ticks):
            gpu.rollout(1, actions=None if actions is None else actions[k:k + 1])
    assert found > 0, "the agents must see edges"
    return found


@pytest.mark.parametrize("Km", [1, 8, 32])
def test_map_against_oracle_town_vehicles(Km):
    town = synthetic.grid_town(seed=0)
    cfg = synthetic.vehicles_config(seed=5, N=6, M=64, T=24, half_extent=200.0)
    scene = synthetic.pack_synthetic(cfg, road_network=town)
    p = abi.default_params()
    p.timestep = cfg.dt
    slots = np.tile(np.arange(64, dtype=np.int32), (cfg.N, 1))
    slots[1, 5:] = -1  # padding agents
    _map_against_oracle(scene, p, cfg.actions, slots, Km, 30.0, (0, 9, 23))


def test_map_crafted_bit_equal():
    """Heading 0: the crafted exact cases read the same bits on the device as on the oracle."""
    for Km, radius in ((1, 20.0), (8, 5.0), (32, 20.0)):
        scene, pose, present, slots = crafted_state()
        p = abi.default_params()
        gpu, cpu = Engine(scene, p), MapOracleEngine(scene, p)
        gpu.reset()
        gpu.tensor("pose").copy_(torch.from_numpy(pose).reshape(gpu.tensor("pose").shape))
        gpu.tensor("present").copy_(torch.from_numpy(present).reshape(gpu.tensor("present").shape))
        cpu.reset()
        cpu.state["pose"][...] = pose
        cpu.state["present"][...] = present
        N, A = slots.shape
        table = abi.map_table(scene.rn_poly_off, scene.rn_edge_off, scene.rn_edges, radius)
        e, keep = _device_spec(scene, slots, Km, radius, table, K=1, look=())
        _, F = cpu.env_spec(slots, 1, 0.0, (), map_edges=Km, map_radius=radius)
        obs, am = torch.zeros(N, A, F, device="cuda"), torch.zeros(N, A, dtype=torch.uint8, device="cuda")
        gpu.env_observe(e, obs, am)
        want, _ = cpu.env_observe()
        got = obs.cpu().numpy()
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (Km, radius)
        assert not got[:, 1:].any() and not got[-1, :, -10 * Km:].any()  # absent / padding agents, no network
        if radius > 5.0:  # (at radius 5 "parallel" and "outside" have every edge at d2 == r * r: nothing selected)
            assert got[:-1, 0, -10 * Km + 9].all()
        else:
            assert np.array_equal(got[:-1, 0, -10 * Km + 9], [1, 1, 0, 0])


@pytest.mark.parametrize("cell", [None, 4.0, math.inf])
def test_map_agents_on_cell_boundaries(cell):
    town = synthetic.grid_town(seed=2, half_extent=60.0)
    cfg = synthetic.vehicles_config(seed=1, N=4, M=32, T=4, half_extent=60.0)
    scene = synthetic.pack_synthetic(cfg, road_network=town)
    radius = 12.0
    t = abi.map_table(scene.rn_poly_off, scene.rn_edge_off, scene.rn_edges, radius, cell=cell)
    ox, oy, c, _ = t["map_grid"][0]
    nx, ny, _ = t["map_dims"][0]
    rng = np.random.default_rng(0)
    gpu = Engine(scene, abi.default_params())
    gpu.reset()
    pose = gpu.get("pose").reshape(6, -1)
    k = pose.shape[1]
    step = c if math.isfinite(c) else 4.0
    i, j = rng.integers(0, min(nx, 30) + 1, k), rng.integers(0, min(ny, 30) + 1, k)
    pose[0], pose[1] = ox + i * step, oy + j * step  # cell corners
    pose[0, ::3] += radius  # the query square's edge on a boundary
    pose[1, 1::3] = rng.uniform(-60, 60, len(pose[1, 1::3]))
    pose[3] = rng.uniform(-np.pi, np.pi, k)
    cpu = MapOracleEngine(scene, abi.default_params())
    cpu.reset()
    gpu.tensor("pose").copy_(torch.from_numpy(pose).reshape(gpu.tensor("pose").shape))
    _copy_state(gpu, cpu)
    slots = np.tile(np.arange(32, dtype=np.int32), (cfg.N, 1))
    e, keep = _device_spec(scene, slots, 16, radius, t)
    _, F = cpu.env_spec(slots, 2, 0.0, (1.0,), map_edges=16, map_radius=radius, table=t)
    obs, am = torch.zeros(cfg.N, 32, F, device="cuda"), torch.zeros(cfg.N, 32, dtype=torch.uint8, device="cuda")
    gpu.env_observe(e, obs, am)
    want, _ = cpu.env_observe()
    assert _check_map(obs.cpu().numpy()[..., F - 160:], want[..., F - 160:], 16) > 0


def test_map_long_edge_appears_once():
    """A 2 km road (its long edges span hundreds of cells) nearest to agents along it: each edge appears once."""
    long_road = Road("long", PolygonArea([(-1000.0, -2.0), (1000.0, -2.0), (1000.0, 2.0), (-1000.0, 2.0)]))
    small = Road("small", PolygonArea([(5.0, 10.0), (7.0, 10.0), (7.0, 12.0), (5.0, 12.0)]))
    net = RoadNetwork(roads=[long_road, small])
    cfg = synthetic.vehicles_config(seed=3, N=2, M=16, T=4, half_extent=1.0)
    scene = synthetic.pack_synthetic(cfg, road_network=net)
    gpu = Engine(scene, abi.default_params())
    gpu.reset()
    pose = gpu.get("pose").reshape(6, -1)
    pose[0] = np.linspace(-900.0, 900.0, pose.shape[1])
    pose[1] = np.linspace(-1.0, 3.0, pose.shape[1])
    pose[3] = 0.0
    gpu.tensor("pose").copy_(torch.from_numpy(pose).reshape(gpu.tensor("pose").shape))
    cpu = MapOracleEngine(scene, abi.default_params())
    cpu.reset()
    _copy_state(gpu, cpu)
    slots = np.tile(np.arange(16, dtype=np.int32), (cfg.N, 1))
    t = abi.map_table(scene.rn_poly_off, scene.rn_edge_off, scene.rn_edges, 8.0, cell=2.0)
    assert t["map_dims"][0, 0] > 500
    e, keep = _device_spec(scene, slots, 8, 8.0, t)
    _, F = cpu.env_spec(slots, 2, 0.0, (1.0,), map_edges=8, map_radius=8.0, table=t)
    obs, am = torch.zeros(cfg.N, 16, F, device="cuda"), torch.zeros(cfg.N, 16, dtype=torch.uint8, device="cuda")
    gpu.env_observe(e, obs, am)
    got, (want, _) = obs.cpu().numpy(), cpu.env_observe()
    got, want = got[..., F - 80:].reshape(-1, 8, 10), want[..., F - 80:].reshape(-1, 8, 10)
    assert np.array_equal(got[..., 6:], want[..., 6:])
    np.testing.assert_allclose(got, want, **F32)
    for row in got:
        ends = [tuple(r[2:6]) for r in row if r[9]]
        assert len(ends) == len(set(ends)) >= 2, "each edge once; both long sides within 8 m"


def test_map_several_networks_in_one_batch():
    t1, t2 = synthetic.grid_town(seed=4, half_extent=50.0), synthetic.grid_town(seed=5, half_extent=50.0)
    cfg = synthetic.vehicles_config(seed=6, N=6, M=16, T=12, half_extent=50.0)
    scene = synthetic.pack_synthetic(cfg)
    nets = [t1, None, t2, crafted_network(), None, t1]
    scene = dataclasses.replace(scene, **dict(zip(RN_FIELDS, pack_road_networks(nets))))
    assert scene.n_networks == 3
    p = abi.default_params()
    p.timestep = cfg.dt
    slots = np.tile(np.arange(16, dtype=np.int32), (cfg.N, 1))
    _map_against_oracle(scene, p, cfg.actions, slots, 8, 20.0, (0, 11))


# ---------------------------------------------------------------------------------------------- env level
def _vehicle_scenes(seed=2, N=6, M=16, town=True, half_extent=40.0):
    cfg = synthetic.vehicles_config(seed=seed, N=N, M=M, T=30, half_extent=half_extent)
    rows = synthetic.two_knot_rows(cfg).reshape(cfg.N, cfg.M, 2, 7)
    ce = CatalogEntry(None, "car1", "car", "Vehicle", BoundingBox(*synthetic.CAR1_BOX))
    rn = synthetic.grid_town(seed=seed, half_extent=half_extent + 20.0) if town else None
    return cfg, [Scenario([Vehicle(ce, trajectory=Trajectory(rows[n, m]), ref="ego" if m == 0 else f"entity_{m}")
                           for m in range(cfg.M)], road_network=rn if n != 1 else None) for n in range(cfg.N)]


def _policy(obs):
    tx, ty = obs[..., 4], obs[..., 5]
    return torch.stack([(torch.sqrt(tx * tx + ty * ty) - obs[..., 0]).clamp(-5.0, 5.0),
                        torch.atan2(ty, tx).clamp(-0.7, 0.7)], -1)


def _make(scs, cfg, **obs):
    return VecScenarioEnv(scs, create_agent=lambda s, e: PolicyAgent(e), timestep=cfg.dt, obs=ObsSpec(**obs))


def _oracle_for(env):
    cpu = MapOracleEngine(env._engine.scene, env._engine.params)
    o = env.obs_spec
    cpu.env_spec(env._slots_host, o.k_neighbours, o.radius, tuple(o.lookahead), o.road, n_rays=o.lidar_rays,
                 ray_range=o.lidar_range, map_edges=o.map_edges, map_radius=o.map_radius)
    return cpu


def test_env_map_with_lidar_and_other_blocks():
    cfg, scs = _vehicle_scenes()
    base = dict(k_neighbours=4, lookahead=(1.0, 2.0), road=True)
    plain = _make(scs, cfg, **base)
    zero = _make(scs, cfg, **base, map_edges=0)
    lid = _make(scs, cfg, **base, lidar_rays=16)
    both = _make(scs, cfg, **base, lidar_rays=16, map_edges=8, map_radius=25.0)
    F0 = plain.n_features
    assert zero.n_features == F0 and both.n_features == F0 + 80 + 16
    cpu = _oracle_for(both)
    obs = [env.reset()[0] for env in (plain, zero, lid, both)]
    seen = 0
    for k in range(cfg.T + 6):
        o0, oz, ol, ob = (o.cpu().numpy() for o in obs)
        assert np.array_equal(oz.view(np.uint32), o0.view(np.uint32)), k
        assert np.array_equal(ob[..., :F0].view(np.uint32), o0.view(np.uint32)), k
        assert np.array_equal(ob[..., -16:].view(np.uint32), ol[..., -16:].view(np.uint32)), k
        _copy_state(both._engine, cpu)
        want, _ = cpu.env_observe()
        seen += _check_map(ob[..., F0:F0 + 80], want[..., F0:F0 + 80], 8)
        a = _policy(obs[0])
        outs = [env.step(a) for env in (plain, zero, lid, both)]
        obs = [out[0] for out in outs]
    assert seen > 0


def test_env_map_step_auto_reset_final_obs_no_sync():
    cfg, scs = _vehicle_scenes(seed=3, N=8, M=8)
    env = _make(scs, cfg, k_neighbours=2, lookahead=(1.0,), map_edges=16, map_radius=30.0)
    cpu = _oracle_for(env)
    F, F0 = env.n_features, env.n_features - 160
    o, _ = env.reset()
    resets = 0
    for k in range(cfg.T + 4):
        a = _policy(o)
        torch.cuda.synchronize()
        torch.cuda.set_sync_debug_mode("error")
        try:
            o, rew, te, tr, info = env.step(a)
        finally:
            torch.cuda.set_sync_debug_mode("default")
        fin = (te | tr).cpu().numpy()
        resets += int(fin.sum())
        # obs after the masked observe of the reset scenarios, against the oracle on the env's state
        _copy_state(env._engine, cpu)
        want, _ = cpu.env_observe()
        _check_map(o.cpu().numpy()[..., F0:], want[..., F0:], 16)
        if fin.any():  # final_obs of the finished scenarios holds the block of their last state (nonzero)
            assert info["final_obs"][torch.from_numpy(fin).cuda()][..., F0 + 9::10].sum() > 0
    assert resets > 0, "the run must cover auto-reset"


def test_branches_final_obs_include_map():
    cfg, scs = _vehicle_scenes(seed=5, N=4, M=8)
    env = _make(scs, cfg, k_neighbours=2, lookahead=(1.0,), map_edges=8, map_radius=30.0)
    o, _ = env.reset()
    for _ in range(3):
        o, *_ = env.step(_policy(o))
    B, H = 3, 5
    br = env.branches(B, H, final_obs=True)
    acts = torch.randn(env.N, B, H, env.A, 2, device="cuda") * 0.5
    out = br.run(acts)
    assert out["final_obs"].shape[-1] == env.n_features
    cpu = _oracle_for(env)
    F0 = env.n_features - 80
    seen = 0
    for b, eng in enumerate(br.engines):
        _copy_state(eng, cpu)
        want, _ = cpu.env_observe()
        seen += _check_map(out["final_obs"][:, b].cpu().numpy()[..., F0:], want[..., F0:], 8)
    assert seen > 0


def test_map_argument_checks():
    cfg, scs = _vehicle_scenes(N=2, M=4)
    for bad in (dict(map_edges=-1), dict(map_edges=33), dict(map_edges=2.5), dict(map_edges=4, map_radius=0.0),
                dict(map_edges=4, map_radius=-1.0), dict(map_edges=4, map_radius=math.inf),
                dict(map_edges=4, map_radius=math.nan)):
        with pytest.raises(ValueError):
            _make(scs, cfg, **bad)
    env = _make(scs, cfg, map_edges=4, map_radius=10.0)
    env.reset()
    eng = env._engine
    for field, value, msg in (("map_edges", 33, "map_edges"), ("map_edges", -1, "map_edges"),
                              ("map_radius", 0.0, "map_radius"), ("map_radius", math.nan, "map_radius"),
                              ("map_networks", 0, "map_networks"), ("map_seg", None, "map table"),
                              ("map_cell_edge", None, "map table")):
        spec = abi.SgEnvSpec.from_buffer_copy(env._spec)
        setattr(spec, field, value)
        with pytest.raises(RuntimeError, match=msg):
            eng.env_observe(spec, env._obs, env._agent_mask)
