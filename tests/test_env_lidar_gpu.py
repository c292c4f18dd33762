"""
GPU tests of the lidar block of sg_env_observe (sg_env_lidar_kernel): the device against the oracle on the
device's own state (vehicles, the reference's test scenes, a 1024-slot crowd in agent chunks), the crafted
exact cases bit for bit, and the lidar through VecScenarioEnv (shapes, the other columns unchanged, auto-reset,
no host synchronisation, argument checks).
"""
import math

import numpy as np
import pytest
import torch

from scenario_gym_b200 import (BoundingBox, CatalogEntry, ObsSpec, PolicyAgent, Scenario, Trajectory,
                               VecScenarioEnv, Vehicle, abi, synthetic)
from scenario_gym_b200.engine import Engine
from scenario_gym_b200.packing import pack_scenarios

from helpers import all_xosc_specs
from lidar_oracle import LidarOracleEngine
from test_env_lidar_cpu import DIRS4, DIRS8, NAMES, RANGE, crafted_expected, crafted_state, slab_terms

pytestmark = pytest.mark.gpu
F32 = dict(rtol=2e-6, atol=2e-5)
SKIP = ("events", "trace_pose", "trace_present", "trace_t", "coll_mask")


def _device_spec(slots, R, ray_range, ray_dir, K=2, look=(1.0,)):
    N, A = slots.shape
    buf = {"agent_slot": torch.from_numpy(slots).cuda(), "snap_dist": torch.zeros(N * A, dtype=torch.float64).cuda(),
           "snap_collided": torch.zeros(N * A, dtype=torch.uint8).cuda(),
           "snap_pair_ticks": torch.zeros(N, dtype=torch.int64).cuda(), "snap_rss": torch.zeros(N, dtype=torch.uint8).cuda(),
           "ray_dir": torch.from_numpy(np.ascontiguousarray(ray_dir, np.float64)).cuda()}
    e = abi.SgEnvSpec()
    e.n_agents, e.k_neighbours, e.radius, e.n_lookahead = A, K, 0.0, len(look)
    for k, v in enumerate(look):
        e.lookahead[k] = v
    for k, t in buf.items():
        setattr(e, k, t.data_ptr())
    e.n_rays, e.ray_range = R, ray_range
    return e, buf


def _copy_state(gpu, cpu):
    for name, _, _ in abi.STATE_FIELDS:
        if name not in SKIP:
            cpu.state[name][...] = gpu.get(name).reshape(cpu.state[name].shape)


def _check_lidar(scene, st, slots, got, want, ray_dir, ray_range):
    """Device vs oracle readings [N, A, R]: equal within F32 except on grazing rays, whose slab margin (some
    box's exit - enter, relative) is below 1e-9; such rays must be rare.  Returns the number of grazing rays."""
    bad = ~np.isclose(got, want, **F32)
    for n, a, k in zip(*np.nonzero(bad)):
        enter, exit_, _ = slab_terms(scene, st, n, slots[n, a], ray_dir[k:k + 1])
        reach = max(float(got[n, a, k]), float(want[n, a, k])) * (1 + 1e-6) + 1e-6
        near = (exit_[:, 0] >= -1e-9) & (np.maximum(enter[:, 0], 0.0) <= reach)
        scale = np.maximum(1.0, np.maximum(np.abs(enter[:, 0]), np.abs(exit_[:, 0])))
        margin = np.abs(exit_[:, 0] - enter[:, 0]) / scale
        assert near.any() and margin[near].min() < 1e-9, (n, a, k, got[n, a, k], want[n, a, k])
    assert bad.sum() <= max(2, got.size // 10000), f"{bad.sum()} grazing mismatches of {got.size}"
    return int(bad.sum())


def _lidar_against_oracle(scene, p, actions, slots, R, ticks, ray_range=RANGE):
    gpu, cpu = Engine(scene, p), LidarOracleEngine(scene, p)
    N, A = slots.shape
    dirs = abi.lidar_directions(R)
    e, keep = _device_spec(slots, R, ray_range, dirs)
    _, F = cpu.env_spec(slots, 2, 0.0, (1.0,), n_rays=R, ray_range=ray_range)
    obs, am = torch.zeros(N, A, F, device="cuda"), torch.zeros(N, A, dtype=torch.uint8, device="cuda")
    gpu.reset()
    hits = 0
    for k in range(max(ticks) + 1):
        if k in ticks:
            _copy_state(gpu, cpu)
            gpu.env_observe(e, obs, am)
            want, want_am = cpu.env_observe()
            got = obs.cpu().numpy()
            assert np.array_equal(am.cpu().numpy(), want_am)
            np.testing.assert_allclose(got[..., :F - R], want[..., :F - R], **F32)
            _check_lidar(scene, cpu.state, slots, got[..., F - R:], want[..., F - R:], dirs, ray_range)
            hits += int((want[..., F - R:][want_am.astype(bool)] < ray_range).sum())
        gpu.rollout(1, actions=None if actions is None else actions[k:k + 1])
    assert hits > 0, "the rays must hit something"


def test_lidar_against_oracle_vehicles():
    cfg = synthetic.vehicles_config(seed=5, N=8, M=64, T=40, half_extent=30.0)
    p = abi.default_params()
    p.timestep = cfg.dt
    slots = np.tile(np.arange(64, dtype=np.int32), (cfg.N, 1))
    _lidar_against_oracle(synthetic.pack_synthetic(cfg), p, cfg.actions, slots, 64, (0, 7, 23, 39))


def test_lidar_against_oracle_xosc_ego():
    specs = all_xosc_specs("xosc")
    scene = pack_scenarios([s for _, s, _, _ in specs])
    assert (scene.etype == abi.ETYPE_PEDESTRIAN).any()
    slots = np.asarray(scene.ego_slot, np.int32).reshape(-1, 1)
    _lidar_against_oracle(scene, abi.default_params(), None, slots, 256, (0, 30, 200))


def test_lidar_against_oracle_crowd_chunks():
    """1024 slots, every one an agent, R = 256: the agents are split over several CTAs per scenario."""
    cfg = synthetic.crowd_config(seed=3, N=1, M=1024, T=8)
    scene = synthetic.pack_synthetic(cfg)
    p = abi.default_params()
    p.timestep = cfg.dt
    slots = np.arange(1024, dtype=np.int32).reshape(1, 1024)
    _lidar_against_oracle(scene, p, None, slots, 256, (0, 3), ray_range=30.0)


@pytest.mark.parametrize("offset", [0.0, 1e5])
@pytest.mark.parametrize("R", [4, 8])
def test_lidar_crafted_bit_equal(R, offset):
    """The crafted exact cases (boxes ahead / behind straddling rays 0 and R/2, corners, edges, inside, range,
    flat and point boxes, absent slots and agents) read the same bits on the device as on the oracle."""
    dirs = DIRS4 if R == 4 else DIRS8
    scene, pose, present, slots = crafted_state(offset)
    p = abi.default_params()
    gpu, cpu = Engine(scene, p), LidarOracleEngine(scene, p)
    gpu.reset()
    gpu.tensor("pose").copy_(torch.from_numpy(pose).reshape(gpu.tensor("pose").shape))
    gpu.tensor("present").copy_(torch.from_numpy(present).reshape(gpu.tensor("present").shape))
    cpu.reset()
    cpu.state["pose"][...] = pose
    cpu.state["present"][...] = present
    N, A = slots.shape
    e, keep = _device_spec(slots, R, RANGE, dirs, K=1, look=())
    _, F = cpu.env_spec(slots, 1, 0.0, (), n_rays=R, ray_range=RANGE, ray_dir=dirs)
    obs, am = torch.zeros(N, A, F, device="cuda"), torch.zeros(N, A, dtype=torch.uint8, device="cuda")
    gpu.env_observe(e, obs, am)
    want, _ = cpu.env_observe()
    got = obs.cpu().numpy()
    assert np.array_equal(got[..., -R:].view(np.uint32), want[..., -R:].view(np.uint32))
    exp = crafted_expected(R)
    for n, name in enumerate(NAMES):
        assert np.array_equal(got[n, 0, -R:], exp[name]), name
    assert not got[:, 1:].any()


# ---------------------------------------------------------------------------------------------- env level
def _vehicle_scenes(seed=2, N=6, M=16):
    cfg = synthetic.vehicles_config(seed=seed, N=N, M=M, T=30, half_extent=20.0)
    rows = synthetic.two_knot_rows(cfg).reshape(cfg.N, cfg.M, 2, 7)
    ce = CatalogEntry(None, "car1", "car", "Vehicle", BoundingBox(*synthetic.CAR1_BOX))
    return cfg, [Scenario([Vehicle(ce, trajectory=Trajectory(rows[n, m]), ref="ego" if m == 0 else f"entity_{m}")
                           for m in range(cfg.M)]) for n in range(cfg.N)]


def _policy(obs):
    tx, ty = obs[..., 4], obs[..., 5]
    return torch.stack([(torch.sqrt(tx * tx + ty * ty) - obs[..., 0]).clamp(-5.0, 5.0),
                        torch.atan2(ty, tx).clamp(-0.7, 0.7)], -1)


def test_env_lidar_columns_and_auto_reset():
    cfg, scs = _vehicle_scenes()
    R = 32
    spec = dict(k_neighbours=4, lookahead=(1.0, 2.0))
    plain = VecScenarioEnv(scs, create_agent=lambda s, e: PolicyAgent(e), timestep=cfg.dt, obs=ObsSpec(**spec))
    lid = VecScenarioEnv(scs, create_agent=lambda s, e: PolicyAgent(e), timestep=cfg.dt,
                         obs=ObsSpec(**spec, lidar_rays=R, lidar_range=40.0))
    F0 = plain.n_features
    assert lid.n_features == F0 + R
    cpu = LidarOracleEngine(lid._engine.scene, lid._engine.params)
    cpu.env_spec(lid._slots_host, 4, lid.obs_spec.radius, (1.0, 2.0), n_rays=R, ray_range=40.0)
    o0, _ = plain.reset()
    o1, _ = lid.reset()
    assert tuple(o1.shape) == (lid.N, lid.A, F0 + R)
    resets = 0
    dirs = abi.lidar_directions(R)
    for k in range(cfg.T + 8):
        assert np.array_equal(o1[..., :F0].cpu().numpy().view(np.uint32), o0.cpu().numpy().view(np.uint32)), k
        _copy_state(lid._engine, cpu)
        want, _ = cpu.env_observe()
        got = o1.cpu().numpy()
        _check_lidar(cpu.scene, cpu.state, lid._slots_host, got[..., F0:], want[..., F0:], dirs, 40.0)
        a = _policy(o0)
        o0, _, te0, tr0, _ = plain.step(a)
        o1, _, te1, tr1, info = lid.step(a)
        assert torch.equal(te0, te1) and torch.equal(tr0, tr1)
        resets += int((te1 | tr1).sum().item())
    assert resets > 0, "the run must cover the observation of scenarios just reset"


def test_env_lidar_no_host_synchronisation():
    cfg, scs = _vehicle_scenes(seed=4, N=8, M=8)
    env = VecScenarioEnv(scs, create_agent=lambda s, e: PolicyAgent(e), timestep=cfg.dt,
                         obs=ObsSpec(lidar_rays=64))
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        o, info = env.reset()
        for _ in range(10):
            o, rew, te, tr, info = env.step(_policy(o))
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    assert torch.isfinite(o).all() and (o[..., -64:] <= 50.0).all()


def test_lidar_argument_checks():
    cfg, scs = _vehicle_scenes(N=1, M=4)
    for bad in (dict(lidar_rays=-1), dict(lidar_rays=257), dict(lidar_rays=8, lidar_range=0.0),
                dict(lidar_rays=8, lidar_range=-1.0), dict(lidar_rays=8, lidar_range=math.inf),
                dict(lidar_rays=8, lidar_range=math.nan)):
        with pytest.raises(ValueError):
            VecScenarioEnv(scs, obs=ObsSpec(**bad))
    env = VecScenarioEnv(scs, obs=ObsSpec(lidar_rays=256, lidar_range=1.0))
    env.reset()
    eng = env._engine
    for field, value, msg in (("n_rays", 257, "n_rays"), ("n_rays", -1, "n_rays"), ("ray_range", 0.0, "ray_range"),
                              ("ray_range", math.nan, "ray_range"), ("ray_dir", None, "ray_dir")):
        spec = abi.SgEnvSpec.from_buffer_copy(env._spec)
        setattr(spec, field, value)
        with pytest.raises(RuntimeError, match=msg):
            eng.env_observe(spec, env._obs, env._agent_mask)
