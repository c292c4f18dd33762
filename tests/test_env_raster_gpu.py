"""
GPU tests of sg_env_raster (sg_env_raster_kernel): the device against the brute-force oracle (tests/raster_oracle.c)
bit for bit on the crafted cases with every heading 0, and on vehicle scenes over a town with random headings, where
a pixel may differ only if its centre lies within 1e-6 m of a ring or box edge (the device's sincos against libm's
cos / sin); several networks in one batch, a scene of more than 256 slots, a long polygon, polygons at the culling
bounds, the masked call, the raster through VecScenarioEnv (nothing else changes, final_raster, the rasters of
reset scenarios, no host synchronisation or allocation) and the argument checks.
"""
import dataclasses
import math

import numpy as np
import pytest
import torch

from scenario_gym_b200 import (BoundingBox, CatalogEntry, ObsSpec, PolicyAgent, ResetSpec, Scenario, Trajectory,
                               VecScenarioEnv, Vehicle, abi, synthetic)
from scenario_gym_b200.engine import Engine
from scenario_gym_b200.packing import pack_road_networks
from scenario_gym_b200.road_network import PolygonArea, Road, RoadNetwork

from raster_oracle import RasterOracleEngine, raster_spec
from test_env_map_cpu import RN_FIELDS, crafted_network
from test_env_raster_cpu import crafted_scene, ring, soup

pytestmark = pytest.mark.gpu
EDGE_TOL = 1e-6


def _device_spec(scene, slots):
    N, A = slots.shape
    buf = {"agent_slot": torch.from_numpy(np.ascontiguousarray(slots, np.int32)).cuda(),
           "snap_dist": torch.zeros(N * A, dtype=torch.float64).cuda(),
           "snap_collided": torch.zeros(N * A, dtype=torch.uint8).cuda(),
           "snap_pair_ticks": torch.zeros(N, dtype=torch.int64).cuda(), "snap_rss": torch.zeros(N, dtype=torch.uint8).cuda()}
    e = abi.SgEnvSpec()
    e.n_agents = A
    for k, t in buf.items():
        setattr(e, k, t.data_ptr())
    return e, buf


def _device_rspec(scene, S, res, ahead):
    r = raster_spec(scene, S, res, ahead)
    box, r.margin = abi.raster_poly_boxes(scene.rn_edge_off, scene.rn_edges, abi.raster_half_diagonal(S, res))
    t = torch.from_numpy(box if len(box) else np.zeros((1, 4))).cuda()
    r.poly_box = t.data_ptr()
    return r, t


def _pair(scene, pose, present, slots):
    """(device engine, oracle) over the same scene and state."""
    gpu = Engine(scene, abi.default_params())
    gpu.reset()
    gpu.tensor("pose").copy_(torch.from_numpy(pose).reshape(gpu.tensor("pose").shape))
    gpu.tensor("present").copy_(torch.from_numpy(present).reshape(gpu.tensor("present").shape))
    cpu = RasterOracleEngine(scene, abi.default_params())
    cpu.reset()
    cpu.state["pose"][...] = pose.reshape(cpu.state["pose"].shape)
    cpu.state["present"][...] = present.reshape(cpu.state["present"].shape)
    cpu.env_spec(slots, 0, 0.0, ())
    return gpu, cpu


def _device_raster(gpu, scene, slots, S, res, ahead, mask=None, out=None):
    e, keep = _device_spec(scene, slots)
    r, box = _device_rspec(scene, S, res, ahead)
    N, A = slots.shape
    if out is None:
        out = torch.zeros(N, A, 5, S, S, dtype=torch.uint8, device="cuda")
    gpu.env_raster(e, r, out, mask=None if mask is None else torch.from_numpy(mask).cuda())
    return out.cpu().numpy()


def _seg_distance(px, py, seg):
    """Distance of each point to the nearest segment of seg [E, 4]."""
    if len(seg) == 0:
        return np.full(len(px), np.inf)
    ax, ay, bx, by = (seg[:, k][None, :] for k in range(4))
    dx, dy = bx - ax, by - ay
    L2 = dx * dx + dy * dy
    t = np.clip(((px[:, None] - ax) * dx + (py[:, None] - ay) * dy) / np.where(L2 > 0, L2, 1.0), 0.0, 1.0)
    qx, qy = ax + t * dx - px[:, None], ay + t * dy - py[:, None]
    return np.sqrt(qx * qx + qy * qy).min(1)


def _box_edges(scene, pose, present, n, skip):
    M = scene.M
    box = scene.box.reshape(4, -1)
    out = []
    for j in range(M):
        b = n * M + j
        if j == skip or not present[b]:
            continue
        c, s = math.cos(pose[3, b]), math.sin(pose[3, b])
        X, Y = pose[0, b] + (box[2, b] * c - box[3, b] * s), pose[1, b] + (box[2, b] * s + box[3, b] * c)
        hl, hw = 0.5 * box[1, b], 0.5 * box[0, b]
        pts = [(X + c * u - s * v, Y + s * u + c * v) for u, v in ((hl, hw), (-hl, hw), (-hl, -hw), (hl, -hw))]
        out += [[*pts[k], *pts[(k + 1) % 4]] for k in range(4)]
    return np.array(out, np.float64).reshape(-1, 4)


def _compare(got, want, scene, pose, present, slots, S, res, ahead):
    """Every pixel where the device and the oracle differ must have its centre within EDGE_TOL of a ring edge of
    its surface or of a box edge.  Returns the number of differing pixels."""
    diff = np.argwhere(got != want)
    h = 0.5 * res
    M = scene.M
    for n, a, ch, i, j in diff:
        slot = int(slots[n, a])
        k = n * M + slot
        x, y, hd = pose[0, k], pose[1, k], pose[3, k]
        c, s = math.cos(hd), math.sin(hd)
        pu, pv = ahead + (S - 1 - 2 * i) * h, (S - 1 - 2 * j) * h
        px, py = np.array([x + (c * pu - s * pv)]), np.array([y + (s * pu + c * pv)])
        if ch < 3:
            r = int(scene.rn_of[n])
            q0, q1 = scene.rn_poly_off[3 * r + ch], scene.rn_poly_off[3 * r + ch + 1]
            seg = scene.rn_edges[scene.rn_edge_off[q0]:scene.rn_edge_off[q1]]
        else:
            seg = _box_edges(scene, pose, present, n, slot)
        d = _seg_distance(px, py, seg)[0]
        assert d <= EDGE_TOL, (int(n), int(a), int(ch), int(i), int(j), d)
    return len(diff)


# ------------------------------------------------------------------------------------------------- exact cases
def test_raster_crafted_bit_equal():
    """Heading 0 everywhere: the crafted cases are bit-equal between the device and the oracle."""
    scene, pose, present, slots = crafted_scene(rot45=False)
    gpu, cpu = _pair(scene, pose, present, slots)
    for S, res, ahead in ((32, 1.0, 0.0), (64, 0.5, 0.0), (32, 1.0, 3.0), (64, 0.25, -1.5), (96, 0.5, 2.0),
                          (256, 0.125, 0.0)):
        got = _device_raster(gpu, scene, slots, S, res, ahead)
        want = cpu.env_raster(raster_spec(scene, S, res, ahead))
        assert np.array_equal(got, want), (S, res, ahead, int((got != want).sum()))
        if S * res >= 32:  # (the smaller windows miss the building)
            assert got[0, 0].any(axis=(1, 2)).all(), "every channel has pixels"
        assert not got[:, 1:].any() and not got[1, 0, :3].any()


def test_raster_culling_bounds():
    """Polygons just inside and just outside the culling square, and one far outside: no pixel, bit for bit."""
    S, res = 32, 1.0
    D = abi.raster_half_diagonal(S, res)
    _, margin = abi.raster_poly_boxes(np.zeros(1, np.int64), np.zeros((0, 4)), D)
    scene, pose, present, slots = crafted_scene(rot45=False)
    polys = [ring((D - 1e-3, 0), (40, 0), (40, 3)), ring((D + 1e-6, -5), (40, -5), (40, -2)),
             ring((-D - 5, D - 1e-3), (-D + 30, D - 1e-3), (-D + 30, D + 4)), ring((200, 200), (210, 200), (210, 210))]
    po, eo, ed = soup([[polys, [], []]])
    scene = dataclasses.replace(scene, **dict(zip(RN_FIELDS, (np.array([0, -1], np.int32), po, eo, ed,
                                                              np.ones(3, np.uint8)))))
    gpu, cpu = _pair(scene, pose, present, slots)
    got = _device_raster(gpu, scene, slots, S, res, 0.0)
    want = cpu.env_raster(raster_spec(scene, S, res, 0.0))
    assert np.array_equal(got, want) and not got[:, :, :3].any()
    assert margin > 0


# ------------------------------------------------------------------------------------------------ random poses
def _town_scene(seed, N, M, half_extent, town_extent, ticks):
    town = synthetic.grid_town(seed=seed, half_extent=town_extent)
    cfg = synthetic.vehicles_config(seed=seed, N=N, M=M, T=max(ticks, 1) + 1, half_extent=half_extent)
    scene = synthetic.pack_synthetic(cfg, road_network=town)
    p = abi.default_params()
    p.timestep = cfg.dt
    gpu = Engine(scene, p)
    gpu.reset()
    if ticks:
        gpu.rollout(ticks, actions=cfg.actions[:ticks])
    pose, present = gpu.get("pose").reshape(6, -1).copy(), gpu.get("present").reshape(-1).copy()
    rng = np.random.default_rng(seed)
    pose[3] = rng.uniform(-math.pi, math.pi, pose.shape[1])
    return scene, pose, present


@pytest.mark.parametrize("S,A,N", [(32, 6, 3), (64, 6, 3), (256, 2, 1)])
def test_raster_random_headings_town(S, A, N):
    scene, pose, present = _town_scene(seed=S, N=N, M=12, half_extent=40.0, town_extent=60.0, ticks=8)
    slots = np.tile(np.arange(A, dtype=np.int32), (N, 1))
    slots[0, A - 1] = -1  # a padding agent
    gpu, cpu = _pair(scene, pose, present, slots)
    res, ahead = 0.5 if S < 256 else 0.25, 6.0
    got = _device_raster(gpu, scene, slots, S, res, ahead)
    want = cpu.env_raster(raster_spec(scene, S, res, ahead))
    n_diff = _compare(got, want, scene, pose, present, slots, S, res, ahead)
    print(f"S={S}: {n_diff} of {got.size} pixels differ, all within {EDGE_TOL} m of an edge")
    assert n_diff <= max(4, got.size // 100000)
    assert want[:, :, 0].any() and want[:, :, 3].any() and not got[0, A - 1].any()


def test_raster_several_networks_in_one_batch():
    t1, t2 = synthetic.grid_town(seed=4, half_extent=50.0), synthetic.grid_town(seed=5, half_extent=50.0)
    cfg = synthetic.vehicles_config(seed=6, N=5, M=8, T=4, half_extent=40.0)
    scene = synthetic.pack_synthetic(cfg)
    nets = [t1, None, t2, crafted_network(), t1]
    scene = dataclasses.replace(scene, **dict(zip(RN_FIELDS, pack_road_networks(nets))))
    assert scene.n_networks == 3
    gpu = Engine(scene, abi.default_params())
    gpu.reset()
    pose, present = gpu.get("pose").reshape(6, -1).copy(), gpu.get("present").reshape(-1).copy()
    pose[3] = np.random.default_rng(1).uniform(-math.pi, math.pi, pose.shape[1])
    slots = np.tile(np.arange(3, dtype=np.int32), (cfg.N, 1))
    gpu, cpu = _pair(scene, pose, present, slots)
    got = _device_raster(gpu, scene, slots, 64, 0.5, 0.0)
    want = cpu.env_raster(raster_spec(scene, 64, 0.5, 0.0))
    _compare(got, want, scene, pose, present, slots, 64, 0.5, 0.0)
    assert not got[1, :, :3].any() and got[0, :, 0].any() and got[2, :, 0].any()


def test_raster_many_slots_pedestrians():
    """M = 300 slots, most of them pedestrians: the box channels at large M (the block's shared memory)."""
    cfg = synthetic.vehicles_config(seed=7, N=2, M=300, T=4, half_extent=12.0)
    scene = synthetic.pack_synthetic(cfg, road_network=synthetic.grid_town(seed=7, half_extent=40.0))
    etype = scene.etype.copy()
    box = scene.box.copy().reshape(4, -1)
    ped = (np.arange(scene.N * scene.M) % scene.M) >= 20
    etype[ped] = abi.ETYPE_PEDESTRIAN
    box[0, ped], box[1, ped] = 0.6, 0.6
    scene = dataclasses.replace(scene, etype=etype, box=np.ascontiguousarray(box))
    gpu = Engine(scene, abi.default_params())
    gpu.reset()
    pose, present = gpu.get("pose").reshape(6, -1).copy(), np.ones(scene.N * scene.M, np.uint8)
    pose[3] = np.random.default_rng(2).uniform(-math.pi, math.pi, pose.shape[1])
    slots = np.tile(np.array([0, 5, 250, 299], np.int32), (scene.N, 1))
    gpu, cpu = _pair(scene, pose, present, slots)
    got = _device_raster(gpu, scene, slots, 64, 0.5, 0.0)
    want = cpu.env_raster(raster_spec(scene, 64, 0.5, 0.0))
    _compare(got, want, scene, pose, present, slots, 64, 0.5, 0.0)
    assert want[:, :, 4].sum() > 100 and want[:, :, 3].any()


def test_raster_long_polygon():
    """A 2 km road crossing the whole raster (most of its edges far outside it)."""
    road = Road("long", PolygonArea([(-1000.0, -3.0), (1000.0, -3.0), (1000.0, 3.0), (-1000.0, 3.0)]))
    cfg = synthetic.vehicles_config(seed=3, N=2, M=6, T=4, half_extent=1.0)
    scene = synthetic.pack_synthetic(cfg, road_network=RoadNetwork(roads=[road]))
    pose = np.zeros((6, scene.N * scene.M))
    pose[0] = np.linspace(-900.0, 900.0, pose.shape[1])
    pose[1] = np.linspace(-2.0, 2.0, pose.shape[1])
    pose[3] = np.random.default_rng(3).uniform(-math.pi, math.pi, pose.shape[1])
    present = np.ones(scene.N * scene.M, np.uint8)
    slots = np.tile(np.arange(scene.M, dtype=np.int32), (scene.N, 1))
    gpu, cpu = _pair(scene, pose, present, slots)
    got = _device_raster(gpu, scene, slots, 64, 0.5, 3.0)
    want = cpu.env_raster(raster_spec(scene, 64, 0.5, 3.0))
    _compare(got, want, scene, pose, present, slots, 64, 0.5, 3.0)
    assert (want[:, :, 0].sum(axis=(2, 3)) > 64).all()


def test_raster_masked_call():
    scene, pose, present = _town_scene(seed=9, N=4, M=8, half_extent=30.0, town_extent=50.0, ticks=0)
    present[1 * 8 + 2] = 0  # an absent agent
    slots = np.tile(np.array([0, 2, 4, -1], np.int32), (4, 1))
    gpu, cpu = _pair(scene, pose, present, slots)
    mask = np.array([0, 1, 1, 0], np.uint8)
    out = torch.full((4, 4, 5, 64, 64), 0xAB, dtype=torch.uint8, device="cuda")
    got = _device_raster(gpu, scene, slots, 64, 0.5, 0.0, mask=mask, out=out)
    want = cpu.env_raster(raster_spec(scene, 64, 0.5, 0.0), mask=mask)
    assert (got[[0, 3]] == 0xAB).all(), "unflagged scenarios are untouched"
    assert not got[1, 1].any() and not got[1:3, 3].any(), "absent and padding agents are zero"
    assert set(np.unique(got[1:3])) <= {0, 1}
    flagged = np.where(mask.astype(bool)[:, None, None, None, None], got, 0)
    _compare(flagged, want, scene, pose, present, slots, 64, 0.5, 0.0)
    assert want[1:3, :, 0].any()


# ----------------------------------------------------------------------------------------------- env level
def _vehicle_scenes(seed=2, N=6, M=8, half_extent=40.0):
    cfg = synthetic.vehicles_config(seed=seed, N=N, M=M, T=30, half_extent=half_extent)
    rows = synthetic.two_knot_rows(cfg).reshape(cfg.N, cfg.M, 2, 7)
    ce = CatalogEntry(None, "car1", "car", "Vehicle", BoundingBox(*synthetic.CAR1_BOX))
    rn = synthetic.grid_town(seed=seed, half_extent=half_extent + 20.0)
    return cfg, [Scenario([Vehicle(ce, trajectory=Trajectory(rows[n, m]), ref="ego" if m == 0 else f"entity_{m}")
                           for m in range(cfg.M)], road_network=rn if n != 1 else None) for n in range(cfg.N)]


def _policy(obs):
    tx, ty = obs[..., 4], obs[..., 5]
    return torch.stack([(torch.sqrt(tx * tx + ty * ty) - obs[..., 0]).clamp(-5.0, 5.0),
                        torch.atan2(ty, tx).clamp(-0.7, 0.7)], -1)


def _make(scs, cfg, reset_spec=None, **obs):
    return VecScenarioEnv(scs, create_agent=lambda s, e: PolicyAgent(e), timestep=cfg.dt,
                          obs=ObsSpec(k_neighbours=2, lookahead=(1.0,), **obs), reset_spec=reset_spec)


@pytest.mark.parametrize("with_spec", [False, True])
def test_env_raster_changes_nothing_else(with_spec):
    cfg, scs = _vehicle_scenes()
    rs = ResetSpec(start_offset=1.0, lon=0.3, heading=0.05, seed=3) if with_spec else None
    plain = _make(scs, cfg, rs, map_edges=4, map_radius=20.0)
    rast = _make(scs, cfg, rs, map_edges=4, map_radius=20.0, raster_size=64, raster_ahead=4.0)
    assert plain.n_features == rast.n_features and "raster" not in plain.reset()[1]
    o1, i1 = plain.reset(seed=1)
    o2, i2 = rast.reset(seed=1)
    assert i2["raster"].shape == (rast.N, rast.A, 5, 64, 64) and i2["raster"].dtype == torch.uint8
    assert rast.raster_channels == ("driveable", "walkable", "impenetrable", "vehicles", "pedestrians")
    resets = 0
    for k in range(60):
        assert torch.equal(o1.view(torch.int32), o2.view(torch.int32)), k
        a = _policy(o1)
        r1, r2 = plain.step(a), rast.step(a)
        for x, y in zip(r1[1:4], r2[1:4]):
            assert torch.equal(x, y), k
        assert set(r2[4]) == set(r1[4]) | {"raster", "final_raster"}
        for key, t in r1[4]["final"].items():
            assert torch.equal(t, r2[4]["final"][key]), (k, key)
        assert torch.equal(r1[4]["final_obs"], r2[4]["final_obs"])
        resets += int((r1[2] | r1[3]).sum())
        o1, o2 = r1[0], r2[0]
    assert resets > 0


def test_env_final_raster_and_reset_rasters():
    cfg, scs = _vehicle_scenes(seed=4, N=5, M=6)
    env = _make(scs, cfg, raster_size=32, raster_resolution=1.0, raster_ahead=2.0)
    o, info = env.reset()
    first = info["raster"].clone()
    assert first[:, :, 0].any() and first[:, :, 3].any()
    twin = Engine(env._engine.scene, env._engine.params)
    twin.reset()
    buf = torch.zeros(1, 2, env.N * twin.M, device="cuda")
    r2 = torch.zeros_like(first)
    resets = 0
    for k in range(45):
        a = _policy(o)
        o, rew, te, tr, info = env.step(a)
        buf[0].index_copy_(1, env._dst, a.reshape(env.N * env.A, 2).index_select(0, env._src).t())
        twin.rollout(1, actions=buf)
        twin.env_raster(env._spec, env._rspec, r2)
        assert torch.equal(info["final_raster"], r2), k
        fin = te | tr
        twin.reset(mask=fin)
        twin.env_raster(env._spec, env._rspec, r2)
        assert torch.equal(info["raster"], r2), k
        if fin.any():
            resets += int(fin.sum())
            assert torch.equal(info["raster"][fin], first[fin]), "a reset scenario's raster is a fresh reset's"
    assert resets > 0


def test_env_raster_step_no_sync_no_allocation():
    cfg, scs = _vehicle_scenes(seed=5, N=4, M=6)
    env = _make(scs, cfg, raster_size=64)
    o, _ = env.reset()
    for _ in range(3):
        o, *_ = env.step(_policy(o))
    for k in range(35):  # (covers auto-resets)
        a = _policy(o)
        torch.cuda.synchronize()
        mem, res = torch.cuda.memory_allocated(), torch.cuda.memory_reserved()
        torch.cuda.set_sync_debug_mode("error")
        try:
            o, rew, te, tr, info = env.step(a)
        finally:
            torch.cuda.set_sync_debug_mode("default")
        # (nothing new is held or reserved; the step's temporaries are freed before it returns)
        assert torch.cuda.memory_allocated() <= mem and torch.cuda.memory_reserved() == res, k
        assert info["raster"] is env._raster and info["final_raster"] is env._final_raster


# ------------------------------------------------------------------------------------------- argument checks
def test_raster_argument_checks():
    cfg, scs = _vehicle_scenes(N=2, M=4)
    env = _make(scs, cfg, raster_size=32)
    env.reset()
    eng = env._engine
    for field, value, msg in (("size", 48, "size"), ("size", 16, "size"), ("size", 288, "size"),
                              ("resolution", 0.0, "resolution"), ("resolution", -0.5, "resolution"),
                              ("resolution", math.nan, "resolution"), ("ahead", math.nan, "ahead"),
                              ("n_networks", env._rspec.n_networks + 1, "n_networks"),
                              ("poly_box", None, "poly_box")):
        r = abi.SgRasterSpec.from_buffer_copy(env._rspec)
        setattr(r, field, value)
        out = env._raster if field != "size" else torch.zeros(env.N, env.A, 5, value, value, dtype=torch.uint8,
                                                              device="cuda")
        with pytest.raises(RuntimeError, match=msg):
            eng.env_raster(env._spec, r, out)
    with pytest.raises(ValueError):
        eng.env_raster(env._spec, env._rspec, env._raster[:, :, :3])
