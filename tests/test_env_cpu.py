"""
CPU tests of the closed-loop environment's entry points on the oracle (sgo_env_observe, sgo_env_reward,
sgo_reset_scenarios) against an independent numpy restatement of include/sg_b200.h (SgEnvSpec).
"""
import math

import numpy as np
import pytest

from oracle import golden_cases
from oracle.env_runner import OracleEnvEngine
from scenario_gym_b200 import abi, synthetic

F32 = dict(rtol=2e-6, atol=2e-5)  # one fp32 rounding of fp64 values (+ libm vs numpy trig)


def _veh_engine(road=None, seed=3, N=3, M=12, T=12, terminal=abi.TERM_MAX_LENGTH):
    cfg = synthetic.vehicles_config(seed=seed, N=N, M=M, T=T, half_extent=14.0)
    scene = synthetic.pack_synthetic(cfg, road_network=road)
    p = abi.default_params()
    p.timestep, p.terminal = cfg.dt, terminal
    return cfg, scene, OracleEnvEngine(scene, p)


def _clamped(rows, t):
    """Trajectory.position_at_t(t) clamped at the ends: numpy's interp per column."""
    return np.array([np.interp(t, rows[:, 0], rows[:, 1 + f]) for f in range(6)])


def _rows(scene, i):
    return scene.traj_rows[scene.traj_off[i]:scene.traj_off[i + 1]]


def _on_segment_dist(px, py, edges):
    a, b = edges[:, :2], edges[:, 2:]
    d = b - a
    L2 = (d * d).sum(1)
    f = np.where(L2 > 0, ((px - a[:, 0]) * d[:, 0] + (py - a[:, 1]) * d[:, 1]) / np.where(L2 > 0, L2, 1), 0)
    f = np.clip(f, 0.0, 1.0)
    c = a + f[:, None] * d
    return float(np.sqrt(((c - [px, py]) ** 2).sum(1).min()))


def _road(scene, n, px, py):
    """(driveable surface contains (px, py), distance to its rings) by ray casting; zeros without area."""
    r = scene.rn_of[n]
    if r < 0 or not scene.rn_has_area[3 * r]:
        return 0.0, 0.0
    q0, q1 = scene.rn_poly_off[3 * r], scene.rn_poly_off[3 * r + 1]
    inside = False
    for q in range(q0, q1):
        E = scene.rn_edges[scene.rn_edge_off[q]:scene.rn_edge_off[q + 1]]
        par = False
        for ax, ay, bx, by in E:
            if (ay > py) != (by > py) and px < ax + (py - ay) * (bx - ax) / (by - ay):
                par = not par
        inside = inside or par
    E = scene.rn_edges[scene.rn_edge_off[q0]:scene.rn_edge_off[q1]]
    return float(inside), _on_segment_dist(px, py, E)


def numpy_observe(scene, st, slots, K, radius, look, road):
    """Observation rows + agent mask + the neighbour slots chosen (numpy restatement)."""
    N, M = scene.N, scene.M
    A = slots.shape[1]
    F = abi.env_n_features(K, len(look), road)
    obs, am = np.zeros((N, A, F)), np.zeros((N, A), np.uint8)
    chosen = {}
    pose, vel = st["pose"], st["vel"]
    for n in range(N):
        for a in range(A):
            s = slots[n, a]
            if s < 0 or not st["present"][n * M + s]:
                continue
            i = n * M + s
            am[n, a] = 1
            x, y, h, vx, vy = pose[0, i], pose[1, i], pose[3, i], vel[0, i], vel[1, i]
            c, sn = math.cos(h), math.sin(h)
            rot = lambda dx, dy: (c * dx + sn * dy, -sn * dx + c * dy)  # noqa: E731
            row = [st["speed"][i], *rot(vx, vy), vel[3, i]]
            for tau in look:
                q = _clamped(_rows(scene, i), st["t"][n] + tau)
                row += [*rot(q[0] - x, q[1] - y), math.remainder(q[3] - h, 2 * math.pi)]
            cand = []
            for j in range(M):
                g = n * M + j
                if j == s or not st["present"][g]:
                    continue
                dx, dy = pose[0, g] - x, pose[1, g] - y
                d2 = dx * dx + dy * dy
                if radius > 0 and not d2 < radius * radius:
                    continue
                cand.append((d2, j))
            cand.sort()
            chosen[(n, a)] = [j for _, j in cand[:K]]
            for q in range(K):
                if q >= len(cand):
                    row += [0.0] * 10
                    continue
                g = n * M + cand[q][1]
                dh = pose[3, g] - h
                row += [*rot(pose[0, g] - x, pose[1, g] - y), math.cos(dh), math.sin(dh),
                        *rot(vel[0, g] - vx, vel[1, g] - vy), scene.box[0, g], scene.box[1, g],
                        float(scene.etype[g] == abi.ETYPE_PEDESTRIAN), 1.0]
            if road:
                row += list(_road(scene, n, x, y))
            obs[n, a] = row
    return obs, am, chosen


def _craft(cfg, eng):
    """Seeded state with duplicate positions, absent slots and a neighbour exactly at the radius."""
    eng.reset()
    eng.rollout(3, actions=cfg.actions)
    st, M = eng.state, cfg.M
    P = st["pose"]
    # scenario 0: agent slot 0 at the origin; slots 1 and 2 at the same place (tie broken by slot),
    # slot 4 at exactly the radius (8 m, excluded), slot 5 just inside it, slot 6 absent
    P[0, 0], P[1, 0] = 0.0, 0.0
    for s, (x, y, h) in {1: (3.0, 4.0, 0.3), 2: (3.0, 4.0, -1.0), 4: (8.0, 0.0, 0.0), 5: (0.0, 7.999, 2.0)}.items():
        P[0, s], P[1, s], P[3, s] = x, y, h
    st["present"][6] = 0
    # scenario 1: an absent agent
    st["present"][M + 3] = 0
    # scenario 2: every slot on one point
    P[0, 2 * M:3 * M], P[1, 2 * M:3 * M] = 1.5, -2.5
    return np.array([[0, 3, 6, -1], [0, 1, 2, 3], [5, -1, -1, -1]], np.int32)


@pytest.mark.parametrize("K,radius,look", [(4, 8.0, (-100.0, 0.5, 100.0)), (16, 0.0, (1.0,)), (0, 5.0, ())])
def test_observe_matches_numpy(K, radius, look):
    cfg, scene, eng = _veh_engine()
    scene.etype[7] = abi.ETYPE_PEDESTRIAN  # (the oracle reads the packed arrays in place)
    slots = _craft(cfg, eng)
    eng.env_spec(slots, k_neighbours=K, radius=radius, lookahead=look)
    obs, am = eng.env_observe()
    want, want_am, chosen = numpy_observe(scene, eng.state, slots, K, radius, look, False)
    assert np.array_equal(am, want_am)
    assert np.array_equal(am[0], [1, 1, 0, 0]) and np.array_equal(am[1], [1, 1, 1, 0])
    np.testing.assert_allclose(obs, want, **F32)
    if K:
        valid = obs[..., 4 + 3 * len(look):4 + 3 * len(look) + 10 * K].reshape(*am.shape, K, 10)[..., 9]
        for (n, a), js in chosen.items():
            assert np.array_equal(valid[n, a], [1.0] * len(js) + [0.0] * (K - len(js)))
    if K == 4:  # scenario 0, agent 0: 1 before 2 (a tie; the headings tell them apart); 4 sits on the radius
        assert chosen[(0, 0)][:2] == [1, 2] and 5 in chosen[(0, 0)] and 4 not in chosen[(0, 0)]
        nb = obs[0, 0, 4 + 9:4 + 9 + 40].reshape(4, 10)
        np.testing.assert_allclose(nb[:2, 3], np.sin([0.3 - eng.state["pose"][3, 0], -1.0 - eng.state["pose"][3, 0]]),
                                   **F32)
    # snapshot
    assert np.array_equal(eng.env["snap_pair_ticks"], eng.state["n_pair_ticks"])
    assert np.array_equal(eng.env["snap_dist"].reshape(slots.shape),
                          np.where(slots >= 0, eng.state["dist"][np.arange(3)[:, None] * cfg.M + np.maximum(slots, 0)], 0))


def test_observe_masked_scenarios_only():
    cfg, scene, eng = _veh_engine()
    slots = _craft(cfg, eng)
    eng.env_spec(slots, k_neighbours=4, radius=0.0, lookahead=(1.0,))
    full, _ = eng.env_observe()
    part, am = eng.env_observe(mask=np.array([0, 1, 0], np.uint8))
    assert np.array_equal(part[1], full[1]) and not part[[0, 2]].any() and not am[[0, 2]].any()


def test_observe_road_block():
    net = golden_cases.road_network(golden_cases.ROAD_VEH_GEOMETRY)
    cfg, scene, eng = _veh_engine(road=net, seed=1, N=4, M=12, T=40)
    eng.reset()
    eng.rollout(30, actions=cfg.actions)
    slots = np.tile(np.arange(12, dtype=np.int32), (4, 1))
    eng.env_spec(slots, k_neighbours=2, radius=0.0, lookahead=(), road=True)
    obs, am = eng.env_observe()
    want, want_am, _ = numpy_observe(scene, eng.state, slots, 2, 0.0, (), True)
    assert np.array_equal(am, want_am)
    np.testing.assert_allclose(obs, want, **F32)
    road = obs[..., -2:][am.astype(bool)]
    assert 0 < road[:, 0].sum() < len(road), "some agents on the road, some off it"


def _terms_numpy(scene, p, before, after, slots, snap_dist, snap_coll, snap_npt, snap_rss):
    N, M = scene.N, scene.M
    A = slots.shape[1]
    terms = np.zeros((N, A, 5))
    te, tr = np.zeros(N, np.uint8), np.zeros(N, np.uint8)
    for n in range(N):
        for a in range(A):
            s = slots[n, a]
            if s < 0 or not after["present"][n * M + s]:
                continue
            i = n * M + s
            x, y = after["pose"][0, i], after["pose"][1, i]
            q = _clamped(_rows(scene, i), after["t"][n])
            terms[n, a] = [after["dist"][i] - snap_dist[n, a],
                           float(after["collided"][i] and not snap_coll[n, a]),
                           float(_road(scene, n, x, y)[0] == 0.0 and scene.rn_of[n] >= 0),
                           -math.hypot(x - q[0], y - q[1]),
                           float(s == scene.ego_slot[n] and (after["rss_flags"][n] & ~snap_rss[n]) != 0)]
        if after["done"][n]:
            fi = n * M + scene.first_slot[n]
            hit = (p.terminal & abi.TERM_COLLISION and after["n_pair_ticks"][n] > snap_npt[n]) or \
                  (p.terminal & abi.TERM_EGO_COLLISION and after["collided"][fi])
            te[n], tr[n] = int(bool(hit)), int(not hit)
    return terms, te, tr


@pytest.mark.parametrize("terminal", [abi.TERM_MAX_LENGTH | abi.TERM_EGO_COLLISION,
                                      abi.TERM_MAX_LENGTH | abi.TERM_COLLISION, abi.TERM_MAX_LENGTH])
def test_reward_terms_and_flags(terminal):
    """Tick by tick on dense random vehicles: terms, weighted rewards and terminated / truncated."""
    cfg = golden_cases.veh_cfg()
    scene = synthetic.pack_synthetic(cfg)
    p = abi.default_params()
    p.timestep, p.terminal = cfg.dt, terminal
    p.features |= abi.FEAT_RSS
    eng = OracleEnvEngine(scene, p)
    eng.reset()
    slots = np.tile(np.arange(3, dtype=np.int32), (cfg.N, 1))
    w = (1.0, -10.0, -1.0, 0.1, -1.0)
    eng.env_spec(slots, k_neighbours=2, lookahead=(0.5,), weights=w)
    seen = {"collision": 0, "terminated": 0, "truncated": 0}
    finished = np.zeros(cfg.N, bool)
    for k in range(cfg.T):
        eng.env_observe()
        snap = (eng.env["snap_dist"].reshape(slots.shape).copy(), eng.env["snap_collided"].reshape(slots.shape).copy(),
                eng.env["snap_pair_ticks"].copy(), eng.env["snap_rss"].copy())
        eng.rollout(1, actions=cfg.actions[k:k + 1])
        rew, terms, te, tr = eng.env_reward()
        want, wte, wtr = _terms_numpy(scene, p, None, eng.state, slots, *snap)
        np.testing.assert_allclose(terms, want, **F32)
        np.testing.assert_allclose(rew, (want * np.array(w)).sum(-1), **F32)
        fresh = ~finished & eng.state["done"].astype(bool)
        assert np.array_equal(te[fresh], wte[fresh]) and np.array_equal(tr[fresh], wtr[fresh])
        assert not (te & tr).any() and np.array_equal((te | tr).astype(bool), eng.state["done"].astype(bool))
        seen["collision"] += int(terms[..., 1].sum())
        seen["terminated"] += int(te[fresh].sum())
        seen["truncated"] += int(tr[fresh].sum())
        finished |= eng.state["done"].astype(bool)
        if finished.all():
            break
    assert seen["collision"] > 0, "case must exercise the collision term"
    if terminal != abi.TERM_MAX_LENGTH:
        assert seen["terminated"] > 0
    else:
        assert seen["terminated"] == 0 and seen["truncated"] == cfg.N


def _scenario_view(name, a, n, N, M):
    """Scenario n's part of state array `name` (None: not a per-scenario array)."""
    spec = dict((f, s) for f, _, s in abi.STATE_FIELDS)[name]
    if "NM" in spec:
        return a[..., n * M:(n + 1) * M]
    if spec[0] == "N":
        return a[n]
    return None


def test_reset_scenarios_masked_rows():
    cfg = golden_cases.rss_cfg()
    scene = synthetic.pack_synthetic(cfg)
    p = abi.default_params()
    p.timestep = cfg.dt
    p.features |= abi.FEAT_RSS
    eng, ref = OracleEnvEngine(scene, p), OracleEnvEngine(scene, p)
    ref.reset()
    eng.reset()
    eng.rollout(25, actions=cfg.actions)
    before = {k: v.copy() for k, v in eng.state.items() if isinstance(v, np.ndarray)}
    mask = np.array([1, 0, 1, 0], np.uint8)
    eng.reset_scenarios(mask)
    assert eng.state["event_count"][0] == before["event_count"][0] and before["event_count"][0] > 0
    for name, _, _ in abi.STATE_FIELDS:
        for n in range(cfg.N):
            got = _scenario_view(name, eng.state[name], n, cfg.N, cfg.M)
            if got is None:
                continue
            want = _scenario_view(name, (ref.state if mask[n] else before)[name], n, cfg.N, cfg.M)
            assert np.array_equal(got, want, equal_nan=True), (name, n)
