"""
CPU tests of branched look-ahead rollouts (VecScenarioEnv.branches, include/sg_b200.h sg_fork_state): the horizon
evaluation -- sg_env_reward once after H ticks, against the state at the fork -- on the oracle against a numpy
restatement, H = 1 against one oracle env step, and the action-scatter index against a loop.
"""
import math

import numpy as np
import pytest

from oracle import golden_cases
from oracle.env_runner import OracleEnvEngine
from scenario_gym_b200 import abi, synthetic
from scenario_gym_b200.env import branch_scatter_index

F32 = dict(rtol=2e-6, atol=2e-5)
W = (1.0, -10.0, -1.0, 0.1, -1.0)
SKIP = ("events", "trace_pose", "trace_present", "trace_t")


def fork(src: OracleEnvEngine, scene, p, slots) -> OracleEnvEngine:
    """sg_fork_state restated on the host: every state array and the snapshot copied, event_count = 0."""
    dst = OracleEnvEngine(scene, p)
    for name, _, _ in abi.STATE_FIELDS:
        if name not in SKIP:
            dst.state[name][...] = src.state[name]
    dst.state["event_count"][...] = 0
    dst.env_spec(slots, k_neighbours=2, lookahead=(0.5,), weights=W)
    for k in ("snap_dist", "snap_collided", "snap_pair_ticks", "snap_rss"):
        dst.env[k][...] = src.env[k]
    return dst


def _clamped(rows, t):
    return np.array([np.interp(t, rows[:, 0], rows[:, 1 + f]) for f in range(6)])


def horizon_numpy(scene, p, fork_state, snap, end, slots):
    """The horizon terms restated from the fork state / snapshot and the end state (no road network here)."""
    N, M = scene.N, scene.M
    A = slots.shape[1]
    sd, sc, snpt, srss = (snap["snap_dist"].reshape(N, A), snap["snap_collided"].reshape(N, A),
                          snap["snap_pair_ticks"], snap["snap_rss"])
    terms = np.zeros((N, A, 5))
    te, tr = np.zeros(N, np.uint8), np.zeros(N, np.uint8)
    for n in range(N):
        for a in range(A):
            s = slots[n, a]
            i = n * M + s
            if s < 0 or not end["present"][i]:
                continue
            rows = scene.traj_rows[scene.traj_off[i]:scene.traj_off[i + 1]]
            q = _clamped(rows, end["t"][n])
            terms[n, a] = [end["dist"][i] - sd[n, a], float(end["collided"][i] and not sc[n, a]), 0.0,
                           -math.hypot(end["pose"][0, i] - q[0], end["pose"][1, i] - q[1]),
                           float(s == scene.ego_slot[n] and (end["rss_flags"][n] & ~srss[n]) != 0)]
        if end["done"][n]:
            fi = n * M + scene.first_slot[n]
            hit = (p.terminal & abi.TERM_COLLISION and end["n_pair_ticks"][n] > snpt[n]) or \
                  (p.terminal & abi.TERM_EGO_COLLISION and end["collided"][fi])
            te[n], tr[n] = int(bool(hit)), int(not hit)
    return terms, te, tr


@pytest.mark.parametrize("terminal", [abi.TERM_MAX_LENGTH | abi.TERM_EGO_COLLISION,
                                      abi.TERM_MAX_LENGTH | abi.TERM_COLLISION, abi.TERM_MAX_LENGTH])
@pytest.mark.parametrize("H", [6, 25])
def test_horizon_evaluation_matches_numpy(terminal, H):
    """Fork at several ticks, roll H ticks, one sgo_env_reward: == the numpy restatement, and the collision term
    == 'collided rose at some tick of the horizon' from stepping a twin one tick at a time."""
    cfg = golden_cases.veh_cfg()
    scene = synthetic.pack_synthetic(cfg)
    p = abi.default_params()
    p.timestep, p.terminal = cfg.dt, terminal
    p.features |= abi.FEAT_RSS
    slots = np.tile(np.arange(3, dtype=np.int32), (cfg.N, 1))
    eng = OracleEnvEngine(scene, p)
    eng.reset()
    eng.env_spec(slots, k_neighbours=2, lookahead=(0.5,), weights=W)
    seen = {"collision": 0, "finished": 0}
    k = 0
    for k0 in (0, 5, 12, 60):
        if k0 > k:
            eng.rollout(k0 - k, actions=cfg.actions[k:k0])
            k = k0
        eng.env_observe()
        acts = np.zeros((H,) + cfg.actions.shape[1:])
        acts[:len(cfg.actions[k:k + H])] = cfg.actions[k:k + H]
        br, twin = fork(eng, scene, p, slots), fork(eng, scene, p, slots)
        br.rollout(H, actions=acts)
        rew, terms, te, tr = br.env_reward()
        want, wte, wtr = horizon_numpy(scene, p, eng.state, twin.env, br.state, slots)
        np.testing.assert_allclose(terms, want, **F32)
        np.testing.assert_allclose(rew, (want * np.array(W)).sum(-1), **F32)
        assert np.array_equal(te, wte) and np.array_equal(tr, wtr)
        rose = np.zeros((cfg.N, 3), bool)
        for h in range(len(acts)):
            twin.rollout(1, actions=acts[h:h + 1])
            coll = twin.state["collided"].reshape(cfg.N, cfg.M)[:, :3].astype(bool)
            rose |= coll & ~twin.env["snap_collided"].reshape(cfg.N, 3).astype(bool)
        for name, _, _ in abi.STATE_FIELDS:  # fused H ticks == H single ticks
            if name not in SKIP:
                assert np.array_equal(twin.state[name], br.state[name], equal_nan=True), name
        present = br.state["present"].reshape(cfg.N, cfg.M)[:, :3].astype(bool)
        assert np.array_equal(terms[..., 1] == 1.0, rose & present)
        seen["collision"] += int(terms[..., 1].sum())
        seen["finished"] += int((te | tr).sum())
    assert seen["collision"] > 0
    if H == 25:
        assert seen["finished"] > 0


def test_h1_equals_one_oracle_env_step():
    """A branch of one tick scores exactly what one env step (rollout(1) + env_reward) scores."""
    cfg = golden_cases.veh_cfg()
    scene = synthetic.pack_synthetic(cfg)
    p = abi.default_params()
    p.timestep, p.terminal = cfg.dt, abi.TERM_MAX_LENGTH | abi.TERM_COLLISION
    p.features |= abi.FEAT_RSS
    slots = np.tile(np.arange(3, dtype=np.int32), (cfg.N, 1))
    slots[1, 2] = -1  # a padding agent
    eng = OracleEnvEngine(scene, p)
    eng.reset()
    eng.env_spec(slots, k_neighbours=2, lookahead=(0.5,), weights=W)
    for k in range(cfg.T):
        eng.env_observe()
        br = fork(eng, scene, p, slots)
        br.rollout(1, actions=cfg.actions[k:k + 1])
        got = br.env_reward()
        eng.rollout(1, actions=cfg.actions[k:k + 1])
        want = eng.env_reward()
        for g, w in zip(got, want):
            assert np.array_equal(g, w), k
        if eng.state["done"].all():
            break


@pytest.mark.parametrize("B,H", [(1, 1), (3, 4), (2, 7)])
def test_scatter_index_matches_loop(B, H):
    rng = np.random.default_rng(B * 10 + H)
    N, M, A = 5, 9, 4
    slots = np.full((N, A), -1, np.int32)
    for n in range(N):
        k = int(rng.integers(0, A + 1))
        slots[n, :k] = rng.choice(M, k, replace=False)
    idx = branch_scatter_index(slots, M, B, H)
    actions = rng.normal(size=(N, B, H, A, 2))
    table = np.zeros(B * H * 2 * N * M + 1)
    table[idx] = actions.reshape(-1)  # (padding agents all land on the trailing element)
    want = np.zeros((B, H, 2, N * M))
    for n in range(N):
        for b in range(B):
            for h in range(H):
                for a in range(A):
                    if slots[n, a] >= 0:
                        for c in range(2):
                            want[b, h, c, n * M + slots[n, a]] = actions[n, b, h, a, c]
    assert np.array_equal(table[:-1].reshape(B, H, 2, N * M), want)
    assert idx.dtype == np.int64 and idx.shape == (N * B * H * A * 2,)
    pad = np.broadcast_to((slots < 0)[:, None, None, :, None], (N, B, H, A, 2)).reshape(-1)
    assert np.all(idx[pad] == B * H * 2 * N * M)
