"""
CPU tests of the lidar block of sg_env_observe on its plain-C restatement (tests/lidar_oracle.c) against an independent,
vectorised numpy restatement of the slab test in include/sg_b200.h (SgEnvSpec), on seeded vehicle scenes
and on crafted scenes whose readings are exact.
"""
import math

import numpy as np
import pytest

from scenario_gym_b200 import abi, synthetic

from lidar_oracle import LidarOracleEngine

F32 = dict(rtol=2e-6, atol=2e-5)  # one fp32 rounding of fp64 values (+ libm vs numpy trig)
RANGE = 50.0
SQ = math.sqrt(0.5)
# direction tables with exact entries (headings 0 make every world direction exact too)
DIRS4 = np.array([[1.0, 0.0], [0.0, 1.0], [-1.0, 0.0], [0.0, -1.0]])
DIRS8 = np.array([[1.0, 0.0], [SQ, SQ], [0.0, 1.0], [-SQ, SQ], [-1.0, 0.0], [-SQ, -SQ], [0.0, -1.0], [SQ, -SQ]])


def slab_terms(scene, st, n, slot, ray_dir):
    """(enter, exit, hit) [J, R] of every other present slot j (js [J]) against the agent's rays."""
    M, nm = scene.M, scene.N * scene.M
    pose, box = st["pose"], scene.box.reshape(4, nm)
    i = n * M + slot
    x, y, h = pose[0, i], pose[1, i], pose[3, i]
    c, s = np.cos(h), np.sin(h)
    ex, ey = ray_dir[:, 0], ray_dir[:, 1]
    ux, uy = c * ex - s * ey, s * ex + c * ey
    js = np.array([j for j in range(M) if j != slot and st["present"][n * M + j]], np.int64)
    g = n * M + js
    cj, sj = np.cos(pose[3, g]), np.sin(pose[3, g])
    X = pose[0, g] + (box[2, g] * cj - box[3, g] * sj)
    Y = pose[1, g] + (box[2, g] * sj + box[3, g] * cj)
    px, py = (x - X)[:, None], (y - Y)[:, None]
    cj, sj = cj[:, None], sj[:, None]
    ox, oy = cj * px + sj * py, -sj * px + cj * py
    dx, dy = cj * ux + sj * uy, -sj * ux + cj * uy

    def axis(o, d, e):
        with np.errstate(divide="ignore", invalid="ignore"):
            t1, t2 = (-e - o) / d, (e - o) / d
        nz = d != 0
        lo = np.where(nz, np.minimum(t1, t2), -np.inf)
        hi = np.where(nz, np.maximum(t1, t2), np.inf)
        return lo, hi, nz | ~(np.abs(o) > e)

    lx, hx, okx = axis(ox, dx, (0.5 * box[1, g])[:, None])
    ly, hy, oky = axis(oy, dy, (0.5 * box[0, g])[:, None])
    enter, exit_ = np.maximum(lx, ly), np.minimum(hx, hy)
    hit = okx & oky & (exit_ >= enter) & (exit_ >= 0)
    return enter, exit_, hit


def numpy_lidar(scene, st, slots, ray_dir, ray_range):
    """The lidar block [N, A, R] (fp32) of every agent: zeros for absent / padding agents."""
    N, A = slots.shape
    R = len(ray_dir)
    out = np.zeros((N, A, R), np.float32)
    for n in range(N):
        for a in range(A):
            s = slots[n, a]
            if s < 0 or not st["present"][n * scene.M + s]:
                continue
            enter, _, hit = slab_terms(scene, st, n, s, ray_dir)
            t = np.where(hit, np.maximum(enter, 0.0), np.inf)
            out[n, a] = np.minimum(ray_range, t.min(0) if len(t) else np.inf).astype(np.float32)
    return out


def _veh_engine(seed, N=3, M=12, T=12):
    cfg = synthetic.vehicles_config(seed=seed, N=N, M=M, T=T, half_extent=14.0)
    scene = synthetic.pack_synthetic(cfg)
    p = abi.default_params()
    p.timestep = cfg.dt
    return cfg, scene, LidarOracleEngine(scene, p)


@pytest.mark.parametrize("R", [1, 7, 64])
def test_lidar_matches_numpy_seeded(R):
    cfg, scene, eng = _veh_engine(seed=11)
    slots = np.tile(np.arange(cfg.M, dtype=np.int32), (cfg.N, 1))
    _, F = eng.env_spec(slots, k_neighbours=2, lookahead=(1.0,), n_rays=R, ray_range=RANGE)
    assert F == abi.env_n_features(2, 1, False) + R
    eng.reset()
    hits = 0
    for k in range(cfg.T):
        if k in (0, 4, 11):
            obs, am = eng.env_observe()
            want = numpy_lidar(scene, eng.state, slots, abi.lidar_directions(R), RANGE)
            np.testing.assert_allclose(obs[..., F - R:], want, **F32)
            hits += int((want < RANGE).sum())
        eng.rollout(1, actions=cfg.actions[k:k + 1])
    assert hits > 0, "the scene must put boxes in front of the rays"


def test_lidar_prefix_is_the_row_without_lidar():
    cfg, scene, eng = _veh_engine(seed=4)
    eng.reset()
    eng.rollout(5, actions=cfg.actions)
    slots = np.array([[0, 3, 5, -1], [2, -1, 1, 7], [11, 10, 9, 8]], np.int32)
    eng.env_spec(slots, k_neighbours=4, radius=10.0, lookahead=(0.5, 2.0))
    plain, am0 = eng.env_observe()
    eng.env_spec(slots, k_neighbours=4, radius=10.0, lookahead=(0.5, 2.0), n_rays=16, ray_range=RANGE)
    lidar, am1 = eng.env_observe()
    F0 = plain.shape[-1]
    assert lidar.shape[-1] == F0 + 16 and np.array_equal(am0, am1)
    assert np.array_equal(lidar[..., :F0].view(np.uint32), plain.view(np.uint32))
    assert not lidar[slots < 0].any()


# ---------------------------------------------------------------------------------------------- crafted
# Each crafted scenario: slot 0 is the agent at the origin (+ offset), heading 0, with a large box of its own
# (it must not see it); slot 2 is absent but would be hit 3 m ahead; slots 1 and 3 are the case's objects.
# (x, y, width, length) per slot; None: absent.  Every heading is 0 and every box centre offset 0.
OWN = (0.0, 0.0, 3.0, 6.0)
HIDDEN = (3.5, 0.0, 2.0, 1.0)
CASES = {
    "ahead": [(12.5, 0.0, 2.0, 5.0), None],                 # near face 10 m ahead on ray 0 (straddles ray 0)
    "behind": [(-12.5, 0.0, 2.0, 5.0), None],               # straddles ray R/2
    "corner": [(7.0, 3.0, 4.0, 4.0), None],                 # corner (5, 5) touches the diagonal
    "edge": [(5.0, 1.0, 2.0, 4.0), None],                   # ray 0 runs along the bottom edge y = 0
    "inside": [(0.5, 0.0, 2.0, 4.0), None],                 # the origin inside the box: every ray reads 0
    "beyond": [(62.5, 0.0, 2.0, 5.0), (0.0, 51.0, 2.0, 4.0)],  # 60 m ahead; near face exactly at 50 m left
    "near_range": [(52.0, 0.0, 2.0, 4.0), (0.0, -50.0, 2.0, 4.0)],  # ahead: face at 50 m; right: 49 m
    "flat": [(5.0, 0.0, 0.0, 4.0), (0.0, 6.0, 0.0, 4.0)],   # zero width: along ray 0; across ray 2
    "points": [(8.0, 0.0, 0.0, 0.0), (4.0, 4.0, 0.0, 0.0)],  # zero-size boxes on ray 0 and on the diagonal
    "empty": [None, None],                                  # nothing but the hidden slot
}
NAMES = list(CASES)


def crafted_state(offset):
    """(scene, pose [6, N*M], present [N*M], slots [N, A]) of the crafted scenes, shifted by `offset` metres."""
    N, M = len(CASES), 4
    cfg = synthetic.vehicles_config(seed=0, N=N, M=M, T=4, half_extent=14.0)
    scene = synthetic.pack_synthetic(cfg)
    box = scene.box.reshape(4, N * M)
    pose = np.zeros((6, N * M))
    present = np.zeros(N * M, np.uint8)
    for n, name in enumerate(NAMES):
        for s, spec in enumerate([OWN, CASES[name][0], HIDDEN, CASES[name][1]]):
            if spec is None:
                continue
            x, y, w, length = spec
            i = n * M + s
            pose[0, i], pose[1, i] = offset + x, offset + y
            box[:, i] = (w, length, 0.0, 0.0)
            present[i] = s != 2
    # agents: slot 0; an absent agent (slot 2); padding
    slots = np.tile(np.array([[0, 2, -1]], np.int32), (N, 1))
    return scene, pose, present, slots


def oracle_crafted(offset, ray_dir):
    scene, pose, present, slots = crafted_state(offset)
    p = abi.default_params()
    eng = LidarOracleEngine(scene, p)
    eng.reset()
    eng.state["pose"][...] = pose
    eng.state["present"][...] = present
    eng.env_spec(slots, k_neighbours=1, lookahead=(), n_rays=len(ray_dir), ray_range=RANGE, ray_dir=ray_dir)
    obs, am = eng.env_observe()
    return scene, eng, slots, obs, am


def crafted_expected(R):
    """The exact readings of agent 0 per case for the R = 4 / R = 8 tables."""
    d8 = {  # ray index of DIRS8 -> reading (every other ray reads the range)
        "ahead": {0: 10.0}, "behind": {4: 10.0}, "corner": {1: 5.0 / SQ}, "edge": {0: 3.0},
        "inside": {k: 0.0 for k in range(8)}, "beyond": {}, "near_range": {6: 49.0}, "flat": {0: 3.0, 2: 6.0},
        "points": {0: 8.0, 1: 4.0 / SQ}, "empty": {},
    }
    out = {}
    for name, hits in d8.items():
        full = np.full(8, RANGE)
        for k, v in hits.items():
            full[k] = v
        out[name] = (full if R == 8 else full[::2]).astype(np.float32)
    return out


@pytest.mark.parametrize("offset", [0.0, 1e5])
@pytest.mark.parametrize("R", [4, 8])
def test_lidar_crafted_exact(R, offset):
    dirs = DIRS4 if R == 4 else DIRS8
    scene, eng, slots, obs, am = oracle_crafted(offset, dirs)
    want = numpy_lidar(scene, eng.state, slots, dirs, RANGE)
    got = obs[..., -R:]
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    exp = crafted_expected(R)
    for n, name in enumerate(NAMES):
        assert np.array_equal(got[n, 0], exp[name]), (name, got[n, 0], exp[name])
    # absent (slot 2) and padding agents: zero rows, agent mask 0
    assert not obs[:, 1:].any() and not am[:, 1:].any() and am[:, 0].all()


def test_lidar_directions_table():
    for R in (1, 7, 64, 256):
        d = abi.lidar_directions(R)
        ang = 2 * np.pi * np.arange(R) / R
        assert d.shape == (R, 2) and d.dtype == np.float64
        assert np.abs(d - np.stack([np.cos(ang), np.sin(ang)], 1)).max() <= 1e-12
