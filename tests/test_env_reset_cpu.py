"""
CPU tests of the randomised episode starts (sg_reset_scenarios_init, include/sg_b200.h; ``ResetSpec``): the numpy
restatement of the start-time uniform and the noise keys against the plain-C oracle, ``abi.start_windows`` on
crafted scenes, the oracle against ``sgo_reset_scenarios`` with nothing drawn, the perturbed rows against the
formulas restated in numpy, and ``ResetSpec``'s validation.
"""
import math

import numpy as np
import pytest

from oracle import golden_cases
from scenario_gym_b200 import ResetSpec, abi, synthetic
from scenario_gym_b200.packing import ScenarioSpec, SlotSpec, pack_scenarios

from helpers import all_xosc_specs
from plan_oracle import noise2_c
from reset_oracle import (ResetOracleEngine, perturb_noise, perturb_rows, reset_init, start_times, tick2,
                          uniform_c, uniform_numpy)

SKIP = ("coll_mask", "events", "trace_pose", "trace_present", "trace_t")


def rss_scene():
    cfg = golden_cases.rss_cfg()
    p = abi.default_params()
    p.timestep, p.features = cfg.dt, p.features | abi.FEAT_RSS
    return synthetic.pack_synthetic(cfg), p, cfg.actions


def xosc_scene():
    return pack_scenarios([s for _, s, _, _ in all_xosc_specs("xosc")]), abi.default_params(), None


def state_of(eng):
    return {name: eng.get(name).copy() for name, _, _ in abi.STATE_FIELDS if name not in SKIP}


def scenario_part(name, a, n, M):
    """Scenario n's part of a state array ([..., N*M] planes or [N, ...])."""
    spec = dict((f, s) for f, _, s in abi.STATE_FIELDS)[name]
    if "NM" in spec:
        return a[..., n * M:(n + 1) * M]
    return a[n] if spec[0] == "N" else a


# ------------------------------------------------------------------------------------------- streams
def test_uniform_numpy_matches_c():
    rng = np.random.default_rng(0)
    i = np.concatenate([-1 - np.arange(64), rng.integers(-2**62, 2**62, 64), [2**40 + 3, -(2**40)]])
    for seed in (0, 1, 2**64 - 1, 0x9E3779B97F4A7C15):
        for k in (0, 1, 7, 2**30, 2**31 + 5, 2**40):
            t = int(tick2(k))
            u = uniform_c(seed, i, t)
            assert np.array_equal(u, uniform_numpy(seed, i, t))
            assert np.all((u >= 0.0) & (u < 1.0))


def test_tick_value_wraps_to_32_bits():
    assert int(tick2(0)) == 0 and int(tick2(3)) == 6
    assert int(tick2(2**30)) == -2**31 and int(tick2(2**31)) == 0 and int(tick2(2**31 + 1)) == 2


def test_perturbation_keys_match_c():
    ctr = np.array([0, 1, 11, 12 * 7 + 3, 2**33 + 5])
    for k in (0, 5, 2**30 - 1, 2**31 + 9):
        z = perturb_noise(42, ctr, k)
        t = int(tick2(k))
        assert np.array_equal(z[..., :2], noise2_c(42, ctr, t))
        assert np.array_equal(z[..., 2:], noise2_c(42, ctr, t + 1))


# ------------------------------------------------------------------------------------------- windows
def _traj(t0, t1, x=0.0, n=None):
    ts = np.linspace(t0, t1, n or int(round((t1 - t0) * 10)) + 1)
    out = np.zeros((len(ts), 7))
    out[:, 0], out[:, 1] = ts, x + 5.0 * ts
    return out


def test_start_windows_crafted():
    V, R, E = abi.KIND_VEHICLE, abi.KIND_REPLAY, abi.KIND_AGENT_REPLAY
    static = np.array([[3.0, 50.0, 0, 0, 0, 0, 0]])
    specs = [
        # a vehicle that ends at 4 s bounds the window: min(10 - 1 - 0, 4 - 0)
        ScenarioSpec([SlotSpec(V, _traj(0, 10)), SlotSpec(V, _traj(0, 4, 20.0))]),
        # a static vehicle (one row) and replay-only slots ending early do not bound it
        ScenarioSpec([SlotSpec(V, _traj(0, 10)), SlotSpec(V, static), SlotSpec(R, _traj(0, 2, 40.0)),
                      SlotSpec(E, _traj(0, 3, 60.0))]),
        # t0 = 2 (the ego's first point); a vehicle absent at t0 (it starts at 5) does not bound it
        ScenarioSpec([SlotSpec(V, _traj(2, 12)), SlotSpec(V, _traj(5, 6, 30.0)), SlotSpec(V, _traj(0, 9, 50.0))]),
        # a PID slot bounds it like a vehicle
        ScenarioSpec([SlotSpec(V, _traj(0, 10)), SlotSpec(abi.KIND_PID, _traj(0, 2.5, 20.0))]),
        # a log shorter than min_remaining: 0
        ScenarioSpec([SlotSpec(V, _traj(0, 0.5))]),
    ]
    scene = pack_scenarios(specs)
    w = abi.start_windows(scene, False, 1.0)
    assert w.dtype == np.float64 and w.shape == (5,)
    assert np.allclose(w, [4.0, 9.0, 7.0, 2.5, 0.0], rtol=0, atol=1e-12)
    # persist: every slot stays present, only the log's end bounds the window
    assert np.allclose(abi.start_windows(scene, True, 1.0), [9.0, 9.0, 9.0, 9.0, 0.0], rtol=0, atol=1e-12)
    # min_remaining longer than every log: all 0
    assert np.array_equal(abi.start_windows(scene, False, 100.0), np.zeros(5))
    assert np.allclose(abi.start_windows(scene, False, 0.0), [4.0, 10.0, 7.0, 2.5, 0.5], rtol=0, atol=1e-12)


def test_start_windows_keep_vehicles_present():
    """At any start inside the window every vehicle present at t0 is still present (its log covers it)."""
    scene, _, _ = rss_scene()
    w = abi.start_windows(scene, False, 0.5)
    M = scene.M
    for n in range(scene.N):
        for s in range(M):
            i = n * M + s
            r = scene.traj_rows[scene.traj_off[i]:scene.traj_off[i + 1]]
            assert r[0, 0] <= scene.t0[n] + w[n] <= r[-1, 0]


# ------------------------------------------------------------------------------------------- the oracle
@pytest.mark.parametrize("which", ["vehicles", "general"])
def test_oracle_without_draws_is_the_masked_reset(which):
    scene, p, actions = rss_scene() if which == "vehicles" else xosc_scene()
    a, b = ResetOracleEngine(scene, p), ResetOracleEngine(scene, p)
    for e in (a, b):
        e.reset()
        e.rollout(20, actions=actions)
    mask = (np.arange(scene.N) % 3 != 1).astype(np.uint8)
    a.reset_scenarios(mask)
    init, keep = reset_init(t_start=scene.t0, counter=np.arange(scene.N) * 5, perturb=np.ones(scene.N * scene.M),
                            seed=9)
    b.reset_init(mask, init)
    sa, sb = state_of(a), state_of(b)
    for name in sa:
        assert np.array_equal(sa[name], sb[name], equal_nan=True), name
    # a zero window draws t0 too
    init, keep = reset_init(start_window=np.zeros(scene.N), counter=np.zeros(scene.N), seed=3)
    b.reset_init(None, init)
    a.reset_scenarios(np.ones(scene.N, np.uint8))
    sa, sb = state_of(a), state_of(b)
    for name in sa:
        if name != "event_count":  # (sgo_reset_scenarios of a full mask and the init reset both keep it)
            assert np.array_equal(sa[name], sb[name], equal_nan=True), name


def test_oracle_drawn_start_times():
    scene, p, _ = rss_scene()
    e = ResetOracleEngine(scene, p)
    win = abi.start_windows(scene, False, 1.0)
    counter = np.array([0, 1, 2**31 + 1, 17])
    init, keep = reset_init(start_window=win, counter=counter, seed=123)
    e.reset_init(None, init)
    want = start_times(scene.t0, win, counter, 123)
    assert np.array_equal(e.get("t"), want)
    assert np.array_equal(e.get("prev_t"), want - 0.1)
    assert np.all((want >= scene.t0) & (want < scene.t0 + win))


@pytest.mark.parametrize("which", ["vehicles", "general"])
def test_oracle_perturbed_rows_follow_the_formulas(which):
    scene, p, actions = rss_scene() if which == "vehicles" else xosc_scene()
    N, M = scene.N, scene.M
    nm = N * M
    rng = np.random.default_rng(1)
    t_start = scene.t0 + rng.uniform(0.0, 1.0, N) * abi.start_windows(scene, False, 1.0)
    mask = np.ones(N, np.uint8)
    mask[1] = 0
    perturb = (rng.random(nm) < 0.6).astype(np.uint8)
    counter = rng.integers(0, 1000, N)
    sigma, seed = (0.7, 0.3, 0.05, 1.5), 77
    base, pert = ResetOracleEngine(scene, p), ResetOracleEngine(scene, p)
    for e in (base, pert):
        e.reset()
        e.rollout(10, actions=actions)
    before = state_of(pert)
    i0, _k0 = reset_init(t_start=t_start, counter=counter)
    base.reset_init(mask, i0)
    i1, _k1 = reset_init(t_start=t_start, counter=counter, perturb=perturb, sigma=sigma, seed=seed)
    pert.reset_init(mask, i1)
    b, q = state_of(base), state_of(pert)
    kind = scene.kind.reshape(-1)
    ctr = np.arange(nm)
    k = np.repeat(counter, M)
    z = np.stack([perturb_noise(seed, ctr[j:j + 1], int(k[j]))[0] for j in range(nm)])
    x, y, h, vx, vy, v = perturb_rows(b["pose"][0], b["pose"][1], b["pose"][3], b["vel"][0], b["vel"][1], z, sigma)
    sel = (np.repeat(mask, M) != 0) & (perturb != 0) & (b["present"] != 0)
    assert sel.sum() > 3
    assert np.array_equal(q["present"], b["present"])
    for got, want, f in ((q["pose"][0], x, "x"), (q["pose"][1], y, "y"), (q["pose"][3], h, "h"),
                         (q["vel"][0], vx, "vx"), (q["vel"][1], vy, "vy")):
        assert np.array_equal(got[sel], want[sel]), f
    ctl = sel & ((kind == abi.KIND_VEHICLE) | (kind == abi.KIND_PID))
    assert np.array_equal(q["speed"][ctl], v[ctl])
    # unflagged or absent slots of the reset scenarios are the plain reset's
    rest = (np.repeat(mask, M) != 0) & ~sel
    for f in ("pose", "vel", "speed", "present"):
        assert np.array_equal(q[f][..., rest], b[f][..., rest]), f
    for f in (2, 4, 5):  # z, pitch, roll never move
        assert np.array_equal(q["pose"][f], b["pose"][f])
    # the ego metrics see the perturbed start
    for n in range(N):
        if mask[n]:
            ei = n * M + scene.ego_slot[n]
            sp = math.sqrt(q["vel"][0, ei] ** 2 + q["vel"][1, ei] ** 2 + q["vel"][2, ei] ** 2)
            assert q["ego_avg_speed"][n] == sp and q["ego_max_speed"][n] == sp
    # the scenario outside the mask is untouched
    for name in q:
        assert np.array_equal(scenario_part(name, q[name], 1, M), scenario_part(name, before[name], 1, M),
                              equal_nan=True), name


def test_zero_sigma_components_are_bit_identical():
    scene, p, _ = rss_scene()
    N, M = scene.N, scene.M
    counter, perturb = np.arange(N), np.ones(N * M)
    base = ResetOracleEngine(scene, p)
    i0, _k0 = reset_init(counter=counter)
    base.reset_init(None, i0)
    b = state_of(base)
    for sigma, same in (((0.0, 0.0, 0.0, 0.0), ("pose", "vel", "speed")),
                        ((0.0, 0.5, 0.0, 0.0), ("vel", "speed")),
                        ((0.0, 0.0, 0.0, 2.0), ("pose",)),
                        ((1.0, 1.0, 0.0, 0.0), ("vel", "speed"))):
        e = ResetOracleEngine(scene, p)
        i1, _k1 = reset_init(counter=counter, perturb=perturb, sigma=sigma, seed=5)
        e.reset_init(None, i1)
        q = state_of(e)
        for f in same:
            assert np.array_equal(q[f], b[f]), (sigma, f)
        assert np.array_equal(q["pose"][3], b["pose"][3]), sigma  # sigma[2] = 0: heading kept
        if sigma[0] == 0.0 and sigma[1] != 0.0:
            assert not np.array_equal(q["pose"][0], b["pose"][0])


def test_oracle_rejects_bad_init():
    scene, p, _ = rss_scene()
    e = ResetOracleEngine(scene, p)
    for sigma in ((-1.0, 0, 0, 0), (0, math.nan, 0, 0), (0, 0, math.inf, 0)):
        init, _keep = reset_init(counter=np.zeros(scene.N), sigma=sigma)
        with pytest.raises(RuntimeError, match="sigma"):
            e.reset_init(None, init)
    init, _keep = reset_init()
    with pytest.raises(RuntimeError, match="counter"):
        e.reset_init(None, init)


# ------------------------------------------------------------------------------------------- ResetSpec
def test_reset_spec_validation():
    ResetSpec()
    ResetSpec(start_offset=3, min_remaining=0.0, lon=0.5, lat=0.2, heading=0.05, speed=1.0, seed=2**70)
    for name in ("start_offset", "min_remaining", "lon", "lat", "heading", "speed"):
        for bad in (-0.1, math.nan, math.inf, -math.inf, True, "1", None):
            with pytest.raises(ValueError, match=name):
                ResetSpec(**{name: bad})
    for bad in (1.5, "3", None, True):
        with pytest.raises(ValueError, match="seed"):
            ResetSpec(seed=bad)
