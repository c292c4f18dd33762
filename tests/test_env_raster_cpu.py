"""
CPU tests of sg_env_raster's semantics (include/sg_b200.h, SgRasterSpec): the plain-C brute-force restatement
(tests/raster_oracle.c) against an independent numpy restatement on crafted cases, the surface channels against
the oracle's strict containment away from the rings, the polygon bounding boxes, and the argument checks of
ObsSpec and of the product's entry point.
"""
import ctypes as C
import dataclasses
import math

import numpy as np
import pytest

from scenario_gym_b200 import ObsSpec, VecScenarioEnv, abi, synthetic

from raster_oracle import RasterOracleEngine, raster_spec
from test_env_map_cpu import RN_FIELDS, ring, soup

# crafted case (S = 32, 1 m pixels, the agent at the origin with heading 0: pixel centres at half-integers,
# pu_i = 15.5 - i, pv_j = 15.5 - j)
ROAD = ring((-14, 9), (14, 9), (14, 13), (-14, 13))               # edges between pixel centres
LANE = ring((-14, 11), (14, 11), (14, 13), (-14, 13))             # inside the road: an OR, not a parity
THROUGH = ring((2.5, -13.5), (6.5, -13.5), (6.5, -9.5), (2.5, -9.5))  # edges through pixel centres
VERTEX = ring((4.5, 2.2), (10, -3), (10, 7))                      # a vertex exactly on row 11 (pu = 4.5)
HOLED = np.concatenate([ring((-12, -12), (-2, -12), (-2, -2), (-12, -2)),
                        ring((-9, -9), (-9, -5), (-5, -5), (-5, -9))])  # a square with a square hole
BUILDING = ring((8, -8), (12, -8), (12, -4), (8, -4))             # walkable and impenetrable


def crafted_scene(rot45=True):
    """Two scenarios of 6 slots: 0 with the crafted network, 1 without one.  Slot 0 is the agent (at the origin,
    heading 0), 1 a vehicle (45 degrees when rot45), 2 a 1 x 1 pedestrian, 3 a flat box (width 0) along a pixel
    row, 4 absent, 5 far away."""
    N, M = 2, 6
    cfg = synthetic.vehicles_config(seed=0, N=N, M=M, T=4, half_extent=1.0)
    scene = synthetic.pack_synthetic(cfg)
    po, eo, ed = soup([[[ROAD, LANE, THROUGH, VERTEX], [HOLED, BUILDING], [BUILDING]]])
    rn = (np.array([0, -1], np.int32), po, eo, ed, np.ones(3, np.uint8))
    etype = np.zeros(N * M, np.uint8)
    box = np.zeros((4, N * M))
    box[0], box[1] = 2.0, 4.0  # width, length
    pose = np.zeros((6, N * M))
    present = np.ones(N * M, np.uint8)
    for n in range(N):
        b = n * M
        pose[:2, b + 1], pose[3, b + 1] = (-6.0, 6.0), (math.pi / 4 if rot45 else 0.0)
        pose[:2, b + 2] = (0.0, -6.0)
        etype[b + 2], box[0, b + 2], box[1, b + 2] = abi.ETYPE_PEDESTRIAN, 1.0, 1.0
        pose[:2, b + 3], box[0, b + 3] = (12.0, 4.5), 0.0
        box[2, b + 3] = 0.0
        present[b + 4] = 0
        pose[:2, b + 5] = (100.0, 100.0)
    scene = dataclasses.replace(scene, etype=etype, box=np.ascontiguousarray(box), **dict(zip(RN_FIELDS, rn)))
    slots = np.tile(np.array([0, 4, -1], np.int32), (N, 1))  # an agent, an absent agent, a padding agent
    return scene, pose, present, slots


def oracle_for(scene, pose, present, slots):
    eng = RasterOracleEngine(scene, abi.default_params())
    eng.reset()
    eng.state["pose"][...] = pose.reshape(eng.state["pose"].shape)
    eng.state["present"][...] = present.reshape(eng.state["present"].shape)
    eng.env_spec(slots, 0, 0.0, ())
    return eng


def numpy_raster(scene, pose, present, slots, S, res, ahead):
    """sg_env_raster restated in numpy, vectorised over the pixels (IEEE fp64, no FMA; cos / sin from libm)."""
    N, M = scene.N, scene.M
    A = slots.shape[1]
    out = np.zeros((N, A, 5, S, S), np.uint8)
    h = 0.5 * res
    k = (S - 1 - 2 * np.arange(S)).astype(np.float64)
    pu, pv = ahead + k * h, k * h
    PU, PV = pu[:, None], pv[None, :]
    box = scene.box.reshape(4, N * M)
    for n in range(N):
        for a in range(A):
            slot = int(slots[n, a])
            if slot < 0 or slot >= M or not present[n * M + slot]:
                continue
            i = n * M + slot
            x, y, hd = pose[0, i], pose[1, i], pose[3, i]
            c, s = math.cos(hd), math.sin(hd)
            rn = int(scene.rn_of[n]) if scene.n_networks > 0 else -1
            for ch in range(3 if rn >= 0 else 0):
                acc = np.zeros((S, S), bool)
                for q in range(int(scene.rn_poly_off[3 * rn + ch]), int(scene.rn_poly_off[3 * rn + ch + 1])):
                    odd = np.zeros((S, S), bool)
                    for e in scene.rn_edges[int(scene.rn_edge_off[q]):int(scene.rn_edge_off[q + 1])]:
                        adx, ady, bdx, bdy = e[0] - x, e[1] - y, e[2] - x, e[3] - y
                        au, av = c * adx + s * ady, -s * adx + c * ady
                        bu, bv = c * bdx + s * bdy, -s * bdx + c * bdy
                        cross = (au > pu) != (bu > pu)
                        if not cross.any():
                            continue
                        vc = av + ((pu[cross] - au) * (bv - av)) / (bu - au)
                        odd[cross] ^= vc[:, None] > pv[None, :]
                    acc |= odd
                out[n, a, ch] = acc
            Px, Py = x + (c * PU - s * PV), y + (s * PU + c * PV)
            for j in range(M):
                b = n * M + j
                if j == slot or not present[b]:
                    continue
                cj, sj = math.cos(pose[3, b]), math.sin(pose[3, b])
                X = pose[0, b] + (box[2, b] * cj - box[3, b] * sj)
                Y = pose[1, b] + (box[2, b] * sj + box[3, b] * cj)
                px, py = Px - X, Py - Y
                ox, oy = cj * px + sj * py, -sj * px + cj * py
                hit = (np.abs(ox) <= 0.5 * box[1, b]) & (np.abs(oy) <= 0.5 * box[0, b])
                out[n, a, 4 if scene.etype[b] == abi.ETYPE_PEDESTRIAN else 3] |= hit.astype(np.uint8)
    return out


@pytest.mark.parametrize("rot45", [True, False])
def test_oracle_matches_numpy_crafted(rot45):
    scene, pose, present, slots = crafted_scene(rot45)
    eng = oracle_for(scene, pose, present, slots)
    for S, res, ahead in ((32, 1.0, 0.0), (64, 0.5, 0.0), (32, 1.0, 3.0), (64, 0.25, -1.5)):
        got = eng.env_raster(raster_spec(scene, S, res, ahead))
        want = numpy_raster(scene, pose, present, slots, S, res, ahead)
        assert np.array_equal(got, want), (S, res, ahead)
        assert not got[:, 1:].any(), "absent and padding agents get zeros"
        assert not got[1, 0, :3].any(), "a scenario without a network gets zero surfaces"
        assert got[1, 0, 3:].any() and np.array_equal(got[1, 0, 3:], got[0, 0, 3:])


def test_oracle_crafted_exact_pixels():
    scene, pose, present, slots = crafted_scene(rot45=False)
    img = oracle_for(scene, pose, present, slots).env_raster(raster_spec(scene, 32, 1.0, 0.0))[0, 0]
    u = 15.5 - np.arange(32.0)  # row i -> u, column j -> v (the same values)

    def cells(ch, u0, u1, v0, v1):
        return img[ch][np.ix_((u >= u0) & (u < u1), (u >= v0) & (u < v1))]

    # road: 28 x 4 pixels, the lane inside it changes nothing
    assert cells(0, -14, 14, 9, 13).all() and img[0][:, (u > 8) & (u < 14)].sum() == 28 * 4
    # through: the rear / right sides in, the front / left sides out
    assert cells(0, 2.5, 6.5, -13.5, -9.5).all() and cells(0, 2.5, 6.5, -13.5, -9.5).size == 16
    assert not img[0][u == 6.5][:, (u >= -13.5) & (u <= -9.5)].any()
    assert not img[0][(u >= 2.5) & (u <= 6.5)][:, u == -9.5].any()
    # the holed square: 100 - 16 pixels
    assert img[1][np.ix_(u < 0, u < 0)].sum() == 84 and not cells(1, -9, -5, -9, -5).any()
    # the building in both surfaces, nowhere in the driveable one
    assert cells(1, 8, 12, -8, -4).all() and cells(2, 8, 12, -8, -4).all() and img[2].sum() == 16
    # boxes: the vehicle 4 x 2 at (-6, 6) (4 x 2 centres), the pedestrian 1 x 1 (2 x 2 centres),
    # the flat box on row v = 4.5 (4 centres), nothing from the absent and far slots
    assert img[4].sum() == 4 and cells(4, -0.5, 1, -6.5, -5).all()
    assert img[3].sum() == 8 + 4 and cells(3, 10, 14, 4.5, 5).all()
    # the vertex on a row: both edges at the apex cross row u = 4.5 at the vertex, so they cancel there
    tri = (u > -3) & (u < 7)
    assert img[0][u == 4.5][:, tri].sum() == 0 and img[0][u == 5.5][:, tri].sum() > 0


def test_raster_poly_boxes_matches_loop():
    po, eo, ed = soup([[[ROAD, LANE], [HOLED], []], [[], [BUILDING], [BUILDING]]])
    eo = np.concatenate([eo, [eo[-1]]])  # a polygon without edges
    box, m = abi.raster_poly_boxes(eo, ed, 10.0)
    assert box.shape == (len(eo) - 1, 4)
    for q in range(len(eo) - 1):
        es = ed[eo[q]:eo[q + 1]]
        if len(es) == 0:
            assert not box[q].any()
            continue
        xs, ys = [v for e in es for v in (e[0], e[2])], [v for e in es for v in (e[1], e[3])]
        assert list(box[q]) == [min(xs), min(ys), max(xs), max(ys)], q
    assert m == 1e-9 * (1.0 + float(np.abs(ed).max()) + 10.0)
    box0, m0 = abi.raster_poly_boxes(np.zeros(1, np.int64), np.zeros((0, 4)), 5.0)
    assert box0.shape == (0, 4) and m0 == 1e-9 * 6.0


def _ring_distance(px, py, edges):
    """Distance of each point to the nearest edge."""
    ax, ay, bx, by = (edges[:, k][None, :] for k in range(4))
    dx, dy = bx - ax, by - ay
    L2 = dx * dx + dy * dy
    t = np.clip(((px[:, None] - ax) * dx + (py[:, None] - ay) * dy) / np.where(L2 > 0, L2, 1.0), 0.0, 1.0)
    qx, qy = ax + t * dx - px[:, None], ay + t * dy - py[:, None]
    return np.sqrt(qx * qx + qy * qy).min(1)


def test_surface_channels_agree_with_surface_contains():
    town = synthetic.grid_town(seed=0)
    cfg = synthetic.vehicles_config(seed=1, N=2, M=4, T=4, half_extent=150.0)
    scene = synthetic.pack_synthetic(cfg, road_network=town)
    rng = np.random.default_rng(0)
    pose = np.zeros((6, scene.N * scene.M))
    pose[0], pose[1] = rng.uniform(-150, 150, pose.shape[1]), rng.uniform(-150, 150, pose.shape[1])
    pose[3] = rng.uniform(-math.pi, math.pi, pose.shape[1])
    present = np.ones(scene.N * scene.M, np.uint8)
    slots = np.tile(np.arange(scene.M, dtype=np.int32), (scene.N, 1))
    eng = oracle_for(scene, pose, present, slots)
    S, res, ahead = 64, 0.5, 4.0
    img = eng.env_raster(raster_spec(scene, S, res, ahead))
    h = 0.5 * res
    k = (S - 1 - 2 * np.arange(S)).astype(np.float64)
    PU, PV = (ahead + k * h)[:, None], (k * h)[None, :]
    checked = inside = 0
    for n in range(scene.N):
        r = int(scene.rn_of[n])
        e0, e1 = int(scene.rn_edge_off[scene.rn_poly_off[3 * r]]), int(scene.rn_edge_off[scene.rn_poly_off[3 * r + 3]])
        edges = scene.rn_edges[e0:e1]
        for a in range(scene.M):
            i = n * scene.M + a
            x, y, hd = pose[0, i], pose[1, i], pose[3, i]
            c, s = math.cos(hd), math.sin(hd)
            Px, Py = (x + (c * PU - s * PV)).reshape(-1), (y + (s * PU + c * PV)).reshape(-1)
            near = (np.maximum(edges[:, 0], edges[:, 2]) > Px.min() - 1) & (np.minimum(edges[:, 0], edges[:, 2]) < Px.max() + 1) \
                & (np.maximum(edges[:, 1], edges[:, 3]) > Py.min() - 1) & (np.minimum(edges[:, 1], edges[:, 3]) < Py.max() + 1)
            far = _ring_distance(Px, Py, edges[near]) > 1e-6 if near.any() else np.ones(len(Px), bool)
            for ch in range(3):
                want = eng.surface_contains(n, ch, Px, Py)
                got = img[n, a, ch].reshape(-1)
                assert np.array_equal(got[far], want[far]), (n, a, ch)
                checked += int(far.sum())
                inside += int(want[far].sum())
    assert inside > 0 and checked > inside, "the poses must see both inside and outside"


def _env_with(**raster):
    return VecScenarioEnv([], obs=ObsSpec(**raster))


@pytest.mark.parametrize("bad", [dict(raster_size=16), dict(raster_size=33), dict(raster_size=288),
                                 dict(raster_size=-32), dict(raster_size=64.5), dict(raster_size=True),
                                 dict(raster_size=64, raster_resolution=0.0),
                                 dict(raster_size=64, raster_resolution=-1.0),
                                 dict(raster_size=64, raster_resolution=math.nan),
                                 dict(raster_size=64, raster_resolution=math.inf),
                                 dict(raster_size=64, raster_ahead=math.nan),
                                 dict(raster_size=64, raster_ahead=math.inf)])
def test_obs_spec_raster_validation(bad):
    with pytest.raises(ValueError, match="raster"):
        _env_with(**bad)


def test_obs_spec_raster_defaults():
    o = ObsSpec()
    assert (o.raster_size, o.raster_resolution, o.raster_ahead) == (0, 0.5, 0.0)
    assert o.n_features == ObsSpec(raster_size=64).n_features, "the raster stays out of the observation rows"


def test_raster_spec_checks_of_the_product():
    """The product's sg_env_raster rejects bad SgRasterSpecs before touching the device."""
    lib = abi.bind(C.CDLL(abi.PRODUCT_LIB), "sg_") if _product_built() else pytest.skip("library not built")
    assert C.sizeof(abi.SgRasterSpec) == lib["sizeof"](9)
    sc, p, st, e = abi.SgScene(), abi.SgParams(), abi.SgState(), abi.SgEnvSpec()
    sc.n_scenarios, sc.n_slots, sc.n_networks = 2, 4, 1
    e.n_agents = 1
    for k in ("agent_slot", "snap_dist", "snap_collided", "snap_pair_ticks", "snap_rss"):
        setattr(e, k, 16)
    fake = 4096

    def call(**kw):
        r = abi.SgRasterSpec()
        r.size, r.n_networks, r.resolution, r.ahead, r.margin, r.poly_box = 64, 1, 0.5, 0.0, 0.0, fake
        for k, v in kw.items():
            setattr(r, k, v)
        rc = lib["env_raster"](C.byref(sc), C.byref(p), C.byref(st), C.byref(e), C.byref(r), None, fake, 0, None)
        return rc, lib["last_error"]().decode()

    for kw, msg in ((dict(size=16), "size"), (dict(size=33), "size"), (dict(size=288), "size"), (dict(size=0), "size"),
                    (dict(resolution=0.0), "resolution"), (dict(resolution=-1.0), "resolution"),
                    (dict(resolution=math.nan), "resolution"), (dict(ahead=math.nan), "ahead"),
                    (dict(ahead=math.inf), "ahead"), (dict(margin=-1.0), "margin"),
                    (dict(n_networks=0), "n_networks"), (dict(poly_box=None), "poly_box")):
        rc, err = call(**kw)
        assert rc != 0 and msg in err, (kw, err)
    rc = lib["env_raster"](C.byref(sc), C.byref(p), C.byref(st), C.byref(e), None, None, fake, 0, None)
    assert rc != 0 and "null" in lib["last_error"]().decode()


def _product_built():
    import os

    return os.path.exists(abi.PRODUCT_LIB)
