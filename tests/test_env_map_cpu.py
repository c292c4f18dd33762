"""
CPU tests of the map block of sg_env_observe: the map-table builder (abi.map_table) against a Python loop, the
culling grid's conservativeness, and the plain-C restatement (tests/map_oracle.c) against an independent numpy
restatement of include/sg_b200.h (SgEnvSpec), on crafted cases whose answers are exact and on a seeded town.
"""
import dataclasses
import math

import numpy as np
import pytest

from scenario_gym_b200 import abi, synthetic
from scenario_gym_b200.packing import pack_road_networks
from scenario_gym_b200.road_network import (Building, Lane, PolygonArea, Pavement, Road, RoadNetwork)

from map_oracle import MapOracleEngine

RN_FIELDS = ("rn_of", "rn_poly_off", "rn_edge_off", "rn_edges", "rn_has_area")


def soup(networks):
    """SgScene.rn_* soups from [[surface0 polys, surface1 polys, surface2 polys], ...] (polys: [E, 4] edges)."""
    poly_off, edge_off, edges = [0], [0], []
    for net in networks:
        for polys in net:
            for e in polys:
                e = np.asarray(e, np.float64).reshape(-1, 4)
                edges.append(e)
                edge_off.append(edge_off[-1] + len(e))
            poly_off.append(len(edge_off) - 1)
    return (np.array(poly_off, np.int64), np.array(edge_off, np.int64),
            np.concatenate(edges) if edges else np.zeros((0, 4)))


def loop_table(poly_off, edge_off, edges, r):
    """The map table of network r by a plain loop over include/sg_b200.h's rules."""
    seen, rows = {}, []
    for k in range(3):
        for q in range(int(poly_off[3 * r + k]), int(poly_off[3 * r + k + 1])):
            for i in range(int(edge_off[q]), int(edge_off[q + 1])):
                x0, y0, x1, y1 = (float(v) for v in edges[i])
                if x0 == x1 and y0 == y1:
                    continue
                key = tuple(sorted([(x0 + 0.0, y0 + 0.0), (x1 + 0.0, y1 + 0.0)]))
                if key not in seen:
                    seen[key] = len(rows)
                    rows.append([[x0, y0, x1, y1], 0])
                rows[seen[key]][1] |= 1 << k
    seg = np.array([s for s, _ in rows], np.float64).reshape(-1, 4)
    return seg, np.array([f for _, f in rows], np.uint8)


def ring(*pts):
    return np.array([[*pts[i], *pts[(i + 1) % len(pts)]] for i in range(len(pts))], np.float64)


def crafted_networks():
    road = ring((0, 0), (10, 0), (10, 4), (0, 4))
    lane0, lane1 = ring((0, 0), (10, 0), (10, 2), (0, 2)), ring((10, 4), (0, 4), (0, 2), (10, 2))  # reversed edges
    pave = ring((0, 4), (10, 4), (10, 6), (0, 6))
    bld = ring((2, 8), (5, 8), (5, 8), (5, 11), (2, 11))  # with a zero-length edge
    a = [[road, lane0, lane1], [pave, bld], [bld]]
    b = [[ring((-0.0, 0.0), (3, 0), (3, 3))], [ring((0.0, -0.0), (3, 3), (3, 0))], []]  # -0.0 equals 0.0
    empty = [[], [], []]
    zero_only = [[np.array([[1.0, 1.0, 1.0, 1.0]])], [], []]
    return [a, empty, b, zero_only]


def test_map_table_matches_loop():
    nets = crafted_networks()
    po, eo, ed = soup(nets)
    t = abi.map_table(po, eo, ed, 5.0)
    assert np.array_equal(t["map_off"][1:] - t["map_off"][:-1], [len(loop_table(po, eo, ed, r)[0]) for r in range(4)])
    for r in range(4):
        seg, fl = loop_table(po, eo, ed, r)
        got = slice(int(t["map_off"][r]), int(t["map_off"][r + 1]))
        assert np.array_equal(t["map_seg"][got], seg), r
        assert np.array_equal(t["map_flags"][got], fl), r
    a = t["map_seg"][: t["map_off"][1]]
    fa = t["map_flags"][: t["map_off"][1]]
    # road: 4 edges, the lanes add their shared middle line (once, although both lanes have it), and their halves
    # of the road's ends; the pavement's lower edge is the road's top edge (driveable + walkable)
    assert list(fa[:4]) == [1, 1, 3, 1]
    assert (fa == 6).sum() == 4, "the building is walkable and impenetrable, its zero-length edge dropped"
    assert len(a) == len(np.unique(np.sort(a.reshape(-1, 2, 2).view(np.complex128).reshape(-1, 2), 1), axis=0))
    assert t["map_off"][2] - t["map_off"][1] == 0 and t["map_off"][4] - t["map_off"][3] == 0
    b = slice(int(t["map_off"][2]), int(t["map_off"][3]))
    assert np.array_equal(t["map_flags"][b], [3, 3, 3]), "triangle b is in both surfaces, oriented as first seen"


def _cells_of_box(t, r, bx0, by0, bx1, by1):
    ox, oy, cell, m = t["map_grid"][r]
    nx, ny, _ = t["map_dims"][r]
    ix = abi.map_cell_index([bx0 - m, bx1 + m], ox, cell, nx)
    iy = abi.map_cell_index([by0 - m, by1 + m], oy, cell, ny)
    return ix, iy


def grid_candidates(t, r, x, y, radius):
    """The edges the device tests from (x, y): each listed edge in the first visited cell listing it (and the
    number of times an edge would be tested, which must be 1)."""
    ox, oy, cell, m = t["map_grid"][r]
    nx, ny, c0 = (int(v) for v in t["map_dims"][r])
    w = radius + m
    ix0, ix1 = (int(v) for v in abi.map_cell_index([x - w, x + w], ox, cell, nx))
    iy0, iy1 = (int(v) for v in abi.map_cell_index([y - w, y + w], oy, cell, ny))
    row0 = int(t["map_off"][r])
    out = []
    for cy in range(iy0, iy1 + 1):
        for cx in range(ix0, ix1 + 1):
            c = c0 + cy * nx + cx
            for e in t["map_cell_edge"][t["map_cell_off"][c]:t["map_cell_off"][c + 1]]:
                lo = t["map_cell0"][row0 + e]
                if max(int(lo[0]), ix0) == cx and max(int(lo[1]), iy0) == cy:
                    out.append(int(e))
    return out


def brute_d2(seg, x, y):
    dx, dy = seg[:, 2] - seg[:, 0], seg[:, 3] - seg[:, 1]
    wx, wy = x - seg[:, 0], y - seg[:, 1]
    L2 = dx * dx + dy * dy
    with np.errstate(divide="ignore", invalid="ignore"):
        t = np.where(L2 > 0, (wx * dx + wy * dy) / L2, 0.0)
    t = np.clip(t, 0.0, 1.0)
    qx, qy = seg[:, 0] + t * dx, seg[:, 1] + t * dy
    return (qx - x) * (qx - x) + (qy - y) * (qy - y), qx, qy


@pytest.mark.parametrize("cell", [None, 7.0, 60.0, math.inf])
@pytest.mark.parametrize("center", [0.0, 1e5])
def test_grid_is_conservative(cell, center):
    town = synthetic.grid_town(seed=3, half_extent=150.0, center=(center, -center))
    _, po, eo, ed, _ = pack_road_networks([town])
    radius = 20.0
    t = abi.map_table(po, eo, ed, radius, cell=cell)
    seg = t["map_seg"]
    ox, oy, c, m = t["map_grid"][0]
    nx, ny, c0 = (int(v) for v in t["map_dims"][0])
    if cell == math.inf:
        assert nx == ny == 1
    # every cell lists (at least) the edges whose bounding box overlaps it
    bx0, bx1 = np.minimum(seg[:, 0], seg[:, 2]), np.maximum(seg[:, 0], seg[:, 2])
    by0, by1 = np.minimum(seg[:, 1], seg[:, 3]), np.maximum(seg[:, 1], seg[:, 3])
    rng = np.random.default_rng(0)
    for cid in rng.choice(nx * ny, min(nx * ny, 200), replace=False):
        cy, cx = divmod(int(cid), nx)
        if math.isfinite(c):
            lo_x, lo_y = ox + cx * c, oy + cy * c
            hit = (bx0 <= lo_x + c) & (bx1 >= lo_x) & (by0 <= lo_y + c) & (by1 >= lo_y)
        else:
            hit = np.ones(len(seg), bool)
        listed = set(t["map_cell_edge"][t["map_cell_off"][c0 + cid]:t["map_cell_off"][c0 + cid + 1]].tolist())
        assert set(np.nonzero(hit)[0].tolist()) <= listed, cid
    # candidates from random points, points on cell boundaries and far outside the town cover the brute force
    pts = list(rng.uniform(-170, 170, (300, 2)) + [center, -center])
    if math.isfinite(c):
        for k in range(60):
            i, j = rng.integers(0, nx + 1), rng.integers(0, ny + 1)
            pts.append((ox + i * c, oy + j * c))  # exactly on a cell corner
            pts.append((ox + i * c, oy + rng.uniform(0, ny * c)))  # on a vertical cell boundary
            pts.append((ox + i * c + radius, oy + j * c - radius))  # the query square's side on a boundary
    pts += [(center + 1e5, -center), (center - 300.0, -center + 10.0)]
    near = 0
    for x, y in pts:
        d2, _, _ = brute_d2(seg, float(x), float(y))
        want = set(np.nonzero(d2 < radius * radius)[0].tolist())
        got = grid_candidates(t, 0, float(x), float(y), radius)
        assert len(got) == len(set(got)), "an edge is tested once"
        assert want <= set(got), (x, y)
        near += len(want)
    assert near > 0


# ---------------------------------------------------------------------------------------------- the oracle
def numpy_map(scene, st, slots, t, Km, radius):
    """The map block [N, A, 10 Km] (fp32) by brute force over the table (numpy's cos / sin for the frame)."""
    N, A = slots.shape
    M, nm = scene.M, scene.N * scene.M
    out = np.zeros((N, A, 10 * Km), np.float32)
    for n in range(N):
        r = int(scene.rn_of[n])
        for a in range(A):
            s = slots[n, a]
            if s < 0 or not st["present"][n * M + s] or r < 0:
                continue
            i = n * M + s
            x, y, h = st["pose"][0, i], st["pose"][1, i], st["pose"][3, i]
            c, sn = np.cos(h), np.sin(h)
            seg = t["map_seg"][t["map_off"][r]:t["map_off"][r + 1]]
            fl = t["map_flags"][t["map_off"][r]:t["map_off"][r + 1]]
            d2, qx, qy = brute_d2(seg, x, y)
            idx = np.nonzero(d2 < radius * radius)[0]
            idx = idx[np.lexsort((idx, d2[idx]))][:Km]
            for q, e in enumerate(idx):
                p = [(qx[e] - x, qy[e] - y), (seg[e, 0] - x, seg[e, 1] - y), (seg[e, 2] - x, seg[e, 3] - y)]
                row = [v for px, py in p for v in (c * px + sn * py, -sn * px + c * py)]
                row += [float((fl[e] >> k) & 1) for k in range(3)] + [1.0]
                out[n, a, 10 * q:10 * q + 10] = np.array(row, np.float64).astype(np.float32)
    return out


def crafted_network():
    """Driveable square (0,0)-(10,10), edges e0 bottom, e1 right, e2 top, e3 left; a walkable strip on top (its
    lower edge is e2 reversed) adds e4 (10,10)->(10,12), e5 (10,12)->(0,12), e6 (0,12)->(0,10)."""
    return RoadNetwork(roads=[Road("r", PolygonArea([(0, 0), (10, 0), (10, 10), (0, 10)]))],
                       pavements=[Pavement("p", PolygonArea([(0, 10), (10, 10), (10, 12), (0, 12)]))])


# agent positions (heading 0): the expected (edge, d2) selections are exact
CRAFTED = {
    "on_edge": (5.0, 0.0),       # d2 = 0 to e0; e1 / e3 tie at 25 (lower e first)
    "vertex": (0.0, 0.0),        # d2 = 0 to e0 and e3 (shared vertex): e0 first
    "parallel": (5.0, 5.0),      # e0..e3 all at d2 = 25: in edge order
    "outside": (15.0, 5.0),      # e1 at 25, then e4 (d2 = 25 + 25), e0 / e2 (25 + 25) ...
}


def crafted_state(networks=None):
    names = list(CRAFTED)
    N, M = len(names) + 1, 3
    cfg = synthetic.vehicles_config(seed=0, N=N, M=M, T=4, half_extent=1.0)
    scene = synthetic.pack_synthetic(cfg)
    nets = networks or ([crafted_network()] * len(names) + [None])
    scene = dataclasses.replace(scene, **dict(zip(RN_FIELDS, pack_road_networks(nets))))
    pose = np.zeros((6, N * M))
    present = np.ones(N * M, np.uint8)
    for n, name in enumerate(names + ["none"]):
        x, y = CRAFTED.get(name, (5.0, 5.0))
        pose[0, n * M:(n + 1) * M], pose[1, n * M:(n + 1) * M] = x, y
        present[n * M + 2] = 0  # slot 2 absent
    slots = np.tile(np.array([0, 2, -1], np.int32), (N, 1))  # an agent, an absent agent, a padding agent
    return scene, pose, present, slots


def _crafted_oracle(Km, radius, networks=None):
    scene, pose, present, slots = crafted_state(networks)
    eng = MapOracleEngine(scene, abi.default_params())
    eng.reset()
    eng.state["pose"][...] = pose
    eng.state["present"][...] = present
    _, F = eng.env_spec(slots, 1, 0.0, (), map_edges=Km, map_radius=radius)
    obs, am = eng.env_observe()
    return scene, eng, slots, obs, am, F


@pytest.mark.parametrize("Km,radius", [(1, 20.0), (4, 20.0), (32, 20.0), (8, 5.0), (8, 7.5)])
def test_oracle_matches_numpy_crafted(Km, radius):
    scene, eng, slots, obs, am, F = _crafted_oracle(Km, radius)
    assert F == abi.env_n_features(1, 0, False, 0, Km)
    t = eng._map
    want = numpy_map(scene, eng.state, slots, t, Km, radius)
    got = obs[..., F - 10 * Km:]
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert not got[:, 1:].any(), "absent and padding agents get zeros"
    assert not got[-1].any(), "a scenario without a network gets zeros"
    sel = {name: [int(v) for v in got[n, 0, 9::10].nonzero()[0]] for n, name in enumerate(CRAFTED)}
    seg = t["map_seg"]
    first = {name: tuple(got[n, 0, 2:6]) for n, name in enumerate(CRAFTED)}
    assert len(seg) == 7 and list(t["map_flags"]) == [1, 1, 3, 1, 2, 2, 2]
    r2 = radius * radius
    if radius == 5.0:  # d2 == r * r is excluded
        assert sel["parallel"] == [] and len(sel["on_edge"]) == 1 and len(sel["vertex"]) == 2
    if Km == 1 and radius == 20.0:
        assert first["on_edge"] == (-5.0, 0.0, 5.0, 0.0)  # e0 from (5, 0)
        assert first["vertex"] == (0.0, 0.0, 10.0, 0.0)   # e0, not e3
    if Km >= 4 and radius == 20.0:
        # parallel: e0 (0,0)->(10,0), e1, e2, e3 in edge order, at distance 5
        ends = got[2, 0, :40].reshape(4, 10)[:, 2:4]
        assert np.array_equal(ends, [[-5.0, -5.0], [5.0, -5.0], [5.0, 5.0], [-5.0, 5.0]])
        assert np.array_equal(got[0, 0, 10:20][2:4], [5.0, 0.0]), "on_edge: e1 before e3 at equal d2"
    n_within = int((brute_d2(seg, 5.0, 5.0)[0] < r2).sum())
    assert len(sel["parallel"]) == min(Km, n_within)


def test_oracle_prefix_and_lidar_unchanged():
    """The oracle's map block sits between the row without it and the lidar, both unchanged."""
    scene, pose, present, slots = crafted_state()
    eng = MapOracleEngine(scene, abi.default_params())
    eng.reset()
    eng.state["pose"][...] = pose
    eng.state["pose"][3] = np.linspace(-3, 3, pose.shape[1])
    eng.state["present"][...] = present
    eng.env_spec(slots, 2, 0.0, (1.0,), n_rays=8)
    base, am0 = eng.env_observe()
    _, F = eng.env_spec(slots, 2, 0.0, (1.0,), n_rays=8, map_edges=5, map_radius=30.0)
    full, am1 = eng.env_observe()
    F0 = base.shape[-1] - 8
    assert np.array_equal(am0, am1)
    assert np.array_equal(full[..., :F0].view(np.uint32), base[..., :F0].view(np.uint32))
    assert np.array_equal(full[..., -8:].view(np.uint32), base[..., -8:].view(np.uint32))
    want = numpy_map(scene, eng.state, slots, eng._map, 5, 30.0)
    np.testing.assert_allclose(full[..., F0:F0 + 50], want, rtol=2e-6, atol=2e-5)


def test_oracle_several_networks_and_town():
    town = synthetic.grid_town(seed=1, half_extent=60.0)
    nets = [town, crafted_network(), None, town]
    scene = dataclasses.replace(crafted_state()[0], **dict(zip(RN_FIELDS, pack_road_networks(nets + [None]))))
    eng = MapOracleEngine(scene, abi.default_params())
    eng.reset()
    rng = np.random.default_rng(2)
    eng.state["pose"][0] = rng.uniform(-60, 60, scene.N * scene.M)
    eng.state["pose"][1] = rng.uniform(-60, 60, scene.N * scene.M)
    eng.state["pose"][3] = rng.uniform(-np.pi, np.pi, scene.N * scene.M)
    slots = np.tile(np.array([0, 1, 2], np.int32), (scene.N, 1))
    _, F = eng.env_spec(slots, 0, 0.0, (), map_edges=16, map_radius=25.0)
    obs, _ = eng.env_observe()
    want = numpy_map(scene, eng.state, slots, eng._map, 16, 25.0)
    np.testing.assert_allclose(obs[..., 4:], want, rtol=2e-6, atol=2e-5)
    assert np.array_equal(obs[..., 4:][..., 6::10], want[..., 6::10])
    assert obs[0, :, 9::10].sum() > 0 and not obs[2, :, 4:].any()


def test_oracle_argument_checks():
    scene, pose, present, slots = crafted_state()
    eng = MapOracleEngine(scene, abi.default_params())
    eng.reset()
    for field, value in (("map_edges", 33), ("map_edges", -1), ("map_radius", 0.0), ("map_radius", math.nan),
                         ("map_networks", 2)):
        e, _ = eng.env_spec(slots, 1, 0.0, (), map_edges=4, map_radius=10.0)
        setattr(e, field, value)
        with pytest.raises(RuntimeError, match="map_"):
            eng.env_observe()


def test_grid_town_is_deterministic():
    a, b, c = synthetic.grid_town(seed=7), synthetic.grid_town(seed=7), synthetic.grid_town(seed=8)
    pa, pb, pc = (pack_road_networks([x]) for x in (a, b, c))
    for u, v in zip(pa, pb):
        assert np.array_equal(u, v)
    assert pa[3].shape != pc[3].shape or not np.array_equal(pa[3], pc[3])
    assert len(a.roads) and len(a.lanes) == 4 * len(a.roads) and len(a.intersections) and len(a.pavements) \
        and len(a.buildings)
    e = pa[3]
    assert e[:, [0, 2]].min() < -200 and e[:, [0, 2]].max() > 200 and e[:, [1, 3]].min() < -200 \
        and e[:, [1, 3]].max() > 200, "the town covers the 400 m square"
    t = abi.map_table(pa[1], pa[2], pa[3], 50.0)
    assert 1000 < len(t["map_seg"]) < len(e)
