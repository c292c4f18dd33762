"""
Synthetic scenario generators for the configurations named in BASELINE.json
(SURVEY.md section 8d): C3 random-action vehicles, C4 social-force crowds,
C5 dense highway with RSS.  Everything is drawn from ``numpy.random.default_rng``
so the reference (golden generation), the CPU oracle and the GPU engine consume
bit-identical inputs.  Scenes are packed vectorised (no per-entity Python objects)
so N = 100k x M = 64 packs in seconds.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import numpy as np

from . import abi
from .action_rng import ActionRng
from .packing import PackedScene

# tests/input_files/Catalogs/Scenario_Gym/VehicleCatalogs/ScenarioGymVehicleCatalog.xosc:8-9 (car1)
CAR1_BOX = (2.0, 4.2, 1.37, 0.0)  # width, length, center_x, center_y
# .../PedestrianCatalogs/ScenarioGymPedestrianCatalog.xosc:7-8 (pedestrian1)
PED1_BOX = (0.69, 0.7, 0.0, 0.0)


@dataclass
class SyntheticConfig:
    """Plain arrays describing N scenarios x M entities."""

    name: str
    N: int
    M: int
    T: int
    dt: float
    x0: np.ndarray  # (N, M)
    y0: np.ndarray
    h0: np.ndarray
    v0: np.ndarray
    box: np.ndarray  # (4,) or (N, M, 4)
    kind: np.ndarray  # (N, M) SgKind
    etype: np.ndarray  # (N, M)
    actions: Optional[np.ndarray] = None  # (T, 2, N*M) accel, steer
    speed_desired: Optional[np.ndarray] = None  # (N, M)
    goal: Optional[np.ndarray] = None  # (N, M, 2) pedestrians' route end point
    # the action table as a description of its place in the numpy stream (device-side action source);
    # always set for the random-action configs, `actions` only when the table was materialised
    action_rng: Optional[ActionRng] = None

    @property
    def t_end(self) -> float:
        # scenario.length chosen so that exactly T ticks run: done when t + dt > length
        return (self.T + 0.5) * self.dt


def two_knot_rows(cfg: SyntheticConfig) -> np.ndarray:
    """Each entity's trajectory: straight line at speed v0 along h0, knots at 0 and t_end."""
    N, M = cfg.N, cfg.M
    rows = np.zeros((N * M, 2, 7))
    te = cfg.t_end
    x0, y0, h0, v0 = (a.reshape(-1) for a in (cfg.x0, cfg.y0, cfg.h0, cfg.v0))
    rows[:, 0, 1], rows[:, 0, 2], rows[:, 0, 4] = x0, y0, h0
    rows[:, 1, 0] = te
    rows[:, 1, 1] = x0 + v0 * np.cos(h0) * te
    rows[:, 1, 2] = y0 + v0 * np.sin(h0) * te
    rows[:, 1, 4] = h0
    return rows


def pack_synthetic(cfg: SyntheticConfig, road_network=None) -> PackedScene:
    """Pack a synthetic configuration; `road_network` (optional) is shared by all its scenarios."""
    from .packing import pack_road_networks

    N, M = cfg.N, cfg.M
    NM = N * M
    rows = two_knot_rows(cfg).reshape(NM * 2, 7)
    box = np.empty((4, NM))
    if cfg.box.ndim == 1:
        box[:] = cfg.box[:, None]
    else:
        box[:] = cfg.box.reshape(NM, 4).T
    if cfg.goal is not None:
        route = np.stack(
            [np.stack([cfg.x0, cfg.y0], -1).reshape(NM, 2), cfg.goal.reshape(NM, 2)], axis=1
        ).reshape(NM * 2, 2)
        route_off = np.arange(NM + 1, dtype=np.int64) * 2
        is_ped = cfg.kind.reshape(-1) == abi.KIND_PEDESTRIAN
        if not is_ped.all():  # non-pedestrians have no route
            cnt = np.where(is_ped, 2, 0)
            route_off = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int64)
            route = route.reshape(NM, 2, 2)[is_ped].reshape(-1, 2)
    else:
        route = np.zeros((0, 2))
        route_off = np.zeros(NM + 1, np.int64)
    if (cfg.kind == abi.KIND_REPLAY).any():
        raise ValueError("synthetic fast path has no batch-replay entities")
    return PackedScene(
        N=N,
        M=M,
        kind=np.ascontiguousarray(cfg.kind.reshape(-1), np.uint8),
        etype=np.ascontiguousarray(cfg.etype.reshape(-1), np.uint8),
        box=box,
        traj_off=np.arange(NM + 1, dtype=np.int64) * 2,
        traj_rows=rows,
        union_off=np.zeros(N + 1, np.int64),
        union_t=np.zeros(0),
        union_x=np.zeros((0, 6, M)),
        t0=np.zeros(N),
        length=np.full(N, cfg.t_end),
        ego_slot=np.zeros(N, np.int32),
        first_slot=np.zeros(N, np.int32),
        ped_speed_desired=(
            np.ascontiguousarray(cfg.speed_desired.reshape(-1))
            if cfg.speed_desired is not None
            else np.zeros(NM)
        ),
        route_off=route_off,
        route_xy=np.ascontiguousarray(route),
        n_entities=np.full(N, M, np.int32),
        **(dict(zip(("rn_of", "rn_poly_off", "rn_edge_off", "rn_edges", "rn_has_area"),
                    pack_road_networks([road_network] * N))) if road_network is not None else {}),
    )


def _uniform_into(rng, out: np.ndarray, low: float, high: float) -> None:
    """Same stream and bits as rng.uniform(low, high, out.shape), written into `out`."""
    rng.random(out=out)
    out *= high - low
    out += low


def vehicles_config(seed: int, N: int, M: int = 64, T: int = 256, dt: float = 0.1,
                    half_extent: float = 200.0, name: str = "C3",
                    actions_out: Optional[np.ndarray] = None, materialise: bool = True) -> SyntheticConfig:
    """
    C3: M VehicleController agents per scenario with random accel/steer actions.
    x,y ~ U(-half_extent, half_extent), h ~ U(-pi, pi), v0 ~ U(0, 15),
    accel ~ U(-6, 6) (exercises the +-5 clip), steer ~ U(-1, 1) (+-0.7 clip).
    The (T, 2, N*M) action table follows the initial conditions in the generator's stream, plane by
    plane (all accel rows, then all steer rows); ``materialise=False`` only describes it
    (``action_rng``) for the device-side action source.
    """
    rng = np.random.default_rng(seed)
    x0 = rng.uniform(-half_extent, half_extent, (N, M))
    y0 = rng.uniform(-half_extent, half_extent, (N, M))
    h0 = rng.uniform(-np.pi, np.pi, (N, M))
    v0 = rng.uniform(0.0, 15.0, (N, M))
    planes = ((-6.0, 6.0), (-1.0, 1.0))
    arng = ActionRng.from_generator(rng, offset=(0, T * N * M), tick_stride=N * M,
                                    low=[lo for lo, _ in planes], high=[hi for _, hi in planes],
                                    n_ticks=T, nm=N * M)
    actions = None
    if materialise or actions_out is not None:
        actions = np.empty((T, 2, N * M)) if actions_out is None else actions_out
        assert actions.shape == (T, 2, N * M) and actions.dtype == np.float64
        # drawn in place: the table can be a view of pinned host memory
        tmp = np.empty(N * M)
        for c, (lo, hi) in enumerate(planes):
            for k in range(T):
                _uniform_into(rng, tmp, lo, hi)
                actions[k, c] = tmp
    return SyntheticConfig(
        name=name, N=N, M=M, T=T, dt=dt, x0=x0, y0=y0, h0=h0, v0=v0,
        box=np.array(CAR1_BOX), kind=np.full((N, M), abi.KIND_VEHICLE, np.uint8),
        etype=np.full((N, M), abi.ETYPE_VEHICLE, np.uint8), actions=actions, action_rng=arng,
    )


def highway_config(seed: int, N: int, M: int = 256, T: int = 256, dt: float = 0.1,
                   lanes: int = 4, name: str = "C5", materialise: bool = True) -> SyntheticConfig:
    """
    C5: `lanes` lanes x (M / lanes) vehicles, lane width 3.7 m, headway U(8, 40) m,
    heading ~ 0 +- 0.02, v0 ~ U(20, 35); small random actions.  Ego = slot 0.
    """
    rng = np.random.default_rng(seed)
    per = M // lanes
    assert per * lanes == M
    headway = rng.uniform(8.0, 40.0, (N, lanes, per))
    x0 = np.cumsum(headway, axis=2).reshape(N, M)
    y0 = np.repeat(np.arange(lanes) * 3.7, per)[None, :] + rng.uniform(-0.3, 0.3, (N, M))
    h0 = rng.uniform(-0.02, 0.02, (N, M))
    v0 = rng.uniform(20.0, 35.0, (N, M))
    # put the ego (slot 0) in the middle of the pack so it has traffic on all sides
    mid = per // 2
    for a in (x0, y0, h0, v0):
        a[:, [0, mid]] = a[:, [mid, 0]]
    arng = ActionRng.from_generator(rng, offset=(0, T * N * M), tick_stride=N * M, low=(-2.0, -0.02),
                                    high=(2.0, 0.02), n_ticks=T, nm=N * M)
    actions = None
    if materialise:
        actions = np.empty((T, 2, N * M))
        actions[:, 0] = rng.uniform(-2.0, 2.0, (T, N * M))
        actions[:, 1] = rng.uniform(-0.02, 0.02, (T, N * M))
    return SyntheticConfig(
        name=name, N=N, M=M, T=T, dt=dt, x0=x0, y0=y0, h0=h0, v0=v0,
        box=np.array(CAR1_BOX), kind=np.full((N, M), abi.KIND_VEHICLE, np.uint8),
        etype=np.full((N, M), abi.ETYPE_VEHICLE, np.uint8), actions=actions, action_rng=arng,
    )


def crowd_config(seed: int, N: int, M: int = 1024, T: int = 128, dt: float = 1.0 / 15.0,
                 side: float = 40.0, name: str = "C4") -> SyntheticConfig:
    """
    C4: slot 0 is an ego vehicle replaying a straight trajectory outside the square;
    slots 1.. are social-force pedestrians starting uniformly in a side x side square
    with a 2-point route to a uniformly drawn goal; speed_desired ~ U(0.5, 1.5) * 1.4.
    """
    rng = np.random.default_rng(seed)
    x0 = rng.uniform(0.0, side, (N, M))
    y0 = rng.uniform(0.0, side, (N, M))
    goal = rng.uniform(0.0, side, (N, M, 2))
    d = goal - np.stack([x0, y0], -1)
    # initial heading / speed deliberately differ from the goal direction / desired speed:
    # otherwise the goal force cancels to rounding noise and the heading atan2(F) of a
    # neighbour-free pedestrian is ill-conditioned (no parity statement is possible)
    h0 = np.arctan2(d[..., 1], d[..., 0]) + rng.uniform(-0.5, 0.5, (N, M))
    speed_desired = rng.uniform(0.5, 1.5, (N, M)) * 1.4
    v0 = speed_desired * rng.uniform(0.3, 0.9, (N, M))
    kind = np.full((N, M), abi.KIND_PEDESTRIAN, np.uint8)
    etype = np.full((N, M), abi.ETYPE_PEDESTRIAN, np.uint8)
    box = np.empty((N, M, 4))
    box[:] = PED1_BOX
    # ego vehicle driving along y = -10
    kind[:, 0] = abi.KIND_AGENT_REPLAY
    etype[:, 0] = abi.ETYPE_VEHICLE
    box[:, 0] = CAR1_BOX
    x0[:, 0], y0[:, 0], h0[:, 0], v0[:, 0] = 0.0, -10.0, 0.0, 5.0
    return SyntheticConfig(
        name=name, N=N, M=M, T=T, dt=dt, x0=x0, y0=y0, h0=h0, v0=v0, box=box, kind=kind,
        etype=etype, speed_desired=speed_desired, goal=goal,
    )


def grid_town(seed: int, half_extent: float = 220.0, center=(0.0, 0.0), spacing: float = 80.0, lanes: int = 2,
              lane_width: float = 3.5, pavement: float = 3.0, buildings: float = 0.8):
    """
    A seeded synthetic town (``RoadNetwork``) covering the square ``center +- half_extent``: a grid of roads
    ``spacing`` metres apart, rotated by an angle and shifted by an offset drawn from ``seed``.  Every road
    segment between two intersections is a ``Road`` split into ``2 * lanes`` ``Lane`` strips (which share their
    edges with each other and with the road); every crossing is an ``Intersection`` square; both sides of a road
    segment carry a ``Pavement`` strip; every block holds up to four ``Building`` lots (each present with
    probability ``buildings``) with jittered footprints.  The same seed gives the same network, float for float.
    """
    from .road_network import Building, Intersection, Lane, PolygonArea, Pavement, Road, RoadNetwork

    rng = np.random.default_rng(seed)
    theta = rng.uniform(0.0, 0.5 * np.pi)
    shift = rng.uniform(-0.5 * spacing, 0.5 * spacing, 2)
    c, s = np.cos(theta), np.sin(theta)
    cx0, cy0 = float(center[0]), float(center[1])

    def world(pts):  # local grid coordinates -> world (the same local point always gives the same floats)
        return [(cx0 + c * (u + shift[0]) - s * (v + shift[1]), cy0 + s * (u + shift[0]) + c * (v + shift[1]))
                for u, v in pts]

    def rect(u0, v0, u1, v1):
        return PolygonArea(world([(u0, v0), (u1, v0), (u1, v1), (u0, v1)]))

    hw = lanes * lane_width  # half width of a road
    n = int(np.ceil((half_extent * np.sqrt(2.0) + spacing) / spacing))
    lines = [k * spacing for k in range(-n, n + 1)]
    roads, inters, paves, blds = [], [], [], []
    for i, a in enumerate(lines):
        for j, b in enumerate(lines):
            inters.append(Intersection(f"x{i}_{j}", rect(a - hw, b - hw, a + hw, b + hw)))
            if i + 1 < len(lines):  # along u from this crossing to the next, and along v (transposed)
                a1 = lines[i + 1]
                for axis in (0, 1):
                    def box(p0, q0, p1, q1):
                        return rect(p0, q0, p1, q1) if axis == 0 else rect(q0, p0, q1, p1)
                    u0, u1 = a + hw, a1 - hw
                    lane_list = [Lane(f"l{axis}_{i}_{j}_{k}", box(u0, b - hw + k * lane_width, u1,
                                                                  b - hw + (k + 1) * lane_width))
                                 for k in range(2 * lanes)]
                    roads.append(Road(f"r{axis}_{i}_{j}", box(u0, b - hw, u1, b + hw), lanes=lane_list))
                    paves.append(Pavement(f"p{axis}_{i}_{j}_0", box(u0, b - hw - pavement, u1, b - hw)))
                    paves.append(Pavement(f"p{axis}_{i}_{j}_1", box(u0, b + hw, u1, b + hw + pavement)))
            if i + 1 < len(lines) and j + 1 < len(lines):  # the block between four roads: 2 x 2 lots
                u0, v0 = a + hw + pavement, b + hw + pavement
                side = 0.5 * (spacing - 2.0 * (hw + pavement))
                for lu in range(2):
                    for lv in range(2):
                        keep = rng.random() < buildings
                        inset = rng.uniform(1.0, 4.0, 4)
                        jitter = rng.uniform(-1.0, 1.0, (4, 2))
                        if not keep:
                            continue
                        p0, q0 = u0 + lu * side, v0 + lv * side
                        corners = [(p0 + inset[0], q0 + inset[1]), (p0 + side - inset[2], q0 + inset[1]),
                                   (p0 + side - inset[2], q0 + side - inset[3]), (p0 + inset[0], q0 + side - inset[3])]
                        pts = [(u + du, v + dv) for (u, v), (du, dv) in zip(corners, jitter)]
                        blds.append(Building(f"b{i}_{j}_{lu}{lv}", PolygonArea(world(pts))))
    # keep the geometries that reach into the covered square (with a road's width of slack)
    lim = half_extent + spacing

    def near(g):
        ext = g.boundary.exterior
        return (np.abs(ext[:, 0] - cx0) <= lim).any() and (np.abs(ext[:, 1] - cy0) <= lim).any()

    keep_roads = [r for r in roads if near(r)]
    return RoadNetwork(name=f"grid_town_{seed}", roads=keep_roads, intersections=[g for g in inters if near(g)],
                       pavements=[g for g in paves if near(g)], buildings=[g for g in blds if near(g)])
