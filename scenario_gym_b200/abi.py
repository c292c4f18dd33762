"""
ctypes mirror of ``include/sg_b200.h`` (the C ABI of the rollout engine).

The structures here are verified against the library at load time with
``sg_sizeof`` so a drifted mirror fails loudly instead of corrupting memory.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from typing import Dict, Optional

ABI_VERSION = 19

# SgKind
KIND_EMPTY, KIND_REPLAY, KIND_AGENT_REPLAY, KIND_VEHICLE, KIND_PEDESTRIAN, KIND_HOST, KIND_PID = range(7)
# SgEntityType
ETYPE_VEHICLE, ETYPE_PEDESTRIAN, ETYPE_MISC = range(3)
# SgTerminal
TERM_MAX_LENGTH, TERM_COLLISION, TERM_EGO_COLLISION, TERM_EGO_OFF_ROAD = 1, 2, 4, 8
# SgFeature
FEAT_COLLISIONS, FEAT_EGO_METRICS, FEAT_RSS, FEAT_COLL_MATRIX, FEAT_NO_GRID, FEAT_SEQUENTIAL = 1, 2, 4, 8, 16, 32
# SgRssRecord
RSS_RECORD_NAMES = {
    0: "safe",
    1: "lateral",
    2: "longitudinal",
    3: "both",
    4: "unsafe_lateral",
    5: "unsafe_longitudinal",
    6: "found",
}
RSS_NONE = 255
SCENE_FLAT_BOXES = 1

_p = C.c_void_p


class SgParams(C.Structure):
    _fields_ = [
        ("timestep", C.c_double),
        ("persist", C.c_int32),
        ("terminal", C.c_int32),
        ("features", C.c_int32),
        ("max_ticks", C.c_int32),
        ("veh_max_steer", C.c_double),
        ("veh_max_accel", C.c_double),
        ("veh_max_speed", C.c_double),
        ("veh_allow_reverse", C.c_int32),
        ("_pad0", C.c_int32),
        ("ped_max_speed", C.c_double),
        ("ped_head_rot_angle", C.c_double),
        ("ped_distance_threshold", C.c_double),
        ("sf_max_speed_factor", C.c_double),
        ("sf_bias_lon", C.c_double),
        ("sf_bias_lat", C.c_double),
        ("sf_sight_weight", C.c_double),
        ("sf_sight_weight_use", C.c_int32),
        ("_pad1", C.c_int32),
        ("sf_sight_angle", C.c_double),
        ("sf_relaxation_time", C.c_double),
        ("sf_ped_repulse_V", C.c_double),
        ("sf_ped_repulse_sigma", C.c_double),
        ("sf_ped_attract_C", C.c_double),
        ("rss_response_time", C.c_double),
        ("rss_min_long_accel", C.c_double),
        ("rss_max_long_accel", C.c_double),
        ("rss_min_safe_clearance", C.c_double),
        ("pid_steer_Kp", C.c_double),
        ("pid_steer_Kd", C.c_double),
        ("pid_accel_Kp", C.c_double),
        ("pid_accel_Kd", C.c_double),
        ("pid_accel_Ki", C.c_double),
        ("sf_boundary_repulse_U", C.c_double),
        ("sf_boundary_repulse_R", C.c_double),
        ("sf_imp_boundary_repulse_U", C.c_double),
        ("sf_imp_boundary_repulse_R", C.c_double),
        ("sf_std_lon", C.c_double),
        ("sf_std_lat", C.c_double),
        ("sf_noise_seed", C.c_uint64),
    ]


class SgScene(C.Structure):
    _fields_ = [
        ("n_scenarios", C.c_int32),
        ("n_slots", C.c_int32),
        ("n_traj_rows", C.c_int64),
        ("n_union_rows", C.c_int64),
        ("n_route_pts", C.c_int64),
        ("kind_mask", C.c_uint32),
        ("scene_flags", C.c_uint32),
        ("kind", _p),
        ("etype", _p),
        ("box", _p),
        ("traj_off", _p),
        ("traj_rows", _p),
        ("union_off", _p),
        ("union_t", _p),
        ("union_x", _p),
        ("t0", _p),
        ("length", _p),
        ("ego_slot", _p),
        ("first_slot", _p),
        ("ped_speed_desired", _p),
        ("route_off", _p),
        ("route_xy", _p),
        ("n_networks", C.c_int32),
        ("_pad1", C.c_int32),
        ("n_rn_polys", C.c_int64),
        ("n_rn_edges", C.c_int64),
        ("rn_of", _p),
        ("rn_poly_off", _p),
        ("rn_edge_off", _p),
        ("rn_edges", _p),
        ("rn_has_area", _p),
        ("veh_limits", _p),
        ("plane_stride", C.c_int64),   # scenario windows (sg_b200.h): 0 = the whole batch
        ("scenario_base", C.c_int32),
        ("_pad2", C.c_int32),
    ]


class SgEvent(C.Structure):
    _fields_ = [
        ("scenario", C.c_int32),
        ("tick", C.c_int32),
        ("slot", C.c_int32),
        ("_pad", C.c_int32),
        ("t", C.c_double),
    ]


class SgState(C.Structure):
    _fields_ = [
        ("pose", _p),
        ("vel", _p),
        ("dist", _p),
        ("present", _p),
        ("t", _p),
        ("prev_t", _p),
        ("tick", _p),
        ("done", _p),
        ("speed", _p),
        ("goal_idx", _p),
        ("force", _p),
        ("cur_own", _p),
        ("cur_union", _p),
        ("ego_avg_speed", _p),
        ("ego_avg_t", _p),
        ("ego_max_speed", _p),
        ("ego_dist", _p),
        ("ego_hits", _p),
        ("coll_mask", _p),
        ("collided", _p),
        ("first_coll_tick", _p),
        ("first_coll_pair", _p),
        ("n_pair_ticks", _p),
        ("events", _p),
        ("event_count", _p),
        ("event_cap", C.c_int32),
        ("trace_cap", C.c_int32),
        ("rss_state", _p),
        ("rss_last", _p),
        ("safe_dist", _p),
        ("safe_ratio", _p),
        ("rss_flags", _p),
        ("trace_pose", _p),
        ("trace_present", _p),
        ("trace_t", _p),
        ("pid_err", _p),
    ]


class SgActionRng(C.Structure):
    _fields_ = [
        ("state_hi", C.c_uint64),
        ("state_lo", C.c_uint64),
        ("inc_hi", C.c_uint64),
        ("inc_lo", C.c_uint64),
        ("offset", C.c_int64 * 2),
        ("tick_stride", C.c_int64),
        ("low", C.c_double * 2),
        ("scale", C.c_double * 2),
    ]


class SgInputs(C.Structure):
    _fields_ = [
        ("actions", _p),
        ("n_action_ticks", C.c_int32),
        ("step_done", C.c_int32),
        ("host_pose", _p),
        ("host_present", _p),
        ("actions_f32", _p),
        ("use_rng", C.c_int32),
        ("rng_tick0", C.c_int32),
        ("rng", SgActionRng),
    ]


class SgHostResults(C.Structure):
    _fields_ = [
        ("ego_avg_speed", _p),
        ("ego_max_speed", _p),
        ("ego_dist", _p),
        ("first_coll_tick", _p),
        ("first_coll_pair", _p),
        ("n_pair_ticks", _p),
        ("rss_flags", _p),
        ("tick", _p),
        ("t", _p),
        ("event_count", _p),
    ]


class SgEnvSpec(C.Structure):
    _fields_ = [
        ("n_agents", C.c_int32),
        ("k_neighbours", C.c_int32),
        ("agent_slot", _p),
        ("radius", C.c_double),
        ("n_lookahead", C.c_int32),
        ("road", C.c_int32),
        ("lookahead", C.c_double * 8),
        ("weights", C.c_double * 5),
        ("snap_dist", _p),
        ("snap_collided", _p),
        ("snap_pair_ticks", _p),
        ("snap_rss", _p),
        ("n_rays", C.c_int32),
        ("_pad0", C.c_int32),
        ("ray_range", C.c_double),
        ("ray_dir", _p),
        ("map_edges", C.c_int32),
        ("map_networks", C.c_int32),
        ("map_radius", C.c_double),
        ("map_off", _p),
        ("map_seg", _p),
        ("map_flags", _p),
        ("map_cell0", _p),
        ("map_grid", _p),
        ("map_dims", _p),
        ("map_cell_off", _p),
        ("map_cell_edge", _p),
    ]


class SgResetInit(C.Structure):
    _fields_ = [
        ("t_start", _p),
        ("start_window", _p),
        ("counter", _p),
        ("perturb", _p),
        ("sigma", C.c_double * 4),
        ("seed", C.c_uint64),
    ]


class SgRasterSpec(C.Structure):
    _fields_ = [
        ("size", C.c_int32),
        ("n_networks", C.c_int32),
        ("resolution", C.c_double),
        ("ahead", C.c_double),
        ("margin", C.c_double),
        ("poly_box", _p),
    ]


# the channels of sg_env_raster, in order
RASTER_CHANNELS = ("driveable", "walkable", "impenetrable", "vehicles", "pedestrians")


def raster_poly_boxes(rn_edge_off, rn_edges, half_diagonal: float):
    """
    ``SgRasterSpec.poly_box`` and ``margin`` of a scene's polygon soups (SgScene.rn_edge_off / rn_edges): [P, 4]
    fp64 min x, min y, max x, max y over each polygon's edges (zeros for a polygon without edges, which toggles
    nothing), and m = 1e-9 * (1 + largest |coordinate| + half_diagonal) (include/sg_b200.h, SgRasterSpec).
    """
    import numpy as np

    off = np.asarray(rn_edge_off, np.int64)
    edges = np.asarray(rn_edges, np.float64).reshape(-1, 4)
    P = len(off) - 1
    box = np.zeros((P, 4), np.float64)
    if len(edges):
        xs, ys = edges[:, 0::2], edges[:, 1::2]
        lo_x, hi_x = xs.min(1), xs.max(1)
        lo_y, hi_y = ys.min(1), ys.max(1)
        full = off[1:] > off[:-1]
        starts = off[:-1][full]
        box[full, 0] = np.minimum.reduceat(lo_x, starts)
        box[full, 1] = np.minimum.reduceat(lo_y, starts)
        box[full, 2] = np.maximum.reduceat(hi_x, starts)
        box[full, 3] = np.maximum.reduceat(hi_y, starts)
    big = float(np.abs(edges).max()) if len(edges) else 0.0
    return box, 1e-9 * (1.0 + big + float(half_diagonal))


def raster_half_diagonal(size: int, resolution: float) -> float:
    """The raster's half-diagonal sqrt(2) * S * h, h = resolution / 2 (the device's value)."""
    return 1.4142135623730951 * (float(size) * (0.5 * float(resolution)))


def start_windows(scene, persist: bool, min_remaining: float):
    """
    [N] fp64, computed on the host from a lowered scene (``PackedScene``): for scenario n the largest w >= 0 with
    t0 + w <= length - min_remaining such that every VEHICLE / PID slot present at t0 stays present over
    [t0, t0 + w], i.e. its last control point is >= t0 + w (static slots, with one row, and every slot under
    ``persist`` stay present anyway).  So a reset at any start in [t0, t0 + w] keeps the vehicles present (the
    promise of SgScene.kind_mask) and leaves at least ``min_remaining`` seconds of the log.
    """
    import numpy as np

    N, M = scene.N, scene.M
    t0 = np.asarray(scene.t0, np.float64)
    w = np.asarray(scene.length, np.float64) - float(min_remaining) - t0
    if not persist:
        kind = np.asarray(scene.kind).reshape(N * M)
        off = np.asarray(scene.traj_off, np.int64)
        rows = np.asarray(scene.traj_rows, np.float64).reshape(-1, 7)
        K = off[1:] - off[:-1]
        ctl = ((kind == KIND_VEHICLE) | (kind == KIND_PID)) & (K > 1)
        idx = np.nonzero(ctl)[0]
        first, last = rows[off[idx], 0], rows[off[idx + 1] - 1, 0]
        n = idx // M
        # present at t0 (within its logged span): bounded by its last control point
        here = (first <= t0[n]) & (t0[n] <= last)
        lim = np.full(N, np.inf)
        np.minimum.at(lim, n[here], last[here] - t0[n[here]])
        w = np.minimum(w, lim)
    return np.maximum(w, 0.0)


# number of reward terms of sg_env_reward: progress, collision, off_road, tracking, rss
ENV_TERMS = ("progress", "collision", "off_road", "tracking", "rss")


def env_n_features(k_neighbours: int, n_lookahead: int, road: bool, n_rays: int = 0, map_edges: int = 0) -> int:
    """Floats per observation row of sg_env_observe (include/sg_b200.h, SgEnvSpec)."""
    return 4 + 3 * n_lookahead + 10 * k_neighbours + (2 if road else 0) + 10 * map_edges + n_rays


# the arrays of the map block's table and grid, in SgEnvSpec order (the field names of SgEnvSpec)
MAP_FIELDS = ("map_off", "map_seg", "map_flags", "map_cell0", "map_grid", "map_dims", "map_cell_off", "map_cell_edge")
# most grid cells one network may have (a finer cell size is widened to stay below it)
MAP_MAX_CELLS = 1 << 20


def map_network_edges(rn_poly_off, rn_edge_off, rn_edges, r: int):
    """The map table of network r (include/sg_b200.h, SgEnvSpec, map block): (seg [E, 4] fp64, flags [E] uint8),
    the edges of its three surfaces walked surface, polygon, edge; zero-length edges dropped; edges with the same
    endpoints (either direction) kept once, at their first occurrence and with its orientation, flag bit k set
    for every surface k they occur in."""
    import numpy as np

    segs, surf = [], []
    for k in range(3):
        p0, p1 = int(rn_poly_off[3 * r + k]), int(rn_poly_off[3 * r + k + 1])
        e0, e1 = int(rn_edge_off[p0]), int(rn_edge_off[p1])
        segs.append(np.asarray(rn_edges[e0:e1], np.float64).reshape(-1, 4))
        surf.append(np.full(e1 - e0, k, np.int64))
    seg, surf = np.concatenate(segs), np.concatenate(surf)
    keep = ~((seg[:, 0] == seg[:, 2]) & (seg[:, 1] == seg[:, 3]))
    seg, surf = seg[keep], surf[keep]
    if len(seg) == 0:
        return np.zeros((0, 4)), np.zeros(0, np.uint8)
    # same endpoints in either direction: compare the endpoints in lexicographic order (-0.0 counts as 0.0)
    key = seg + 0.0
    swap = (key[:, 0] > key[:, 2]) | ((key[:, 0] == key[:, 2]) & (key[:, 1] > key[:, 3]))
    key[swap] = key[swap][:, [2, 3, 0, 1]]
    key = np.ascontiguousarray(key).view(np.dtype((np.void, 32))).reshape(-1)
    _, first, inv = np.unique(key, return_index=True, return_inverse=True)
    flags = np.zeros(len(first), np.uint8)
    np.bitwise_or.at(flags, inv.reshape(-1), (1 << surf).astype(np.uint8))
    order = np.argsort(first, kind="stable")
    return np.ascontiguousarray(seg[first[order]]), flags[order]


def map_cell_index(v, o: float, cell: float, n: int):
    """The grid cell of coordinates v along one axis: floor((v - o) / cell) clamped to [0, n - 1] (int64)."""
    import numpy as np

    return np.clip(np.floor((np.asarray(v, np.float64) - o) / cell), 0, n - 1).astype(np.int64)


def map_table(rn_poly_off, rn_edge_off, rn_edges, radius: float, cell: Optional[float] = None):
    """
    The map block's table and culling grid of every network of a scene (SgScene.rn_* as numpy arrays), as the
    numpy arrays of ``MAP_FIELDS``.  Per network: margin m = 1e-9 * (1 + largest |coordinate| + radius), origin
    the table's bounding box minus m, square cells of side ``cell`` (None: radius / 2, widened where the network
    would need more than ``MAP_MAX_CELLS`` cells; ``math.inf``: a single cell, i.e. brute force), every edge
    listed, in ascending order, in the cells its bounding box widened by m overlaps (include/sg_b200.h).
    """
    import numpy as np

    radius = float(radius)
    if not (math.isfinite(radius) and radius > 0.0):
        raise ValueError(f"map radius must be finite and > 0, got {radius}")
    if cell is not None and not float(cell) > 0.0:
        raise ValueError(f"map grid cell size must be > 0, got {cell}")
    R = (len(rn_poly_off) - 1) // 3
    off, segs, flags, cell0, grid, dims, cell_off, cell_edge = [0], [], [], [], [], [], [np.zeros(1, np.int64)], []
    n_cells = n_listed = 0
    for r in range(R):
        seg, fl = map_network_edges(rn_poly_off, rn_edge_off, rn_edges, r)
        E = len(seg)
        bx0, bx1 = np.minimum(seg[:, 0], seg[:, 2]), np.maximum(seg[:, 0], seg[:, 2])
        by0, by1 = np.minimum(seg[:, 1], seg[:, 3]), np.maximum(seg[:, 1], seg[:, 3])
        big = float(np.abs(seg).max()) if E else 0.0
        m = 1e-9 * (1.0 + big + radius)
        ox, oy = (float(bx0.min()) - m, float(by0.min()) - m) if E else (0.0, 0.0)
        ex, ey = (float(bx1.max()) + m - ox, float(by1.max()) + m - oy) if E else (0.0, 0.0)
        c = 0.5 * radius if cell is None else float(cell)
        if math.isfinite(c):
            c = max(c, math.sqrt(ex * ey / MAP_MAX_CELLS), max(ex, ey) / MAP_MAX_CELLS)
        nx = int(math.floor(ex / c)) + 1 if E else 1
        ny = int(math.floor(ey / c)) + 1 if E else 1
        ix0, ix1 = map_cell_index(bx0 - m, ox, c, nx), map_cell_index(bx1 + m, ox, c, nx)
        iy0, iy1 = map_cell_index(by0 - m, oy, c, ny), map_cell_index(by1 + m, oy, c, ny)
        wx, cnt = ix1 - ix0 + 1, (ix1 - ix0 + 1) * (iy1 - iy0 + 1)
        ed = np.repeat(np.arange(E, dtype=np.int64), cnt)
        local = np.arange(len(ed), dtype=np.int64) - np.repeat(np.cumsum(cnt) - cnt, cnt)
        cid = (iy0[ed] + local // wx[ed]) * nx + ix0[ed] + local % wx[ed]
        order = np.lexsort((ed, cid))
        counts = np.bincount(cid, minlength=nx * ny)
        off.append(off[-1] + E)
        segs.append(seg)
        flags.append(fl)
        cell0.append(np.stack([ix0, iy0], 1).astype(np.int32).reshape(-1, 2))
        grid.append([ox, oy, c, m])
        dims.append([nx, ny, n_cells])
        cell_off.append(n_listed + np.cumsum(counts))
        cell_edge.append(ed[order].astype(np.int32))
        n_cells += nx * ny
        n_listed += len(ed)
    return {
        "map_off": np.array(off, np.int64),
        "map_seg": np.ascontiguousarray(np.concatenate(segs) if segs else np.zeros((0, 4)), np.float64),
        "map_flags": np.concatenate(flags).astype(np.uint8) if flags else np.zeros(0, np.uint8),
        "map_cell0": np.ascontiguousarray(np.concatenate(cell0) if cell0 else np.zeros((0, 2)), np.int32),
        "map_grid": np.array(grid, np.float64).reshape(R, 4),
        "map_dims": np.array(dims, np.int64).reshape(R, 3),
        "map_cell_off": np.concatenate(cell_off).astype(np.int64),
        "map_cell_edge": np.concatenate(cell_edge).astype(np.int32) if cell_edge else np.zeros(0, np.int32),
    }


def lidar_directions(n_rays: int):
    """The [R, 2] fp64 ray directions of SgEnvSpec.ray_dir: (cos, sin)(2 pi k / R), numpy's values."""
    import numpy as np

    ang = 2.0 * np.pi * np.arange(n_rays) / n_rays
    return np.ascontiguousarray(np.stack([np.cos(ang), np.sin(ang)], 1))


# (field, dtype, shape spec) of every SgState array; shape tokens: N, M, NM, W, E, T
STATE_FIELDS = [
    ("pose", "float64", ("6", "NM")),
    ("vel", "float64", ("6", "NM")),
    ("dist", "float64", ("NM",)),
    ("present", "uint8", ("NM",)),
    ("t", "float64", ("N",)),
    ("prev_t", "float64", ("N",)),
    ("tick", "int32", ("N",)),
    ("done", "uint8", ("N",)),
    ("speed", "float64", ("NM",)),
    ("goal_idx", "int32", ("NM",)),
    ("force", "float64", ("2", "NM")),
    ("cur_own", "int32", ("NM",)),
    ("cur_union", "int32", ("N",)),
    ("ego_avg_speed", "float64", ("N",)),
    ("ego_avg_t", "float64", ("N",)),
    ("ego_max_speed", "float64", ("N",)),
    ("ego_dist", "float64", ("N",)),
    ("ego_hits", "uint32", ("N", "W")),
    ("coll_mask", "uint32", ("N", "M", "W")),
    ("collided", "uint8", ("NM",)),
    ("first_coll_tick", "int32", ("N",)),
    ("first_coll_pair", "int32", ("N", "2")),
    ("n_pair_ticks", "int64", ("N",)),
    ("events", "event", ("E",)),
    ("event_count", "int32", ("1",)),
    ("rss_state", "uint8", ("NM",)),
    ("rss_last", "uint8", ("NM",)),
    ("safe_dist", "float64", ("2", "NM")),
    ("safe_ratio", "float64", ("2", "NM")),
    ("rss_flags", "uint8", ("N",)),
    ("trace_pose", "float64", ("T", "6", "NM")),
    ("trace_present", "uint8", ("T", "NM")),
    ("trace_t", "float64", ("T", "N")),
    ("pid_err", "float64", ("3", "NM")),
]

SCENE_FIELDS = [
    "kind", "etype", "box", "traj_off", "traj_rows", "union_off", "union_t", "union_x",
    "t0", "length", "ego_slot", "first_slot", "ped_speed_desired", "route_off", "route_xy",
    "rn_of", "rn_poly_off", "rn_edge_off", "rn_edges", "rn_has_area", "veh_limits",
]


def default_params() -> SgParams:
    """Defaults of the reference constructors (same values as sg_default_params)."""
    p = SgParams()
    p.timestep = 1.0 / 30.0
    p.persist = 0
    p.terminal = TERM_MAX_LENGTH
    p.features = FEAT_COLLISIONS | FEAT_EGO_METRICS
    p.max_ticks = 1 << 20
    p.veh_max_steer = 0.7
    p.veh_max_accel = 5.0
    p.veh_max_speed = math.nan
    p.veh_allow_reverse = 0
    p.ped_max_speed = 5.0
    p.ped_head_rot_angle = 0.0
    p.ped_distance_threshold = 1.0
    p.sf_max_speed_factor = 1.3
    p.sf_bias_lon = 0.0
    p.sf_bias_lat = 0.0
    p.sf_sight_weight = 0.5
    p.sf_sight_weight_use = 1
    p.sf_sight_angle = 200.0
    p.sf_relaxation_time = 1.5
    p.sf_ped_repulse_V = 1.0
    p.sf_ped_repulse_sigma = 1.0
    p.sf_ped_attract_C = 0.0
    p.rss_response_time = 0.6
    p.rss_min_long_accel = 1.2 * 9.81
    p.rss_max_long_accel = 1.2 * 9.81
    p.rss_min_safe_clearance = 0.1
    p.pid_steer_Kp, p.pid_steer_Kd = 0.03054, 1.5709
    p.pid_accel_Kp, p.pid_accel_Kd, p.pid_accel_Ki = 0.3753, 1.8970, 0.0204
    p.sf_boundary_repulse_U, p.sf_boundary_repulse_R = 10.0, 0.2
    p.sf_imp_boundary_repulse_U, p.sf_imp_boundary_repulse_R = 2.0, 0.1
    return p


EXPORTS = [
    "abi_version", "sizeof", "last_error", "default_params", "reset", "rollout",
    "test_box_pairs", "future_collisions", "fill_random_actions", "rollout_host", "host_h2d_bytes",
    "host_d2h_bytes", "reset_scenarios", "env_observe", "env_reward", "fork_state", "plan_sample", "plan_update",
    "reset_scenarios_init", "env_raster",
]


def bind(lib: C.CDLL, prefix: str) -> Dict[str, object]:
    """Attach prototypes for the entry points of include/sg_b200.h."""
    f = {}

    def get(name, restype, argtypes, required=True):
        try:
            fn = getattr(lib, prefix + name)
        except AttributeError:
            if required:
                raise
            return None
        fn.restype = restype
        fn.argtypes = argtypes
        f[name] = fn
        return fn

    get("abi_version", C.c_int, [])
    get("sizeof", C.c_int64, [C.c_int])
    get("last_error", C.c_char_p, [])
    get("default_params", None, [C.POINTER(SgParams)])
    get("reset", C.c_int, [C.POINTER(SgScene), C.POINTER(SgParams), C.POINTER(SgState), C.c_int, _p])
    # the closed-loop environment's entry points: the product exports them (tests/test_abi.py checks every
    # declared symbol); of the CPU oracle's libraries only libsg_env_oracle.so does (oracle/env_runner.py)
    get("reset_scenarios", C.c_int,
        [C.POINTER(SgScene), C.POINTER(SgParams), C.POINTER(SgState), _p, C.c_int, _p], required=False)
    get("env_observe", C.c_int,
        [C.POINTER(SgScene), C.POINTER(SgParams), C.POINTER(SgState), C.POINTER(SgEnvSpec), _p, _p, _p,
         C.c_int, _p], required=False)
    get("env_reward", C.c_int,
        [C.POINTER(SgScene), C.POINTER(SgParams), C.POINTER(SgState), C.POINTER(SgEnvSpec), _p, _p, _p, _p,
         C.c_int, _p], required=False)
    # sg_fork_state: the product exports it; the CPU oracle has no counterpart (a host fork is a numpy copy)
    get("fork_state", C.c_int,
        [C.POINTER(SgScene), C.POINTER(SgState), C.POINTER(C.POINTER(SgState)), C.c_int, C.POINTER(SgEnvSpec),
         C.POINTER(C.POINTER(SgEnvSpec)), C.c_int, _p], required=False)
    # sg_plan_sample / sg_plan_update: the product exports them; the CPU oracle has none (tests restate them)
    get("plan_sample", C.c_int,
        [C.POINTER(SgEnvSpec), C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_int, C.POINTER(C.c_double), _p,
         _p, _p, C.c_int, C.c_int, _p], required=False)
    get("plan_update", C.c_int,
        [C.POINTER(SgEnvSpec), C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, _p, _p, C.c_int, _p, _p, C.c_int,
         _p, _p, _p, C.c_int, _p], required=False)
    # sg_reset_scenarios_init: the product exports it; its oracle is test code (tests/reset_oracle.c)
    get("reset_scenarios_init", C.c_int,
        [C.POINTER(SgScene), C.POINTER(SgParams), C.POINTER(SgState), _p, C.POINTER(SgResetInit), C.c_int, _p],
        required=False)
    # sg_env_raster: the product exports it; its oracle is test code (tests/raster_oracle.c)
    get("env_raster", C.c_int,
        [C.POINTER(SgScene), C.POINTER(SgParams), C.POINTER(SgState), C.POINTER(SgEnvSpec), C.POINTER(SgRasterSpec),
         _p, _p, C.c_int, _p], required=False)
    get("rollout", C.c_int,
        [C.POINTER(SgScene), C.POINTER(SgParams), C.POINTER(SgState), C.POINTER(SgInputs),
         C.c_int, C.c_int, _p])
    get("test_box_pairs", C.c_int, [_p, _p, _p, _p, _p, C.c_int64, C.c_int, _p])
    get("future_collisions", C.c_int,
        [C.POINTER(SgScene), _p, _p, C.c_double, C.c_int, _p, C.c_int, _p])
    get("fill_random_actions", C.c_int,
        [C.POINTER(SgActionRng), C.c_int, C.c_int, C.c_int64, _p, C.c_int, _p])
    get("entities_in_radius", C.c_int,
        [C.POINTER(SgState), C.c_int, C.c_int, _p, _p, _p, _p, C.c_int, _p])
    get("build_union_x", C.c_int, [C.POINTER(SgScene), C.c_int, _p])
    get("test_trajectory", C.c_int,
        [_p, C.c_int64, _p, C.c_int64, C.c_int, _p, _p, _p, C.c_int, _p])
    get("measure_fp64_peak", C.c_int, [C.POINTER(C.c_double), C.c_int, _p], required=False)
    get("rollout_host", C.c_int,
        [C.POINTER(SgScene), C.POINTER(SgScene), C.POINTER(SgParams), C.POINTER(SgState),
         C.POINTER(SgInputs), C.POINTER(SgInputs), C.POINTER(SgHostResults), C.c_int, C.c_int, _p],
        required=False)
    get("host_h2d_bytes", C.c_int64, [C.POINTER(SgScene), C.POINTER(SgInputs), C.c_int], required=False)
    get("host_d2h_bytes", C.c_int64, [C.POINTER(SgScene)], required=False)

    if f["abi_version"]() != ABI_VERSION:
        raise RuntimeError(f"ABI version mismatch: lib {f['abi_version']()} != {ABI_VERSION}")
    structs = [SgParams, SgScene, SgState, SgInputs, SgEvent, SgActionRng, SgHostResults]
    if "env_observe" in f:  # (a library that takes SgEnvSpec knows its size)
        structs.append(SgEnvSpec)
        if "reset_scenarios_init" in f:
            structs.append(SgResetInit)
            if "env_raster" in f:
                structs.append(SgRasterSpec)
    for which, st in enumerate(structs):
        if f["sizeof"](which) != C.sizeof(st):
            raise RuntimeError(
                f"ABI struct {st.__name__}: lib {f['sizeof'](which)} B != ctypes {C.sizeof(st)} B"
            )
    return f


_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PRODUCT_LIB = os.environ.get(
    "SG_B200_LIB", os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc", "libsg_b200.so"))

_product: Optional[Dict[str, object]] = None


def load_product() -> Dict[str, object]:
    """Load the CUDA engine.  There is no CPU fallback: a missing library is fatal."""
    global _product
    if _product is None:
        if not os.path.exists(PRODUCT_LIB):
            raise RuntimeError(
                f"{PRODUCT_LIB} not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(the engine has no CPU fallback)"
            )
        _product = bind(C.CDLL(PRODUCT_LIB), "sg_")
    return _product
