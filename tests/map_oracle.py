"""
TEST INFRASTRUCTURE ONLY -- ``MapOracleEngine``: ``LidarOracleEngine`` whose ``env_observe`` builds the map block of
include/sg_b200.h (SgEnvSpec) by brute force from its plain-C restatement, ``tests/map_oracle.c``, between the road
block and the lidar.  The library is compiled on first use into a temporary directory (removed at exit), so
nothing is written into the tree.
"""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile
from typing import Dict, Optional

import numpy as np

from oracle.env_runner import _CFLAGS
from oracle.runner import _ptr
from scenario_gym_b200 import abi

from lidar_oracle import LidarOracleEngine

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(os.path.dirname(_HERE), "oracle")
_lib: Optional[Dict[str, object]] = None


def load_map_oracle() -> Dict[str, object]:
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="sg_map_oracle_")
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, "libmap_oracle.so")
        cc = os.environ.get("CC", "gcc")
        subprocess.check_call([cc] + _CFLAGS + ["-shared", "-I", _ORACLE, "-I", _HERE, "-o", out,
                               os.path.join(_HERE, "map_oracle.c"), "-lm"])
        cdll = C.CDLL(out)
        f = abi.bind(cdll, "sgo_")
        fn = cdll.sgo_env_observe_map
        fn.restype = C.c_int
        fn.argtypes = [C.POINTER(abi.SgScene), C.POINTER(abi.SgParams), C.POINTER(abi.SgState),
                       C.POINTER(abi.SgEnvSpec), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        f["env_observe_map"] = fn
        _lib = f
    return _lib


class MapOracleEngine(LidarOracleEngine):
    """``LidarOracleEngine`` with the map block: ``env_spec(..., map_edges, map_radius, table)`` and an
    ``env_observe`` whose rows have ``abi.env_n_features(K, L, road, n_rays, map_edges)`` floats."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.lib = load_map_oracle()

    def env_spec(self, agent_slot: np.ndarray, k_neighbours: int = 8, radius: float = 0.0, lookahead=(),
                 road: bool = False, weights=(0.0,) * 5, n_rays: int = 0, ray_range: float = 50.0,
                 ray_dir: Optional[np.ndarray] = None, map_edges: int = 0, map_radius: float = 50.0,
                 table: Optional[Dict[str, np.ndarray]] = None):
        """As ``LidarOracleEngine.env_spec``; ``map_edges`` > 0 adds the map block over ``table`` (None:
        ``abi.map_table`` of the scene).  Returns (spec, F)."""
        e, F = super().env_spec(agent_slot, k_neighbours, radius, lookahead, road, weights, n_rays, ray_range, ray_dir)
        e.map_edges, e.map_radius = int(map_edges), float(map_radius)
        e.map_networks = self.scene.n_networks
        if map_edges > 0 and self.scene.n_networks > 0:
            sc = self.scene
            t = abi.map_table(sc.rn_poly_off, sc.rn_edge_off, sc.rn_edges, map_radius) if table is None else table
            self._map = {k: np.ascontiguousarray(t[k]) for k in abi.MAP_FIELDS}
            for k, a in self._map.items():
                setattr(e, k, a.ctypes.data if a.size else 0)
        return e, F + 10 * int(map_edges)

    def env_observe(self, mask: Optional[np.ndarray] = None):
        """(obs [N, A, F] fp32, agent_mask [N, A]) of the spec made by env_spec (rows of masked-out scenarios: 0)."""
        e = self._env_spec
        N, A = self.scene.N, e.n_agents
        F = abi.env_n_features(e.k_neighbours, e.n_lookahead, bool(e.road), e.n_rays, e.map_edges)
        obs, am = np.zeros((N, A, F), np.float32), np.zeros((N, A), np.uint8)
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        rc = self.lib["env_observe_map"](C.byref(self._sc), C.byref(self.params), C.byref(self._st), C.byref(e),
                                         _ptr(m), obs.ctypes.data, am.ctypes.data, 0, None)
        if rc:
            raise RuntimeError(self.lib["last_error"]().decode())
        return obs, am
