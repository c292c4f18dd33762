"""
TEST INFRASTRUCTURE ONLY -- ``LidarOracleEngine``: ``OracleEnvEngine`` whose ``env_observe`` appends the lidar
block of include/sg_b200.h (SgEnvSpec) from its plain-C restatement, ``tests/lidar_oracle.c``.  The library is
compiled on first use into a temporary directory (removed at exit), so nothing is written into the tree.
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

from oracle.env_runner import _CFLAGS, OracleEnvEngine
from oracle.runner import _ptr
from scenario_gym_b200 import abi

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(os.path.dirname(_HERE), "oracle")
_lib: Optional[Dict[str, object]] = None


def load_lidar_oracle() -> Dict[str, object]:
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="sg_lidar_oracle_")
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, "liblidar_oracle.so")
        cc = os.environ.get("CC", "gcc")
        subprocess.check_call([cc] + _CFLAGS + ["-shared", "-I", _ORACLE, "-o", out,
                               os.path.join(_HERE, "lidar_oracle.c"), "-lm"])
        cdll = C.CDLL(out)
        f = abi.bind(cdll, "sgo_")
        fn = cdll.sgo_env_observe_lidar
        fn.restype = C.c_int
        fn.argtypes = [C.POINTER(abi.SgScene), C.POINTER(abi.SgParams), C.POINTER(abi.SgState),
                       C.POINTER(abi.SgEnvSpec), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        f["env_observe_lidar"] = fn
        _lib = f
    return _lib


class LidarOracleEngine(OracleEnvEngine):
    """``OracleEnvEngine`` with the lidar block: ``env_spec(..., n_rays, ray_range, ray_dir)`` and an
    ``env_observe`` whose rows have ``abi.env_n_features(K, L, road, n_rays)`` floats."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.lib = load_lidar_oracle()

    def env_spec(self, agent_slot: np.ndarray, k_neighbours: int = 8, radius: float = 0.0, lookahead=(),
                 road: bool = False, weights=(0.0,) * 5, n_rays: int = 0, ray_range: float = 50.0,
                 ray_dir: Optional[np.ndarray] = None):
        """As ``OracleEnvEngine.env_spec``; ``n_rays`` > 0 adds the lidar with the [R, 2] directions ``ray_dir``
        (None: numpy's cos / sin of 2 pi k / R).  Returns (spec, F)."""
        e, F = super().env_spec(agent_slot, k_neighbours, radius, lookahead, road, weights)
        e.n_rays, e.ray_range = int(n_rays), float(ray_range)
        if n_rays > 0:
            d = abi.lidar_directions(int(n_rays)) if ray_dir is None else np.ascontiguousarray(ray_dir, np.float64)
            assert d.shape == (n_rays, 2), d.shape
            self._ray_dir = d
            e.ray_dir = d.ctypes.data
        return e, F + int(n_rays)

    def env_observe(self, mask: Optional[np.ndarray] = None):
        """(obs [N, A, F] fp32, agent_mask [N, A]) of the spec made by env_spec (rows of masked-out scenarios: 0)."""
        e = self._env_spec
        N, A = self.scene.N, e.n_agents
        F = abi.env_n_features(e.k_neighbours, e.n_lookahead, bool(e.road), e.n_rays)
        obs, am = np.zeros((N, A, F), np.float32), np.zeros((N, A), np.uint8)
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        rc = self.lib["env_observe_lidar"](C.byref(self._sc), C.byref(self.params), C.byref(self._st), C.byref(e),
                                           _ptr(m), obs.ctypes.data, am.ctypes.data, 0, None)
        if rc:
            raise RuntimeError(self.lib["last_error"]().decode())
        return obs, am
