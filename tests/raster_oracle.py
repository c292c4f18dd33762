"""
TEST INFRASTRUCTURE ONLY -- ``RasterOracleEngine``: ``OracleEnvEngine`` with ``env_raster``, the brute-force
plain-C restatement of sg_env_raster (include/sg_b200.h, SgRasterSpec) in ``tests/raster_oracle.c``, and
``surface_contains``, a wrapper of the oracle's strict containment test.  The library is compiled on first use into
a temporary directory (removed at exit), so nothing is written into the tree.
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


def load_raster_oracle() -> Dict[str, object]:
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="sg_raster_oracle_")
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, "libraster_oracle.so")
        cc = os.environ.get("CC", "gcc")
        subprocess.check_call([cc] + _CFLAGS + ["-shared", "-I", _ORACLE, "-o", out,
                               os.path.join(_HERE, "raster_oracle.c"), "-lm"])
        cdll = C.CDLL(out)
        f = abi.bind(cdll, "sgo_")
        fn = cdll.sgo_env_raster_brute
        fn.restype = C.c_int
        fn.argtypes = [C.POINTER(abi.SgScene), C.POINTER(abi.SgParams), C.POINTER(abi.SgState),
                       C.POINTER(abi.SgEnvSpec), C.POINTER(abi.SgRasterSpec), C.c_void_p, C.c_void_p]
        f["env_raster_brute"] = fn
        fn = cdll.sgo_test_surface_contains
        fn.restype = C.c_int
        fn.argtypes = [C.POINTER(abi.SgScene), C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
        f["test_surface_contains"] = fn
        _lib = f
    return _lib


def raster_spec(scene, size: int, resolution: float = 0.5, ahead: float = 0.0) -> abi.SgRasterSpec:
    """An SgRasterSpec over ``scene`` (poly_box / margin left unset: the oracle does not read them)."""
    r = abi.SgRasterSpec()
    r.size, r.n_networks, r.resolution, r.ahead = int(size), scene.n_networks, float(resolution), float(ahead)
    return r


class RasterOracleEngine(OracleEnvEngine):
    """``OracleEnvEngine`` with ``env_raster(rspec, mask)`` over the agents of the spec made by ``env_spec``."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.lib = load_raster_oracle()

    def env_raster(self, rspec: abi.SgRasterSpec, mask: Optional[np.ndarray] = None) -> np.ndarray:
        """uint8 [N, A, 5, S, S] (rasters of masked-out scenarios: 0)."""
        e = self._env_spec
        S = int(rspec.size)
        out = np.zeros((self.scene.N, e.n_agents, 5, S, S), np.uint8)
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        rc = self.lib["env_raster_brute"](C.byref(self._sc), C.byref(self.params), C.byref(self._st), C.byref(e),
                                          C.byref(rspec), _ptr(m), out.ctypes.data)
        if rc:
            raise RuntimeError(self.lib["last_error"]().decode())
        return out

    def surface_contains(self, n: int, k: int, px: np.ndarray, py: np.ndarray) -> np.ndarray:
        """The oracle's surface_contains(scene, n, k, px, py) for arrays of points (uint8)."""
        px, py = np.ascontiguousarray(px, np.float64).reshape(-1), np.ascontiguousarray(py, np.float64).reshape(-1)
        out = np.zeros(len(px), np.uint8)
        self.lib["test_surface_contains"](C.byref(self._sc), int(n), int(k), px.ctypes.data, py.ctypes.data,
                                          len(px), out.ctypes.data)
        return out
