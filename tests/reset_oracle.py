"""
TEST INFRASTRUCTURE ONLY -- sg_reset_scenarios_init (include/sg_b200.h) on the CPU: ``ResetOracleEngine``, an
``OracleEnvEngine`` whose ``reset_init`` runs the plain-C restatement ``tests/reset_oracle.c``, and the same
semantics restated in numpy (``uniform_numpy``, ``start_times``, ``perturb_rows``) to check the C against.  The
library is compiled on first use into a temporary directory (removed at exit), so nothing is written into the tree.
"""
from __future__ import annotations

import atexit
import ctypes as C
import math
import os
import shutil
import subprocess
import tempfile
from typing import Dict, Optional

import numpy as np

from oracle.env_runner import _CFLAGS, OracleEnvEngine
from oracle.runner import _ptr
from scenario_gym_b200 import abi

from plan_oracle import _GOLDEN, _splitmix64, noise2_numpy

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(os.path.dirname(_HERE), "oracle")
_lib: Optional[Dict[str, object]] = None
_cos, _sin = (np.frompyfunc(f, 1, 1) for f in (math.cos, math.sin))


def load_reset_oracle() -> Dict[str, object]:
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="sg_reset_oracle_")
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, "libreset_oracle.so")
        cc = os.environ.get("CC", "gcc")
        subprocess.check_call([cc] + _CFLAGS + ["-shared", "-I", _ORACLE, "-o", out,
                               os.path.join(_HERE, "reset_oracle.c"), "-lm"])
        cdll = C.CDLL(out)
        init = cdll.sgo_reset_scenarios_init
        init.restype = C.c_int
        init.argtypes = [C.POINTER(abi.SgScene), C.POINTER(abi.SgParams), C.POINTER(abi.SgState), C.c_void_p,
                         C.POINTER(abi.SgResetInit), C.c_int, C.c_void_p]
        uni = cdll.sgr_uniform
        uni.restype = None
        uni.argtypes = [C.c_uint64, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]
        last = cdll.sgo_last_error
        last.restype = C.c_char_p
        _lib = {"reset_scenarios_init": init, "uniform": uni, "last_error": last}
    return _lib


def tick2(k) -> np.ndarray:
    """The tick value 2k of draw index k, as the 32-bit int the stream's key takes."""
    return ((np.asarray(k, np.int64).astype(np.uint64) * np.uint64(2)) & np.uint64(0xFFFFFFFF)).astype(np.uint32) \
        .view(np.int32)


def uniform_c(seed: int, i, tick: int) -> np.ndarray:
    i = np.ascontiguousarray(i, np.int64)
    u = np.empty(i.shape, np.float64)
    load_reset_oracle()["uniform"](int(seed) & (2**64 - 1), i.ctypes.data, i.size, int(tick), u.ctypes.data)
    return u


def uniform_numpy(seed: int, i, tick) -> np.ndarray:
    """(a >> 11) * 2^-53 with a = splitmix64(seed ^ splitmix64(i * golden + (uint32) tick)), in numpy."""
    i = np.asarray(i, np.int64).astype(np.uint64)
    t = np.asarray(tick, np.int64).astype(np.uint64) & np.uint64(0xFFFFFFFF)
    with np.errstate(over="ignore"):
        a = _splitmix64(np.uint64(int(seed) & (2**64 - 1)) ^ _splitmix64(i * _GOLDEN + t))
    return (a >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


def start_times(t0, window, counter, seed: int, base: int = 0) -> np.ndarray:
    """The drawn start times t0 + u * window of sg_reset_scenarios_init (no t_start)."""
    N = len(t0)
    u = np.array([uniform_numpy(seed, -1 - (base + n), int(tick2(counter[n]))) for n in range(N)])
    return np.asarray(t0, np.float64) + u * np.asarray(window, np.float64)


def perturb_rows(x, y, h, vx, vy, z, sigma):
    """The perturbation of include/sg_b200.h restated element-wise: z [..., 4] the noise (z0, z1, z2, z3).
    Returns (x, y, h, vx, vy, v)."""
    x, y, h, vx, vy = (np.array(a, np.float64) for a in (x, y, h, vx, vy))
    s0, s1, s2, s3 = (float(s) for s in sigma)
    v0 = np.sqrt(vx * vx + vy * vy)
    v = v0.copy()
    if s0 != 0.0 or s1 != 0.0:
        c, s = _cos(h).astype(np.float64), _sin(h).astype(np.float64)
        lon, lat = s0 * z[..., 0], s1 * z[..., 1]
        x, y = x + (c * lon - s * lat), y + (s * lon + c * lat)
    dh = np.zeros_like(h)
    if s2 != 0.0:
        dh = s2 * z[..., 2]
        h = h + dh
    if s2 != 0.0 or s3 != 0.0:
        v = np.maximum(v0 + s3 * z[..., 3], 0.0)
        cd, sd = _cos(dh).astype(np.float64), _sin(dh).astype(np.float64)
        rot = v0 > 0.0
        fresh = ~rot & (v > 0.0)
        with np.errstate(divide="ignore", invalid="ignore"):  # (v / v0 is only used where v0 > 0)
            f = v / v0
            nvx = np.where(rot, (cd * vx - sd * vy) * f, np.where(fresh, v * _cos(h).astype(np.float64), vx))
            nvy = np.where(rot, (sd * vx + cd * vy) * f, np.where(fresh, v * _sin(h).astype(np.float64), vy))
        vx, vy = nvx, nvy
    return x, y, h, vx, vy, v


def perturb_noise(seed: int, ctr, k) -> np.ndarray:
    """[..., 4] the noise (z0, z1, z2, z3) of slot counters ``ctr`` at draw index k (numpy restatement)."""
    t = int(tick2(k))
    return np.concatenate([noise2_numpy(seed, ctr, t), noise2_numpy(seed, ctr, t + 1)], -1)


def reset_init(t_start=None, start_window=None, counter=None, perturb=None, sigma=(0.0,) * 4, seed: int = 0):
    """(SgResetInit over host arrays, the arrays to keep alive)."""
    keep = {}
    r = abi.SgResetInit()
    for name, a, dt in (("t_start", t_start, np.float64), ("start_window", start_window, np.float64),
                        ("counter", counter, np.int64), ("perturb", perturb, np.uint8)):
        if a is not None:
            keep[name] = np.ascontiguousarray(a, dt)
            setattr(r, name, keep[name].ctypes.data)
    for k, v in enumerate(sigma):
        r.sigma[k] = float(v)
    r.seed = int(seed) & (2**64 - 1)
    return r, keep


class ResetOracleEngine(OracleEnvEngine):
    """``OracleEnvEngine`` plus ``reset_init(mask, init)``: sgo_reset_scenarios_init on the oracle's state."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.reset_lib = load_reset_oracle()

    def reset_init(self, mask: Optional[np.ndarray], init: abi.SgResetInit):
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        rc = self.reset_lib["reset_scenarios_init"](C.byref(self._sc), C.byref(self.params), C.byref(self._st),
                                                    _ptr(m), C.byref(init), 0, None)
        if rc:
            raise RuntimeError(self.reset_lib["last_error"]().decode())
