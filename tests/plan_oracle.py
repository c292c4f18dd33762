"""
TEST INFRASTRUCTURE ONLY -- the MPPI planner of include/sg_b200.h (sg_plan_sample / sg_plan_update) restated in
numpy, with the noise from the oracle's plain-C ``noise2`` (``tests/plan_oracle.c``, compiled on first use into a
temporary directory removed at exit, so nothing is written into the tree), and ``noise2_numpy``, the same
splitmix64 + Box-Muller written in numpy.
"""
from __future__ import annotations

import atexit
import ctypes as C
import math
import os
import shutil
import subprocess
import tempfile
from typing import Optional

import numpy as np

from oracle.env_runner import _CFLAGS

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(os.path.dirname(_HERE), "oracle")
_fn: Optional[object] = None
_GOLDEN = np.uint64(0x9E3779B97F4A7C15)
_log, _cos, _sin = (np.frompyfunc(f, 1, 1) for f in (math.log, math.cos, math.sin))


def _load():
    global _fn
    if _fn is None:
        tmp = tempfile.mkdtemp(prefix="sg_plan_oracle_")
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, "libplan_oracle.so")
        cc = os.environ.get("CC", "gcc")
        subprocess.check_call([cc] + _CFLAGS + ["-shared", "-I", _ORACLE, "-o", out,
                               os.path.join(_HERE, "plan_oracle.c"), "-lm"])
        fn = C.CDLL(out).sgp_noise2
        fn.restype = None
        fn.argtypes = [C.c_uint64, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]
        _fn = fn
    return _fn


def noise2_c(seed: int, i, k: int) -> np.ndarray:
    """[..., 2] fp64: the oracle's noise2(seed, i, k) for every counter of ``i``."""
    i = np.ascontiguousarray(i, np.int64)
    z = np.empty(i.shape + (2,), np.float64)
    _load()(int(seed) & (2**64 - 1), i.ctypes.data, i.size, int(k), z.ctypes.data)
    return z


def _splitmix64(z):
    with np.errstate(over="ignore"):
        z = z + _GOLDEN
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def noise2_numpy(seed: int, i, k: int) -> np.ndarray:
    """noise2 restated in numpy (uint64 arithmetic wraps as in C)."""
    i = np.asarray(i, np.int64).astype(np.uint64)
    with np.errstate(over="ignore"):
        ctr = i * _GOLDEN + np.uint64(int(k) & 0xFFFFFFFF)
    a = _splitmix64(np.uint64(int(seed) & (2**64 - 1)) ^ _splitmix64(ctr))
    b = _splitmix64(a)
    u1 = ((a >> np.uint64(11)).astype(np.float64) + 1.0) * (1.0 / 9007199254740992.0)
    u2 = (b >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)
    # (the C library's log / cos / sin, element by element: numpy's vectorised ones may differ in the last place)
    r = np.sqrt(-2.0 * _log(u1).astype(np.float64))
    ang = 2.0 * np.pi * u2
    return np.stack([r * _cos(ang).astype(np.float64), r * _sin(ang).astype(np.float64)], -1)


def sample_noise(slots: np.ndarray, B: int, H: int, seed: int, k: int, sigma) -> np.ndarray:
    """eps [N, B, H, A, 2] of sg_plan_sample: sigma_c * z_c of counter ((n*A + a)*B + b)*H + h, 0 for b = 0
    (padding agents get 0 too)."""
    N, A = slots.shape
    i = ((np.arange(N * A).reshape(N, 1, 1, A) * B + np.arange(B).reshape(1, B, 1, 1)) * H
         + np.arange(H).reshape(1, 1, H, 1))
    eps = noise2_c(seed, i, k) * np.asarray(sigma, np.float64)
    eps[:, 0] = 0.0
    eps.transpose(0, 3, 1, 2, 4)[slots < 0] = 0.0  # padding (n, a), every b, h
    return eps


def sample(mu: np.ndarray, reset, slots: np.ndarray, B: int, H: int, seed: int, k: int, sigma, dtype):
    """
    sg_plan_sample restated: (mu0, table) with mu0 = mu [N, H, A, 2] with the rows of scenarios with reset[n] != 0
    zeroed (reset None: none) and table [N, B, H, A, 2] the values it stores, round(mu0 + eps) in ``dtype``
    (branch 0: mu0).
    """
    mu0 = np.array(mu, np.float64)
    if reset is not None:
        mu0[np.asarray(reset) != 0] = 0.0
    eps = sample_noise(slots, B, H, seed, k, sigma)
    return mu0, (mu0[:, None] + eps).astype(dtype)


def update(mu: np.ndarray, table: np.ndarray, reward: np.ndarray, lam: float):
    """
    sg_plan_update restated: mu [N, H, A, 2] fp64, table [N, B, H, A, 2] (the stored values), reward [N, B, A]
    fp32.  Returns (mu' [N, H, A, 2], action [N, A, 2] fp32, shifted [N, H, A, 2], best_branch [N, A],
    best_reward [N, A]) for every (n, a); the device leaves padding agents alone.
    """
    R = reward.astype(np.float64)
    rmax = R.max(axis=1)                                          # [N, A]
    w = np.exp((R - rmax[:, None]) / lam)                         # [N, B, A]
    eps_hat = table.astype(np.float64) - mu[:, None]              # [N, B, H, A, 2]
    acc = np.zeros_like(mu)
    wsum = np.zeros_like(rmax)
    for b in range(R.shape[1]):                                   # ascending b, as the device sums
        acc += w[:, b, None, :, None] * eps_hat[:, b]
        wsum += w[:, b]
    new = mu + acc / wsum[:, None, :, None]
    shifted = np.zeros_like(new)
    shifted[:, :-1] = new[:, 1:]
    best = np.argmax(R, axis=1).astype(np.int32)                  # (the first maximum)
    return new, new[:, 0].astype(np.float32), shifted, best, rmax.astype(np.float32)
