"""
TEST INFRASTRUCTURE ONLY -- drives ``oracle/_build/libsg_env_oracle.so`` (``sg_env_oracle.c``: the oracle plus
the plain-C restatement of the closed-loop environment's entry points) through the same ABI as the CUDA
engine, with numpy host buffers.  Imported only by tests/.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Dict, Optional

import numpy as np

from scenario_gym_b200 import abi

from .runner import OracleEngine, _ptr

_HERE = os.path.dirname(os.path.abspath(__file__))
ENV_ORACLE_LIB = os.path.join(_HERE, "_build", "libsg_env_oracle.so")
# the flags of oracle/Makefile (no FMA contraction: the reference has none on this path)
_CFLAGS = ["-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wextra", "-std=gnu11"]


def build_env_oracle(force: bool = False) -> str:
    srcs = [os.path.join(_HERE, f) for f in ("sg_env_oracle.c", "sg_oracle.c")]
    srcs.append(os.path.join(_HERE, "..", "include", "sg_b200.h"))
    stale = force or not os.path.exists(ENV_ORACLE_LIB) or \
        os.path.getmtime(ENV_ORACLE_LIB) < max(os.path.getmtime(s) for s in srcs)
    if stale:
        os.makedirs(os.path.dirname(ENV_ORACLE_LIB), exist_ok=True)
        cc = os.environ.get("CC", "gcc")
        subprocess.check_call([cc] + _CFLAGS + ["-shared", "-o", ENV_ORACLE_LIB, srcs[0], "-lm"])
    return ENV_ORACLE_LIB


_lib: Optional[Dict[str, object]] = None


def load_env_oracle() -> Dict[str, object]:
    global _lib
    if _lib is None:
        build_env_oracle()
        _lib = abi.bind(C.CDLL(ENV_ORACLE_LIB), "sgo_")
    return _lib


class OracleEnvEngine(OracleEngine):
    """``OracleEngine`` plus the environment's entry points (sgo_reset_scenarios, sgo_env_observe,
    sgo_env_reward); mirrors ``Engine.reset(mask)`` / ``env_observe`` / ``env_reward``."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.lib = load_env_oracle()

    def reset_scenarios(self, mask: np.ndarray):
        m = np.ascontiguousarray(mask, np.uint8)
        assert m.shape == (self.scene.N,), m.shape
        rc = self.lib["reset_scenarios"](C.byref(self._sc), C.byref(self.params), C.byref(self._st),
                                         m.ctypes.data, 0, None)
        if rc:
            raise RuntimeError(self.lib["last_error"]().decode())

    def env_spec(self, agent_slot: np.ndarray, k_neighbours: int = 8, radius: float = 0.0,
                 lookahead=(), road: bool = False, weights=(0.0,) * 5):
        """
        An SgEnvSpec over host buffers (kept on the engine): agent_slot [N, A].  Returns (spec, F);
        ``self.env`` holds the snapshot arrays.
        """
        N = self.scene.N
        slots = np.ascontiguousarray(agent_slot, np.int32)
        A = slots.shape[1]
        self.env = {"agent_slot": slots, "snap_dist": np.zeros(N * A), "snap_collided": np.zeros(N * A, np.uint8),
                    "snap_pair_ticks": np.zeros(N, np.int64), "snap_rss": np.zeros(N, np.uint8)}
        e = abi.SgEnvSpec()
        e.n_agents, e.k_neighbours, e.radius = A, int(k_neighbours), float(radius)
        e.n_lookahead, e.road = len(lookahead), int(bool(road))
        for k, v in enumerate(lookahead):
            e.lookahead[k] = float(v)
        for k, v in enumerate(weights):
            e.weights[k] = float(v)
        for k, a in self.env.items():
            setattr(e, k, a.ctypes.data)
        self._env_spec = e
        return e, abi.env_n_features(int(k_neighbours), len(lookahead), road)

    def env_observe(self, mask: Optional[np.ndarray] = None):
        """(obs [N, A, F] fp32, agent_mask [N, A]) of the spec made by env_spec (rows of masked-out scenarios: 0)."""
        e = self._env_spec
        N, A = self.scene.N, e.n_agents
        F = abi.env_n_features(e.k_neighbours, e.n_lookahead, bool(e.road))
        obs, am = np.zeros((N, A, F), np.float32), np.zeros((N, A), np.uint8)
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        rc = self.lib["env_observe"](C.byref(self._sc), C.byref(self.params), C.byref(self._st), C.byref(e),
                                     _ptr(m), obs.ctypes.data, am.ctypes.data, 0, None)
        if rc:
            raise RuntimeError(self.lib["last_error"]().decode())
        return obs, am

    def env_reward(self):
        """(reward [N, A], terms [N, A, 5], terminated [N], truncated [N]) against the last observe's snapshot."""
        e = self._env_spec
        N, A = self.scene.N, e.n_agents
        rew, terms = np.zeros((N, A), np.float32), np.zeros((N, A, 5), np.float32)
        te, tr = np.zeros(N, np.uint8), np.zeros(N, np.uint8)
        rc = self.lib["env_reward"](C.byref(self._sc), C.byref(self.params), C.byref(self._st), C.byref(e),
                                    rew.ctypes.data, terms.ctypes.data, te.ctypes.data, tr.ctypes.data, 0, None)
        if rc:
            raise RuntimeError(self.lib["last_error"]().decode())
        return rew, terms, te, tr

