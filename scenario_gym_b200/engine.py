"""
Host-side driver of the CUDA rollout engine (``csrc/libsg_b200.so``).

PyTorch is used for plumbing only: device allocations, streams and (in
``distributed.py``) the final NCCL gather.  All arithmetic happens inside the
library's sm_100a kernels, reached through the C ABI of ``include/sg_b200.h``.
There is no CPU fallback: constructing an ``Engine`` without a CUDA device or
without the built library raises.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Sequence, Union

import numpy as np
import torch

from . import abi
from .action_rng import ActionRng
from .packing import PackedScene

EVENT_DTYPE = np.dtype(
    [("scenario", "<i4"), ("tick", "<i4"), ("slot", "<i4"), ("_pad", "<i4"), ("t", "<f8")]
)

_TORCH_DTYPES = {
    "float64": torch.float64,
    "uint8": torch.uint8,
    "int32": torch.int32,
    "uint32": torch.int32,  # bit-identical storage; viewed as uint32 on the host
    "int64": torch.int64,
}


class Engine:
    """N scenarios x M slots resident on one GPU."""

    def __init__(self, scene: PackedScene, params: Optional[abi.SgParams] = None,
                 device: Union[int, str, torch.device] = 0, event_cap: int = 1 << 20,
                 trace_cap: int = 0, coll_matrix: Optional[bool] = None):
        if not torch.cuda.is_available():
            raise RuntimeError("scenario_gym_b200 needs a CUDA device (no CPU fallback)")
        self.lib = abi.load_product()
        self.device = torch.device(device if not isinstance(device, int) else f"cuda:{device}")
        self.dev_index = self.device.index or 0
        self.scene = scene
        self.params = params if params is not None else abi.default_params()
        self.N, self.M, self.W = scene.N, scene.M, scene.W
        if coll_matrix is None:
            coll_matrix = bool(self.params.features & abi.FEAT_COLL_MATRIX)
        elif not coll_matrix:
            self.params.features &= ~abi.FEAT_COLL_MATRIX
        self.event_cap, self.trace_cap = int(event_cap), int(trace_cap)

        # --- scene -> device
        self._scene_t: Dict[str, torch.Tensor] = {}
        self._sc = abi.SgScene()
        self._sc.n_scenarios, self._sc.n_slots = scene.N, scene.M
        self._sc.n_traj_rows = scene.traj_rows.shape[0]
        self._sc.n_union_rows = scene.union_t.shape[0]
        self._sc.n_route_pts = scene.route_xy.shape[0]
        self._sc.n_networks = scene.n_networks
        self._sc.n_rn_polys = len(scene.rn_edge_off) - 1
        self._sc.n_rn_edges = scene.rn_edges.shape[0]
        self._sc.kind_mask = scene.kind_mask()
        self._sc.scene_flags = scene.scene_flags()
        # a union table that was not built on the host is built here from the uploaded control points
        device_union = not scene.union_ready and scene.union_on_device_ok()
        for k, a in scene.arrays(union_rows=not device_union).items():
            t = torch.from_numpy(np.ascontiguousarray(a)).to(self.device)
            if t.numel() == 0:  # keep a valid pointer for empty tables
                t = torch.zeros(8, dtype=t.dtype, device=self.device)
            self._scene_t[k] = t
            setattr(self._sc, k, t.data_ptr())
        if device_union:
            t = torch.empty((scene.union_t.shape[0], 6, scene.M), dtype=torch.float64, device=self.device)
            self._scene_t["union_x"] = t
            self._sc.union_x = t.data_ptr()
            self.build_union_on_device()

        self._alloc_state(coll_matrix)

    @classmethod
    def sharing_scene(cls, other: "Engine", event_cap: int = 1024, trace_cap: int = 0) -> "Engine":
        """
        A second state over ``other``'s device scene: the same scene tensors (nothing is uploaded or packed
        again), a copy of its parameters and a state of its own, sized like ``other``'s (pair matrix included
        when ``other`` has one).  What a fork (``fork_into``) needs: branches that do not keep many collision
        events take a small ``event_cap``.
        """
        eng = cls.__new__(cls)
        eng.lib, eng.device, eng.dev_index = other.lib, other.device, other.dev_index
        eng.scene = other.scene
        eng.params = abi.SgParams.from_buffer_copy(other.params)
        eng.N, eng.M, eng.W = other.N, other.M, other.W
        eng.event_cap, eng.trace_cap = int(event_cap), int(trace_cap)
        eng._scene_t = other._scene_t
        eng._sc = abi.SgScene.from_buffer_copy(other._sc)
        eng._alloc_state(other._coll_matrix)
        return eng

    def _alloc_state(self, coll_matrix: bool) -> None:
        N, M, W = self.N, self.M, self.W
        self._coll_matrix = bool(coll_matrix)
        dims = {"N": N, "M": M, "NM": N * M, "W": W, "E": max(self.event_cap, 1),
                "T": max(self.trace_cap, 1)}
        self._state_t: Dict[str, torch.Tensor] = {}
        self._st = abi.SgState()
        for name, dtype, shape in abi.STATE_FIELDS:
            shp = tuple(dims[s] if s in dims else int(s) for s in shape)
            if name == "coll_mask" and not coll_matrix:
                shp = (1,)
            if dtype == "event":
                t = torch.zeros((shp[0] * EVENT_DTYPE.itemsize,), dtype=torch.uint8, device=self.device)
            else:
                t = torch.zeros(shp, dtype=_TORCH_DTYPES[dtype], device=self.device)
            self._state_t[name] = t
            setattr(self._st, name, t.data_ptr())
        self._st.event_cap = self.event_cap
        self._st.trace_cap = self.trace_cap
        self._dtypes = {name: dtype for name, dtype, _ in abi.STATE_FIELDS}
        self._actions_t: Optional[torch.Tensor] = None

    # ------------------------------------------------------------------ helpers
    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def _check(self, rc: int):
        if rc:
            raise RuntimeError(f"sg_b200: {self.lib['last_error']().decode()} (rc={rc})")

    def state_bytes(self) -> int:
        return int(sum(t.numel() * t.element_size() for t in self._state_t.values()))

    # ------------------------------------------------------------------ API
    def reset(self, mask: Optional[torch.Tensor] = None) -> None:
        """
        State.reset + metric/controller resets for every scenario (sg_reset), or -- ``mask``: a uint8 / bool
        device tensor [N] -- for the scenarios with ``mask[n] != 0`` only (sg_reset_scenarios; the other
        scenarios and the event count are left as they are).
        """
        if mask is None:
            self._check(self.lib["reset"](C.byref(self._sc), C.byref(self.params), C.byref(self._st),
                                          self.dev_index, self._stream()))
            return
        m = self._scenario_mask(mask)
        self._check(self.lib["reset_scenarios"](C.byref(self._sc), C.byref(self.params), C.byref(self._st),
                                                m.data_ptr(), self.dev_index, self._stream()))

    def fork_into(self, engines: Sequence["Engine"], spec: Optional[abi.SgEnvSpec] = None,
                  specs: Optional[Sequence[abi.SgEnvSpec]] = None) -> None:
        """
        sg_fork_state: copy this engine's state into every engine of ``engines`` (same scene size, no trace)
        in one device pass, on the current stream.  The destinations' event counts are set to 0.  With
        ``spec`` / ``specs`` (the source's SgEnvSpec and one per destination) the snapshot arrays are
        copied too, so the destinations' env_reward compares against this engine's last observation.
        """
        self._check(self.lib["fork_state"](*self.fork_args(engines, spec, specs), self.dev_index, self._stream()))

    def fork_args(self, engines: Sequence["Engine"], spec: Optional[abi.SgEnvSpec] = None,
                  specs: Optional[Sequence[abi.SgEnvSpec]] = None) -> tuple:
        """The checked arguments of ``fork_into`` but the device and the stream (callers that fork repeatedly
        build them once)."""
        engines = list(engines)
        if not engines:
            raise ValueError("fork_into needs at least one destination engine")
        for e in engines:
            if not isinstance(e, Engine) or (e.N, e.M) != (self.N, self.M) or e.device != self.device:
                raise ValueError(f"fork_into: every destination must be an Engine of {self.N} x {self.M} "
                                 f"slots on {self.device}")
            if e is self:
                raise ValueError("fork_into: the source cannot be a destination")
        if (spec is None) != (specs is None) or (specs is not None and len(specs) != len(engines)):
            raise ValueError("fork_into: give spec and one spec per destination, or neither")
        # (ctypes pointers and arrays keep the structures they point to alive)
        dst = (C.POINTER(abi.SgState) * len(engines))(*[C.pointer(e._fork_view()) for e in engines])
        src_spec = dst_spec = None
        if spec is not None:
            dst_spec = (C.POINTER(abi.SgEnvSpec) * len(specs))(*[C.pointer(s) for s in specs])
            src_spec = C.pointer(spec)
        return (C.byref(self._sc), C.byref(self._fork_view()), dst, len(engines), src_spec, dst_spec)

    def _fork_view(self) -> abi.SgState:
        """The SgState sg_fork_state sees: coll_mask NULL when the pair matrix is not allocated."""
        if self._coll_matrix:
            return self._st
        if getattr(self, "_fork_st", None) is None:
            self._fork_st = abi.SgState.from_buffer_copy(self._st)
            self._fork_st.coll_mask = None
        return self._fork_st

    def _scenario_mask(self, mask: torch.Tensor) -> torch.Tensor:
        if not isinstance(mask, torch.Tensor) or mask.device != self.device or mask.numel() != self.N \
                or mask.dtype not in (torch.uint8, torch.bool):
            raise ValueError(f"mask must be a uint8 / bool tensor of {self.N} entries on {self.device}")
        return mask.contiguous().view(torch.uint8) if mask.dtype == torch.bool else mask.contiguous()

    def env_observe(self, spec: abi.SgEnvSpec, obs: torch.Tensor, agent_mask: torch.Tensor,
                    mask: Optional[torch.Tensor] = None) -> None:
        """sg_env_observe into preallocated ``obs`` (fp32 [N, A, F]) / ``agent_mask`` (uint8 [N, A])."""
        m = None if mask is None else self._scenario_mask(mask)
        self._check(self.lib["env_observe"](C.byref(self._sc), C.byref(self.params), C.byref(self._st),
                                            C.byref(spec), None if m is None else m.data_ptr(), obs.data_ptr(),
                                            agent_mask.data_ptr(), self.dev_index, self._stream()))

    def env_reward(self, spec: abi.SgEnvSpec, reward: torch.Tensor, terms: torch.Tensor,
                   terminated: torch.Tensor, truncated: torch.Tensor) -> None:
        """sg_env_reward into preallocated reward (fp32 [N, A]), terms (fp32 [N, A, 5]) and flags (uint8 [N])."""
        self._check(self.lib["env_reward"](C.byref(self._sc), C.byref(self.params), C.byref(self._st),
                                           C.byref(spec), reward.data_ptr(), terms.data_ptr(),
                                           terminated.data_ptr(), truncated.data_ptr(), self.dev_index,
                                           self._stream()))

    def plan_sample(self, spec: abi.SgEnvSpec, B: int, H: int, seed: int, k: int, sigma, mu: torch.Tensor,
                    reset: Optional[torch.Tensor], table: torch.Tensor) -> None:
        """sg_plan_sample: the B branches' actions drawn around the mean ``mu`` (fp64 [N, H, A, 2]) into the flat
        branch table ``table`` ([B][H][2][N*M], fp32 or fp64); ``reset`` (uint8 / bool [N] or None): the scenarios
        whose mean is zeroed first."""
        sig = (C.c_double * 2)(float(sigma[0]), float(sigma[1]))
        r = None if reset is None else self._scenario_mask(reset).data_ptr()
        self._check(self.lib["plan_sample"](C.byref(spec), self.N, self.M, int(B), int(H), int(seed) & (2**64 - 1),
                                            int(k), sig, mu.data_ptr(), r, table.data_ptr(),
                                            int(table.dtype == torch.float64), self.dev_index, self._stream()))

    def plan_update(self, spec: abi.SgEnvSpec, B: int, H: int, lam: float, reward: torch.Tensor,
                    table: torch.Tensor, mu_in: torch.Tensor, mu_out: torch.Tensor, finish: bool,
                    action: Optional[torch.Tensor], best_branch: torch.Tensor, best_reward: torch.Tensor) -> None:
        """sg_plan_update: the mean ``mu_in`` moved to the reward-weighted average of the branches (``reward`` fp32
        [B, N, A]) into ``mu_out``; with ``finish`` also the first action (fp32 [N, A, 2]) and the shift."""
        self._check(self.lib["plan_update"](C.byref(spec), self.N, self.M, int(B), int(H), float(lam),
                                            reward.data_ptr(), table.data_ptr(), int(table.dtype == torch.float64),
                                            mu_in.data_ptr(), mu_out.data_ptr(), int(bool(finish)),
                                            None if action is None else action.data_ptr(), best_branch.data_ptr(),
                                            best_reward.data_ptr(), self.dev_index, self._stream()))

    def build_union_on_device(self) -> torch.Tensor:
        """
        Recompute the resident BatchReplayEntity union table from the uploaded control points and knot
        times (sg_build_union_x; entity/batch.py:80-112); returns the device tensor (rows, 6, M).
        """
        self._check(self.lib["build_union_x"](C.byref(self._sc), self.dev_index, self._stream()))
        return self._scene_t["union_x"]

    def set_actions(self, actions) -> torch.Tensor:
        """Upload a (T, 2, N*M) VehicleAction table (accel, steer; fp64 or fp32) and keep it resident."""
        if isinstance(actions, np.ndarray):
            if actions.dtype != np.float32:
                actions = np.ascontiguousarray(actions, np.float64)
            actions = torch.from_numpy(np.ascontiguousarray(actions))
        if actions.dtype != torch.float32:
            actions = actions.to(dtype=torch.float64)
        actions = actions.to(self.device).contiguous()
        if actions.dim() != 3 or tuple(actions.shape[1:]) != (2, self.N * self.M):
            raise ValueError(f"actions must be (T, 2, {self.N * self.M}), got {tuple(actions.shape)}")
        self._actions_t = actions
        return actions

    def fill_actions(self, rng: ActionRng, tick0: int = 0, n_ticks: Optional[int] = None) -> torch.Tensor:
        """Rows [tick0, tick0 + n_ticks) of the table `rng` describes, drawn on the device (fp64)."""
        n_ticks = rng.n_ticks - tick0 if n_ticks is None else n_ticks
        if rng.nm != self.N * self.M:
            raise ValueError(f"ActionRng describes {rng.nm} slots, the engine has {self.N * self.M}")
        out = torch.empty((max(n_ticks, 0), 2, rng.nm), dtype=torch.float64, device=self.device)
        r = rng.struct()
        self._check(self.lib["fill_random_actions"](C.byref(r), int(tick0), int(n_ticks), int(rng.nm),
                                                    out.data_ptr(), self.dev_index, self._stream()))
        return out

    def _wants_f64_table(self) -> bool:
        """Vehicle-only scenes rolled out with a trace / pair matrix take an fp64 table (sg_api.cu)."""
        mask = self._sc.kind_mask
        veh_only = bool(mask & (1 << abi.KIND_VEHICLE)) and not (
            mask & ~((1 << abi.KIND_VEHICLE) | (1 << abi.KIND_EMPTY)))
        f, term = self.params.features, self.params.terminal
        need_coll = bool(f & abi.FEAT_COLLISIONS) or bool(term & (abi.TERM_COLLISION | abi.TERM_EGO_COLLISION))
        lean = need_coll and self.trace_cap <= 0 and not (f & abi.FEAT_COLL_MATRIX)
        return veh_only and not lean

    def rollout(self, n_ticks: int = -1, actions=None, tick0: int = 0, host_pose=None,
                host_present=None, step_done: bool = False) -> None:
        """
        ``n_ticks`` x ScenarioGym.step() fused on the device; ``n_ticks < 0`` runs every
        scenario to ``is_done`` (ScenarioGym.rollout).  ``actions``: a (T, 2, N*M) table (fp64 or
        fp32), consumed from row ``tick0``, or an ``ActionRng`` (the rows are then drawn inside the
        kernel from numpy's PCG64 stream; nothing is uploaded).
        """
        inp = abi.SgInputs()
        inp.step_done = int(step_done)
        keep = []
        if isinstance(actions, ActionRng) and self._wants_f64_table():
            rows = actions.n_ticks - tick0 if n_ticks < 0 else min(n_ticks, actions.n_ticks - tick0)
            actions, tick0 = self.fill_actions(actions, tick0, rows), 0
            self._actions_t = actions
        if isinstance(actions, ActionRng):
            if actions.nm != self.N * self.M:
                raise ValueError(f"ActionRng describes {actions.nm} slots, the engine has {self.N * self.M}")
            inp.use_rng, inp.rng_tick0 = 1, int(tick0)
            inp.rng = actions.struct()
            inp.n_action_ticks = max(actions.n_ticks - tick0, 0)
        elif actions is not None:
            a = self.set_actions(actions) if not (
                isinstance(actions, torch.Tensor) and actions is self._actions_t) else actions
            if a.dtype == torch.float32 and self._wants_f64_table():
                a = a.to(torch.float64)
            if tick0:
                a = a[tick0:]
            if a.dtype == torch.float32:
                inp.actions_f32 = a.data_ptr()
            else:
                inp.actions = a.data_ptr()
            inp.n_action_ticks = a.shape[0]
            keep.append(a)
        elif (self.scene.kind == abi.KIND_VEHICLE).any():
            raise ValueError("scene has VehicleController slots: an action table or ActionRng is required")
        if host_pose is not None:
            hp = torch.from_numpy(np.ascontiguousarray(host_pose, np.float64)).to(self.device)
            hm = torch.from_numpy(np.ascontiguousarray(host_present, np.uint8)).to(self.device)
            inp.host_pose, inp.host_present = hp.data_ptr(), hm.data_ptr()
            keep += [hp, hm]
        self._check(self.lib["rollout"](C.byref(self._sc), C.byref(self.params), C.byref(self._st),
                                        C.byref(inp), int(n_ticks), self.dev_index, self._stream()))
        self._keep = keep

    def future_collisions(self, t=None, horizon: float = 5.0, n_samples: int = 10, slot=None) -> np.ndarray:
        """
        ``FutureCollisionDetector._step`` (reference sensor/common.py:88-105) for every scenario of
        the batch in one launch: does the sensor entity (``slot[n]``, default the ego) meet any other
        entity within ``horizon`` of ``t[n]`` (default: the current ``state.t``)?  Returns bool [N].
        """
        tt = self._state_t["t"] if t is None else torch.as_tensor(
            np.ascontiguousarray(t, np.float64)).to(self.device)
        if tt.numel() != self.N:
            raise ValueError(f"t must have {self.N} entries")
        sl = None
        if slot is not None:
            sl = torch.as_tensor(np.ascontiguousarray(slot, np.int32)).to(self.device)
        out = torch.zeros(self.N, dtype=torch.uint8, device=self.device)
        self._check(self.lib["future_collisions"](
            C.byref(self._sc), tt.data_ptr(), None if sl is None else sl.data_ptr(), float(horizon),
            int(n_samples), out.data_ptr(), self.dev_index, self._stream()))
        return out.cpu().numpy().astype(bool)

    def entities_in_radius(self, x, y, r) -> np.ndarray:
        """
        ``State.get_entities_in_radius`` for every scenario in one launch: bool [N, M], slot s of
        scenario n present and strictly inside ``Point(x[n], y[n]).buffer(r[n])`` (r[n] <= 0: skipped).
        """
        args = [torch.from_numpy(np.array(np.broadcast_to(np.asarray(a, np.float64), (self.N,)))).to(self.device)
                for a in (x, y, r)]
        out = torch.zeros(self.N * self.M, dtype=torch.uint8, device=self.device)
        self._check(self.lib["entities_in_radius"](C.byref(self._st), self.N, self.M, args[0].data_ptr(),
                                                   args[1].data_ptr(), args[2].data_ptr(), out.data_ptr(),
                                                   self.dev_index, self._stream()))
        return out.cpu().numpy().astype(bool).reshape(self.N, self.M)

    def tensor(self, name: str) -> torch.Tensor:
        """The device tensor behind a state field (no copy)."""
        return self._state_t[name]

    def get(self, name: str) -> np.ndarray:
        """Host copy of a state array."""
        a = self._state_t[name].cpu().numpy()
        if self._dtypes[name] == "uint32":
            a = a.view(np.uint32)
        return a

    def events(self) -> np.ndarray:
        """Ego collision rising-edge events, sorted by (scenario, tick, slot)."""
        n = int(self._state_t["event_count"].item())
        if n > self.event_cap:
            raise RuntimeError(f"{n} collision events exceed event_cap={self.event_cap}")
        raw = self._state_t["events"][: n * EVENT_DTYPE.itemsize].cpu().numpy()
        ev = raw.view(EVENT_DTYPE)
        return ev[np.lexsort((ev["slot"], ev["tick"], ev["scenario"]))]

    def synchronize(self) -> None:
        torch.cuda.synchronize(self.device)
