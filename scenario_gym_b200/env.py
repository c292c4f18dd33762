"""
``VecScenarioEnv`` -- a closed-loop, batched environment on the device: a policy chooses every step's
VehicleActions from observations, and observations, rewards, termination and the reset of finished
scenarios are all computed by the library's kernels (``sg_env_observe``, ``sg_env_reward``,
``sg_reset_scenarios`` / ``sg_reset_scenarios_init``; semantics in ``include/sg_b200.h``).  ``step()`` and
``reset()`` enqueue their work on the current CUDA stream with no per-scenario Python and no device -> host
synchronisation; every buffer is allocated once, when the env is built.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Callable, Dict, List, Mapping, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import abi
from .entity import Entity
from .gym import ScenarioGym
from .plugins import PolicyAgent, RSSDistances, StateCallback
from .scenario import Scenario

# default weights of the reward terms (abi.ENV_TERMS order): progress, collision, off_road, tracking, rss
DEFAULT_REWARD_WEIGHTS = {"progress": 1.0, "collision": -10.0, "off_road": -1.0, "tracking": 0.1, "rss": -1.0}

# the per-scenario results ``info["final"]`` carries: key -> State field
_FINAL_FIELDS = {"ego_avg_speed": "ego_avg_speed", "ego_max_speed": "ego_max_speed",
                 "ego_distance_travelled": "ego_dist", "first_coll_tick": "first_coll_tick",
                 "rss_flags": "rss_flags", "tick": "tick", "t": "t"}


@dataclass
class ObsSpec:
    """What each agent observes (include/sg_b200.h, SgEnvSpec): ``k_neighbours`` (0..32) nearest present
    entities within ``radius`` metres (<= 0: no cut-off), its own trajectory ``lookahead`` seconds ahead
    (at most 8 times), with ``road`` whether it is on the driveable surface and how far its edge is, and with
    ``lidar_rays`` = R (0..256) a planar lidar: R rays at angles 2 pi k / R from its heading, each reading the
    distance to the first box of another present entity, at most ``lidar_range`` metres.  With ``map_edges`` = Km
    (0..32) it also sees the Km road-network edges (of the driveable, walkable and impenetrable surfaces) nearest to
    it within ``map_radius`` metres: the nearest point and both end points in its frame, which surfaces the edge
    bounds, and a valid flag (10 floats each, between the road block and the lidar).  With ``raster_size`` = S
    (0, or a multiple of 32 in 32..256) each agent also gets a bird's-eye raster, uint8 [5, S, S] of 0 / 1 in
    ``info["raster"]``, kept out of the observation rows: ``raster_resolution`` metres per pixel, centred
    ``raster_ahead`` metres ahead of the agent, row 0 ahead and column 0 to the left, with channels
    ``VecScenarioEnv.raster_channels`` (include/sg_b200.h, SgRasterSpec)."""
    k_neighbours: int = 8
    radius: float = 50.0
    lookahead: Sequence[float] = (1.0, 2.0, 3.0)
    road: bool = False
    lidar_rays: int = 0
    lidar_range: float = 50.0
    map_edges: int = 0
    map_radius: float = 50.0
    raster_size: int = 0
    raster_resolution: float = 0.5
    raster_ahead: float = 0.0

    @property
    def n_features(self) -> int:
        return abi.env_n_features(int(self.k_neighbours), len(self.lookahead), bool(self.road),
                                  int(self.lidar_rays), int(self.map_edges))


@dataclass
class ResetSpec:
    """Randomised episode starts of a ``VecScenarioEnv`` (include/sg_b200.h, sg_reset_scenarios_init).  Every
    reset, the auto-reset in ``step()`` included, starts scenario n at t0 + u * window[n], u uniform in [0, 1),
    window[n] = min(``start_offset``, ``env.start_window[n]``): the longest delay that keeps every vehicle of the
    log present and leaves ``min_remaining`` seconds of it.  Each agent's start is then moved by N(0, std)
    noise: ``lon`` / ``lat`` metres along / across its heading, ``heading`` radians and ``speed`` m/s (the speed
    is kept >= 0 and the velocity turns with the heading).  The draws are a pure function of ``seed``, the
    scenario, the agent and the scenario's episode count, so a seeded sequence of episodes repeats.  A start
    whose box overlaps another entity's collides at the first tick; nothing rejects it."""
    start_offset: float = 0.0
    min_remaining: float = 1.0
    lon: float = 0.0
    lat: float = 0.0
    heading: float = 0.0
    speed: float = 0.0
    seed: int = 0

    def __post_init__(self):
        for name in ("start_offset", "min_remaining", "lon", "lat", "heading", "speed"):
            v = getattr(self, name)
            if isinstance(v, bool) or not isinstance(v, (int, float)) or not (math.isfinite(v) and v >= 0.0):
                raise ValueError(f"ResetSpec.{name} must be a finite number >= 0, got {v!r}")
        if isinstance(self.seed, bool) or not isinstance(self.seed, (int, np.integer)):
            raise ValueError(f"ResetSpec.seed must be an int, got {self.seed!r}")


def _ego_policy(scenario: Scenario, entity: Entity):
    """Default ``create_agent`` of the env: the ego is driven by the policy, everything else is replayed."""
    return PolicyAgent(entity) if entity is scenario.ego else None


class VecScenarioEnv:
    """
    N scenarios stepped together; agent ``a`` of scenario ``n`` is the ``a``-th ``PolicyAgent`` of that
    scenario (``agent_slots`` / ``agent_entities(n)``), ``A`` the most any scenario has (the others are padded:
    zero observations, ``agent_mask`` 0, actions ignored).

    The batch is lowered by ``ScenarioGym`` and must run entirely on the device: host-side agents or
    policies, custom ``Metric`` / ``StateCallback`` classes (``RSSDistances`` is on the device), callable
    terminal conditions and ``record=True`` raise ``NotImplementedError``, as do ``ActionTableAgent`` /
    ``RandomActionAgent`` (their tables are indexed from the start of a rollout, not per episode).  Scenario
    actions (``UpdateStateVariableAction``) only write host-side entity state and are not applied here.

    ``step()`` returns the env's own buffers (overwritten by the next step; clone what you keep):
    ``obs`` [N, A, F] fp32, ``reward`` [N, A] fp32, ``terminated`` / ``truncated`` [N] bool.  A scenario that
    finishes is reset in the same step: ``obs`` holds the first observation of its next episode,
    ``info["final_obs"]`` the observation it finished with, ``info["final"]`` its episode results (rows of
    scenarios that did not finish hold their running values).

    ``reset_spec`` (a ``ResetSpec``): every reset, the auto-reset included, starts at a drawn time inside the log
    with the agents' starts perturbed (``sg_reset_scenarios_init``); ``start_window`` [N] fp64 holds the longest
    delay after t0 each scenario allows (every vehicle of the log still present, ``min_remaining`` seconds left).
    A pedestrian starting later restarts at the first point of its route, as at t0: routes are not re-targeted.

    With ``ObsSpec(raster_size=S)`` every agent also gets a bird's-eye raster (``sg_env_raster``): ``reset()`` and
    ``step()`` return ``info["raster"]`` uint8 [N, A, 5, S, S] (channels ``raster_channels``), and ``step()``
    ``info["final_raster"]``, the raster of the state each scenario ended the step in, before its reset.
    """

    def __init__(self, scenarios: List[Scenario], create_agent: Callable = _ego_policy,
                 timestep: float = 1.0 / 30.0, terminal_conditions: Optional[List[Union[str, Callable]]] = None,
                 state_callbacks: Optional[List[StateCallback]] = None, obs: Optional[ObsSpec] = None,
                 reward_weights: Optional[Union[Mapping[str, float], Sequence[float]]] = None,
                 device: Union[int, str, torch.device] = 0, record: bool = False,
                 reset_spec: Optional[ResetSpec] = None):
        if reset_spec is not None and not isinstance(reset_spec, ResetSpec):
            raise ValueError(f"reset_spec must be a ResetSpec or None, got {type(reset_spec).__name__}")
        if record:
            raise NotImplementedError("VecScenarioEnv keeps no pose trace (record=True needs ScenarioGym)")
        terminal_conditions = ["max_length"] if terminal_conditions is None else list(terminal_conditions)
        if any(callable(c) for c in terminal_conditions):
            raise NotImplementedError("callable terminal conditions run on the host: not available in the env")
        state_callbacks = list(state_callbacks or [])
        if any(not isinstance(cb, RSSDistances) for cb in state_callbacks):
            raise NotImplementedError("the env runs RSSDistances only (custom StateCallbacks run on the host)")
        self.obs_spec = obs if obs is not None else ObsSpec()
        if not 0 <= int(self.obs_spec.k_neighbours) <= 32 or len(self.obs_spec.lookahead) > 8:
            raise ValueError("ObsSpec: k_neighbours must be in 0..32 and lookahead have at most 8 times")
        R = int(self.obs_spec.lidar_rays)
        if not 0 <= R <= 256:
            raise ValueError(f"ObsSpec: lidar_rays must be in 0..256, got {self.obs_spec.lidar_rays}")
        if R > 0 and not (math.isfinite(float(self.obs_spec.lidar_range)) and float(self.obs_spec.lidar_range) > 0):
            raise ValueError(f"ObsSpec: lidar_range must be finite and > 0, got {self.obs_spec.lidar_range}")
        Km = int(self.obs_spec.map_edges)
        if Km != self.obs_spec.map_edges or not 0 <= Km <= 32:
            raise ValueError(f"ObsSpec: map_edges must be in 0..32, got {self.obs_spec.map_edges}")
        if Km > 0 and not (math.isfinite(float(self.obs_spec.map_radius)) and float(self.obs_spec.map_radius) > 0):
            raise ValueError(f"ObsSpec: map_radius must be finite and > 0, got {self.obs_spec.map_radius}")
        S = self.obs_spec.raster_size
        if isinstance(S, bool) or int(S) != S or not (S == 0 or (32 <= S <= 256 and int(S) % 32 == 0)):
            raise ValueError(f"ObsSpec: raster_size must be 0 or a multiple of 32 in 32..256, got {S}")
        S = int(S)
        if S > 0 and not (math.isfinite(float(self.obs_spec.raster_resolution))
                          and float(self.obs_spec.raster_resolution) > 0):
            raise ValueError(f"ObsSpec: raster_resolution must be finite and > 0, got {self.obs_spec.raster_resolution}")
        if S > 0 and not math.isfinite(float(self.obs_spec.raster_ahead)):
            raise ValueError(f"ObsSpec: raster_ahead must be finite, got {self.obs_spec.raster_ahead}")
        w = dict(DEFAULT_REWARD_WEIGHTS)
        if isinstance(reward_weights, Mapping):
            unknown = set(reward_weights) - set(abi.ENV_TERMS)
            if unknown:
                raise ValueError(f"unknown reward terms {sorted(unknown)}; known: {abi.ENV_TERMS}")
            w.update(reward_weights)
        elif reward_weights is not None:
            if len(reward_weights) != len(abi.ENV_TERMS):
                raise ValueError(f"reward_weights needs {len(abi.ENV_TERMS)} values {abi.ENV_TERMS}")
            w = dict(zip(abi.ENV_TERMS, reward_weights))
        self.reward_weights = w

        dev_index = device if isinstance(device, int) else (torch.device(device).index or 0)
        gym = ScenarioGym(timestep=timestep, terminal_conditions=terminal_conditions,
                          state_callbacks=state_callbacks, device=dev_index)
        gym.set_scenarios(list(scenarios), create_agent=create_agent)
        if gym._host_mode:
            raise NotImplementedError("the batch has host-side agents / policies: they cannot run in the env")
        if gym._action_table is not None or gym._action_rng is not None:
            raise NotImplementedError("ActionTableAgent / RandomActionAgent cannot run in the env")
        self._gym = gym
        eng = self._engine = gym._engine
        # the reward and info["final"] read the collision book-keeping and the ego metrics
        eng.params.features |= abi.FEAT_COLLISIONS | abi.FEAT_EGO_METRICS
        self.device = eng.device
        N, M = eng.N, eng.M
        self.N = N
        self.A = max(len(s) for s in gym._env_slots)
        if self.A == 0:
            raise ValueError("no PolicyAgent in any scenario: nothing for a policy to drive")
        slots = np.full((N, self.A), -1, np.int32)
        for n, ss in enumerate(gym._env_slots):
            slots[n, : len(ss)] = ss
        self._slots_host = slots
        src = np.nonzero(slots.reshape(-1) >= 0)[0]
        dst = (src // self.A) * M + slots.reshape(-1)[src]
        dev = self.device

        def zeros(*shape, dtype=torch.float32):
            return torch.zeros(shape, dtype=dtype, device=dev)

        self.agent_slots = torch.from_numpy(slots).to(dev)
        self._src = torch.from_numpy(src.astype(np.int64)).to(dev)
        self._dst = torch.from_numpy(dst.astype(np.int64)).to(dev)
        self._act = {torch.float32: zeros(1, 2, N * M), torch.float64: zeros(1, 2, N * M, dtype=torch.float64)}
        F = self.obs_spec.n_features
        self.n_features = F
        self._obs, self._final_obs = zeros(N, self.A, F), zeros(N, self.A, F)
        self._agent_mask = zeros(N, self.A, dtype=torch.uint8)
        self._reward, self._terms = zeros(N, self.A), zeros(N, self.A, len(abi.ENV_TERMS))
        self._terminated, self._truncated = zeros(N, dtype=torch.uint8), zeros(N, dtype=torch.uint8)
        self._finished = zeros(N, dtype=torch.uint8)
        self._episode = zeros(N, dtype=torch.int64)
        self._resets = 0  # reset() calls so far
        self._final = {k: torch.zeros_like(eng.tensor(f)) for k, f in _FINAL_FIELDS.items()}
        self._snap = {"snap_dist": zeros(N * self.A, dtype=torch.float64),
                      "snap_collided": zeros(N * self.A, dtype=torch.uint8),
                      "snap_pair_ticks": zeros(N, dtype=torch.int64), "snap_rss": zeros(N, dtype=torch.uint8)}
        spec = abi.SgEnvSpec()
        spec.n_agents, spec.k_neighbours = self.A, int(self.obs_spec.k_neighbours)
        spec.radius = float(self.obs_spec.radius)
        spec.n_lookahead, spec.road = len(self.obs_spec.lookahead), int(bool(self.obs_spec.road))
        for k, v in enumerate(self.obs_spec.lookahead):
            spec.lookahead[k] = float(v)
        for k, name in enumerate(abi.ENV_TERMS):
            spec.weights[k] = float(w[name])
        spec.agent_slot = self.agent_slots.data_ptr()
        spec.n_rays, spec.ray_range = R, float(self.obs_spec.lidar_range)
        # the lidar's ray directions, built once from numpy's values (the env keeps the tensor alive)
        self._ray_dir = torch.from_numpy(abi.lidar_directions(R)).to(dev) if R > 0 else None
        if R > 0:
            spec.ray_dir = self._ray_dir.data_ptr()
        spec.map_edges, spec.map_radius = Km, float(self.obs_spec.map_radius)
        # the map table and its grid, built once per network from the lowered scene (the env keeps them alive)
        self._map = {}
        if Km > 0:
            sc = eng.scene
            spec.map_networks = sc.n_networks
            if sc.n_networks > 0:
                table = abi.map_table(sc.rn_poly_off, sc.rn_edge_off, sc.rn_edges, spec.map_radius)
                for k, a in table.items():  # (an empty array still gets an address)
                    a = a if a.size else np.zeros((1,) + a.shape[1:], a.dtype)
                    self._map[k] = torch.from_numpy(np.ascontiguousarray(a)).to(dev)
                    setattr(spec, k, self._map[k].data_ptr())
        for k, t in self._snap.items():
            setattr(spec, k, t.data_ptr())
        self._spec = spec
        self._info = {"agent_mask": self._agent_mask, "episode_step": eng.tensor("tick"), "episode": self._episode}

        # the raster (sg_env_raster): its buffers and the polygons' bounding boxes, built once
        self.raster_channels = abi.RASTER_CHANNELS
        self._raster = self._final_raster = None
        if S > 0:
            sc = eng.scene
            rspec = abi.SgRasterSpec()
            rspec.size, rspec.n_networks = S, sc.n_networks
            rspec.resolution, rspec.ahead = float(self.obs_spec.raster_resolution), float(self.obs_spec.raster_ahead)
            box, rspec.margin = abi.raster_poly_boxes(sc.rn_edge_off, sc.rn_edges,
                                                      abi.raster_half_diagonal(S, rspec.resolution))
            self._poly_box = torch.from_numpy(box if len(box) else np.zeros((1, 4))).to(dev)
            rspec.poly_box = self._poly_box.data_ptr()
            self._rspec = rspec
            self._raster = zeros(N, self.A, 5, S, S, dtype=torch.uint8)
            self._final_raster = zeros(N, self.A, 5, S, S, dtype=torch.uint8)
            self._info["raster"] = self._raster

        # episode starts (sg_reset_scenarios_init): the valid windows are decided once, on the host
        self.reset_spec = reset_spec
        rs = reset_spec if reset_spec is not None else ResetSpec()
        win = abi.start_windows(eng.scene, bool(eng.params.persist), rs.min_remaining)
        self.start_window = torch.from_numpy(win).to(dev)
        self._draw_window = torch.from_numpy(np.minimum(win, float(rs.start_offset))).to(dev)
        self._t_start = zeros(N, dtype=torch.float64)
        self._counter = zeros(N, dtype=torch.int64)
        perturb = np.zeros(N * M, np.uint8)
        perturb[dst] = 1
        self._perturb = torch.from_numpy(perturb).to(dev)
        self._init = abi.SgResetInit()  # draws the start (reset() and step())
        self._init.start_window = self._draw_window.data_ptr()
        self._init.counter = self._counter.data_ptr()
        if reset_spec is not None:
            self._init.perturb = self._perturb.data_ptr()
            for k, v in enumerate((rs.lon, rs.lat, rs.heading, rs.speed)):
                self._init.sigma[k] = float(v)
        self._init.seed = int(rs.seed) & (2**64 - 1)
        self._init_at = abi.SgResetInit.from_buffer_copy(self._init)  # starts at the times of reset(start_time)
        self._init_at.t_start = self._t_start.data_ptr()

    # ------------------------------------------------------------------ API
    def agent_entities(self, n: int) -> List[Entity]:
        """The entities behind agents 0 .. of scenario ``n`` (shorter than ``A`` where the row is padded)."""
        ents = self._gym._entity_of[n]
        return [ents[s] for s in self._gym._env_slots[n]]

    def branches(self, B: int, H: int, final_obs: bool = False) -> "BranchRollout":
        """
        A ``BranchRollout`` of ``B`` branches over ``H`` ticks from this env's current state (see there).
        Everything it needs is allocated here, once.
        """
        return BranchRollout(self, B, H, final_obs)

    def planner(self, B: int = 64, H: int = 30, sigma: Sequence[float] = (1.0, 0.1), temperature: float = 1.0,
                iterations: int = 1, seed: int = 0) -> "MPPIPlanner":
        """An ``MPPIPlanner`` over ``B`` branches of ``H`` ticks from this env (see there).  Everything it needs is
        allocated here, once."""
        return MPPIPlanner(self, B, H, sigma, temperature, iterations, seed)

    def reset(self, seed: Optional[int] = None, start_time: Optional[torch.Tensor] = None
              ) -> Tuple[torch.Tensor, Dict[str, torch.Tensor]]:
        """
        Every scenario back to its start and observed; episode counters restart at 0.  Without a ``ResetSpec``
        the start is the log's (sg_reset), with one it is drawn as the spec says.  ``seed``: the draws' seed from
        now on, with every scenario's draw count back at 0, so the same seed replays the same episodes.
        ``start_time`` (fp64 [N] on the env's device, with or without a spec): start scenario n that many seconds
        after its t0, clamped on the device to [0, ``start_window[n]``] (NaN counts as 0); a spec's perturbation
        still applies.
        """
        eng = self._engine
        if seed is not None:
            if isinstance(seed, bool) or not isinstance(seed, (int, np.integer)):
                raise ValueError(f"seed must be an int, got {seed!r}")
            self._init.seed = self._init_at.seed = int(seed) & (2**64 - 1)
            self._counter.zero_()
        if start_time is not None:
            if not isinstance(start_time, torch.Tensor) or tuple(start_time.shape) != (self.N,) \
                    or start_time.dtype != torch.float64 or start_time.device != self.device:
                raise ValueError(f"start_time must be a float64 tensor of shape ({self.N},) on {self.device}")
            torch.nan_to_num(start_time, nan=0.0, out=self._t_start)
            torch.clamp(self._t_start, min=0.0, out=self._t_start)
            torch.minimum(self._t_start, self.start_window, out=self._t_start)
            self._t_start.add_(eng._scene_t["t0"])
            init = self._init_at
        else:
            init = self._init if self.reset_spec is not None else None
        if init is None:
            eng.reset()
        else:
            eng.reset(init=init)
            eng.tensor("event_count").zero_()  # (as sg_reset)
            self._counter.add_(1)
        self._episode.zero_()
        self._resets += 1  # (a planner cannot see this reset in the episode counters when they were 0)
        eng.env_observe(self._spec, self._obs, self._agent_mask)
        if self._raster is not None:
            eng.env_raster(self._spec, self._rspec, self._raster)
        return self._obs, dict(self._info)

    def step(self, actions: torch.Tensor):
        """
        One tick of every scenario with the policy's ``actions`` [N, A, 2] (accel, steer; fp32 or fp64, on the
        env's device).  Returns ``(obs, reward, terminated, truncated, info)``; see the class docstring.
        """
        if not isinstance(actions, torch.Tensor):
            raise ValueError("actions must be a torch.Tensor [N, A, 2]")
        if tuple(actions.shape) != (self.N, self.A, 2):
            raise ValueError(f"actions must have shape ({self.N}, {self.A}, 2), got {tuple(actions.shape)}")
        if actions.dtype not in self._act:
            raise ValueError(f"actions must be float32 or float64, got {actions.dtype}")
        if actions.device != self.device:
            raise ValueError(f"actions must be on {self.device}, got {actions.device}")
        eng = self._engine
        buf = self._act[actions.dtype]
        vals = actions.reshape(self.N * self.A, 2).index_select(0, self._src)
        buf[0].index_copy_(1, self._dst, vals.t())
        eng.rollout(1, actions=buf)
        eng.env_reward(self._spec, self._reward, self._terms, self._terminated, self._truncated)
        eng.env_observe(self._spec, self._obs, self._agent_mask)
        self._final_obs.copy_(self._obs)
        if self._raster is not None:
            eng.env_raster(self._spec, self._rspec, self._raster)
            self._final_raster.copy_(self._raster)
        for k, f in _FINAL_FIELDS.items():
            self._final[k].copy_(eng.tensor(f))
        torch.bitwise_or(self._terminated, self._truncated, out=self._finished)
        if self.reset_spec is None:
            eng.reset(mask=self._finished)
        else:
            eng.reset(mask=self._finished, init=self._init)
            self._counter.add_(self._finished)
        eng.env_observe(self._spec, self._obs, self._agent_mask, mask=self._finished)
        if self._raster is not None:
            eng.env_raster(self._spec, self._rspec, self._raster, mask=self._finished)
        self._episode.add_(self._finished)
        eng.tensor("event_count").zero_()  # ego collision events are not kept across steps
        info = dict(self._info, final_obs=self._final_obs, final=self._final, terms=self._terms)
        if self._raster is not None:
            info["final_raster"] = self._final_raster
        return self._obs, self._reward, self._terminated.view(torch.bool), self._truncated.view(torch.bool), info


def branch_scatter_index(slots: np.ndarray, M: int, B: int, H: int) -> np.ndarray:
    """
    Where ``index_copy_`` puts each element of a contiguous ``actions [N, B, H, A, 2]`` in the flat branch action
    table ``[B][H][2][N*M]`` (plus one trailing element): element (n, b, h, a, c) goes to
    ``((b*H + h)*2 + c)*N*M + n*M + slots[n, a]``, padding agents (slot -1) to the trailing element, which no
    rollout reads.  The env's ``_src`` / ``_dst`` scatter of one step, extended over B and H.
    """
    slots = np.asarray(slots, np.int64)
    N, A = slots.shape
    NM = N * M
    n = np.arange(N).reshape(N, 1, 1, 1, 1)
    b = np.arange(B).reshape(1, B, 1, 1, 1)
    h = np.arange(H).reshape(1, 1, H, 1, 1)
    c = np.arange(2).reshape(1, 1, 1, 1, 2)
    s = slots.reshape(N, 1, 1, A, 1)
    idx = ((b * H + h) * 2 + c) * NM + n * M + s
    idx = np.where(s >= 0, idx, B * H * 2 * NM)
    return np.array(np.broadcast_to(idx, (N, B, H, A, 2))).reshape(-1)


class BranchRollout:
    """
    Branched look-ahead rollouts from a ``VecScenarioEnv``'s live state: ``run(actions)`` forks the env's state
    (and the snapshot its next reward compares against) into ``B`` branch states in one device pass
    (``sg_fork_state``), rolls branch ``b`` out for ``H`` ticks with the fused rollout, consuming
    ``actions[:, b]``, and scores every branch against the state at the fork.  This is what sampling-based
    planners (random shooting, CEM, MPPI) and counterfactual questions ("would any of these manoeuvres have
    avoided the collision?") need, at the cost of B x H fused ticks instead of B x H env steps.

    Horizon semantics: ``sg_env_reward`` evaluated once, after the H ticks, against the state at the fork:
      progress   dist_H - dist_0
      collision  collided rose at any tick of the horizon (it is sticky)
      off_road / tracking   at the end state (a branch that finished is frozen where it finished)
      rss        rss_flags gained a bit over the horizon
      terminated / truncated   how a branch that finished within the horizon finished (both 0 otherwise)
    This is not the sum of per-tick rewards.  With H = 1 it is exactly what ``env.step`` computes.  Branches
    stop where their scenario finishes: ``ticks`` says how many ticks each advanced.

    ``run()`` enqueues everything on the current stream, with no host synchronisation and no device allocation
    (an ``actions`` tensor that is not contiguous is copied first), and does not touch the env's state, snapshot,
    observations or episode counters.  It returns views into this object's buffers (overwritten by the next
    ``run()``), in ``[N, B, ...]`` order, permuted views of ``[B, N, ...]`` storage:
      ``reward`` [N, B, A] fp32, ``terms`` [N, B, A, 5] fp32, ``terminated`` / ``truncated`` [N, B] bool,
      ``ticks`` [N, B] int32, ``agent_mask`` [N, B, A] uint8 (the agent is present at the end of the branch),
      ``final_obs`` [N, B, A, F] fp32 (the observation at the end of the branch, with ``final_obs=True``).
    """

    def __init__(self, env: VecScenarioEnv, B: int, H: int, final_obs: bool = False):
        if int(B) != B or int(H) != H or B < 1 or H < 1:
            raise ValueError(f"branches need B >= 1 and H >= 1, got B={B}, H={H}")
        B, H = int(B), int(H)
        src = env._engine
        # every env state can be forked: the env keeps no trace and sg_fork_state copies everything else
        assert src.trace_cap == 0, "VecScenarioEnv states have no trace"
        self.env, self.B, self.H, self.final_obs = env, B, H, bool(final_obs)
        N, A, M, F = env.N, env.A, src.M, env.n_features
        dev = env.device
        self._engines = [type(src).sharing_scene(src, event_cap=1024) for _ in range(B)]
        # flat action tables [B][H][2][N*M] + one element the padding agents are scattered into
        size = B * H * 2 * N * M
        self._flat = {dt: torch.zeros(size + 1, dtype=dt, device=dev) for dt in (torch.float32, torch.float64)}
        self._tables = {dt: [t[b * H * 2 * N * M:(b + 1) * H * 2 * N * M].view(H, 2, N * M) for b in range(B)]
                        for dt, t in self._flat.items()}
        self._index = torch.from_numpy(branch_scatter_index(env._slots_host, M, B, H)).to(dev)
        # the branches' SgEnvSpecs: the env's, with snapshot arrays of their own
        self._snaps, self._specs = [], []
        for _ in range(B):
            snap = {k: torch.zeros_like(t) for k, t in env._snap.items()}
            spec = abi.SgEnvSpec.from_buffer_copy(env._spec)
            for k, t in snap.items():
                setattr(spec, k, t.data_ptr())
            self._snaps.append(snap)
            self._specs.append(spec)
        self._fork_args = src.fork_args(self._engines, env._spec, self._specs)

        def zeros(*shape, dtype=torch.float32):
            return torch.zeros(shape, dtype=dtype, device=dev)

        self._reward, self._terms = zeros(B, N, A), zeros(B, N, A, len(abi.ENV_TERMS))
        self._terminated, self._truncated = zeros(B, N, dtype=torch.uint8), zeros(B, N, dtype=torch.uint8)
        self._ticks = zeros(B, N, dtype=torch.int32)
        self._agent_mask = zeros(B, N, A, dtype=torch.uint8)
        self._final_obs = zeros(B, N, A, F) if self.final_obs else None
        slots = env._slots_host
        self._present_idx = torch.from_numpy(
            (np.arange(N)[:, None] * M + np.maximum(slots, 0)).reshape(-1).astype(np.int64)).to(dev)
        self._valid = torch.from_numpy((slots >= 0).reshape(-1).astype(np.uint8)).to(dev)
        out = {"reward": self._reward.permute(1, 0, 2), "terms": self._terms.permute(1, 0, 2, 3),
               "terminated": self._terminated.view(torch.bool).t(), "truncated": self._truncated.view(torch.bool).t(),
               "ticks": self._ticks.t(), "agent_mask": self._agent_mask.permute(1, 0, 2)}
        if self.final_obs:
            out["final_obs"] = self._final_obs.permute(1, 0, 2, 3)
        self._out = out

    @property
    def engines(self):
        """The B branch engines (their state is the end state of the last ``run()``)."""
        return list(self._engines)

    def run(self, actions: torch.Tensor) -> Dict[str, torch.Tensor]:
        """
        Fork, roll every branch ``H`` ticks and score it; ``actions`` [N, B, H, A, 2] (accel, steer; fp32 or
        fp64, on the env's device): branch ``b`` consumes ``actions[:, b, h]`` at its h-th tick.  Returns the
        views described in the class docstring.
        """
        env = self.env
        shape = (env.N, self.B, self.H, env.A, 2)
        if not isinstance(actions, torch.Tensor):
            raise ValueError(f"actions must be a torch.Tensor {list(shape)}")
        if tuple(actions.shape) != shape:
            raise ValueError(f"actions must have shape {shape}, got {tuple(actions.shape)}")
        if actions.dtype not in self._flat:
            raise ValueError(f"actions must be float32 or float64, got {actions.dtype}")
        if actions.device != env.device:
            raise ValueError(f"actions must be on {env.device}, got {actions.device}")
        self._flat[actions.dtype].index_copy_(0, self._index, actions.reshape(-1))
        self._roll(self._tables[actions.dtype])
        return dict(self._out)

    def _roll(self, tables: List[torch.Tensor]) -> None:
        """Fork, roll branch ``b`` ``H`` ticks on ``tables[b]`` ([H][2][N*M]) and score it into the buffers."""
        src = self.env._engine
        self._check(src.lib["fork_state"](*self._fork_args, src.dev_index, src._stream()))
        tick0 = src.tensor("tick")
        for b, eng in enumerate(self._engines):
            eng.rollout(self.H, actions=tables[b])
            eng.env_reward(self._specs[b], self._reward[b], self._terms[b], self._terminated[b], self._truncated[b])
            torch.sub(eng.tensor("tick"), tick0, out=self._ticks[b])
            if self.final_obs:
                eng.env_observe(self._specs[b], self._final_obs[b], self._agent_mask[b])
            else:
                mask = self._agent_mask[b].view(-1)
                torch.index_select(eng.tensor("present"), 0, self._present_idx, out=mask)
                mask.mul_(self._valid)

    def _check(self, rc: int):
        self.env._engine._check(rc)


class MPPIPlanner:
    """
    MPPI (model-predictive path integral) planning on the device, over a ``BranchRollout`` of ``B`` branches and
    ``H`` ticks: ``plan()`` repeats ``iterations`` times
      sample   ``sg_plan_sample`` draws branch b's actions, mean + sigma * N(0, 1) (branch 0: the mean itself),
               straight into the branch action table (no [N, B, H, A, 2] tensor, no scatter);
      roll     fork the env's state, roll every branch H ticks and score it (``BranchRollout``'s horizon reward);
      update   ``sg_plan_update`` moves the mean to the average of the branches weighted by
               exp((R_b - max R) / temperature), reading the noise back from the same table (it is never stored),
    per agent and independently.  The last update also returns the first action of the refined mean and shifts the
    mean one tick for the next ``plan()`` (its last tick starts at 0).  The mean of a scenario whose episode
    changed since the last ``plan()`` (auto-reset in ``env.step``, or ``env.reset()``) restarts at 0.  Semantics:
    include/sg_b200.h, sg_plan_sample / sg_plan_update.

    The noise is a pure function of (seed, agent, branch, tick, call counter), so two planners with the same seed
    driving equal envs plan the same actions.  ``plan()`` enqueues everything on the current stream, with no host
    synchronisation and no allocation, and leaves the env's state, snapshot, observations and episode counters
    alone.  Each agent plans for its own reward (there is no scenario-level objective), and actions are bounded
    only by the controller's clipping.
    """

    def __init__(self, env: VecScenarioEnv, B: int = 64, H: int = 30, sigma: Sequence[float] = (1.0, 0.1),
                 temperature: float = 1.0, iterations: int = 1, seed: int = 0):
        if int(B) != B or B < 2:
            raise ValueError(f"the planner needs B >= 2 branches (branch 0 is the mean), got B={B}")
        if int(H) != H or H < 1:
            raise ValueError(f"the planner needs H >= 1, got H={H}")
        if int(iterations) != iterations or iterations < 1:
            raise ValueError(f"iterations must be >= 1, got {iterations}")
        sigma = tuple(float(s) for s in sigma)
        if len(sigma) != 2 or not all(math.isfinite(s) and s >= 0.0 for s in sigma):
            raise ValueError(f"sigma must be two finite values >= 0 (accel, steer), got {sigma}")
        temperature = float(temperature)
        if not (math.isfinite(temperature) and temperature > 0.0):
            raise ValueError(f"temperature must be finite and > 0, got {temperature}")
        self.env, self.B, self.H = env, int(B), int(H)
        self.sigma, self.temperature, self.iterations, self.seed = sigma, temperature, int(iterations), int(seed)
        self.branches = BranchRollout(env, self.B, self.H)
        br, N, A, dev = self.branches, env.N, env.A, env.device
        # the table type the branch rollouts consume without a conversion
        dt = torch.float64 if br._engines[0]._wants_f64_table() else torch.float32
        self._table, self._tables = br._flat[dt], br._tables[dt]
        self._mean = torch.zeros(2, N, self.H, A, 2, dtype=torch.float64, device=dev)  # ping-pong
        self._cur = 0
        self._action = torch.zeros(N, A, 2, device=dev)
        self._best_branch = torch.zeros(N, A, dtype=torch.int32, device=dev)
        self._best_reward = torch.zeros(N, A, device=dev)
        self._seen = env._episode.clone()
        self._resets = env._resets
        self._changed = torch.zeros(N, dtype=torch.bool, device=dev)
        self._all = torch.ones(N, dtype=torch.uint8, device=dev)
        self._k = 0  # sample passes so far: the noise counter

    def plan(self) -> Tuple[torch.Tensor, Dict[str, torch.Tensor]]:
        """
        One planning step from the env's current state.  Returns views into the planner's buffers (overwritten by
        the next ``plan()``): ``actions`` [N, A, 2] fp32, the first action of the refined mean, and ``info`` with
        ``mean`` [N, H, A, 2] fp64 (the refined mean shifted one tick: where the next ``plan()`` starts),
        ``reward`` [N, B, A] (the branch rewards of the last iteration), ``best_branch`` [N, A] int32 and
        ``best_reward`` [N, A] fp32 (the smallest b with the largest reward, and that reward).
        """
        env, br, B, H = self.env, self.branches, self.B, self.H
        eng, spec = env._engine, env._spec
        if self._resets != env._resets:
            self._resets = env._resets
            reset = self._all
        else:
            reset = torch.ne(env._episode, self._seen, out=self._changed)
        self._seen.copy_(env._episode)
        for it in range(self.iterations):
            mu = self._mean[self._cur]
            eng.plan_sample(spec, B, H, self.seed, self._k, self.sigma, mu, reset if it == 0 else None, self._table)
            self._k += 1
            br._roll(self._tables)
            self._cur ^= 1
            last = it == self.iterations - 1
            eng.plan_update(spec, B, H, self.temperature, br._reward, self._table, mu, self._mean[self._cur], last,
                            self._action if last else None, self._best_branch, self._best_reward)
        info = {"mean": self._mean[self._cur], "reward": br._out["reward"], "best_branch": self._best_branch,
                "best_reward": self._best_reward}
        return self._action, info
