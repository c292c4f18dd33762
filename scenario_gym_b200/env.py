"""
``VecScenarioEnv`` -- a closed-loop, batched environment on the device: a policy chooses every step's
VehicleActions from observations, and observations, rewards, termination and the reset of finished
scenarios are all computed by the library's kernels (``sg_env_observe``, ``sg_env_reward``,
``sg_reset_scenarios``; semantics in ``include/sg_b200.h``).  ``step()`` and ``reset()`` enqueue their work
on the current CUDA stream with no per-scenario Python and no device -> host synchronisation; every buffer
is allocated once, when the env is built.
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
    distance to the first box of another present entity, at most ``lidar_range`` metres."""
    k_neighbours: int = 8
    radius: float = 50.0
    lookahead: Sequence[float] = (1.0, 2.0, 3.0)
    road: bool = False
    lidar_rays: int = 0
    lidar_range: float = 50.0

    @property
    def n_features(self) -> int:
        return abi.env_n_features(int(self.k_neighbours), len(self.lookahead), bool(self.road),
                                  int(self.lidar_rays))


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
    """

    def __init__(self, scenarios: List[Scenario], create_agent: Callable = _ego_policy,
                 timestep: float = 1.0 / 30.0, terminal_conditions: Optional[List[Union[str, Callable]]] = None,
                 state_callbacks: Optional[List[StateCallback]] = None, obs: Optional[ObsSpec] = None,
                 reward_weights: Optional[Union[Mapping[str, float], Sequence[float]]] = None,
                 device: Union[int, str, torch.device] = 0, record: bool = False):
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
        for k, t in self._snap.items():
            setattr(spec, k, t.data_ptr())
        self._spec = spec
        self._info = {"agent_mask": self._agent_mask, "episode_step": eng.tensor("tick"), "episode": self._episode}

    # ------------------------------------------------------------------ API
    def agent_entities(self, n: int) -> List[Entity]:
        """The entities behind agents 0 .. of scenario ``n`` (shorter than ``A`` where the row is padded)."""
        ents = self._gym._entity_of[n]
        return [ents[s] for s in self._gym._env_slots[n]]

    def reset(self) -> Tuple[torch.Tensor, Dict[str, torch.Tensor]]:
        """Every scenario back to its start (sg_reset) and observed; episode counters restart at 0."""
        eng = self._engine
        eng.reset()
        self._episode.zero_()
        eng.env_observe(self._spec, self._obs, self._agent_mask)
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
        for k, f in _FINAL_FIELDS.items():
            self._final[k].copy_(eng.tensor(f))
        torch.bitwise_or(self._terminated, self._truncated, out=self._finished)
        eng.reset(mask=self._finished)
        eng.env_observe(self._spec, self._obs, self._agent_mask, mask=self._finished)
        self._episode.add_(self._finished)
        eng.tensor("event_count").zero_()  # ego collision events are not kept across steps
        info = dict(self._info, final_obs=self._final_obs, final=self._final, terms=self._terms)
        return self._obs, self._reward, self._terminated.view(torch.bool), self._truncated.view(torch.bool), info
