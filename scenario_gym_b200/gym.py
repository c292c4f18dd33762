"""
``ScenarioGym`` -- the reference's engine class (reference scenario_gym/scenario_gym.py:13-319)
on top of the B200 rollout engine.  Same constructor arguments and methods
(``load_scenario``, ``set_scenario``, ``reset_scenario``, ``step``, ``rollout``, ``get_metrics``,
``add_metrics``, ``run_scenarios``); in addition ``load_scenarios`` / ``set_scenarios`` take a
list and roll all of them out as one batch on the device.

Lowering: what ``create_agent`` returns decides each entity's device slot kind
  None                          -> batch replay            (entity/batch.py)
  ReplayTrajectoryAgent         -> clamped replay agent    (agent.py:118-128)
  ActionTableAgent              -> VehicleController, whole action table on device
  PolicyAgent                   -> VehicleController on device, actions from VecScenarioEnv.step (env only)
  Agent + VehicleController     -> VehicleController on device, policy ``_step`` on the host per tick
  PedestrianAgent + SocialForce -> social force on device
  any other Agent               -> pose from ``agent.step(state)`` on the host per tick
Built-in metrics / ``RSSDistances`` are accumulated on the device; custom ``Metric`` /
``StateCallback`` subclasses and callable terminal conditions run on the host after every tick
on a materialised ``State``.  A rollout without host-side plugins is a single fused launch.
"""
from __future__ import annotations

from copy import deepcopy
from typing import Any, Callable, Dict, List, Optional, Union

import numpy as np

from . import abi
from .entity import Entity
from .packing import ScenarioSpec, SlotSpec, pack_scenarios
from .plugins import (ActionTableAgent, Agent, CollisionMetric, EgoLocalizationSensor, Metric,
                      PedestrianAgent, PIDAgent, PIDController, PolicyAgent, RandomActionAgent, ReplayTrajectoryAgent, ReplayTrajectoryController, RSSDistances,
                      SocialForce, StateCallback, VehicleAction, VehicleController, _create_agent,
                      _DeviceMetric)
from .scenario import Scenario
from .state import State
from .xosc import import_scenario, import_scenarios

_TERMINAL_BITS = {"max_length": abi.TERM_MAX_LENGTH, "collision": abi.TERM_COLLISION,
                  "ego_collision": abi.TERM_EGO_COLLISION, "ego_off_road": abi.TERM_EGO_OFF_ROAD}


class ScenarioGym:
    """Loads and runs scenarios."""

    @classmethod
    def run_scenarios(cls, paths: List[str], render: bool = False, **kwargs) -> "ScenarioGym":
        """
        Reference scenario_gym.py:16-27 loads and rolls the paths out one by one; here they are
        ingested together and rolled out as ONE device batch (scenarios are independent).
        """
        gym = cls(**kwargs)
        gym.load_scenarios(list(paths))
        gym.rollout(render=render)
        return gym

    def __init__(self, timestep: float = 1.0 / 30.0, persist: bool = False, viewer_class=None,
                 terminal_conditions: Optional[List[Union[str, Callable]]] = None,
                 state_callbacks: Optional[List[StateCallback]] = None,
                 metrics: Optional[List[Metric]] = None, device: int = 0, record: bool = False,
                 **viewer_parameters):
        self.timestep = timestep
        self.persist = persist
        self.device = device
        # record=True keeps a device-side trace of every tick's poses so that
        # state.recorded_poses() / state.to_scenario() also work after a fused rollout
        self.record = record
        self.viewer_parameters = viewer_parameters.copy()
        self.terminal_conditions = ["max_length"] if terminal_conditions is None else terminal_conditions
        self.state_callbacks = [] if state_callbacks is None else state_callbacks
        self.viewer = None
        self.states: List[State] = []
        self.metrics: List[Metric] = []
        self._engine = None
        if metrics is not None:
            self.add_metrics(metrics)

    # ------------------------------------------------------------------ reference API
    @property
    def state(self) -> Optional[State]:
        return self.states[0] if self.states else None

    def reset_gym(self) -> None:
        self.states = []
        self.metrics = []
        self._engine = None

    def add_metrics(self, metrics: List[Metric]) -> None:
        self.metrics.extend(metrics)

    def load_scenario(self, scenario_path: str, create_agent=_create_agent, relabel: bool = False,
                      **kwargs) -> None:
        if str(scenario_path).endswith(".json"):  # reference scenario_gym.py:145-146
            scenario = Scenario.from_json(scenario_path, **kwargs)
        else:
            scenario = import_scenario(scenario_path, relabel=relabel, **kwargs)
        self.set_scenario(scenario, scenario_path=scenario_path, create_agent=create_agent)

    def load_scenarios(self, scenario_paths: List[str], create_agent=_create_agent,
                       relabel: bool = False, workers: Optional[int] = None) -> None:
        """N scenario files as one device batch (batched ingest: xosc.import_scenarios)."""
        self.set_scenarios(import_scenarios(scenario_paths, relabel=relabel, workers=workers),
                           scenario_paths=scenario_paths, create_agent=create_agent)

    def set_scenario(self, scenario: Scenario, scenario_path: Optional[str] = None,
                     create_agent=_create_agent) -> None:
        self.set_scenarios([scenario], scenario_paths=[scenario_path], create_agent=create_agent)

    def set_scenarios(self, scenarios: List[Scenario], scenario_paths=None,
                      create_agent=_create_agent) -> None:
        paths = scenario_paths or [None] * len(scenarios)
        self.states = [State(self, n, sc, scenario_path=p) for n, (sc, p) in enumerate(zip(scenarios, paths))]
        self.create_agents(create_agent=create_agent)
        self._build()
        self.reset_scenario(force=True)

    def create_agents(self, create_agent=_create_agent) -> None:
        """Call ``create_agent(scenario, entity)`` once per entity (reference :188-211)."""
        for st in self.states:
            st.agents = {}
            for entity in st.scenario.entities:
                agent = create_agent(st.scenario, entity)
                if agent is not None:
                    st.agents[entity] = agent

    def get_start_time(self, scenario: Scenario) -> float:
        return max((0.0, scenario.ego.trajectory.min_t))

    def reset_scenario(self, force: bool = False) -> None:
        """Reset the state to the beginning of the scenario(s) (reference :217-225)."""
        if not self.states:
            return
        if not force and self._ticks_since_reset == 0:
            return
        self._sync_params()
        self._engine.reset()
        self._ticks_since_reset = 0
        self._epoch += 1
        self._cache = {}
        self._host_done = [False] * len(self.states)
        self._last_tick = np.zeros(len(self.states), np.int32)
        for n, st in enumerate(self.states):
            st._invalidate()
            st._recorded = {e: [] for e in st.scenario.entities}
            st.next_t = None
            st._reset_actions()
            st.update_actions()  # reference State.reset, state.py:136
        if self._host_mode:
            for n, st in enumerate(self.states):
                st._record()
                for cb in self._host_callbacks[n]:
                    cb.reset(st)
                for agent in st.agents.values():
                    if self._agent_kind[agent] in ("host", "host_policy"):
                        agent.reset(st)
                for m in self._host_metrics[n]:
                    m.reset(st)
        for m in self.metrics:
            if isinstance(m, _DeviceMetric):
                m._value = None

    def _refuse_env_agents(self) -> None:
        if getattr(self, "_any_env_policy", False):
            raise RuntimeError("the batch has PolicyAgents, whose actions come from a policy: "
                               "run it through VecScenarioEnv")

    def step(self) -> None:
        """One tick for every scenario that is not done (reference :227-254)."""
        self._refuse_env_agents()
        self._sync_params()
        eng = self._engine
        N, M = eng.N, eng.M
        actions = None
        host_pose = host_present = None
        if self._host_mode:
            if self._any_host_policy:
                actions = np.zeros((1, 2, N * M))
            if self._any_host_agent:
                host_pose = np.zeros((6, N * M))
                host_present = np.zeros(N * M, np.uint8)
            for n, st in enumerate(self.states):
                if st.is_done and not (len(self.states) == 1):
                    continue
                st.next_t = st.t + self.timestep
                for entity, agent in st.agents.items():
                    kind = self._agent_kind[agent]
                    i = n * M + self._slot_of[n][entity]
                    if entity not in st.poses:
                        continue
                    if kind == "host_policy":
                        act = agent._step(agent.sensor.step(st))
                        agent.last_action = act
                        a = (act.acceleration, act.steering) if isinstance(act, VehicleAction) else act
                        actions[0, 0, i], actions[0, 1, i] = a
                    elif kind == "host":
                        pose = agent.step(st)
                        if pose is not None:
                            host_pose[:, i] = pose
                            host_present[i] = 1
        force = len(self.states) == 1  # the reference's step() has no is_done guard
        if self._ticks_since_reset < 0:
            raise RuntimeError("step() after a fused rollout(): call reset_scenario() first")
        if self._action_table is not None:
            k, T = self._ticks_since_reset, self._action_table_host.shape[0]
            if k >= T and self._table_scenarios_live():
                raise IndexError(f"ActionTableAgent: the action table has {T} rows, step {k + 1} needs another")
            if actions is not None:  # merge the host policies' row into the resident table's row
                row = self._action_table_host[k].copy() if k < T else np.zeros((2, N * M))
                mask = self._host_policy_mask
                row[:, mask] = actions[0][:, mask]
                eng.rollout(1, actions=row[None], host_pose=host_pose, host_present=host_present, step_done=force)
            elif k < T:
                eng.rollout(1, actions=self._action_table, tick0=k,
                            host_pose=host_pose, host_present=host_present, step_done=force)
            else:  # only finished table scenarios are left: a zero row keeps the others stepping
                eng.rollout(1, actions=np.zeros((1, 2, N * M)), host_pose=host_pose,
                            host_present=host_present, step_done=force)
        elif self._action_rng is not None:
            eng.rollout(1, actions=self._action_rng, tick0=self._ticks_since_reset, host_pose=host_pose,
                        host_present=host_present, step_done=force)
        else:
            eng.rollout(1, actions=actions, host_pose=host_pose, host_present=host_present, step_done=force)
        self._ticks_since_reset += 1
        self._epoch += 1
        self._cache = {}
        for st in self.states:
            st._invalidate()
            st.update_actions()
        if self._host_mode:
            self._after_tick_host()

    def rollout(self, render: bool = False, video_path: Optional[str] = None) -> None:
        """Roll every scenario out to ``is_done`` (reference :256-267)."""
        if render:
            raise ValueError("rendering is out of scope of the device engine (no viewer)")
        self._refuse_env_agents()
        self.reset_scenario()
        if self._host_mode:
            while not all(st.is_done for st in self.states):
                self.step()
        else:
            self._sync_params()
            self._engine.rollout(-1, actions=self._action_rng if self._action_rng is not None else self._action_table,
                                 tick0=self._ticks_since_reset)
            self._ticks_since_reset = -1  # unknown per scenario; forces the next reset
            self._epoch += 1
            self._cache = {}
            for st in self.states:
                st._invalidate()
            self._replay_scenario_actions()
            for m in self.metrics:  # cache_metric / cache_mean on device metrics: one step on the final state
                if isinstance(m, _DeviceMetric) and getattr(m, "_sg_cached", False):
                    for n, st in enumerate(self.states):
                        m._n = n
                        m._step(st)
                    m._n = 0
            if (self._action_table is not None or self._action_rng is not None) and not self._fetch("done").all():
                if self._action_rng is not None:
                    raise IndexError(f"RandomActionSource: a scenario is not done after its {self._action_rng.n_ticks} rows")
                # the device stops a scenario whose ActionTableAgents ran out of rows; the
                # reference's agent would have raised on its next table lookup
                n = int(np.nonzero(self._fetch("done") == 0)[0][0])
                raise IndexError(f"ActionTableAgent: scenario {n} is not done after the "
                                 f"{self._action_table_host.shape[0]} rows of its action table")
        for st in self.states:
            for agent in st.agents.values():
                agent.finish(st)

    def get_metrics(self):
        """Metric states; a dict for one scenario, a list of dicts for a batch (reference :308-319)."""
        out = []
        self._cache = {}
        for n in range(len(self.states)):
            values = {}
            for metric in self._metrics_for(n):
                if isinstance(metric, _DeviceMetric):
                    metric._n = n
                value = metric.get_state()
                if isinstance(value, dict):
                    for k, v in value.items():
                        if isinstance(k, str):
                            values[f"{metric.name}_{k}"] = v
                elif value is not None:
                    values[metric.name] = value
            out.append(values)
        for metric in self.metrics:
            if isinstance(metric, _DeviceMetric):
                metric._n = 0
        return out[0] if len(out) == 1 else out

    def get_metric_arrays(self) -> Dict[str, np.ndarray]:
        """
        The device-side metrics of the whole batch as arrays indexed by scenario -- what ``get_metrics()`` reports
        scenario by scenario (a Python loop: ~4 us per scenario and metric), read back once.  Keys follow
        ``get_metrics()``: ``ego_avg_speed``, ``ego_max_speed``, ``ego_distance_travelled``,
        ``RSS_safe_longitudinal`` / ``RSS_safe_lateral``; ``CollisionMetric`` gives ``collisions_count`` and the
        batch's ``collisions_events`` records (scenario, tick, slot, t; ``slot_entities(n)[slot]`` is the hazard).
        Host-side (custom) metrics have no array
        form and are left to ``get_metrics()``.
        """
        if self._engine is None:
            return {}
        self._cache = {}
        out: Dict[str, np.ndarray] = {}
        for metric in self.metrics:
            if isinstance(metric, _DeviceMetric):
                try:
                    out.update(metric._arrays(self))
                except NotImplementedError:
                    pass
        return out

    def slot_entities(self, n: int = 0) -> List[Entity]:
        """The entities of scenario ``n`` in device slot order (agents first): what a ``slot`` index refers to."""
        return list(self._entity_of[n])

    def close(self) -> None:
        pass

    # ------------------------------------------------------------------ lowering
    def _metrics_for(self, n: int) -> List[Metric]:
        host = {id(m0): m for m0, m in zip(self._host_metric_protos, self._host_metrics[n])} \
            if self._host_metrics[n] else {}
        return [host.get(id(m), m) for m in self.metrics]

    def _build(self) -> None:
        from .engine import Engine

        specs, self._slot_of, self._entity_of = [], [], []
        self._agent_kind: Dict[Agent, str] = {}
        self._env_slots: List[List[int]] = [[] for _ in self.states]  # PolicyAgent slots per scenario
        veh_params, ped_params, pid_params = set(), set(), set()
        tables, random_agents = {}, {}
        for n, st in enumerate(self.states):
            sc = st.scenario
            ents = [e for e in sc.entities if e in st.agents] + [e for e in sc.entities if e not in st.agents]
            slots = []
            for s, e in enumerate(ents):
                agent = st.agents.get(e)
                kw = dict(traj=np.asarray(e.trajectory.data), etype=e.etype(), ref=e.ref or "",
                          box=(e.bounding_box.width, e.bounding_box.length, e.bounding_box.center_x,
                               e.bounding_box.center_y))
                if agent is None:
                    kind = abi.KIND_REPLAY
                elif type(agent) is ReplayTrajectoryAgent and type(agent.controller) is ReplayTrajectoryController \
                        and agent._trajectory is None:
                    kind, self._agent_kind[agent] = abi.KIND_AGENT_REPLAY, "device"
                elif isinstance(agent, PedestrianAgent) and type(agent.behaviour) is SocialForce:
                    kind, self._agent_kind[agent] = abi.KIND_PEDESTRIAN, "device"
                    kw.update(speed_desired=agent.speed_desired, route=np.array(agent.route))
                    pr = agent.behaviour.params
                    ped_params.add((agent.max_speed, agent.head_rot_angle, agent.distance_threshold,
                                    pr.max_speed_factor, pr.bias_lon, pr.bias_lat, pr.sight_weight,
                                    bool(pr.sight_weight_use), pr.sight_angle, pr.relaxation_time,
                                    pr.ped_repulse_V, pr.ped_repulse_sigma, pr.ped_attract_C,
                                    pr.boundary_repulse_U, pr.boundary_repulse_R,
                                    pr.imp_boundary_repulse_U, pr.imp_boundary_repulse_R,
                                    pr.std_lon, pr.std_lat, agent.behaviour.noise_seed))
                elif type(agent) is PIDAgent and type(agent.controller) is PIDController \
                        and agent._trajectory is None:
                    kind, self._agent_kind[agent] = abi.KIND_PID, "device"
                    c = agent.controller
                    veh_params.add((c.max_steer, c.max_accel, c.max_speed, bool(c.allow_reverse)))
                    kw.update(veh_limits=(c.max_steer, c.max_accel, c.max_speed, bool(c.allow_reverse)))
                    pid_params.add((c.steer_Kp, c.steer_Kd, c.accel_Kp, c.accel_Kd, c.accel_Ki))
                elif type(agent.controller) is VehicleController:
                    kind = abi.KIND_VEHICLE
                    c = agent.controller
                    veh_params.add((c.max_steer, c.max_accel, c.max_speed, bool(c.allow_reverse)))
                    kw.update(veh_limits=(c.max_steer, c.max_accel, c.max_speed, bool(c.allow_reverse)))
                    if type(agent) is ActionTableAgent:
                        self._agent_kind[agent] = "device"
                        tables[(n, s)] = agent.table
                    elif type(agent) is PolicyAgent:
                        self._agent_kind[agent] = "env_policy"
                        self._env_slots[n].append(s)
                    elif type(agent) is RandomActionAgent:
                        self._agent_kind[agent] = "device"
                        random_agents[(n, s)] = agent
                    else:
                        self._agent_kind[agent] = "host_policy"
                else:
                    if isinstance(agent, PedestrianAgent):
                        raise NotImplementedError(
                            "PedestrianAgent is integrated on the device with a SocialForce behaviour only "
                            f"(got {type(agent.behaviour).__name__})")
                    if agent.controller is None or agent.sensor is None:
                        raise NotImplementedError(f"{type(agent).__name__} needs a controller and a sensor to "
                                                  "run as a host-side agent")
                    kind, self._agent_kind[agent] = abi.KIND_HOST, "host"
                slots.append(SlotSpec(kind=kind, **kw))
            specs.append(ScenarioSpec(slots=slots, ego_slot=ents.index(sc.ego),
                                      first_slot=ents.index(sc.entities[0]),
                                      t0=self.get_start_time(sc), length=sc.length, name=sc.name or "",
                                      road_network=sc.road_network))
            self._slot_of.append({e: s for s, e in enumerate(ents)})
            self._entity_of.append(ents)
        if len(ped_params) > 1 or len(pid_params) > 1:
            raise NotImplementedError("pedestrian behaviour / PID gain parameters must be equal across agents")
        if len(veh_params) <= 1:  # one set of VehicleController limits: it travels in SgParams (fast kernels)
            for sp in specs:
                for sl in sp.slots:
                    sl.veh_limits = None
        self._veh_params = next(iter(veh_params)) if len(veh_params) == 1 else None
        self._ped_params = next(iter(ped_params)) if ped_params else None
        scene = pack_scenarios(specs, union_rows=False)  # knot times only: the rows are built on the device
        N, M = scene.N, scene.M
        for n, st in enumerate(self.states):  # device rows behind agent.force / agent.goal_idx
            for e, a in st.agents.items():
                if isinstance(a, PedestrianAgent) and self._agent_kind.get(a) == "device":
                    a._bound = (self, n * M + self._slot_of[n][e])
        for m in self.metrics:
            if isinstance(m, _DeviceMetric):
                m._gym, m._n = self, 0

        # host-side plugins
        self._host_metric_protos = [m for m in self.metrics if not isinstance(m, _DeviceMetric)]
        self._host_metrics = [[deepcopy(m) for m in self._host_metric_protos] if N > 1 else
                              list(self._host_metric_protos) for _ in range(N)]
        host_cbs = [cb for cb in self.state_callbacks if not getattr(cb, "_device", False)]
        self._host_callbacks = [[deepcopy(cb) for cb in host_cbs] if N > 1 else list(host_cbs)
                                for _ in range(N)]
        self._host_terminal = [c for c in self.terminal_conditions if callable(c)]
        kinds = set(self._agent_kind.values())
        self._any_host_policy = "host_policy" in kinds
        self._any_host_agent = "host" in kinds
        self._any_env_policy = "env_policy" in kinds
        self._host_mode = bool(self._host_metric_protos or host_cbs or self._host_terminal
                               or self._any_host_policy or self._any_host_agent)

        # parameters
        p = abi.default_params()
        p.terminal = 0
        for c in self.terminal_conditions:
            if callable(c):
                continue
            if c not in _TERMINAL_BITS:
                raise NotImplementedError(f"terminal condition {c!r} is out of scope of the device engine")
            p.terminal |= _TERMINAL_BITS[c]
        p.features = 0
        if any(isinstance(m, CollisionMetric) for m in self.metrics) or self._host_mode:
            p.features |= abi.FEAT_COLLISIONS
        if any(isinstance(m, _DeviceMetric) and not isinstance(m, CollisionMetric) for m in self.metrics) \
                or self._host_mode:
            p.features |= abi.FEAT_EGO_METRICS
        self._rss_cb = next((cb for cb in self.state_callbacks if isinstance(cb, RSSDistances)), None)
        if self._rss_cb is not None:
            p.features |= abi.FEAT_RSS
        if self._host_mode:
            p.features |= abi.FEAT_COLL_MATRIX
        for m in self.metrics:  # required callbacks must be present (reference metrics/base.py:44-53)
            for CB in m.required_callbacks:
                if not any(isinstance(cb, CB) for cb in self.state_callbacks):
                    raise ValueError("Cannot run metric {} without callback {}.".format(
                        m.__class__.__name__, CB.__name__))
        if self._veh_params:
            p.veh_max_steer, p.veh_max_accel = self._veh_params[0], self._veh_params[1]
            p.veh_max_speed = float("nan") if self._veh_params[2] is None else self._veh_params[2]
            p.veh_allow_reverse = int(self._veh_params[3])
        if pid_params:
            (p.pid_steer_Kp, p.pid_steer_Kd, p.pid_accel_Kp, p.pid_accel_Kd, p.pid_accel_Ki) = next(iter(pid_params))
        if self._ped_params:
            (p.ped_max_speed, p.ped_head_rot_angle, p.ped_distance_threshold, p.sf_max_speed_factor,
             p.sf_bias_lon, p.sf_bias_lat, p.sf_sight_weight, suse, p.sf_sight_angle,
             p.sf_relaxation_time, p.sf_ped_repulse_V, p.sf_ped_repulse_sigma, p.sf_ped_attract_C,
             p.sf_boundary_repulse_U, p.sf_boundary_repulse_R, p.sf_imp_boundary_repulse_U,
             p.sf_imp_boundary_repulse_R, p.sf_std_lon, p.sf_std_lat, p.sf_noise_seed) = self._ped_params
            p.sf_sight_weight_use = int(suse)
        self._params = p
        trace_cap = 0
        if self.record and not self._host_mode:
            ts = float(self.timestep)
            trace_cap = int(max((sp.length - sp.t0) / ts for sp in specs)) + 8
        self._engine = Engine(scene, p, device=self.device, trace_cap=trace_cap)

        # RandomActionAgents: the actions are drawn inside the kernel when one source feeds every vehicle
        # agent of the batch; otherwise their columns join the resident table below
        self._action_rng = None
        for (n, s_), a in random_agents.items():
            a._column = (N * M, n * M + s_)
        sources = {id(a.source): a.source for a in random_agents.values()}
        if random_agents and len(sources) == 1 and not tables and not self._any_host_policy:
            self._action_rng = next(iter(sources.values())).action_rng(N * M)
        else:
            for (n, s_), a in random_agents.items():
                tables[(n, s_)] = a.source.table(N * M)[:, :, n * M + s_]
        # resident action table of ActionTableAgents
        self._action_table = self._action_table_host = None
        if tables or self._any_host_policy:
            T = max((len(t) for t in tables.values()), default=0)
            if self._any_host_policy:
                T = max(T, 1)
            tab = np.zeros((max(T, 1), 2, N * M))
            for (n, s), t in tables.items():
                tab[: len(t), :, n * M + s] = t
            self._action_table_host = tab
            if tables:
                self._action_table = self._engine.set_actions(tab)
            mask = np.zeros(N * M, bool)
            for n, st in enumerate(self.states):
                for e, a in st.agents.items():
                    if self._agent_kind[a] == "host_policy":
                        mask[n * M + self._slot_of[n][e]] = True
            self._host_policy_mask = mask
        self._table_slots = np.array(sorted(n * M + s_ for (n, s_) in tables), np.int64)
        self._ticks_since_reset = 1
        self._epoch = 0
        self._host_done = [False] * N
        self._cache: Dict[str, np.ndarray] = {}

    def _replay_scenario_actions(self) -> None:
        """
        Scenario actions after a fused rollout: the tick times of a scenario are t0 plus the timestep
        added tick by tick (the sum the device accumulates, scenario_gym.py:229); every pending
        action is applied at the first of them that satisfies its trigger condition.
        """
        pending = [n for n, st in enumerate(self.states) if st.unapplied_actions]
        if not pending:
            return
        ticks, t0 = self._fetch("tick"), self._engine.scene.t0
        for n in pending:
            times, t = [], float(t0[n])
            for _ in range(int(ticks[n])):
                t = t + self.timestep
                times.append(t)
            self.states[n]._replay_actions(times)

    def _entities_in_radius(self, n: int, x: float, y: float, r: float) -> np.ndarray:
        """Present slots of scenario n strictly inside Point(x, y).buffer(r) (device query)."""
        N = len(self.states)
        xs, ys, rs = np.zeros(N), np.zeros(N), np.full(N, -1.0)
        xs[n], ys[n], rs[n] = x, y, r
        return self._engine.entities_in_radius(xs, ys, rs)[n]

    def _table_scenarios_live(self) -> bool:
        """Is any scenario with an ActionTableAgent still running (it would need another table row)?"""
        if not len(self._table_slots):
            return False
        done = self._fetch("done")
        return bool((done[np.unique(self._table_slots // self._engine.M)] == 0).any())

    def _sync_params(self) -> None:
        self._params.timestep = self.timestep
        self._params.persist = int(self.persist)

    # ------------------------------------------------------------------ device -> host views
    def _fetch(self, name: str) -> np.ndarray:
        if name not in self._cache:
            self._cache[name] = self._engine.get(name)
        return self._cache[name]

    def _materialise(self, n: int) -> dict:
        """
        Host view of scenario n.  The planes come from ONE device->host copy per field for the whole
        batch (``_fetch`` caches them until the state advances), sliced here.
        """
        M = self._engine.M
        sl = slice(n * M, (n + 1) * M)
        if "poseT" not in self._cache:  # entity-major rows, transposed once per tick for the whole batch
            self._cache["poseT"] = np.ascontiguousarray(self._fetch("pose").T)
            self._cache["velT"] = np.ascontiguousarray(self._fetch("vel").T)
        ents = self._entity_of[n]
        k = len(ents)
        dist, present = self._fetch("dist")[sl], self._fetch("present")[n * M:n * M + k]
        rows_p, rows_v = self._cache["poseT"][n * M:n * M + k], self._cache["velT"][n * M:n * M + k]
        if present.all():
            here, rows_p, rows_v = ents, rows_p.copy(), rows_v.copy()
        else:
            idx = np.nonzero(present)[0]
            here, rows_p, rows_v = [ents[i] for i in idx], rows_p[idx], rows_v[idx]
        poses, vels = dict(zip(here, rows_p)), dict(zip(here, rows_v))  # (rows of this scenario's own copies)
        if self._rss_cb is not None:
            self._sync_rss(n, ents, sl)
        return {
            "t": float(self._fetch("t")[n]), "prev_t": float(self._fetch("prev_t")[n]),
            "done": bool(self._fetch("done")[n]), "poses": poses, "velocities": vels,
            "distances": dict(zip(ents, dist[: len(ents)].tolist())),
        }

    def _sync_rss(self, n: int, ents, sl) -> None:
        cb = self._rss_cb
        sd, ratio, rec = self._fetch("safe_dist")[:, sl], self._fetch("safe_ratio")[:, sl], self._fetch("rss_last")[sl]
        cb.safe_distances = {e: [float(sd[0, s]), float(sd[1, s])] for s, e in enumerate(ents)
                             if rec[s] != abi.RSS_NONE}
        cb.entity_safe_ratios = {e: [float(ratio[0, s]), float(ratio[1, s])] for s, e in enumerate(ents)}
        cb.intersect = {e: [abi.RSS_RECORD_NAMES[int(rec[s])]] for s, e in enumerate(ents)
                        if rec[s] != abi.RSS_NONE}

    def _device_trace(self, n: int):
        """Recorded (t, pose) rows per entity from the device trace of a fused rollout."""
        eng = self._engine
        if eng.trace_cap <= 0:
            return None
        M = eng.M
        T = int(eng.tensor("tick")[n].item()) + 1
        if T > eng.trace_cap:
            raise RuntimeError("trace buffer too short (timestep changed after set_scenario?)")
        sl = slice(n * M, (n + 1) * M)
        pose = eng.tensor("trace_pose")[:T, :, sl].cpu().numpy()
        present = eng.tensor("trace_present")[:T, sl].cpu().numpy().astype(bool)
        ts = eng.tensor("trace_t")[:T, n].cpu().numpy()
        out = {}
        for s, e in enumerate(self._entity_of[n]):
            k = np.nonzero(present[:, s])[0]
            out[e] = np.concatenate([ts[k, None], pose[k, :, s]], axis=1) if len(k) else np.empty((0, 7))
        return out

    def _future_collision(self, n: int, entity: Entity, horizon: float, n_samples: int) -> bool:
        """
        FutureCollisionDetector for scenario ``n``: answered from one batched device launch per
        (tick, horizon, sensor slots); the result is cached until the state advances.
        """
        slot = self._slot_of[n][entity]
        key = (id(self._engine), self._epoch, float(horizon), int(n_samples))
        cache = getattr(self, "_future_cache", None)
        if cache is None or cache[0] != key or cache[1][n] != slot:
            slots = np.array([self._slot_of[k].get(self.states[k].scenario.ego, 0)
                              for k in range(len(self.states))], np.int32)
            if cache is not None and cache[0] == key:
                slots = cache[1].copy()
            slots[n] = slot
            flags = self._engine.future_collisions(None, horizon, n_samples, slots)
            cache = self._future_cache = (key, slots, flags)
        return bool(cache[2][n])

    def _collisions(self, n: int) -> Dict[Entity, List[Entity]]:
        eng = self._engine
        ents = self._entity_of[n]
        present = self._fetch("present")[n * eng.M:(n + 1) * eng.M]
        if not (self._params.features & abi.FEAT_COLL_MATRIX):
            # no per-tick pair matrix on this run (it is kept whenever a host-side plugin is
            # present): test the present entities' current boxes pairwise on the device
            return self._collisions_on_demand(n, ents, present)
        rows = self._fetch("coll_mask")[n]  # [M, W] uint32 (one copy per tick for the whole batch)
        bits = np.unpackbits(rows.view(np.uint8), axis=1, bitorder="little")[:, : len(ents)]
        out = {}
        for a in np.nonzero(present[: len(ents)])[0]:
            out[ents[a]] = [ents[b] for b in np.nonzero(bits[a])[0]]
        return out

    def _collisions_on_demand(self, n: int, ents, present) -> Dict[Entity, List[Entity]]:
        import ctypes as C

        import torch

        eng = self._engine
        M = eng.M
        idx = [a for a in range(len(ents)) if present[a]]
        out = {ents[a]: [] for a in idx}
        pairs = [(a, b) for i, a in enumerate(idx) for b in idx[i + 1:]]
        if not pairs:
            return out
        pose = eng.tensor("pose").view(6, -1)[:, n * M:(n + 1) * M].cpu().numpy()
        box = eng._scene_t["box"].view(4, -1)[:, n * M:(n + 1) * M].cpu().numpy()
        ia, ib = np.array([a for a, _ in pairs]), np.array([b for _, b in pairs])
        dev = eng.device
        pa = torch.from_numpy(np.ascontiguousarray(pose[[0, 1, 3]][:, ia].T)).to(dev)
        pb = torch.from_numpy(np.ascontiguousarray(pose[[0, 1, 3]][:, ib].T)).to(dev)
        ba = torch.from_numpy(np.ascontiguousarray(box[:, ia].T)).to(dev)
        bb = torch.from_numpy(np.ascontiguousarray(box[:, ib].T)).to(dev)
        hit = torch.zeros(len(pairs), dtype=torch.uint8, device=dev)
        eng._check(eng.lib["test_box_pairs"](pa.data_ptr(), ba.data_ptr(), pb.data_ptr(), bb.data_ptr(),
                                             hit.data_ptr(), len(pairs), eng.dev_index, eng._stream()))
        for (a, b), h in zip(pairs, hit.cpu().numpy()):
            if h:
                out[ents[a]].append(ents[b])
                out[ents[b]].append(ents[a])
        return out

    def _collision_events(self, n: int) -> list:
        if "events_by_scenario" not in self._cache:  # one pass over the batch's event list, kept in order
            ev = self._engine.events()  # sorted by (scenario, tick, slot)
            starts = np.searchsorted(ev["scenario"], np.arange(len(self.states) + 1))
            self._cache["events_by_scenario"] = (ev, starts)
        ev, starts = self._cache["events_by_scenario"]
        ev = ev[starts[n]:starts[n + 1]]
        ents = self._entity_of[n]
        out = []
        for e in ev:
            hazard = ents[int(e["slot"])]
            ctype = "non_vehicle" if hazard.catalog_entry.catalog_type != "Vehicle" else "vehicle"
            out.append((float(e["t"]), hazard.ref, ctype))
        return out

    def _after_tick_host(self) -> None:
        """Host-side callbacks, terminal conditions and metrics for the scenarios that ticked."""
        eng = self._engine
        ticks = eng.get("tick")
        for n, st in enumerate(self.states):
            if ticks[n] == self._last_tick[n]:
                continue  # done scenario of a batch: the device skipped it
            st._record()
            for cb in self._host_callbacks[n]:
                cb(st)
            if any(cond(st) for cond in self._host_terminal):
                self._host_done[n] = True
                eng.tensor("done")[n] = 1
            for m in self._host_metrics[n]:
                m.step(st)
        self._last_tick = ticks.copy()
