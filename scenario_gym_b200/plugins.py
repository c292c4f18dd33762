"""
Plugin API -- the reference's subclassing surface for this path, with the same names,
constructor arguments and hook methods (reference scenario_gym/action.py, agent.py,
controller.py, sensor/base.py, sensor/common.py, observation.py, callback.py, metrics/*.py,
pedestrian/*.py).  ``ScenarioGym`` (gym.py) inspects what ``create_agent`` returned and lowers
the recognised classes to device slot kinds; anything else keeps working through a per-tick
host call on a materialised ``State`` (drop-in, just slower).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Any, Dict, List, Optional, Tuple, Type

import numpy as np

from .entity import Entity, Pedestrian
from .trajectory import Trajectory


# ------------------------------------------------------------------------------ actions
class Action:
    """Base class for actions that agents communicate to controllers."""


class TeleportAction(Action):
    """Desired coordinates for the next pose (reference action.py:12-63)."""

    def __init__(self, x=0.0, y=0.0, z=0.0, h=0.0, r=0.0, p=0.0, pose: Optional[np.ndarray] = None):
        self.x = pose[0] if pose is not None else x
        self.y = pose[1] if pose is not None else y
        self.z = pose[2] if pose is not None else z
        self.h = pose[3] if pose is not None else h
        self.r = pose[4] if pose is not None else r
        self.p = pose[5] if pose is not None else p

    @property
    def pose(self) -> np.ndarray:
        return np.array([self.x, self.y, self.z, self.h, self.r, self.p])


class VehicleAction(Action):
    """An acceleration and a steering update (reference action.py:66-83)."""

    def __init__(self, accel: float, steer: float):
        self.acceleration = accel
        self.steering = steer


@dataclass
class PedestrianAction(Action):
    speed: float
    heading: float


# ------------------------------------------------------------------------------ observations
@dataclass
class Observation:
    pass


@dataclass
class SingleEntityObservation(Observation):
    entity: Entity
    t: float
    next_t: float
    pose: np.ndarray
    velocity: np.ndarray
    distance_travelled: float
    recorded_poses: np.ndarray
    entity_state: Any


# ------------------------------------------------------------------------------ sensors
class Sensor:
    """Produce an observation for an entity from the global state (reference sensor/base.py)."""

    def __init__(self, entity: Entity):
        self.entity = entity
        self.initial_observation = None
        self.last_observation = None

    def reset(self, state):
        self.last_observation = None
        self.initial_observation = self._reset(state)
        return self.initial_observation

    def step(self, state):
        self.last_observation = self._step(state)
        return self.last_observation

    def _reset(self, state):
        raise NotImplementedError

    def _step(self, state):
        raise NotImplementedError


class EgoLocalizationSensor(Sensor):
    """Observation with the base entity information (reference sensor/common.py:39-50)."""

    def _reset(self, state):
        return self._step(state)

    def _step(self, state):
        return SingleEntityObservation(self.entity, *state.get_entity_data(self.entity))


def combine_observations(*obs_classes, prefixes=None):
    """
    A dataclass holding the fields of several observation classes (reference observation.py:31-83):
    the first class that defines a field name provides it; with ``prefixes`` a repeated name is
    kept as ``f"{prefix}_{name}"`` instead of being skipped.  The class gets ``from_obs(*obs)``.
    """
    import dataclasses

    if prefixes is not None and len(prefixes) != len(obs_classes):
        raise ValueError
    spec, source = [], []
    for idx, oc in enumerate(obs_classes):
        if not dataclasses.is_dataclass(oc):
            raise TypeError(f"Observation {oc} is not a dataclass.")
        for f in dataclasses.fields(oc):
            name = f.name
            if any(name == n for n, _ in spec):
                if prefixes is None:
                    continue
                name = f"{prefixes[idx]}_{f.name}"
                if any(name == n for n, _ in spec):
                    raise ValueError(f"Prefix {prefixes[idx]} still leads to duplicate name for {name}.")
            spec.append((name, f.type))
            source.append((idx, f.name))

    def from_obs(cls, *obs):
        return cls(*(getattr(obs[i], name) for i, name in source))

    return dataclasses.make_dataclass("CombinedObservation", spec, bases=(Observation,),
                                      namespace={"from_obs": classmethod(from_obs)})


class CombinedSensor(Sensor):
    """Combines the observations of several sensors of one entity (reference sensor/common.py:18-36)."""

    def __init__(self, entity: Entity, *sensors: Sensor):
        super().__init__(entity)
        self.sensors = sensors
        self.obs_class = None

    def _reset(self, state):
        init_obs = [s.reset(state) for s in self.sensors]
        self.obs_class = combine_observations(*(o.__class__ for o in init_obs))
        return self.obs_class.from_obs(*init_obs)

    def _step(self, state):
        return self.obs_class.from_obs(*(s.step(state) for s in self.sensors))


@dataclass
class CollisionObservation(SingleEntityObservation):
    """Observation with detected collisions (reference sensor/common.py:108-112)."""

    collisions: Any = None


class GlobalCollisionDetector(Sensor):
    """Returns the collisions observed in the scene (reference sensor/common.py:115-128)."""

    def _reset(self, state):
        return self._step(state)

    def _step(self, state):
        return CollisionObservation(self.entity, *state.get_entity_data(self.entity), state.collisions())


@dataclass
class FutureCollisionObservation(SingleEntityObservation):
    """Observation with future collision information (reference sensor/common.py:53-57)."""

    future_collision: bool = False


class FutureCollisionDetector(Sensor):
    """
    Detects any future collision with the sensor's entity over ``horizon`` seconds from the
    entities' trajectories (reference sensor/common.py:60-105).  The look-ahead runs on the device
    for the whole batch (``sg_future_collisions``): one launch per tick serves the detectors of
    every scenario with the same horizon.
    """

    N_SAMPLES = 10  # np.linspace(state.t, state.t + horizon, 10), sensor/common.py:94

    def __init__(self, entity: Entity, horizon: float = 5.0):
        super().__init__(entity)
        self.horizon = horizon

    def _reset(self, state):
        return self._step(state)

    def _step(self, state):
        flag = state._gym._future_collision(state._n, self.entity, self.horizon, self.N_SAMPLES)
        return FutureCollisionObservation(self.entity, *state.get_entity_data(self.entity), bool(flag))


# ------------------------------------------------------------------------------ controllers
class Controller:
    """Takes the agent's action and returns the pose (reference controller.py:12-42)."""

    def __init__(self, entity: Entity):
        self.entity = entity

    def reset(self, state) -> None:
        self._reset(state)

    def step(self, state, action):
        return self._step(state, action)

    def _reset(self, state) -> None:
        raise NotImplementedError

    def _step(self, state, action):
        raise NotImplementedError


class ReplayTrajectoryController(Controller):
    def _reset(self, state) -> None:
        pass

    def _step(self, state, action: TeleportAction):
        return action.pose


class VehicleController(Controller):
    """
    Kinematic bicycle with clipped acceleration / steering (reference controller.py:57-140).
    Agents that use this exact class are integrated on the device; ``_step`` is the host
    implementation used only when a subclass overrides behaviour.
    """

    def __init__(self, entity: Entity, max_steer: float = 0.7, max_accel: float = 5.0,
                 max_speed: Optional[float] = None, allow_reverse: bool = False):
        super().__init__(entity)
        self.max_steer = max_steer
        self.max_accel = max_accel
        self.allow_reverse = allow_reverse
        self.max_speed = max_speed

    def _reset(self, state) -> None:
        self.speed = np.linalg.norm(state.velocities[self.entity][:2])
        self.l = self.entity.catalog_entry.bounding_box.length

    def _step(self, state, action):
        if isinstance(action, VehicleAction):
            accel, steer = action.acceleration, action.steering
        else:
            accel, steer = action
        accel = np.clip(accel, -self.max_accel, self.max_accel)
        steer = np.clip(steer, -self.max_steer, self.max_steer)
        pose = state.poses[self.entity].copy()
        dt = state.next_t - state.t
        h = pose[3]
        dx, dy = self.speed * np.cos(h), self.speed * np.sin(h)
        dh = self.speed * np.tan(steer) / self.l
        pose[[0, 1]] += np.array([dx, dy]) * dt
        pose[3] += dh * dt
        speed = self.speed + accel * dt
        if not self.allow_reverse:
            speed = np.maximum(0.0, speed)
        if self.max_speed is not None:
            speed = np.minimum(self.max_speed, speed)
        self.speed = speed
        return pose


class PIDController(VehicleController):
    """
    PID steering / acceleration towards a target point (reference controller.py:143-258); runs
    on the device for ``PIDAgent``.  Keyword arguments go to the underlying vehicle model.
    """

    def __init__(self, entity: Entity, steer_Kp: float = 0.03054, steer_Kd: float = 1.5709,
                 accel_Kp: float = 0.3753, accel_Kd: float = 1.8970, accel_Ki: float = 0.0204,
                 **kwargs):
        super().__init__(entity, **kwargs)
        self.steer_Kp, self.steer_Kd = steer_Kp, steer_Kd
        self.accel_Kp, self.accel_Ki, self.accel_Kd = accel_Kp, accel_Ki, accel_Kd

    # host implementation: used when the agent is not lowered to the device PID kind (a PIDAgent
    # subclass, or one that follows a trajectory other than its entity's)
    def _reset(self, state) -> None:
        self.e_lon_prev = self.e_lon_int = self.e_lat_prev = 0.0
        VehicleController._reset(self, state)

    def _step(self, state, action):
        tx, ty = action.pose[0], action.pose[1]
        x, y, h = (state.poses[self.entity][k] for k in (0, 1, 3))
        ch, sh = np.cos(h), np.sin(h)
        ex, ey = tx - x, ty - y
        e_lon, e_lat = ch * ex + sh * ey, -sh * ex + ch * ey  # error in the vehicle frame
        v = self.speed
        gain = 1.0 - 0.9 * (v - 5.0) / 10.0 if 5.0 < v <= 15 else (0.1 if v > 15 else 1.0)
        dt = state.dt
        steer = self.steer_Kp * gain * e_lat + self.steer_Kd * gain * ((e_lat - self.e_lat_prev) / dt)
        integ = self.e_lon_int + e_lon * dt
        accel = 0.0
        if abs(e_lon) > 0.1:
            accel = self.accel_Kp * e_lon + self.accel_Kd * ((e_lon - self.e_lon_prev) / dt) + self.accel_Ki * integ
        self.e_lat_prev, self.e_lon_prev, self.e_lon_int = e_lat, e_lon, integ
        return VehicleController._step(self, state, VehicleAction(accel, steer))


# ------------------------------------------------------------------------------ agents
class Agent:
    """Processes observations to select an action (reference agent.py:18-115)."""

    def __init__(self, entity: Entity, controller: Controller, sensor: Sensor):
        self.entity = entity
        self.controller = controller
        self.sensor = sensor
        self.last_action = None
        self.last_reward = None
        self._trajectory: Optional[Trajectory] = None

    def reset(self, state) -> None:
        self.last_action = None
        self.last_reward = None
        self.sensor.reset(state)
        self.controller.reset(state)
        self._reset()

    def step(self, state):
        obs = self.sensor.step(state)
        action = self._step(obs)
        self.last_action = action
        return self.controller.step(state, action)

    def _reset(self) -> None:
        pass

    def _step(self, observation) -> Action:
        pass

    def finish(self, state) -> None:
        pass

    @property
    def trajectory(self) -> Trajectory:
        return self._trajectory if self._trajectory is not None else self.entity.trajectory

    @trajectory.setter
    def trajectory(self, trajectory: Trajectory):
        self._trajectory = trajectory

    def reward(self, state):
        r = self._reward(state)
        if r is not None:
            self.last_reward = r
        return r

    def _reward(self, state):
        pass


class ReplayTrajectoryAgent(Agent):
    """Follows the predefined trajectory (reference agent.py:118-128)."""

    def _step(self, observation) -> Action:
        return TeleportAction(pose=self.trajectory.position_at_t(observation.next_t))


class PIDAgent(Agent):
    """Follows its trajectory with a PID controller (reference agent.py:131-148)."""

    def __init__(self, entity: Entity, **controller_kwargs):
        super().__init__(entity, PIDController(entity, **controller_kwargs), EgoLocalizationSensor(entity))

    def _step(self, observation) -> TeleportAction:
        pos = self.trajectory.position_at_t(observation.next_t)
        return TeleportAction(x=pos[0], y=pos[1], z=pos[2])


class ActionTableAgent(Agent):
    """
    Vehicle agent that plays back a pre-drawn ``(T, 2)`` table of (accel, steer) through a
    ``VehicleController``: row k is the action of the k-th step after reset.  The whole table is
    uploaded once, so rollouts of such agents run fused on the device.
    """

    def __init__(self, entity: Entity, table: np.ndarray, **controller_kwargs):
        super().__init__(entity, VehicleController(entity, **controller_kwargs),
                         EgoLocalizationSensor(entity))
        self.table = np.ascontiguousarray(table, dtype=np.float64).reshape(-1, 2)
        self.k = 0

    def _reset(self) -> None:
        self.k = 0

    def _step(self, observation) -> VehicleAction:
        a = self.table[self.k]
        self.k += 1
        return VehicleAction(a[0], a[1])


class RandomActionSource:
    """
    The random policy of the "random accel / steer" configurations: a ``(n_ticks, 2, N*M)`` table of
    uniform actions drawn from ``numpy.random.default_rng(seed)``, accelerations first
    (``rng.uniform(low[0], high[0], (n_ticks, N*M))``), then steering.  Agents sharing one source read
    their own column; when every vehicle agent of a batch is a ``RandomActionAgent`` of one source the
    table is never built -- the kernels evaluate numpy's PCG64 stream in place (``ActionRng``).
    """

    def __init__(self, seed: int, n_ticks: int, low=(-6.0, -1.0), high=(6.0, 1.0)):
        self.seed, self.n_ticks = int(seed), int(n_ticks)
        self.low, self.high = (float(low[0]), float(low[1])), (float(high[0]), float(high[1]))
        self._table = None

    def action_rng(self, nm: int):
        from .action_rng import ActionRng

        return ActionRng.from_generator(self.seed, offset=(0, self.n_ticks * nm), tick_stride=nm,
                                        low=self.low, high=self.high, n_ticks=self.n_ticks, nm=nm)

    def table(self, nm: int) -> np.ndarray:
        if self._table is None or self._table.shape[2] != nm:
            rng = np.random.default_rng(self.seed)
            tab = np.empty((self.n_ticks, 2, nm))
            for c in range(2):
                tab[:, c] = rng.uniform(self.low[c], self.high[c], (self.n_ticks, nm))
            self._table = tab
        return self._table


class RandomActionAgent(Agent):
    """Vehicle agent whose VehicleActions are the columns of a ``RandomActionSource`` (see there)."""

    def __init__(self, entity: Entity, source: RandomActionSource, **controller_kwargs):
        super().__init__(entity, VehicleController(entity, **controller_kwargs), EgoLocalizationSensor(entity))
        self.source = source
        self.k = 0
        self._column = None  # (nm, flat slot index), set when the agent is lowered

    def _reset(self) -> None:
        self.k = 0

    def _step(self, observation) -> VehicleAction:
        if self._column is None:
            raise RuntimeError("RandomActionAgent is not part of a gym yet")
        nm, i = self._column
        a = self.source.table(nm)[self.k, :, i]
        self.k += 1
        return VehicleAction(float(a[0]), float(a[1]))


class PolicyAgent(Agent):
    """
    Vehicle agent whose VehicleActions come from the policy of a ``VecScenarioEnv``: the env scatters
    each step's action tensor into the device's action rows, so the agent has no host-side ``_step``.
    It runs only inside an env; ``ScenarioGym.step`` / ``rollout`` refuse a batch that contains one.
    """

    def __init__(self, entity: Entity, **controller_kwargs):
        super().__init__(entity, VehicleController(entity, **controller_kwargs), EgoLocalizationSensor(entity))

    def _step(self, observation) -> VehicleAction:
        raise RuntimeError("PolicyAgent takes its actions from VecScenarioEnv.step()")


def _create_agent(scenario, entity) -> Optional[Agent]:
    """Default: a replay agent for the entity named "ego" (reference agent.py:151-169)."""
    if entity.ref == "ego":
        return ReplayTrajectoryAgent(entity, ReplayTrajectoryController(entity),
                                     EgoLocalizationSensor(entity))
    return None


# ------------------------------------------------------------------------------ callbacks / metrics
class StateCallback:
    """Per-tick callback on the state (reference callback.py:9-41)."""

    required_callbacks: List[Type["StateCallback"]] = []

    def __init__(self):
        self.callbacks: List[StateCallback] = []

    def reset(self, state) -> None:
        self.callbacks.clear()
        for req in self.required_callbacks:
            cb = state.get_callback(req)
            if cb is None:
                raise ValueError(f"Callback {req.__name__} is required for {self.__class__}.")
            self.callbacks.append(cb)
        self._reset(state)

    def _reset(self, state) -> None:
        pass

    def __call__(self, state) -> None:
        raise NotImplementedError


class Metric:
    """Base class for metrics (reference metrics/base.py:8-73)."""

    name: Optional[str] = None
    required_callbacks: List[Type[StateCallback]] = []

    def __init__(self, name: Optional[str] = None):
        if name is not None:
            self.name = name
        elif self.name is None:
            self.name = self.__class__.__name__
        self.callbacks: List[StateCallback] = []

    def reset(self, state) -> None:
        self.callbacks.clear()
        for CB in self.required_callbacks:
            cb = state.get_callback(CB)
            if cb is None:
                raise ValueError("Cannot run metric {} without callback {}.".format(
                    self.__class__.__name__, CB.__name__))
            self.callbacks.append(cb)
        self._reset(state)

    def step(self, state) -> None:
        self._step(state)

    def _reset(self, state) -> None:
        raise NotImplementedError

    def _step(self, state) -> None:
        raise NotImplementedError

    def get_state(self) -> Any:
        raise NotImplementedError


class _DeviceMetric(Metric):
    """Built-in metric whose value is accumulated on the device; ``_pull`` reads it back."""

    _device = True
    _gym = None   # bound by ScenarioGym when the scenarios are built
    _n = 0        # scenario of the batch get_state() reports (get_metrics() walks over all of them)
    _value = None

    def _reset(self, state) -> None:
        self._value = None

    def _step(self, state) -> None:
        pass

    def _pull(self, gym, n: int) -> None:
        raise NotImplementedError

    def get_state(self):
        if self._gym is not None and self._gym._engine is not None:
            self._pull(self._gym, self._n)
        return self._value

    def _arrays(self, gym) -> Dict[str, np.ndarray]:
        """The metric over the whole batch as arrays indexed by scenario (ScenarioGym.get_metric_arrays)."""
        raise NotImplementedError


class EgoAvgSpeed(_DeviceMetric):
    """Time-weighted average ego speed (reference metrics/trajectory.py:8-28)."""

    name = "ego_avg_speed"

    def _pull(self, gym, n):
        self._value = float(gym._fetch("ego_avg_speed")[n])

    def _arrays(self, gym):
        return {self.name: gym._fetch("ego_avg_speed").copy()}


class EgoMaxSpeed(_DeviceMetric):
    name = "ego_max_speed"

    def _pull(self, gym, n):
        self._value = float(gym._fetch("ego_max_speed")[n])

    def _arrays(self, gym):
        return {self.name: gym._fetch("ego_max_speed").copy()}


class EgoDistanceTravelled(_DeviceMetric):
    name = "ego_distance_travelled"

    def _pull(self, gym, n):
        self._value = float(gym._fetch("ego_dist")[n])

    def _arrays(self, gym):
        return {self.name: gym._fetch("ego_dist").copy()}


class CollisionMetric(_DeviceMetric):
    """
    Records ``(t, ref, type)`` for every entity that starts colliding with the ego
    (reference metrics/collision.py:46-86).  Non-vehicle hazards are ``"non_vehicle"`` as in the
    reference; vehicle hazards -- whose classification raises AttributeError in the reference
    (collision.py:94) -- are reported as ``"vehicle"``.
    """

    name = "collisions"

    def __init__(self, c_tol: float = 0.4, name: Optional[str] = None):
        self.c_tol = c_tol
        super().__init__(name=name)

    def _pull(self, gym, n):
        self._value = gym._collision_events(n)

    def get_state(self):
        super().get_state()
        return list(self._value or [])

    def _arrays(self, gym):
        # the batch's rising edges as one record array (scenario, tick, slot, t), sorted by scenario, and how many
        # each scenario has; `slot` indexes ScenarioGym.slot_entities(n)
        ev = gym._engine.events()
        counts = np.bincount(ev["scenario"], minlength=len(gym.states)).astype(np.int64)
        return {f"{self.name}_events": ev, f"{self.name}_count": counts}


class RSSParameters:
    """RSS parameters (reference metrics/rss/callback.py:21-31)."""

    RESPONSE_TIME = 0.6
    MIN_LONG_ACCEL = 1.2 * 9.81
    MAX_LONG_ACCEL = 1.2 * 9.81
    MIN_SAFE_CLEARANCE = 0.1


class RSSDistances(StateCallback):
    """
    Per-tick safe longitudinal / lateral distances and buffer-intersection records per entity
    (reference metrics/rss/callback.py:34-505), computed on the device.  After a step
    ``safe_distances[entity] = [lat, long]``, ``entity_safe_ratios[entity]`` and ``intersect[entity]``
    (the record appended this tick) are available.
    """

    _device = True

    def _reset(self, state) -> None:
        self.safe_distances: Dict[Entity, List[float]] = {}
        self.entity_safe_ratios: Dict[Entity, List[float]] = {}
        self.intersect: Dict[Entity, List[str]] = {}

    def __call__(self, state) -> None:
        pass


class RSS(_DeviceMetric):
    """``safe_longitudinal`` / ``safe_lateral`` booleans (reference metrics/rss/rss.py:106-163)."""

    required_callbacks = [RSSDistances]

    def _pull(self, gym, n):
        flags = int(gym._fetch("rss_flags")[n])
        self._value = {"safe_longitudinal": not (flags & 1), "safe_lateral": not (flags & 2)}

    def _arrays(self, gym):
        flags = gym._fetch("rss_flags")
        return {f"{self.name}_safe_longitudinal": (flags & 1) == 0, f"{self.name}_safe_lateral": (flags & 2) == 0}


def cache_metric(Met: Type[Metric]) -> Type[Metric]:
    """Keep the metric's value of the last finished scenario in ``previous_value`` (metrics/base.py:76-89)."""
    prev_step = Met._step
    Met.previous_value = None
    Met._sg_cached = True  # device metrics: ScenarioGym calls _step once a fused rollout has finished

    def new_step(self, state):
        prev_step(self, state)
        if state.is_done:
            self.previous_value = self.get_state()

    Met._step = new_step
    return Met


def cache_mean(Met: Type[Metric]) -> Type[Metric]:
    """
    Running mean of the metric's value over finished scenarios; reading ``previous_value`` returns it
    and starts a new mean (metrics/base.py:92-113).
    """

    def previous_value(self):
        val = self._previous_value
        self._previous_value = 0.0
        self._prev_count = 0
        return val

    prev_step = Met._step
    Met._previous_value = 0.0
    Met._prev_count = 0
    Met.previous_value = property(previous_value)
    Met._sg_cached = True

    def new_step(self, state):
        prev_step(self, state)
        if state.is_done:
            self._prev_count += 1
            self._previous_value += (self.get_state() - self._previous_value) / self._prev_count

    Met._step = new_step
    return Met


def _clip_convex(subject: np.ndarray, clip: np.ndarray) -> np.ndarray:
    """Sutherland-Hodgman: the part of convex polygon `subject` inside convex polygon `clip` (vertex rows)."""
    def area2(p):
        return float(np.dot(p[:, 0], np.roll(p[:, 1], -1)) - np.dot(np.roll(p[:, 0], -1), p[:, 1]))

    if area2(clip) < 0:
        clip = clip[::-1]
    out = subject
    for k in range(len(clip)):
        a, b = clip[k], clip[(k + 1) % len(clip)]
        if len(out) == 0:
            break
        side = (b[0] - a[0]) * (out[:, 1] - a[1]) - (b[1] - a[1]) * (out[:, 0] - a[0])
        nxt = []
        for i in range(len(out)):
            j = (i + 1) % len(out)
            if side[i] >= 0:
                nxt.append(out[i])
            if (side[i] >= 0) != (side[j] >= 0):
                t = side[i] / (side[i] - side[j])
                nxt.append(out[i] + t * (out[j] - out[i]))
        out = np.array(nxt).reshape(-1, 2)
    return out


def _centroid(p: np.ndarray) -> np.ndarray:
    if len(p) == 0:
        return np.array([np.nan, np.nan])
    x, y = p[:, 0], p[:, 1]
    xn, yn = np.roll(x, -1), np.roll(y, -1)
    cr = x * yn - xn * y
    a = cr.sum() / 2.0
    if a == 0.0:
        return p.mean(axis=0)
    return np.array([((x + xn) * cr).sum() / (6 * a), ((y + yn) * cr).sum() / (6 * a)])


class CollisionPointMetric(Metric):
    """
    ``(ref, point, angle)`` of every entity that starts colliding with the ego: the centroid of the
    overlap of the two boxes and the relative heading in [0, 2 pi) (reference metrics/collision.py:
    206-262).  Host-side metric (it runs per tick on the materialised state).  The reference reads the
    headings from ``entity.pose``, an attribute entities do not have at v0.3.1 (AttributeError on the
    first collision); the headings of ``state.poses`` -- the evident intent -- are used here.
    """

    name = "collision_points"

    def __init__(self, name: Optional[str] = None):
        self.ego: Optional[Entity] = None
        self.collisions: List[Tuple[str, np.ndarray, float]] = []
        super().__init__(name=name)

    def _reset(self, state) -> None:
        self.ego = state.scenario.ego
        self.collisions = []
        self.last_timestep: List[Entity] = []

    def _step(self, state) -> None:
        now = state.collisions().get(self.ego, [])
        for other in now:
            if other not in self.last_timestep:
                self.collisions.append(self.record_collision_position(state, other))
        self.last_timestep = list(now)

    def get_state(self):
        return self.collisions

    def record_collision_position(self, state, hazard: Entity):
        ego_box = self.ego.get_bounding_box_points(state.poses[self.ego])
        hazard_box = hazard.get_bounding_box_points(state.poses[hazard])
        point = _centroid(_clip_convex(ego_box, hazard_box))
        angle = (state.poses[hazard][3] - state.poses[self.ego][3]) % (np.pi * 2)
        return hazard.ref, point, float(angle)


# ------------------------------------------------------------------------------ pedestrians
class BehaviourParameters:
    max_speed_factor = 1.3

    def __init__(self, **kwargs):
        for k, v in kwargs.items():
            setattr(self, k, v)


class RandomWalkParameters(BehaviourParameters):
    bias_lon = 0.0
    bias_lat = 0.0
    std_lon = 0.000002
    std_lat = 0.0000001


class SocialForceParameters(RandomWalkParameters):
    """Parameters of the social force model (reference pedestrian/social_force.py:16-30)."""

    distance_threshold = 3
    sight_weight = 0.5
    sight_weight_use = True
    sight_angle = 200
    relaxation_time = 1.5
    ped_repulse_V = 1.0
    ped_repulse_sigma = 1.0
    ped_attract_C = 0.0
    boundary_repulse_U = 10.0
    boundary_repulse_R = 0.2
    imp_boundary_repulse_U = 2.0
    imp_boundary_repulse_R = 0.1


class SocialForce:
    """
    Social force behaviour (reference pedestrian/social_force.py:33-222), run on the device.

    With ``std_lon = std_lat = 0`` the rollout reproduces the reference.  With non-zero standard
    deviations (the reference's defaults are 2e-6 / 1e-7) the reference draws its fluctuations from
    numpy's global generator; the engine then adds N(0, std) noise from its own counter-based stream
    (``noise_seed``): statistically the same model, not the same numbers.
    """

    def __init__(self, params: SocialForceParameters, noise_seed: int = 0):
        self.params = params
        self.max_speed_factor = params.max_speed_factor
        self.noise_seed = int(noise_seed)


@dataclass
class PedestrianObservation(SingleEntityObservation):
    """Observation of a pedestrian (reference pedestrian/observation.py)."""

    head_rot_angle: float = 0.0
    near_peds: Any = None
    walkable_surface: Any = None
    impenetrable_surface: Any = None


class PedestrianSensor(Sensor):
    """
    Pedestrians within ``distance_threshold`` plus the road-network surfaces (reference
    pedestrian/sensor.py:9-64).  On the device the query is part of the fused tick; this host class
    serves custom agents that want the same observation.
    """

    def __init__(self, entity: Entity, head_rot_angle: float = 0.0, distance_threshold: float = 1.0):
        super().__init__(entity)
        self.head_rot_angle = head_rot_angle
        self.distance_threshold = distance_threshold

    def _reset(self, state):
        return self._step(state)

    def _step(self, state):
        rn = state.scenario.road_network
        return PedestrianObservation(
            self.entity, *state.get_entity_data(self.entity), self.head_rot_angle,
            self.get_nearby_pedestrians(state),
            None if rn is None else rn.walkable_surface, None if rn is None else rn.impenetrable_surface)

    def get_nearby_pedestrians(self, state):
        x, y = state.poses[self.entity][:2]
        return [(e, state.poses[e], state.velocities[e])
                for e in state.get_entities_in_radius(x, y, self.distance_threshold)
                if (isinstance(e, Pedestrian) or e.type == "Pedestrian") and e != self.entity]


class PedestrianController(Controller):
    """Moves the pedestrian by speed and heading (reference pedestrian/controller.py:9-46)."""

    def __init__(self, entity: Entity, max_speed: float = 5.0):
        super().__init__(entity)
        self.max_speed = max_speed

    def _reset(self, state) -> None:
        self.speed = np.linalg.norm(state.velocities[self.entity][:2])

    def _step(self, state, action: PedestrianAction):
        speed = np.clip(action.speed, -self.max_speed, self.max_speed)
        pose = state.poses[self.entity].copy()
        pose[0] += speed * state.dt * np.cos(action.heading)  # state.dt: the previous interval
        pose[1] += speed * state.dt * np.sin(action.heading)
        pose[3] = action.heading
        self.speed = speed
        return pose


class PedestrianAgent(Agent):
    """
    Pedestrian following a route with a behaviour model (reference pedestrian/agent.py:15-69).
    ``force`` and ``goal_idx`` read the device rows of the agent's slot once it is part of a gym.
    """

    def __init__(self, entity: Entity, route: List[np.ndarray], speed_desired: float,
                 behaviour: SocialForce, max_speed: float = 5.0, head_rot_angle: float = 0.0,
                 distance_threshold: float = 1.0):
        super().__init__(entity, PedestrianController(entity, max_speed=max_speed),
                         PedestrianSensor(entity, head_rot_angle=head_rot_angle,
                                          distance_threshold=distance_threshold))
        self.route = [np.asarray(r, dtype=np.float64) for r in route]
        self.speed_desired = speed_desired
        self.behaviour = behaviour
        self.max_speed = max_speed
        self.head_rot_angle = head_rot_angle
        self.distance_threshold = distance_threshold
        self._bound = None  # (gym, flat slot index) once lowered to the device
        self._goal_idx = 0
        self._force = np.array([0.0, 0.0])

    @property
    def force(self) -> np.ndarray:
        if self._bound is not None and self._bound[0]._engine is not None:
            gym, i = self._bound
            return np.array(gym._fetch("force")[:, i])
        return self._force

    @force.setter
    def force(self, value) -> None:
        self._force = np.asarray(value, dtype=np.float64)

    @property
    def goal_idx(self) -> int:
        if self._bound is not None and self._bound[0]._engine is not None:
            gym, i = self._bound
            return int(gym._fetch("goal_idx")[i])
        return self._goal_idx

    @goal_idx.setter
    def goal_idx(self, value: int) -> None:
        self._goal_idx = int(value)

    def reset(self, state) -> None:
        self._goal_idx = 0
        self._force = np.array([0.0, 0.0])
