"""
scenario_gym_b200 -- B200-native batched rollout engine behind Scenario Gym's plugin API.

The names exported here mirror ``scenario_gym/__init__.py`` of the reference for the per-tick
rollout path; the arithmetic runs in hand-written sm_100a kernels (``csrc/``) reached through
the C ABI of ``include/sg_b200.h``.  Importing the package does not need a GPU; constructing a
gym / engine does (there is no CPU fallback).
"""
from .actions import FixedTAction, ScenarioAction, UpdateStateVariableAction, UserDefinedAction
from .entity import BoundingBox, CatalogEntry, Entity, MiscObject, Pedestrian, Vehicle
from .env import ObsSpec, VecScenarioEnv
from .gym import ScenarioGym
from .plugins import (RSS, Action, ActionTableAgent, Agent, CollisionMetric, CollisionObservation,
                      CombinedSensor, Controller, GlobalCollisionDetector, combine_observations,
                      EgoAvgSpeed, EgoDistanceTravelled, EgoLocalizationSensor, EgoMaxSpeed,
                      FutureCollisionDetector, FutureCollisionObservation, Metric,
                      Observation, PedestrianAction, PedestrianAgent, PIDAgent, PIDController, PolicyAgent, ReplayTrajectoryAgent,
                      ReplayTrajectoryController, RSSDistances, RSSParameters, Sensor,
                      SingleEntityObservation, SocialForce, SocialForceParameters, StateCallback,
                      TeleportAction, VehicleAction, VehicleController, cache_mean, cache_metric,
                      CollisionPointMetric, PedestrianController, RandomActionAgent, RandomActionSource, PedestrianObservation, PedestrianSensor)
from .road_network import RoadNetwork
from .scenario import Scenario
from .state import State
from .trajectory import Trajectory
from .xosc import import_scenario, import_scenarios, read_catalog, relabel_scenario

__all__ = [n for n in dir() if not n.startswith("_")]
