"""CPU tests of the host-side mirror of the reference interface (no device calls)."""
import os

import numpy as np
import pytest

from scenario_gym_b200 import (BoundingBox, CatalogEntry, Entity, Metric, Scenario, ScenarioGym,
                               Trajectory, Vehicle, import_scenario)
from scenario_gym_b200.packing import build_union_table, call_linear_clamped

from helpers import golden, manifest, sub

DATA = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data")


def test_position_at_t_truth_table():
    """The reference's own truth table, tests/test_trajectory.py:166-228."""
    data = np.array([[0, 0, 0], [1, 1, 1], [2, 2, 2]])
    traj = Trajectory(data, fields=["t", "x", "y"])
    assert np.allclose(traj.position_at_t(0.5, extrapolate=True)[:2], [0.5, 0.5])
    assert np.allclose(traj.position_at_t(1.5, extrapolate=True)[:2], [1.5, 1.5])
    traj.position_at_t(1)
    assert np.allclose(traj.position_at_t(2.5, extrapolate=True)[:2], [2.5, 2.5])
    assert np.allclose(traj.position_at_t(-1.0, extrapolate=True)[:2], [-1.0, -1.0])
    assert traj.position_at_t(-1.0, extrapolate=False) is None
    assert traj.position_at_t(3.0, extrapolate=False) is None
    assert np.allclose(traj.position_at_t(-1.0, extrapolate=(False, True))[:2], [0.0, 0.0])
    assert np.allclose(traj.position_at_t(-1.0, extrapolate=(True, True))[:2], [-1.0, -1.0])
    assert np.allclose(traj.position_at_t(3.0, extrapolate=(True, False))[:2], [2.0, 2.0])
    assert np.allclose(traj.position_at_t(3.0, extrapolate=(True, True))[:2], [3.0, 3.0])
    assert np.allclose(traj.position_at_t(data[:, 0], extrapolate=True)[:, :2], data[:, 1:])
    x = np.array([-1.0, 3.0])
    assert np.allclose(traj.position_at_t(x, extrapolate=True)[:, :2], [[-1.0, -1.0], [3.0, 3.0]])
    assert np.allclose(traj.position_at_t(x, extrapolate=False)[:, :2], [[0.0, 0.0], [2.0, 2.0]])
    assert np.allclose(traj.position_at_t(x, extrapolate=(False, True))[:, :2], [[0, 0], [3.0, 3.0]])
    assert np.allclose(traj.position_at_t(x, extrapolate=(True, False))[:, :2], [[-1.0, -1.0], [2.0, 2.0]])


def test_trajectory_construction():
    """Dedup, heading fill, z/p/r fill (reference tests/test_trajectory.py:49-110)."""
    traj = Trajectory(np.array([[0.0, 0, 0, 0], [1.0, 0, 0, 0], [1.0, 0, 0, 0], [2.0, 0, 0, 0],
                                [3.0, 0, 0, 0.5]]), fields=["t", "x", "y", "h"])
    assert traj.data.shape[0] == 4
    traj = Trajectory(np.array([[0, 0, 0], [1, 1, 1], [2, 2, 2]]), fields=["t", "x", "y"])
    assert np.allclose(traj.h, np.ones(3) * np.pi / 4)
    assert np.allclose(traj.z, 0) and np.allclose(traj.p, 0) and np.allclose(traj.r, 0)
    with pytest.raises(ValueError):
        Trajectory(np.zeros((3, 2)), fields=["t", "x"])
    with pytest.raises(ValueError):
        traj.data[0, 0] = 1.0  # read-only


def test_trajectory_matches_reference_vectors():
    g = sub(golden("unit"), "unit")
    tr = Trajectory(g["traj_data"])
    assert np.array_equal(tr.data, g["traj_data"])
    for mode, ext in ((0, False), (1, (False, False)), (2, True)):
        for t, want in zip(g["traj_ts"], g[f"traj_pos_mode{mode}"]):
            got = tr.position_at_t(float(t), extrapolate=ext)
            if np.isnan(want).all():
                assert got is None
            else:
                assert np.array_equal(got, want)
    for t, want in zip(g["traj_ts"], g["traj_vel"]):
        assert np.array_equal(tr.velocity_at_t(float(t)), want)
    one = Trajectory(g["traj1_data"])
    for t, want in zip(g["traj_ts"], g["traj1_pos_mode2"]):
        assert np.array_equal(one.position_at_t(float(t), extrapolate=True), want)


def test_bounding_box_points_match_reference():
    g = sub(golden("unit"), "unit")
    W, L, cx, cy = manifest()["unit"]["box"]
    e = Entity(CatalogEntry(None, "x", "car", "Vehicle", BoundingBox(W, L, cx, cy)), ref="x")
    for pose, want in zip(g["box_pose"], g["box_points"]):
        assert np.array_equal(e.get_bounding_box_points(pose), want)


def test_union_table_matches_scipy():
    """BatchReplayEntity table restated in numpy equals scipy's interp1d bit for bit."""
    interp1d = pytest.importorskip("scipy.interpolate").interp1d
    rng = np.random.default_rng(0)
    trajs = []
    for K in (1, 5, 9):
        d = np.zeros((K, 7))
        d[:, 0] = np.sort(rng.uniform(0, 10, K))
        d[:, 1:] = rng.normal(size=(K, 6))
        trajs.append(d)
    ts, X = build_union_table(trajs)
    for j, d in enumerate(trajs):
        d = d.copy()
        if len(d) == 1:
            d = np.repeat(d, 2, axis=0)
            d[-1, 0] += 1e-1
        want = interp1d(d[:, 0], d[:, 1:].T, bounds_error=False, fill_value=(d[0, 1:], d[-1, 1:]))(ts).T
        assert np.array_equal(X[:, j], want)


def test_import_demo_scenario():
    sc = import_scenario(os.path.join(DATA, "Scenarios", "demo.xosc"))
    assert [e.ref for e in sc.entities] == ["ego", "vehicle_0", "pedestrian_0", "vehicle_1"]
    assert sc.ego is sc.entities[0]
    assert sc.entities[3].is_static() and not sc.entities[1].is_static()
    bb = sc.entities[0].bounding_box
    assert (bb.width, bb.length, bb.center_x, bb.center_y) == (1.9, 4.1, 1.3, 0.0)
    assert sc.entities[2].type == "Pedestrian" and sc.entities[2].etype() == 1
    assert np.isclose(sc.length, 10.0)
    assert np.allclose(sc.entities[1].trajectory.h, np.pi)  # given headings are kept (unwrapped)
    assert np.allclose(sc.entities[2].trajectory.h, np.pi / 2)  # filled from the direction of travel
    unl = import_scenario(os.path.join(DATA, "Scenarios", "demo.xosc"), relabel=False)
    assert [e.ref for e in unl.entities] == ["ego", "oncoming", "crossing", "parked"]
    with pytest.raises(FileNotFoundError):
        import_scenario("/nonexistent.xosc")


def test_missing_required_callback_raises():
    """reference metrics/base.py:44-53"""
    import torch

    from scenario_gym_b200 import RSS

    sc = import_scenario(os.path.join(DATA, "Scenarios", "demo.xosc"))
    gym = ScenarioGym(metrics=[RSS()])
    if torch.cuda.is_available():
        with pytest.raises(ValueError, match="without callback"):
            gym.set_scenario(sc)
    else:
        with pytest.raises((ValueError, RuntimeError)):
            gym.set_scenario(sc)


def test_batched_ingest_matches_single_imports():
    """import_scenarios (catalog cache, optional process pool) == a loop of import_scenario."""
    import os

    from scenario_gym_b200.xosc import import_scenario, import_scenarios

    f = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data", "Scenarios", "demo.xosc")
    one = import_scenario(f)
    for workers in (1, 2):
        many = import_scenarios([f] * 5, workers=workers)
        assert len(many) == 5
        for sc in many:
            assert [e.ref for e in sc.entities] == [e.ref for e in one.entities]
            for a, b in zip(sc.entities, one.entities):
                assert np.array_equal(a.trajectory.data, b.trajectory.data)
                assert a.bounding_box == b.bounding_box
    with pytest.raises(FileNotFoundError):
        import_scenarios([f, f + ".missing"])


def test_combine_observations_fields_and_prefixes():
    """Reference observation.py:31-83: first definition of a field wins; prefixes keep repeats."""
    import dataclasses

    from scenario_gym_b200.plugins import (CollisionObservation, FutureCollisionObservation,
                                           SingleEntityObservation, combine_observations)

    C = combine_observations(SingleEntityObservation, FutureCollisionObservation, CollisionObservation)
    names = [f.name for f in dataclasses.fields(C)]
    assert names[:8] == [f.name for f in dataclasses.fields(SingleEntityObservation)]
    assert names[8:] == ["future_collision", "collisions"]
    a = SingleEntityObservation("e", 1.0, 2.0, "pose", "vel", 3.0, "rec", None)
    b = FutureCollisionObservation("e", 1.0, 2.0, "pose", "vel", 3.0, "rec", None, True)
    c = CollisionObservation("e", 1.0, 2.0, "pose", "vel", 3.0, "rec", None, {"x": []})
    obs = C.from_obs(a, b, c)
    assert obs.entity == "e" and obs.future_collision is True and obs.collisions == {"x": []}
    P = combine_observations(SingleEntityObservation, FutureCollisionObservation, prefixes=("a", "b"))
    pn = [f.name for f in dataclasses.fields(P)]
    assert "b_pose" in pn and "future_collision" in pn and pn.count("pose") == 1
    with pytest.raises(ValueError):
        combine_observations(SingleEntityObservation, prefixes=("a", "b"))


def test_scenario_json_round_trip_and_actions(tmp_path):
    """Scenario.to_json / from_json (reference scenario.py:186-319) incl. actions; action trigger rules."""
    import numpy as np

    from scenario_gym_b200 import (BoundingBox, CatalogEntry, Pedestrian, Scenario, Trajectory,
                                   UpdateStateVariableAction, Vehicle)

    ce = CatalogEntry(None, "car1", "car", "Vehicle", BoundingBox(2.0, 4.2, 1.37, 0.0), {"mass": 1.0}, ["m.osgb"])
    pe = CatalogEntry(None, "ped", "pedestrian", "Pedestrian", BoundingBox(0.69, 0.7, 0.0, 0.0))
    ego = Vehicle(ce, trajectory=Trajectory(np.array([[0.0, 0, 0, 0, 0, 0, 0], [4.0, 20, 1, 0, 0.1, 0, 0]])), ref="ego")
    ped = Pedestrian(pe, trajectory=Trajectory(np.array([[1.0, 5, 5, 0, 0, 0, 0]])), ref="ped_0")
    sc = Scenario([ego, ped], name="rt", properties={"k": 1})
    sc.add_action(UpdateStateVariableAction(3.0, "TestAction", "ego", {"var": 1.0}), inplace=True)
    path = str(tmp_path / "rt.json")
    sc.to_json(path)
    back = Scenario.from_json(path)
    assert [type(e).__name__ for e in back.entities] == ["Vehicle", "Pedestrian"]
    for a, b in zip(sc.entities, back.entities):
        assert a.ref == b.ref and np.array_equal(a.trajectory.data, b.trajectory.data)
        assert a.catalog_entry == b.catalog_entry
    assert back.properties == {"k": 1} and back.name == "rt" and back.road_network is None
    act = back.actions[0]
    assert isinstance(act, UpdateStateVariableAction) and act.t == 3.0 and act.action_variables == {"var": 1.0}
    shifted = back.reset_start(back.entities[1])  # pedestrian starts at t = 1
    assert shifted.entities[0].trajectory.min_t == -1.0 and shifted.actions[0].t == 2.0 and back.actions[0].t == 3.0

    class FakeState:
        def __init__(self, t):
            self.t = t
            self.entity_state = {ego: None}

    assert not act.trigger_condition(FakeState(3.0)) and act.trigger_condition(FakeState(3.0000001))
    st = FakeState(3.5)
    act.apply(st, ego)
    assert st.entity_state[ego] == {"var": 1.0}


def test_road_network_surfaces_host():
    """RoadNetwork surfaces: class flags, point membership incl. holes, packing for the device."""
    from oracle import golden_cases
    from scenario_gym_b200.packing import pack_road_networks

    rn = golden_cases.road_network(golden_cases.ROAD_PED_GEOMETRY)
    d, w, i = rn.surfaces()
    assert (len(d), len(w), len(i)) == (1, 3, 2)  # buildings are walkable too (reference class flags)
    assert i.contains(2.0, 2.0) and not i.contains(1.8, 2.0) and not i.contains(4.5, 1.3)  # boundary / L notch
    pav = w.polygons[0]
    assert pav.contains(3.0, 3.0) and not pav.contains(0.5, 4.2) and pav.point_side(0.2, 4.0) == 0  # hole
    assert abs(pav.area - (81.0 - 0.49)) < 1e-12
    names, geoms = rn.get_geometries_at_point(2.0, 2.0)
    assert sorted(names) == ["Building", "Pavement"]
    rn_of, poly_off, edge_off, edges, has_area = pack_road_networks([rn, None, rn])
    assert rn_of.tolist() == [0, -1, 0] and poly_off.tolist() == [0, 1, 4, 6] and has_area.tolist() == [1, 1, 1]
    assert edges.shape == (edge_off[-1], 4) and edge_off[1] == 4 and edge_off[2] - edge_off[1] == 8


def test_union_times_equal_the_set_formulation():
    """packing.build_union_times (numpy) == sorted(set(...)) over the trajectories as BatchReplayEntity holds them
    (entity/batch.py:88-99): NaN times become 0, a single control point is held twice 0.1 s apart, duplicates merge."""
    from scenario_gym_b200.packing import _batch_data, build_union_times

    rng = np.random.default_rng(5)
    for trial in range(100):
        trajs = []
        for _ in range(int(rng.integers(1, 7))):
            K = int(rng.integers(1, 9))
            d = rng.normal(size=(K, 7))
            d[:, 0] = np.sort(rng.choice(np.arange(24) * 0.125, K, replace=False))
            if rng.random() < 0.2:
                d[int(rng.integers(0, K)), 0] = np.nan
            trajs.append(d)
        want = np.array(sorted(set(t for data in trajs for t in _batch_data(data)[:, 0])))
        got = build_union_times(trajs)
        assert got.dtype == np.float64 and np.array_equal(got, want), trial
    assert build_union_times([]).shape == (0,)
