#!/usr/bin/env python
"""
bench_env.py -- throughput of the closed-loop environment (VecScenarioEnv) and where its step goes.

    python tools/bench_env.py [--out FILE] [--lidar R] [--map Km] [--reset]   # one JSON line per workload on
                              [--raster S [--raster-brute LIB]]               # stdout (and appended to FILE)

Workloads:
  vehicles  12 500 scenarios x 64 VehicleController entities (synthetic.vehicles_config, 625 distinct
            scenarios each 20 times: building 800 000 host-side entities one by one would dominate the run),
            every vehicle a PolicyAgent: the lean vehicle kernel, one tick per launch.
  xosc      4096 replicas of the reference's 23 test scenarios with the ego a PolicyAgent: the general kernel.
Observation: K = 8 neighbours within 50 m, lookahead 1 / 2 / 3 s, and with --lidar R > 0 a lidar of R rays
reaching 50 m (ObsSpec.lidar_rays; 0, the default, leaves the workloads as they were).  With --map Km > 0 every
scenario drives over a synthetic town (synthetic.grid_town: the vehicles' 400 m square, or one town over the 23 test
scenes' trajectory points, 0.5 .. 99.5 % range) and observes its Km nearest road-network edges within 50 m (ObsSpec.map_edges; 0, the default, attaches no
town and leaves the workloads as they were).  --raster S > 0 attaches the same town and gives every agent a bird's-eye
raster of S x S pixels of 0.5 m (ObsSpec.raster_size).  The policy is a trivial
torch function of the observation (steer toward the first lookahead point).  SG_B200_LIB selects the library
(e.g. a variant built by tools/build_variant.sh); `library` in the record names it.

Reported per workload:
  env_steps_per_s / agent_steps_per_s   step() + policy, host clock over >= 1 s ending in a synchronise
  host_enqueue_us_per_step              host time of step() + policy without a synchronise
  device_us_per_step                    a separate pass with CUDA events between the phases of a step:
                                        tick (action scatter + one-tick rollout), reward, observe, reset, observe_reset
  fused_us_per_tick                     rollout() of the same scene, 64 ticks in one launch, actions drawn in the kernel
  observe_bytes / observe_GBps          bytes sg_env_observe writes (obs, agent mask, snapshot) over its kernel time
  lidar_rays / lidar_bytes              R and the bytes of the lidar block (part of observe_bytes)
  map_edges / map_table_edges / map_bytes   Km, the edges of the town's map table, the bytes of the map block
  map_us / map_brute_us                 the map kernel's time per observe (observe with the map block minus observe
                                        without it, CUDA events over 50 calls each), with the env's culling grid and
                                        with the same table built as a single cell (brute force, same kernel)
  reset_{full,1pct}_{plain,init}_us     with --reset (the envs are then built with RESET_SPEC: randomised starts
                                        and perturbed agents): the masked reset's device time (CUDA events over 20
                                        calls) with every scenario / every 100th selected, through the plain kernel
                                        (sg_reset_scenarios) and the init kernel (sg_reset_scenarios_init)
  env_steps_per_s_spec / _plain         with --reset: step() + policy with the spec's auto-reset, and with the plain
                                        one (env.reset_spec = None), host clock over >= 1 s each
  raster_size / raster_bytes            with --raster: S and the bytes one sg_env_raster call writes (N*A*5*S*S)
  raster_us / raster_TBps / raster_floor_us   its device time per call (CUDA events over 20 calls, every scenario),
                                        the write rate, and the time the bytes take at 7.7 TB/s
  raster_brute_us                       with --raster-brute LIB: the same call through LIB, a library built with
                                        -DSG_RASTER_BRUTE (tools/build_variant.sh), on the same buffers
  env_steps_per_s_raster / _no_raster   with --raster: step() + policy with the raster, and without it (the same env
                                        with its raster switched off), host clock over >= 1 s each
  device / power_limit_w                the card and its power limit
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import time

sys.dont_write_bytecode = True
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from scenario_gym_b200 import (BoundingBox, CatalogEntry, Entity, ObsSpec, Pedestrian, PolicyAgent,  # noqa: E402
                               ResetSpec, Scenario, Trajectory, VecScenarioEnv, Vehicle, abi, synthetic)
from scenario_gym_b200.engine import Engine  # noqa: E402


def policy(obs):
    tx, ty = obs[..., 4], obs[..., 5]
    return torch.stack([(torch.sqrt(tx * tx + ty * ty) - obs[..., 0]).clamp(-5.0, 5.0),
                        torch.atan2(ty, tx).clamp(-0.7, 0.7)], -1)


# --reset: episodes start up to 2 s into the log with every agent's start perturbed
RESET_SPEC = ResetSpec(start_offset=2.0, min_remaining=1.0, lon=0.5, lat=0.2, heading=0.05, speed=1.0, seed=0)


def vehicles_env(obs, reset_spec=None):
    distinct, reps, M = 625, 20, 64
    cfg = synthetic.vehicles_config(seed=0, N=distinct, M=M, T=256)
    rows = synthetic.two_knot_rows(cfg).reshape(distinct, M, 2, 7)
    ce = CatalogEntry(None, "car1", "car", "Vehicle", BoundingBox(*synthetic.CAR1_BOX))
    town = synthetic.grid_town(seed=0, half_extent=200.0) if obs.map_edges > 0 or obs.raster_size > 0 else None
    scs = [Scenario([Vehicle(ce, trajectory=Trajectory(rows[n, m]), ref="ego" if m == 0 else f"entity_{m}")
                     for m in range(M)], road_network=town) for n in range(distinct)]
    return VecScenarioEnv(scs * reps, create_agent=lambda s, e: PolicyAgent(e), timestep=cfg.dt, obs=obs,
                          reset_spec=reset_spec)


def xosc_env(obs, reset_spec=None):
    sys.path.insert(0, os.path.join(REPO, "tests"))
    from helpers import golden, manifest, sub

    g, man = golden("xosc"), manifest()["xosc"]
    cls = {abi.ETYPE_VEHICLE: (Vehicle, "Vehicle"), abi.ETYPE_PEDESTRIAN: (Pedestrian, "Pedestrian")}
    scs = []
    for name in sorted(man):
        inp = sub(g, f"xosc/{name}/in")
        ents = []
        for i in range(int(inp["n_entities"])):
            C, ctype = cls.get(int(inp["etype"][i]), (Entity, "MiscObject"))
            ce = CatalogEntry(None, "entry", None, ctype, BoundingBox(*[float(v) for v in inp["box"][i]]))
            ents.append(C(ce, trajectory=Trajectory(inp[f"traj{i}"]), ref=man[name]["refs"][i]))
        scs.append(Scenario(ents))
    if obs.map_edges > 0 or obs.raster_size > 0:  # one town over the test scenes: the 0.5 .. 99.5 % range of their trajectory points
        # (one scene has a stray point thousands of km away, which a town cannot sensibly cover)
        xy = np.concatenate([np.asarray(e.trajectory.data)[:, 1:3] for sc in scs for e in sc.entities])
        lo, hi = np.quantile(xy, 0.005, axis=0), np.quantile(xy, 0.995, axis=0)
        town = synthetic.grid_town(seed=0, half_extent=float((hi - lo).max()) / 2 + 20.0, center=(lo + hi) / 2)
        for sc in scs:
            sc.road_network = town
    return VecScenarioEnv([scs[k % len(scs)] for k in range(4096)], obs=obs, reset_spec=reset_spec)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(out.splitlines()[0])
    except Exception:  # the limit is reported as unknown rather than guessed
        power = None
    return name, power


def measure(name, env, brute_lib=None):
    eng = env._engine
    stream = torch.cuda.current_stream()
    o, _ = env.reset()
    for _ in range(20):  # warm-up: module loads, allocator, every launch shape of a step
        o, *_ = env.step(policy(o))
    torch.cuda.synchronize()
    # host enqueue time (no synchronise inside the window)
    t0 = time.perf_counter()
    n_enq = 30
    for _ in range(n_enq):
        o, *_ = env.step(policy(o))
    enqueue_us = (time.perf_counter() - t0) / n_enq * 1e6
    torch.cuda.synchronize()
    # end to end over >= 1 s
    steps, t0 = 0, time.perf_counter()
    while True:
        for _ in range(10):
            o, *_ = env.step(policy(o))
        steps += 10
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if dt >= 1.0:
            break
    n_agents = int((env.agent_slots >= 0).sum().item())
    # device split: the phases of VecScenarioEnv.step with events between them (same calls, same order)
    names = ("tick", "reward", "observe", "reset", "observe_reset")
    acc = dict.fromkeys(names, 0.0)
    reps = 50
    for _ in range(reps):
        a = policy(o)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(names) + 1)]
        ev[0].record(stream)
        buf = env._act[a.dtype]
        buf[0].index_copy_(1, env._dst, a.reshape(env.N * env.A, 2).index_select(0, env._src).t())
        eng.rollout(1, actions=buf)
        ev[1].record(stream)
        eng.env_reward(env._spec, env._reward, env._terms, env._terminated, env._truncated)
        ev[2].record(stream)
        eng.env_observe(env._spec, env._obs, env._agent_mask)
        ev[3].record(stream)
        env._final_obs.copy_(env._obs)
        for k, f in (("ego_avg_speed", "ego_avg_speed"), ("ego_max_speed", "ego_max_speed"),
                     ("ego_distance_travelled", "ego_dist"), ("first_coll_tick", "first_coll_tick"),
                     ("rss_flags", "rss_flags"), ("tick", "tick"), ("t", "t")):
            env._final[k].copy_(eng.tensor(f))
        torch.bitwise_or(env._terminated, env._truncated, out=env._finished)
        eng.reset(mask=env._finished)
        ev[4].record(stream)
        eng.env_observe(env._spec, env._obs, env._agent_mask, mask=env._finished)
        env._episode.add_(env._finished)
        eng.tensor("event_count").zero_()
        ev[5].record(stream)
        o = env._obs
        torch.cuda.synchronize()
        for k, nm in enumerate(names):
            acc[nm] += ev[k].elapsed_time(ev[k + 1]) * 1e3 / reps
    # fused rollout of the same scene: 64 ticks in one launch, actions from the in-kernel PCG64 stream
    fused = Engine(eng.scene, eng.params, device=eng.dev_index)
    rng = synthetic.vehicles_config(seed=1, N=eng.N, M=eng.M, T=64, materialise=False).action_rng
    fused.reset()
    fused.rollout(8, actions=rng)
    fused.reset()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    fused.rollout(64, actions=rng)
    e1.record(stream)
    torch.cuda.synchronize()
    fused_tick_us = e0.elapsed_time(e1) * 1e3 / 64
    assert int(fused.get("tick").min()) == 64, "every scenario must run the 64 timed ticks"
    del fused
    maps = map_times(env) if env.obs_spec.map_edges > 0 else {}
    resets = reset_times(env) if env.reset_spec is not None else {}
    rasters = raster_times(env, brute_lib) if env.obs_spec.raster_size > 0 else {}
    F = env.n_features
    obs_bytes = env.N * env.A * (4 * F + 1 + 9) + env.N * 9
    dev, power = card()
    return {
        "workload": name, "N": env.N, "M": eng.M, "A": env.A, "agents": n_agents, "F": F,
        "k_neighbours": env.obs_spec.k_neighbours, "lookahead": list(env.obs_spec.lookahead),
        "env_steps_per_s": steps / dt, "agent_steps_per_s": steps * n_agents / dt, "timed_steps": steps,
        "timed_s": dt, "host_enqueue_us_per_step": enqueue_us,
        "device_us_per_step": {k: round(v, 2) for k, v in acc.items()},
        "device_us_per_step_total": round(sum(acc.values()), 2),
        "fused_us_per_tick": fused_tick_us,
        "observe_bytes": obs_bytes, "observe_GBps": obs_bytes / (acc["observe"] * 1e-6) / 1e9,
        "lidar_rays": int(env.obs_spec.lidar_rays), "lidar_bytes": env.N * env.A * 4 * int(env.obs_spec.lidar_rays),
        "map_edges": int(env.obs_spec.map_edges), "map_bytes": env.N * env.A * 40 * int(env.obs_spec.map_edges),
        **maps, **resets, **rasters,
        "library": os.path.basename(abi.PRODUCT_LIB),
        "device": dev, "power_limit_w": power,
    }


def map_times(env):
    """The map kernel's time per observe: observe with the env's spec minus observe with map_edges = 0, and the
    same with the table built as a single cell (brute force through the same kernel)."""
    eng, sc, stream = env._engine, env._engine.scene, torch.cuda.current_stream()
    plain = abi.SgEnvSpec.from_buffer_copy(env._spec)
    plain.map_edges = 0
    brute = abi.SgEnvSpec.from_buffer_copy(env._spec)
    table = abi.map_table(sc.rn_poly_off, sc.rn_edge_off, sc.rn_edges, env.obs_spec.map_radius, cell=math.inf)
    keep = {k: torch.from_numpy(np.ascontiguousarray(a)).to(env.device) for k, a in table.items()}
    for k, t in keep.items():
        setattr(brute, k, t.data_ptr())

    def observe_us(spec, reps=50):
        for _ in range(3):
            eng.env_observe(spec, env._obs, env._agent_mask)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            eng.env_observe(spec, env._obs, env._agent_mask)
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / reps

    base, grid, flat = observe_us(plain), observe_us(env._spec), observe_us(brute)
    dims = env._map["map_dims"].cpu().numpy()
    return {"map_table_edges": int(env._map["map_off"][-1].item()), "map_grid_cells": int((dims[:, 0] * dims[:, 1]).sum()),
            "map_cell_m": float(env._map["map_grid"][0, 2].item()), "observe_no_map_us": round(base, 2),
            "map_us": round(grid - base, 2), "map_brute_us": round(flat - base, 2)}


def raster_times(env, brute_lib=None):
    """sg_env_raster's device time per call (every scenario), through the product and, given a library built with
    -DSG_RASTER_BRUTE, through it on the same buffers; the env's steps per second with and without its raster."""
    import ctypes as C

    eng, stream = env._engine, torch.cuda.current_stream()
    S = int(env.obs_spec.raster_size)

    def raster_us(call, reps):
        for _ in range(2):
            call()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            call()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / reps

    nbytes = env._raster.numel()
    out = {"raster_size": S, "raster_resolution": float(env.obs_spec.raster_resolution), "raster_bytes": nbytes,
           "raster_polygons": int(len(eng.scene.rn_edge_off) - 1)}
    us = raster_us(lambda: eng.env_raster(env._spec, env._rspec, env._raster), 20)
    out.update(raster_us=round(us, 2), raster_TBps=round(nbytes / (us * 1e-6) / 1e12, 3),
               raster_floor_us=round(nbytes / 7.7e12 * 1e6, 2))
    if brute_lib:
        lib = abi.bind(C.CDLL(os.path.abspath(brute_lib)), "sg_")
        want = env._raster.clone()

        def brute():
            rc = lib["env_raster"](C.byref(eng._sc), C.byref(eng.params), C.byref(eng._st), C.byref(env._spec),
                                   C.byref(env._rspec), None, env._raster.data_ptr(), eng.dev_index, eng._stream())
            if rc:
                raise RuntimeError(lib["last_error"]().decode())

        out["raster_brute_us"] = round(raster_us(brute, 3), 2)
        out["raster_brute_equal"] = bool(torch.equal(want, env._raster))
        out["raster_brute_library"] = os.path.basename(brute_lib)
        del want
    out["env_steps_per_s_raster"] = steps_per_s(env)
    keep, env._raster = env._raster, None  # (step() skips the raster)
    out["env_steps_per_s_no_raster"] = steps_per_s(env)
    env._raster = keep
    return out


def steps_per_s(env):
    """step() + policy per second, host clock over >= 1 s ending in a synchronise (after 20 warm-up steps)."""
    o, _ = env.reset()
    for _ in range(20):
        o, *_ = env.step(policy(o))
    torch.cuda.synchronize()
    steps, t0 = 0, time.perf_counter()
    while True:
        for _ in range(10):
            o, *_ = env.step(policy(o))
        steps += 10
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if dt >= 1.0:
            return steps / dt


def reset_times(env):
    """The masked reset's device time through the plain and the init kernel, for a full and a 1 % mask, and the
    env's steps per second with its spec and with the plain auto-reset."""
    eng, stream = env._engine, torch.cuda.current_stream()
    n = torch.arange(env.N, device=env.device)
    masks = {"full": torch.ones(env.N, dtype=torch.uint8, device=env.device),
             "1pct": (n % 100 == 0).to(torch.uint8)}

    def reset_us(mask, init, reps=20):
        for _ in range(3):
            eng.reset(mask=mask, init=init)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            eng.reset(mask=mask, init=init)
        e1.record(stream)
        torch.cuda.synchronize()
        return round(e0.elapsed_time(e1) * 1e3 / reps, 2)

    out = {"reset_spec": {k: getattr(env.reset_spec, k) for k in ("start_offset", "min_remaining", "lon", "lat",
                                                                   "heading", "speed")}}
    for k, m in masks.items():
        out[f"reset_{k}_plain_us"] = reset_us(m, None)
        out[f"reset_{k}_init_us"] = reset_us(m, env._init)
    spec = env.reset_spec
    out["env_steps_per_s_spec"] = steps_per_s(env)
    env.reset_spec = None  # (the env's plain auto-reset: sg_reset_scenarios)
    out["env_steps_per_s_plain"] = steps_per_s(env)
    env.reset_spec = spec
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--workloads", default="vehicles,xosc")
    ap.add_argument("--lidar", type=int, default=0, help="lidar rays R of the observation (0: no lidar block)")
    ap.add_argument("--map", type=int, default=0, help="map edges Km of the observation (0: no town, no map block)")
    ap.add_argument("--reset", action="store_true", help="build the envs with RESET_SPEC and time the resets")
    ap.add_argument("--raster", type=int, default=0, help="raster size S (0: no town, no raster)")
    ap.add_argument("--raster-brute", default=None, help="a library built with -DSG_RASTER_BRUTE to time as well")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_env.py measures the GPU engine: no CUDA device")
    obs = ObsSpec(k_neighbours=8, radius=50.0, lookahead=(1.0, 2.0, 3.0), lidar_rays=args.lidar, lidar_range=50.0,
                  map_edges=args.map, map_radius=50.0, raster_size=args.raster, raster_resolution=0.5)
    for w in args.workloads.split(","):
        t0 = time.time()
        env = {"vehicles": vehicles_env, "xosc": xosc_env}[w](obs, RESET_SPEC if args.reset else None)
        build_s = time.time() - t0
        rec = measure(w, env, args.raster_brute)
        rec["build_s"] = round(build_s, 1)
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")
        del env
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
