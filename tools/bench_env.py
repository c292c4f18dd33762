#!/usr/bin/env python
"""
bench_env.py -- throughput of the closed-loop environment (VecScenarioEnv) and where its step goes.

    python tools/bench_env.py [--out FILE] [--lidar R]   # one JSON line per workload on stdout (and appended to FILE)

Workloads:
  vehicles  12 500 scenarios x 64 VehicleController entities (synthetic.vehicles_config, 625 distinct
            scenarios each 20 times: building 800 000 host-side entities one by one would dominate the run),
            every vehicle a PolicyAgent: the lean vehicle kernel, one tick per launch.
  xosc      4096 replicas of the reference's 23 test scenarios with the ego a PolicyAgent: the general kernel.
Observation: K = 8 neighbours within 50 m, lookahead 1 / 2 / 3 s, and with --lidar R > 0 a lidar of R rays
reaching 50 m (ObsSpec.lidar_rays; 0, the default, leaves the workloads as they were).  The policy is a trivial
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
  device / power_limit_w                the card and its power limit
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

sys.dont_write_bytecode = True
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

import torch  # noqa: E402

from scenario_gym_b200 import (BoundingBox, CatalogEntry, Entity, ObsSpec, Pedestrian, PolicyAgent,  # noqa: E402
                               Scenario, Trajectory, VecScenarioEnv, Vehicle, abi, synthetic)
from scenario_gym_b200.engine import Engine  # noqa: E402


def policy(obs):
    tx, ty = obs[..., 4], obs[..., 5]
    return torch.stack([(torch.sqrt(tx * tx + ty * ty) - obs[..., 0]).clamp(-5.0, 5.0),
                        torch.atan2(ty, tx).clamp(-0.7, 0.7)], -1)


def vehicles_env(obs):
    distinct, reps, M = 625, 20, 64
    cfg = synthetic.vehicles_config(seed=0, N=distinct, M=M, T=256)
    rows = synthetic.two_knot_rows(cfg).reshape(distinct, M, 2, 7)
    ce = CatalogEntry(None, "car1", "car", "Vehicle", BoundingBox(*synthetic.CAR1_BOX))
    scs = [Scenario([Vehicle(ce, trajectory=Trajectory(rows[n, m]), ref="ego" if m == 0 else f"entity_{m}")
                     for m in range(M)]) for n in range(distinct)]
    return VecScenarioEnv(scs * reps, create_agent=lambda s, e: PolicyAgent(e), timestep=cfg.dt, obs=obs)


def xosc_env(obs):
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
    return VecScenarioEnv([scs[k % len(scs)] for k in range(4096)], obs=obs)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(out.splitlines()[0])
    except Exception:  # the limit is reported as unknown rather than guessed
        power = None
    return name, power


def measure(name, env):
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
        "library": os.path.basename(abi.PRODUCT_LIB),
        "device": dev, "power_limit_w": power,
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--workloads", default="vehicles,xosc")
    ap.add_argument("--lidar", type=int, default=0, help="lidar rays R of the observation (0: no lidar block)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_env.py measures the GPU engine: no CUDA device")
    obs = ObsSpec(k_neighbours=8, radius=50.0, lookahead=(1.0, 2.0, 3.0), lidar_rays=args.lidar, lidar_range=50.0)
    for w in args.workloads.split(","):
        t0 = time.time()
        env = {"vehicles": vehicles_env, "xosc": xosc_env}[w](obs)
        build_s = time.time() - t0
        rec = measure(w, env)
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
