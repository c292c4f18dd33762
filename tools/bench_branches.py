#!/usr/bin/env python
"""
bench_branches.py -- cost of branched look-ahead rollouts (VecScenarioEnv.branches / BranchRollout.run) against
stepping the env.

    python tools/bench_branches.py [--out FILE]   # one JSON line per workload on stdout (and appended to FILE)

Workloads (the two of tools/bench_env.py, same observation: K = 8 within 50 m, lookahead 1 / 2 / 3 s):
  vehicles  12 500 scenarios x 64 PolicyAgent vehicles, B = 8 branches of H = 30 ticks (the lean vehicle kernel)
  xosc      4096 replicas of the reference's test scenarios, ego a PolicyAgent, B = 64, H = 30 (general kernel)
The env is stepped 10 times with the bench_env policy first, so the fork starts from a live mid-episode state;
branch actions are uniform random fp32.

Reported per workload (device times from CUDA events, averaged over repeated passes after a warm-up):
  fork_us / fork_bytes / fork_GBps   sg_fork_state of the env's state and snapshot into B branches; bytes = the
                                     bytes of one copy x (1 read + B writes).  The test scenes' state (7.6 MB)
                                     fits in the 126 MB L2, so its read may be served from there on repeated
                                     passes; the vehicle state (165 MB) does not.
  scatter_us                         the index_copy_ of the [N, B, H, A, 2] actions into the branch table
  rollout_us_per_branch_tick         the B fused sg_rollout(H) calls over B x H
  reward_us / observe_us             the B sg_env_reward calls / the B final observations (final_obs=True)
  run_ms                             one whole BranchRollout.run (final_obs=False), events around the call
  env_step_us                        one env.step with fixed actions (device time, events around 20 steps)
  env_steps_equiv_ms                 B x H x env_step_us: the same branch-ticks done by stepping B env copies
  branch_ticks_per_s / speedup       B x H x N / run time, and env_steps_equiv_ms / run_ms
  device / power_limit_w             the card and its power limit
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

sys.dont_write_bytecode = True
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (REPO, os.path.join(REPO, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

from bench_env import card, policy, vehicles_env, xosc_env  # noqa: E402
from scenario_gym_b200 import ObsSpec, abi  # noqa: E402

SKIP = ("events", "trace_pose", "trace_present", "trace_t", "event_count")


def fork_bytes(env) -> int:
    """Bytes of one copy of what sg_fork_state moves: the state arrays and the snapshot arrays."""
    eng = env._engine
    n = sum(eng.tensor(k).numel() * eng.tensor(k).element_size() for k, _, _ in abi.STATE_FIELDS
            if k not in SKIP and (k != "coll_mask" or eng._coll_matrix))
    return n + sum(t.numel() * t.element_size() for t in env._snap.values()) + 4


def timed(fn, reps, stream):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    e0.record(stream)
    for _ in range(reps):
        fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / reps  # microseconds


def measure(name, env, B, H):
    stream = torch.cuda.current_stream()
    o, _ = env.reset()
    for _ in range(10):
        o, *_ = env.step(policy(o))
    torch.cuda.synchronize()
    g = torch.Generator(device="cuda").manual_seed(0)
    acts = (torch.rand((env.N, B, H, env.A, 2), generator=g, device="cuda") * torch.tensor([8.0, 1.2], device="cuda")
            - torch.tensor([4.0, 0.6], device="cuda"))
    br = env.branches(B, H, final_obs=True)
    src = env._engine
    br.run(acts)  # warm-up: every launch shape
    torch.cuda.synchronize()
    fork = timed(lambda: src._check(src.lib["fork_state"](*br._fork_args, src.dev_index, src._stream())), 20, stream)
    scatter = timed(lambda: br._flat[torch.float32].index_copy_(0, br._index, acts.reshape(-1)), 20, stream)
    tables = br._tables[torch.float32]
    reps = 3

    def rollouts():
        src._check(src.lib["fork_state"](*br._fork_args, src.dev_index, src._stream()))
        for b, eng in enumerate(br._engines):
            eng.rollout(H, actions=tables[b])

    # the fork is part of each pass (the branches must start from the fork); subtract it
    roll = (timed(rollouts, reps, stream) - fork) / (B * H)

    def rewards():
        for b, eng in enumerate(br._engines):
            eng.env_reward(br._specs[b], br._reward[b], br._terms[b], br._terminated[b], br._truncated[b])

    def observes():
        for b, eng in enumerate(br._engines):
            eng.env_observe(br._specs[b], br._final_obs[b], br._agent_mask[b])

    reward, observe = timed(rewards, 10, stream), timed(observes, 5, stream)
    plain = env.branches(B, H)
    run_ms = timed(lambda: plain.run(acts), reps, stream) / 1e3
    # env.step with fixed actions: device time per step (reset scenarios included, as a real loop pays them)
    a = policy(o)
    step = timed(lambda: env.step(a), 20, stream)
    nbytes = fork_bytes(env)
    dev, power = card()
    equiv_ms = B * H * step / 1e3
    return {
        "workload": name, "N": env.N, "M": src.M, "A": env.A, "B": B, "H": H,
        "fork_us": round(fork, 1), "fork_bytes": nbytes * (1 + B), "fork_copy_bytes": nbytes,
        "fork_GBps": round(nbytes * (1 + B) / (fork * 1e-6) / 1e9, 1),
        "scatter_us": round(scatter, 1), "rollout_us_per_branch_tick": round(roll, 2),
        "reward_us": round(reward, 1), "observe_us": round(observe, 1),
        "run_ms": round(run_ms, 3), "env_step_us": round(step, 1), "env_steps_equiv_ms": round(equiv_ms, 2),
        "branch_ticks_per_s": B * H * env.N / (run_ms * 1e-3), "speedup": round(equiv_ms / run_ms, 2),
        "device": dev, "power_limit_w": power,
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--workloads", default="vehicles,xosc")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_branches.py measures the GPU engine: no CUDA device")
    obs = ObsSpec(k_neighbours=8, radius=50.0, lookahead=(1.0, 2.0, 3.0))
    shapes = {"vehicles": (vehicles_env, 8, 30), "xosc": (xosc_env, 64, 30)}
    for w in args.workloads.split(","):
        make, B, H = shapes[w]
        t0 = time.time()
        env = make(obs)
        build_s = time.time() - t0
        rec = measure(w, env, B, H)
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
