#!/usr/bin/env python
"""
bench_plan.py -- cost of on-device MPPI planning (VecScenarioEnv.planner / MPPIPlanner.plan) against the same MPPI
step written in torch around BranchRollout.run.

    python tools/bench_plan.py [--out FILE]   # one JSON line per workload on stdout (and appended to FILE)

Workloads (those of tools/bench_branches.py): vehicles, 12 500 x 64 PolicyAgent vehicles, B = 8, H = 30 (the lean
vehicle kernel); xosc, 4096 replicas of the reference's test scenarios, B = 64, H = 30 (the general kernel).  The
env is stepped 10 times with the bench_env policy first.  sigma = (1.0, 0.1), temperature 1.

Reported per workload (device times from CUDA events, after a warm-up):
  sample_us / sample_bytes / sample_GBps   sg_plan_sample into the branch table: B x H x N x A normal pairs (fp64
                                           splitmix64 + Box-Muller), bytes = the table entries written + the mean
  scatter_us                               for comparison: BranchRollout.run's index_copy_ of a [N, B, H, A, 2] fp32
                                           tensor into the same table (what sampling into the table replaces)
  update_us                                sg_plan_update (finish: action and shift included)
  fork_us / rollout_us_per_branch_tick / reward_us   the parts of one iteration, split as in bench_branches.py
  plan_ms                                  one plan() at iterations = 1 (events around the call)
  torch_ms                                 the torch path a user would write: torch.randn noise [N, B, H, A, 2] fp32,
                                           actions = mean + noise, BranchRollout.run, softmax weights, the weighted
                                           noise average into the fp64 mean, the first action and the shift.  Timed
                                           in the same process, alternating with plan() (medians of the rounds)
  torch_noise_bytes                        the size of the noise tensor the torch path holds
  device / power_limit_w                   the card and its power limit
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

sys.dont_write_bytecode = True
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (REPO, os.path.join(REPO, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

from bench_branches import timed  # noqa: E402
from bench_env import card, policy, vehicles_env, xosc_env  # noqa: E402
from scenario_gym_b200 import ObsSpec  # noqa: E402

SIGMA, LAM = (1.0, 0.1), 1.0


class TorchMPPI:
    """One MPPI step in torch around BranchRollout.run (the mean is fp64 [N, H, A, 2], as the planner's)."""

    def __init__(self, env, B, H):
        self.br = env.branches(B, H)
        self.mean = torch.zeros(env.N, H, env.A, 2, dtype=torch.float64, device="cuda")
        self.sigma = torch.tensor(SIGMA, device="cuda")
        self.g = torch.Generator(device="cuda").manual_seed(0)
        self.shape = (env.N, B, H, env.A, 2)

    def step(self):
        noise = torch.randn(self.shape, generator=self.g, device="cuda") * self.sigma
        noise[:, 0] = 0.0
        res = self.br.run(self.mean[:, None].float() + noise)
        r = res["reward"].double()
        w = torch.softmax(r / LAM, dim=1)                              # [N, B, A]
        self.mean += torch.einsum("nba,nbhac->nhac", w, noise.double())
        action = self.mean[:, 0].float()
        self.mean = torch.cat([self.mean[:, 1:], torch.zeros_like(self.mean[:, :1])], 1)
        return action


def measure(name, env, B, H):
    stream = torch.cuda.current_stream()
    o, _ = env.reset()
    for _ in range(10):
        o, *_ = env.step(policy(o))
    torch.cuda.synchronize()
    pl = env.planner(B=B, H=H, sigma=SIGMA, temperature=LAM, iterations=1, seed=0)
    br, eng, spec = pl.branches, env._engine, env._spec
    pl.plan()  # warm-up: every launch shape
    torch.cuda.synchronize()
    mu, other = pl._mean[0], pl._mean[1]
    sample = timed(lambda: eng.plan_sample(spec, B, H, 0, 1, SIGMA, mu, None, pl._table), 20, stream)
    update = timed(lambda: eng.plan_update(spec, B, H, LAM, br._reward, pl._table, mu, other, True, pl._action,
                                           pl._best_branch, pl._best_reward), 20, stream)
    acts = torch.randn((env.N, B, H, env.A, 2), device="cuda")
    scatter = timed(lambda: br._flat[torch.float32].index_copy_(0, br._index, acts.reshape(-1)), 20, stream)
    del acts
    src = eng
    fork = timed(lambda: src._check(src.lib["fork_state"](*br._fork_args, src.dev_index, src._stream())), 20, stream)

    def rollouts():
        src._check(src.lib["fork_state"](*br._fork_args, src.dev_index, src._stream()))
        for b, e in enumerate(br._engines):
            e.rollout(H, actions=pl._tables[b])

    roll = (timed(rollouts, 3, stream) - fork) / (B * H)

    def rewards():
        for b, e in enumerate(br._engines):
            e.env_reward(br._specs[b], br._reward[b], br._terms[b], br._terminated[b], br._truncated[b])

    reward = timed(rewards, 10, stream)
    tm = TorchMPPI(env, B, H)
    tm.step()
    torch.cuda.synchronize()
    plan_ms, torch_ms = [], []
    for _ in range(5):  # alternate the two paths
        plan_ms.append(timed(pl.plan, 3, stream) / 1e3)
        torch_ms.append(timed(tm.step, 3, stream) / 1e3)
    table_bytes = B * H * 2 * env.N * env.A * pl._table.element_size()
    sample_bytes = table_bytes + env.N * H * env.A * 2 * 8
    dev, power = card()
    return {
        "workload": name, "N": env.N, "M": eng.M, "A": env.A, "B": B, "H": H,
        "table_dtype": str(pl._table.dtype).replace("torch.", ""), "normal_pairs": B * H * env.N * env.A,
        "sample_us": round(sample, 1), "sample_bytes": sample_bytes,
        "sample_GBps": round(sample_bytes / (sample * 1e-6) / 1e9, 1), "scatter_us": round(scatter, 1),
        "update_us": round(update, 1), "fork_us": round(fork, 1), "rollout_us_per_branch_tick": round(roll, 2),
        "reward_us": round(reward, 1), "plan_ms": round(statistics.median(plan_ms), 3),
        "plan_ms_rounds": [round(x, 3) for x in plan_ms], "torch_ms": round(statistics.median(torch_ms), 3),
        "torch_ms_rounds": [round(x, 3) for x in torch_ms], "torch_noise_bytes": B * H * 2 * env.N * env.A * 4,
        "device": dev, "power_limit_w": power,
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--workloads", default="vehicles,xosc")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_plan.py measures the GPU engine: no CUDA device")
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
