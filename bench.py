#!/usr/bin/env python
"""
bench.py -- entity-steps/s of the batched rollout + collision path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # B200 engine
    python bench.py --impl reference --steps K --warmup W     # CPU arm (oracle port, all cores)
    python bench.py --steps K --warmup W --dump-outputs DIR  # + the results of the last timed step as .npy

A "step" is one full rollout (reset + T ticks) of this rank's batch of synthetic scenarios.  Every
timed region of the headline workload runs K steps; the sub-records run --sub-steps.  The inputs are
seeded, so two runs with the same arguments roll out the same scenarios and actions.

Headline workload = BASELINE.json configs[2] per-GPU shard (C3): 12 500 scenarios x 64
VehicleController entities x 256 ticks of dt = 0.1 with random accel/steer actions,
CollisionMetric + EgoAvgSpeed/EgoMaxSpeed/EgoDistanceTravelled + RSSDistances/RSS; weak scaling
(every GPU gets its own 12 500 scenarios, seed = rank), no per-tick communication, one NCCL
all-gather of the per-scenario records at the end.  The random actions come from
numpy.random.default_rng(seed): the engine draws that PCG64 stream inside the kernel
(``ActionRng``), the table-fed path is measured beside it (``table_path``).

The other BASELINE configurations ride along as sub-records of the same JSON line
(``workloads``: C2 4096 replicas of the reference's test scenarios, C4 1000 x 1024 social-force
pedestrians, C5 10 000 x 256 highway vehicles with RSS), each at its stated TOTAL size, sharded
over the ranks (strong scaling), with its own value / e2e / roofline / parity stamp.

value  : device-timed (CUDA events on the launching stream, max over ranks), inputs resident in HBM.
e2e    : the same metric through sg_rollout_host with pinned HOST buffers: scene (+ action table
         for the table path) H2D and result D2H inside the timed region; at N > 1 the NCCL gather
         of the records is inside it too.
parity_checked : the GPU's results of the first n scenarios of the timed batch against the CPU
         oracle rolled out on the same inputs (same run that yields cpu_baseline): discrete fields
         exact, continuous fields 1e-9 absolute-or-relative.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True  # the benchmark writes nothing into the source tree (which may be read-only)
REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

from scenario_gym_b200 import abi, synthetic  # noqa: E402
from scenario_gym_b200.distributed import shard_range  # noqa: E402
from scenario_gym_b200.packing import slice_scene  # noqa: E402

METRIC = "entity-steps/s, batched rollout+collision"
UNIT = "entity-steps/s"
TOL = 1e-9

# total sizes of the configurations (BASELINE.json configs[1..4]); C3 is per GPU (weak scaling)
SIZES = {"c2": 4096, "c3": 12500, "c4": 1000, "c5": 10000}
KERNELS = {"c3": "sg_vehicle_kernel<RSS=%d, lean>", "c5": "sg_vehicle_kernel<RSS=%d, sorted, lean>",
           "c2": "sg_replay_kernel (tick-parallel)", "c4": "sg_crowd_kernel"}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c3", choices=["c2", "c3", "c4", "c5"])
    ap.add_argument("--scenarios", type=int, default=0,
                    help="scenarios (per GPU for c3, in total for the others); 0 = the configuration's size")
    ap.add_argument("--scenarios-per-gpu", type=int, default=0, help="alias of --scenarios for c3")
    ap.add_argument("--ticks", type=int, default=256)
    ap.add_argument("--no-rss", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-subs", action="store_true", help="headline workload only (no `workloads` sub-records)")
    ap.add_argument("--actions", default="rng", choices=["rng", "table"],
                    help="action source of the headline value for c3 / c5 (the other one is reported beside it)")
    ap.add_argument("--sub-steps", type=int, default=5)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the headline workload computed as DIR/<name>.npy "
                         "(rank 0's batch)")
    return ap.parse_args()


# ------------------------------------------------------------------------------ workloads
class Workload:
    """One configuration on one rank: scene, parameters, action source, expectations."""

    def __init__(self, name: str, args, rank: int, world: int, n_override: int = 0):
        self.name, self.rank, self.world = name, rank, world
        self.rss = (not args.no_rss) and name in ("c3", "c5")
        self.action_rng = self.cfg = None
        T = args.ticks
        if name == "c3":  # weak scaling: every rank its own batch
            self.N_total = (n_override or SIZES["c3"]) * world
            self.N = n_override or SIZES["c3"]
            self.lo = rank * self.N
            self.M, self.T, self.dt = 64, T, 0.1
            self.cfg = synthetic.vehicles_config(seed=rank, N=self.N, M=64, T=T, dt=0.1, materialise=False)
            self.scene = synthetic.pack_synthetic(self.cfg)
            self.action_rng = self.cfg.action_rng
            self.scaling = "weak"
        else:  # strong scaling: the configuration's total size, sharded by contiguous blocks
            self.N_total = n_override or SIZES[name]
            self.lo, hi = shard_range(self.N_total, rank, world)
            self.N = hi - self.lo
            self.scaling = "strong"
            if name == "c5":
                self.M, self.T, self.dt = 256, T, 0.1
                self.cfg = synthetic.highway_config(seed=0, N=self.N_total, M=256, T=T, dt=0.1, materialise=False)
                full = synthetic.pack_synthetic(self.cfg)
                self.scene = slice_scene(full, self.lo, hi) if world > 1 else full
                self.action_rng = self.cfg.action_rng.shard(self.lo * 256, self.N * 256)
            elif name == "c4":
                self.M, self.T, self.dt = 1024, min(T, 128), 1.0 / 15.0
                self.cfg = synthetic.crowd_config(seed=0, N=self.N_total, M=1024, T=self.T, dt=self.dt)
                full = synthetic.pack_synthetic(self.cfg)
                self.scene = slice_scene(full, self.lo, hi) if world > 1 else full
            else:  # c2
                full, self._c2_steps, self._c2_ticks = c2_scene(self.N_total)
                self.scene = slice_scene(full, self.lo, hi) if world > 1 else full
                self.M, self.T, self.dt = self.scene.M, 0, 1.0 / 30.0
        self.p = abi.default_params()
        self.p.timestep = self.dt
        self.p.features = abi.FEAT_COLLISIONS | abi.FEAT_EGO_METRICS | (abi.FEAT_RSS if self.rss else 0)
        if name == "c2":
            idx = np.arange(self.lo, self.lo + self.N)
            self.steps_expected = int(self._c2_steps[idx % len(self._c2_steps)].sum())
            self.expected_ticks = self._c2_ticks[idx % len(self._c2_ticks)]
        else:
            self.steps_expected = self.N * self.M * self.T
            self.expected_ticks = np.full(self.N, self.T)

    # SURVEY.md section 8d B_tick (per-tick streaming design, fp64 SoA)
    @property
    def bytes_per_entity_step(self) -> int:
        return {"c2": 290, "c4": 305}.get(self.name, 259 if self.rss else 225)

    @property
    def kernel(self) -> str:
        k = KERNELS[self.name]
        return k % (1 if self.rss else 0) if "%d" in k else k

    def traffic_key(self) -> str:
        return f"{self.name}{'' if self.rss or self.name in ('c2', 'c4') else '_norss'}_{self.N}x{self.M}x{self.T}"

    def describe(self) -> str:
        return {
            "c2": f"C2: {self.N_total} replicas of the reference's 23 test scenarios (1-9 entities, 324-722 ticks "
                  "at 30 Hz), trajectory replay + CollisionMetric/ego metrics (BASELINE.json configs[1])",
            "c3": f"C3: {self.N} scenarios/GPU x {self.M} VehicleController entities x {self.T} ticks, random "
                  "accel/steer actions (BASELINE.json configs[2] per-GPU shard)",
            "c4": f"C4: {self.N_total} scenarios x {self.M} social-force pedestrians x {self.T} ticks "
                  "(BASELINE.json configs[3])",
            "c5": f"C5: {self.N_total} scenarios x {self.M} highway vehicles x {self.T} ticks, RSS + SafeDistance "
                  "(BASELINE.json configs[4])",
        }[self.name]

    def config_json(self, extra=None) -> dict:
        mets = ["CollisionMetric", "EgoAvgSpeed", "EgoMaxSpeed", "EgoDistanceTravelled"]
        if self.rss:
            mets += ["RSSDistances", "RSS"]
        c = {"workload": self.describe(), "scenarios_per_gpu": self.N, "scenarios_total": self.N_total,
             "entities": self.M, "ticks": self.T, "timestep": self.dt, "metrics": mets,
             "actions": ("uniform random accel/steer drawn from numpy.random.default_rng(seed) (PCG64)"
                         if self.name in ("c3", "c5") else None),
             "l2_policy": "L2 flushed between steps: a 256 MiB scratch buffer is rewritten before every step "
                          "(and the reset kernel rewrites every state plane)"}
        if extra:
            c.update(extra)
        return c

    def oracle_sample(self, n: int):
        """(scene, actions) of this rank's first n scenarios, for the CPU oracle (numpy draws the table)."""
        sc = slice_scene(self.scene, 0, n)
        actions = None
        if self.action_rng is not None:
            actions = self.action_rng.shard(0, n * self.M).table()
        return sc, actions


def c2_scene(n_scen: int):
    """C2: replicas of the reference's 23 test scenarios (inputs committed under tests/golden)."""
    sys.path.insert(0, os.path.join(REPO, "tests"))
    from helpers import all_xosc_specs

    from scenario_gym_b200.packing import pack_scenarios, tile_scene

    specs = all_xosc_specs("xosc")
    base = pack_scenarios([s for _, s, _, _ in specs])
    reps = -(-n_scen // base.N)
    per = np.array([int(o["present"][1:].sum()) for _, _, _, o in specs], np.int64)
    tk = np.array([int(o["n_ticks"]) for _, _, _, o in specs], np.int64)
    return slice_scene(tile_scene(base, reps), 0, n_scen), per, tk


# ------------------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock / throttle-reason samples taken DURING the timed regions.

    NVML is polled from a thread every few ms (the timed region of a short run is < 100 ms, too
    short for `nvidia-smi -lms`); `nvidia-smi` is the fall-back when NVML cannot be loaded.
    """

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index: int, uuid: str = None, period_s: float = 0.004):
        self.index, self.uuid, self.period = index, uuid, period_s
        self.proc = None
        self.nvml = None
        self.samples = []  # (wall time, sm MHz, max MHz, watts, set of reasons)
        self._stop = threading.Event()
        self.thread = None

    def _nvml_open(self):
        import pynvml as nv

        nv.nvmlInit()
        h = None
        if self.uuid:
            for u in (self.uuid, "GPU-" + self.uuid):
                try:
                    h = nv.nvmlDeviceGetHandleByUUID(u.encode() if isinstance(u, str) else u)
                    break
                except Exception:
                    h = None
        if h is None:
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
        self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        self.nvml, self.handle = nv, h

    def _nvml_loop(self):
        nv, h = self.nvml, self.handle
        bits = [(nv.nvmlClocksEventReasonHwSlowdown, "hw_slowdown"),
                (nv.nvmlClocksEventReasonHwThermalSlowdown, "hw_thermal_slowdown"),
                (nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_thermal_slowdown"),
                (nv.nvmlClocksEventReasonSwPowerCap, "sw_power_cap")]
        while not self._stop.is_set():
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
                try:
                    watts = nv.nvmlDeviceGetPowerUsage(h) / 1e3
                except Exception:
                    watts = float("nan")
                self.samples.append((time.time(), mhz, self.max_mhz, watts,
                                     {nm for b, nm in bits if r & b}))
            except Exception:
                pass
            self._stop.wait(self.period)

    def _smi_loop(self):
        for line in self.proc.stdout:
            parts = [x.strip() for x in line.strip().split(",")]
            if len(parts) < 7:
                continue
            try:
                self.samples.append((time.time(), float(parts[0]), float(parts[1]), float(parts[2]),
                                     {nm for nm, v in zip(self.NAMES, parts[3:7])
                                      if v.lower().startswith("active")}))
            except ValueError:
                continue

    def start(self):
        try:
            self._nvml_open()
            self.thread = threading.Thread(target=self._nvml_loop, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._smi_loop, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def report(self, t0: float, t1: float) -> dict:
        """Summary of the samples taken inside [t0, t1] (a timed region)."""
        if self.nvml is None and self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["no NVML / nvidia-smi"]}
        inside = [s for s in list(self.samples) if t0 <= s[0] <= t1]
        reasons = set()
        for s in inside:
            reasons |= s[4]
        power = [s[3] for s in inside if s[3] == s[3]]
        return {
            "sm_mhz": float(np.median([s[1] for s in inside])) if inside else None,
            "sm_max_mhz": float(max(s[2] for s in inside)) if inside else None,
            "power_w_max": float(max(power)) if power else None,
            "samples": len(inside),
            "source": "nvml" if self.nvml is not None else "nvidia-smi",
            "reasons": sorted(reasons),
        }

    def stop(self):
        self._stop.set()
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()
        if self.thread is not None:
            self.thread.join(timeout=2)


# ------------------------------------------------------------------------------ CPU arms
_W = {}


def _worker_init(args_dict, per_worker):
    import argparse as _ap

    from oracle.runner import OracleEngine

    args = _ap.Namespace(**args_dict)
    ident = os.getpid()
    wl = Workload(args.workload, args, rank=1000 + ident % 1000, world=1, n_override=per_worker)
    scene, actions = wl.oracle_sample(wl.N)
    _W["eng"] = OracleEngine(scene, wl.p, event_cap=1 << 16)
    _W["actions"], _W["M"] = actions, scene.M
    _W["steps"] = wl.steps_expected if wl.name == "c2" else None


def _worker_step(_):
    eng = _W["eng"]
    t0 = time.perf_counter()
    eng.reset()
    eng.rollout(-1, actions=_W["actions"])
    steps = _W["steps"] if _W["steps"] is not None else int(eng.get("tick").sum()) * _W["M"]
    return steps, time.perf_counter() - t0


def result_fields(wl: Workload):
    """The state fields a rollout of `wl` computes: (discrete per scenario, discrete per entity,
    continuous per scenario, continuous per entity)."""
    disc_n = ("tick", "done", "first_coll_tick", "first_coll_pair", "n_pair_ticks", "rss_flags", "t")
    disc_nm = ("present", "collided") + (("rss_state", "rss_last") if wl.rss else ())
    cont_n = ("ego_avg_speed", "ego_max_speed", "ego_dist")
    cont_nm = ("pose", "vel", "dist", "speed") + (("safe_dist", "safe_ratio") if wl.rss else ()) + \
        (("force",) if wl.name == "c4" else ())
    if wl.name == "c4":
        disc_nm += ("goal_idx",)
    return disc_n, disc_nm, cont_n, cont_nm


DUMP_ENTITIES = 1 << 16  # per-entity planes of at most this many entities are written (~13 MB)
DUMP_LIMIT = 64 << 20


def dump_outputs(wl: Workload, eng, out_dir: str) -> None:
    """
    Write what the last rollout of `eng` computed as out_dir/<name>.npy (float64), so that two builds can be
    compared output for output: every per-scenario field over the whole batch, and the per-entity planes
    and ego collision events (rows: scenario, tick, slot, t) of a fixed, seeded sample of scenarios
    (`sample_scenarios`; the full planes of C3 take ~100 MB).  Per-entity planes keep the engine's layout,
    restricted to the sampled scenarios' slots.  Every value written is finite.
    """
    disc_n, disc_nm, cont_n, cont_nm = result_fields(wl)
    n = min(wl.N, max(1, DUMP_ENTITIES // wl.M))
    sample = np.sort(np.random.default_rng(0).choice(wl.N, n, replace=False))
    cols = (sample[:, None] * wl.M + np.arange(wl.M)).ravel()
    out = {"sample_scenarios": sample}
    out.update({k: eng.get(k) for k in disc_n + cont_n})
    out.update({k: eng.get(k)[..., cols] for k in disc_nm + cont_nm})
    ev = eng.events()
    ev = ev[np.isin(ev["scenario"], sample)]
    out["events"] = np.stack([ev[f].astype(np.float64) for f in ("scenario", "tick", "slot", "t")], axis=1)
    if "safe_ratio" in out:  # no hazard: the ratio is +inf (as in the reference); written as 0, flagged in safe_ratio_inf
        inf = np.isposinf(out["safe_ratio"])
        out["safe_ratio_inf"] = inf
        out["safe_ratio"] = np.where(inf, 0.0, out["safe_ratio"])
    out = {k: np.ascontiguousarray(v, np.float64) for k, v in out.items()}
    bad = [k for k, v in out.items() if not np.isfinite(v).all()]
    assert not bad, f"--dump-outputs: non-finite values in {bad}"
    total = sum(v.nbytes for v in out.values())
    assert total <= DUMP_LIMIT, f"--dump-outputs would write {total} bytes"
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def oracle_parity_and_baseline(wl: Workload, gpu, budget_s: float = 10.0, n_min: int = 4, n_max: int = 2048):
    """
    Roll the first n scenarios of this rank's batch out on the CPU oracle (one core, ~budget_s of work),
    time it (cpu_baseline) and compare the GPU engine's results on the same scenarios with it
    (parity_checked).  `gpu` holds the final state of a rollout of the whole batch.
    """
    from oracle.runner import OracleEngine

    n_min = {"c2": 23, "c4": 1, "c5": 2}.get(wl.name, n_min)
    disc_n, disc_nm, cont_n, cont_nm = result_fields(wl)
    n = min(n_min, wl.N)
    while True:
        scene, actions = wl.oracle_sample(n)
        eng = OracleEngine(scene, wl.p, event_cap=1 << 20)
        t0 = time.perf_counter()
        eng.reset()
        eng.rollout(-1, actions=actions)
        dt = time.perf_counter() - t0
        if dt >= budget_s / 4 or n >= min(n_max, wl.N):
            break
        n = min(n_max, wl.N, max(n * 2, int(n * budget_s / max(dt, 1e-3) / 2)))
    M = wl.M
    if wl.name == "c2":
        idx = np.arange(wl.lo, wl.lo + n)
        steps = int(wl._c2_steps[idx % len(wl._c2_steps)].sum())
    else:
        steps = int(eng.get("tick").sum()) * M
    cpu = {
        "value": steps / dt, "unit": UNIT, "cores": 1, "kind": "port",
        "sample": f"the first {n} scenarios of the timed batch x {M} entities x {wl.T or 'all'} ticks "
                  f"({steps} entity-steps in {dt:.2f} s), oracle/sg_oracle.c single thread",
    }
    # ---- parity: GPU rows of the same scenarios
    sl = slice(0, n * M)
    mism, max_err = [], 0.0
    for k in disc_n:
        if not np.array_equal(gpu.get(k)[:n], eng.get(k), equal_nan=True):
            mism.append(k)
    for k in disc_nm:
        if not np.array_equal(gpu.get(k)[sl], eng.get(k)):
            mism.append(k)
    ge = gpu.events()
    ge = ge[ge["scenario"] < n]
    ce = eng.events()
    if not (len(ge) == len(ce) and all(np.array_equal(ge[f], ce[f]) for f in ("scenario", "tick", "slot", "t"))):
        mism.append("events")
    pres = eng.get("present").astype(bool)

    def err(a, b):
        a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
        e = np.abs(a - b) / np.maximum(1.0, np.abs(b))
        e[(a == b) | (np.isnan(a) & np.isnan(b))] = 0.0
        return float(np.nanmax(e)) if e.size else 0.0

    for k in cont_n:
        max_err = max(max_err, err(gpu.get(k)[:n], eng.get(k)))
    for k in cont_nm:
        a, b = gpu.get(k)[..., sl], eng.get(k)
        if k in ("pose", "vel"):
            a, b = a[:, pres], b[:, pres]
        elif k == "safe_ratio":
            fin = np.isfinite(b)
            a, b = a[fin], b[fin]
        max_err = max(max_err, err(a, b))
    parity = {"ok": not mism and max_err <= TOL, "n_scenarios": n, "ticks": wl.T or "all (324-722)",
              "entity_steps": steps, "max_err": max_err, "tolerance": TOL, "discrete_mismatches": mism,
              "discrete_fields": list(disc_n + disc_nm) + ["events"], "continuous_fields": list(cont_n + cont_nm),
              "collisions_in_sample": {"pair_ticks": int(eng.get("n_pair_ticks").sum()), "ego_events": int(len(ce))}}
    return cpu, parity


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp

    from oracle.runner import build_oracle

    build_oracle()
    cores = os.cpu_count() or 1
    M = {"c2": 9, "c3": 64, "c4": 1024, "c5": 256}[args.workload]
    T = {"c2": 500, "c4": min(args.ticks, 128)}.get(args.workload, args.ticks)
    per_worker = max(1, int(round(4e5 / (M * max(T, 200)))))  # ~0.2-0.4 s of work per step per core
    if args.workload == "c2":
        per_worker = 23
    args_dict = vars(args)
    ctx = mp.get_context("fork")
    with ctx.Pool(cores, initializer=_worker_init, initargs=(args_dict, per_worker)) as pool:
        for _ in range(args.warmup):
            pool.map(_worker_step, range(cores), chunksize=1)
        t0 = time.perf_counter()
        total = 0
        for _ in range(args.steps):
            res = pool.map(_worker_step, range(cores), chunksize=1)
            total += sum(r[0] for r in res)
        dt = time.perf_counter() - t0
    value = total / dt
    sample = (f"{cores} processes x {per_worker} scenarios x {M} entities x {T} ticks per step; "
              "plain-C port of the reference path (oracle/sg_oracle.c); the Python reference itself "
              "cannot travel to the GPU box (measured in the authoring container: ~1.5e4 entity-steps/s/core)")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": reference_config(args),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def reference_config(args) -> dict:
    """The B200 arm's `config` for the same command line (without building the scenes)."""
    n = args.scenarios or args.scenarios_per_gpu or SIZES[args.workload]
    M = {"c2": 9, "c3": 64, "c4": 1024, "c5": 256}[args.workload]
    T = {"c2": 0, "c4": min(args.ticks, 128)}.get(args.workload, args.ticks)
    dt = {"c2": 1.0 / 30.0, "c4": 1.0 / 15.0}.get(args.workload, 0.1)
    stub = Workload.__new__(Workload)
    stub.name, stub.N, stub.M, stub.T, stub.dt = args.workload, n, M, T, dt
    stub.N_total = n * (args.gpus if args.workload == "c3" else 1)
    if args.workload != "c3":
        stub.N = -(-n // max(args.gpus, 1))
    stub.rss = (not args.no_rss) and args.workload in ("c3", "c5")
    return stub.config_json({"parallelism": f"scenario-sharded x{args.gpus}, no per-tick communication"})


# ------------------------------------------------------------------------------ B200 arm
class Bench:
    def __init__(self, args):
        import torch
        import torch.distributed as dist

        from scenario_gym_b200.distributed import init_from_env

        self.torch, self.dist, self.args = torch, dist, args
        self.rank, self.world, self.local = init_from_env()
        if not torch.cuda.is_available():
            raise SystemExit("bench.py --impl b200 needs a CUDA device (no CPU fallback)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device(f"cuda:{self.local}")
        self.stream = torch.cuda.current_stream(self.dev)
        self.flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)
        try:
            uuid = str(torch.cuda.get_device_properties(self.local).uuid)
        except Exception:
            uuid = None
        self.sampler = ClockSampler(self.local, uuid)
        if self.rank == 0:
            self.sampler.start()
        peaks_path = os.path.join(REPO, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            self.peak, self.peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
        else:
            self.peak, self.peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        tpath = os.path.join(REPO, "profiles", "traffic.json")
        self.traffic = json.load(open(tpath)) if os.path.exists(tpath) else {}
        self.fp64_peak = None
        self.launches = 0

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def allreduce(self, x: float, op: str) -> float:
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=getattr(self.dist.ReduceOp, op))
        return float(t.item())

    def flush_l2(self):
        self.flush_buf.zero_()

    # -------------------------------------------------------------- device-resident timing
    def time_device(self, eng, actions, steps: int, warmup: int):
        torch = self.torch
        for _ in range(warmup):
            self.flush_l2()
            eng.reset()
            eng.rollout(-1, actions=actions)
        self.barrier()
        t_wall0 = time.time()
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record(self.stream)
        for k in range(steps):
            self.flush_l2()
            ev[k][0].record(self.stream)
            eng.reset()
            ev[k][1].record(self.stream)
            eng.rollout(-1, actions=actions)
            ev[k][2].record(self.stream)
        stop.record(self.stream)
        self.barrier()
        t_wall1 = time.time()
        self.launches += 2 * steps
        elapsed_ms = self.allreduce(start.elapsed_time(stop), "MAX")
        kern_ms = float(np.mean([e[1].elapsed_time(e[2]) for e in ev]))
        reset_ms = float(np.mean([e[0].elapsed_time(e[1]) for e in ev]))
        clocks = self.sampler.report(t_wall0, t_wall1) if self.rank == 0 else None
        return elapsed_ms, kern_ms, reset_ms, clocks

    # -------------------------------------------------------------- end to end (host buffers)
    def time_e2e(self, wl: Workload, eng, act_mode, steps: int, warmup: int, ref: dict):
        """
        sg_rollout_host (scenario_gym_b200.hostpath.HostRollout) from pinned host buffers: scene H2D
        (+ action table H2D for act_mode = "table" / "table_f32"), reset, rollout, results D2H; at
        world > 1 followed by the NCCL gather of the per-scenario records (the caller's view of a
        finished batch).  Returns the e2e dict.
        """
        from scenario_gym_b200.distributed import gather_records, pack_records
        from scenario_gym_b200.hostpath import HostRollout

        torch, N = self.torch, wl.N
        actions = None
        if act_mode == "rng":
            actions = wl.action_rng
        elif act_mode in ("table", "table_f32"):
            dt_ = torch.float64 if act_mode == "table" else torch.float32
            act_host = torch.empty((wl.T, 2, N * wl.M), dtype=dt_, pin_memory=True)
            dev_tab = eng.fill_actions(wl.action_rng)  # the same rows, drawn on the device ...
            act_host.copy_(dev_tab.to(dt_))            # ... staged in pinned host memory as a policy would
            del dev_tab
            actions = act_host
        hr = HostRollout(eng, actions)
        rec_fields = ("ego_avg_speed", "ego_max_speed", "ego_dist", "first_coll_tick", "first_coll_pair",
                      "n_pair_ticks", "rss_flags", "tick", "t")
        gathered = [None]

        def e2e_step():
            hr.launch()
            if self.world > 1:  # the only collective of the path: the final gather of the records
                gathered[0] = gather_records(pack_records({k: eng.tensor(k) for k in rec_fields}), wl.N_total)
            self.stream.synchronize()  # the caller reads the results after every rollout

        for _ in range(max(1, min(warmup, 2))):
            e2e_step()
        self.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            e2e_step()
        self.torch.cuda.synchronize(self.dev)
        wall = time.perf_counter() - t0
        self.launches += 2 * steps
        # the host-buffer path must reproduce the resident path bit for bit
        for k, v in ref.items():
            got = hr.results[k].numpy()
            assert np.array_equal(got, v, equal_nan=True), f"e2e path: {k} differs from the resident path"
        gather_checked = None
        if self.world > 1:  # content of the gather: this rank's slice equals its local records
            rec = gathered[0]
            local = pack_records({k: eng.tensor(k) for k in rec_fields})
            assert rec.shape[0] == wl.N_total
            assert bool(self.torch.equal(rec[wl.lo:wl.lo + N], local)), "gathered records differ from the local slice"
            gather_checked = True
        wall = self.allreduce(wall, "MAX")
        total = self.allreduce(float(wl.steps_expected), "SUM")
        return {"value": total * steps / wall, "unit": UNIT, "h2d_bytes_per_step": hr.h2d_bytes,
                "d2h_bytes_per_step": hr.d2h_bytes, "ms_per_step": 1e3 * wall / steps, "steps": steps, "action_source": act_mode,
                "includes_gather": self.world > 1, "gather_content_checked": gather_checked}

    # -------------------------------------------------------------- one workload
    def run_workload(self, wl: Workload, steps: int, warmup: int, headline: bool):
        from scenario_gym_b200.engine import Engine

        args, torch = self.args, self.torch
        eng = Engine(wl.scene, wl.p, device=self.dev, event_cap=1 << 22)
        has_actions = wl.action_rng is not None
        primary = args.actions if has_actions else None
        table_dev = None

        def source(mode):
            nonlocal table_dev
            if mode == "rng":
                return wl.action_rng
            if mode == "table":
                if table_dev is None:
                    table_dev = eng.fill_actions(wl.action_rng)
                return table_dev
            return None

        elapsed_ms, kern_ms, reset_ms, clocks = self.time_device(eng, source(primary), steps, warmup)
        ticks = eng.get("tick")
        assert np.array_equal(ticks, wl.expected_ticks), "every scenario must run its full number of ticks"
        if headline and args.dump_outputs and self.rank == 0:
            dump_outputs(wl, eng, args.dump_outputs)
        total_steps = self.allreduce(float(wl.steps_expected), "SUM")
        value = total_steps * steps / (elapsed_ms / 1e3)
        ref = {k: eng.get(k).copy() for k in ("ego_avg_speed", "ego_max_speed", "ego_dist", "first_coll_tick",
                                               "first_coll_pair", "n_pair_ticks", "rss_flags", "tick", "t")}
        collisions = {"pair_ticks": int(ref["n_pair_ticks"].sum()),
                      "scenarios_with_collision": int((ref["first_coll_tick"] >= 0).sum()),
                      "ego_events": int(eng.tensor("event_count").item())}

        # parity + CPU baseline on the first scenarios of the batch (rank 0; state of the timed rollout)
        cpu = parity = None
        if self.rank == 0 and not args.no_cpu_baseline:
            cpu, parity = oracle_parity_and_baseline(wl, eng, budget_s=10.0 if headline else 5.0)

        bpe = wl.bytes_per_entity_step
        achieved = wl.steps_expected * bpe / (kern_ms / 1e3) / 1e9
        tr = self.traffic.get(wl.traffic_key()) or {}
        if not isinstance(tr, dict):
            tr = {"dram_bytes": tr}
        roofline = {
            "bound": "hbm", "achieved": achieved, "peak": self.peak, "unit": "GB/s", "frac": achieved / self.peak,
            "traffic": tr.get("dram_bytes"), "kernel": wl.kernel, "kernel_ms": kern_ms, "reset_kernel_ms": reset_ms,
            "algorithmic_bytes_per_entity_step": bpe, "entity_steps_per_launch": wl.steps_expected,
            "peak_source": self.peak_src,
            "note": "achieved = SURVEY 8d per-tick-streaming bytes (B_tick) x entity-steps / kernel time, of measured "
                    "HBM copy bandwidth; the fused kernels keep State rows on chip across ticks, so their real DRAM "
                    "traffic (`traffic`, ncu) is far below B_tick: the fp64 block is the ceiling that binds",
        }
        if self.fp64_peak and tr.get("fp64_inst"):
            a = tr["fp64_inst"] / (kern_ms / 1e3)
            roofline["fp64"] = {"achieved": a, "peak": self.fp64_peak, "unit": "fp64 thread-instructions/s",
                                "frac": a / self.fp64_peak, "fp64_inst_per_launch": tr["fp64_inst"],
                                "fp64_inst_per_entity_step": tr["fp64_inst"] / wl.steps_expected,
                                "peak_source": "DFMA micro-benchmark of this run (sg_measure_fp64_peak), same clocks",
                                "inst_source": "ncu smsp__sass_thread_inst_executed_op_d{add,mul,fma}_pred_on "
                                               "(profiles/traffic.json)"}
        out = {"value": value, "unit": UNIT, "ms_per_step": elapsed_ms / steps, "steps": steps, "warmup": warmup,
               "scaling": wl.scaling, "clocks": clocks, "roofline": roofline, "collisions": collisions,
               "action_source": primary, "cpu_baseline": cpu, "parity_checked": parity}

        if not args.no_e2e:
            out["e2e"] = self.time_e2e(wl, eng, primary, steps, warmup, ref)
        if has_actions and headline:  # the other action source beside it
            other = "table" if primary == "rng" else "rng"
            e2, k2, _, _ = self.time_device(eng, source(other), steps, 2)
            for k, v in ref.items():
                assert np.array_equal(eng.get(k), v, equal_nan=True), f"{other} action source: {k} differs"
            rec = {"value": total_steps * steps / (e2 / 1e3), "kernel_ms": k2, "action_source": other,
                   "bit_equal_to_headline": True}
            if not args.no_e2e:
                table_dev = None  # free the resident table before the e2e buffers are allocated
                rec["e2e"] = self.time_e2e(wl, eng, other, steps, 2, ref)
                if other == "table":
                    r32 = self.time_e2e(wl, eng, "table_f32", steps, 2, {"tick": ref["tick"]})
                    rec["e2e_fp32_table"] = r32
            out["table_path" if other == "table" else "rng_path"] = rec
        del eng
        torch.cuda.empty_cache()
        return out


def api_records(bench, n_fused: int = 4096, n_host: int = 64) -> dict:
    """
    The C2 workload through the reference-facing Python API: ScenarioGym.set_scenarios -> rollout ->
    get_metrics on `n_fused` replicas of the reference's test scenarios (one fused launch), and on
    `n_host` replicas with a custom host-side Metric (per-tick host mode: every tick the batch's planes
    are copied back once and the metric runs on the materialised states).
    """
    sys.path.insert(0, os.path.join(REPO, "tests"))
    from helpers import golden, manifest, sub

    from scenario_gym_b200 import (BoundingBox, CatalogEntry, CollisionMetric, EgoAvgSpeed, Entity, Metric,
                                   Pedestrian, Scenario, ScenarioGym, Trajectory, Vehicle)

    g, man = golden("xosc"), manifest()["xosc"]
    names = sorted(man)
    cls = {abi.ETYPE_VEHICLE: (Vehicle, "Vehicle"), abi.ETYPE_PEDESTRIAN: (Pedestrian, "Pedestrian")}

    def build(name):
        inp = sub(g, f"xosc/{name}/in")
        ents = []
        for i in range(int(inp["n_entities"])):
            C_, ctype = cls.get(int(inp["etype"][i]), (Entity, "MiscObject"))
            ce = CatalogEntry(None, "entry", None, ctype, BoundingBox(*[float(v) for v in inp["box"][i]]))
            ents.append(C_(ce, trajectory=Trajectory(inp[f"traj{i}"]), ref=man[name]["refs"][i]))
        return Scenario(ents, name=name)

    per = {n: int(sub(g, f"xosc/{n}/out")["present"][1:].sum()) for n in names}
    want = {n: float(sub(g, f"xosc/{n}/out")["ego_avg_speed"]) for n in names}

    class MaxEntities(Metric):  # a user metric the engine knows nothing about
        name = "max_entities"

        def _reset(self, state):
            self.value = len(state.poses)

        def _step(self, state):
            self.value = max(self.value, len(state.poses))

        def get_state(self):
            return self.value

    out = {}
    for tag, n_scen, metrics in (("fused", n_fused, lambda: [CollisionMetric(), EgoAvgSpeed()]),
                                 ("host_metric", n_host, lambda: [EgoAvgSpeed(), MaxEntities()])):
        order = [names[k % len(names)] for k in range(n_scen)]
        t0 = time.perf_counter()
        scenarios = [build(n) for n in order]
        gym = ScenarioGym(metrics=metrics(), device=bench.local)
        gym.set_scenarios(scenarios)
        t_set = time.perf_counter() - t0
        gym.rollout()  # warm-up
        gym.get_metrics()
        bench.torch.cuda.synchronize(bench.dev)
        reps = 3 if tag == "fused" else 1
        t0 = time.perf_counter()
        for _ in range(reps):
            gym.rollout()
            bench.torch.cuda.synchronize(bench.dev)
        t_roll = (time.perf_counter() - t0) / reps
        t0 = time.perf_counter()
        ms = gym.get_metrics()
        t_get = time.perf_counter() - t0
        ms = ms if isinstance(ms, list) else [ms]
        ok = all(abs(m["ego_avg_speed"] - want[n]) <= 1e-9 * max(1.0, abs(want[n])) for m, n in zip(ms, order))
        t0 = time.perf_counter()
        arr = gym.get_metric_arrays()  # the batch-wide form of the device metrics (no per-scenario Python)
        t_arr = time.perf_counter() - t0
        ok = ok and all(arr["ego_avg_speed"][k] == m["ego_avg_speed"] for k, m in enumerate(ms))
        steps = sum(per[n] for n in order)
        out[tag] = {"scenarios": n_scen, "entity_steps": steps, "value": steps / (t_roll + t_get), "unit": UNIT,
                    "ms_set_scenarios": 1e3 * t_set, "ms_rollout": 1e3 * t_roll, "ms_get_metrics": 1e3 * t_get,
                    "ms_get_metric_arrays": 1e3 * t_arr, "value_with_metric_arrays": steps / (t_roll + t_arr),
                    "metrics_match_reference_goldens": bool(ok),
                    "path": "ScenarioGym.set_scenarios -> rollout -> get_metrics" +
                            ("" if tag == "fused" else " with a custom host Metric (per-tick host mode)")}
    return out


def measure_fp64_peak(dev_index: int, stream) -> float:
    """DFMA thread-instructions/s of this GPU at its current clocks (library micro-benchmark)."""
    import ctypes as C

    lib = abi.load_product()
    out = C.c_double(0.0)
    rc = lib["measure_fp64_peak"](C.byref(out), dev_index, stream)
    if rc:
        raise RuntimeError(lib["last_error"]().decode())
    return float(out.value)


def run_b200(args):
    b = Bench(args)
    rank, world = b.rank, b.world
    try:
        b.fp64_peak = measure_fp64_peak(b.local, b.stream.cuda_stream)
    except Exception as e:  # noqa: BLE001
        b.fp64_peak = None
        print(f"fp64 micro-benchmark unavailable: {e}", file=sys.stderr)
    n_over = args.scenarios or args.scenarios_per_gpu
    wl = Workload(args.workload, args, rank, world, n_override=n_over)
    main = b.run_workload(wl, args.steps, args.warmup, headline=True)
    subs = {}
    if not args.no_subs and args.workload == "c3" and not n_over:
        for name in ("c5", "c2", "c4"):
            try:
                sw = Workload(name, args, rank, world)
                subs[name] = b.run_workload(sw, args.sub_steps, 3, headline=False)
                subs[name]["config"] = sw.config_json()
            except Exception as e:  # noqa: BLE001 -- a failing sub-workload must not take the headline with it
                import traceback

                subs[name] = {"error": f"{type(e).__name__}: {e}", "trace": traceback.format_exc()[-600:]}
    if rank == 0:
        out = {
            "metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True,
            "scaling": wl.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": wl.config_json({"parallelism": f"scenario-sharded x{world}, no per-tick communication"}),
            "action_source": main["action_source"],
            "clocks": main["clocks"], "e2e": main.get("e2e"), "gpu_launches": b.launches,
            "roofline": main["roofline"], "cpu_baseline": main["cpu_baseline"],
            "parity_checked": main["parity_checked"], "collisions": main["collisions"],
            "fp64_peak_inst_per_s": b.fp64_peak,
        }
        for k in ("table_path", "rng_path"):
            if k in main:
                out[k] = main[k]
        if subs:
            out["workloads"] = subs
        if world == 1 and not args.no_subs and args.workload == "c3" and not n_over:
            try:
                out["python_api"] = api_records(b)
            except Exception as e:  # noqa: BLE001
                out["python_api"] = {"error": f"{type(e).__name__}: {e}"}
        print(json.dumps(out))
    b.sampler.stop()
    if world > 1:
        b.dist.barrier()
        b.dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
