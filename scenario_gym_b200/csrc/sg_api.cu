// sg_api.cu -- the C ABI of include/sg_b200.h: argument checks, kernel selection, host-buffer path.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "sg_internal.h"

static thread_local char g_err[512];
static int set_err(const char* what, cudaError_t e) {
  snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
  return -2;
}
static int set_msg(const char* what) {
  snprintf(g_err, sizeof(g_err), "%s", what);
  return -1;
}

// launch-uniform form of an SgActionRng for rows starting at `tick0` (sg_pcg.cuh)
static SgRngDev make_rng_dev(const SgActionRng& r, int tick0) {
  SgRngDev d;
  memset(&d, 0, sizeof(d));
  const sg_u128 s0 = sg_u128_make(r.state_hi, r.state_lo), inc = sg_u128_make(r.inc_hi, r.inc_lo);
  for (int c = 0; c < 2; ++c) {
    const sg_u128 sc = sg_pcg_advance(s0, inc, (sg_u128)(r.offset[c] + (int64_t)tick0 * r.tick_stride));
    d.s_hi[c] = (uint64_t)(sc >> 64);
    d.s_lo[c] = (uint64_t)sc;
    d.low[c] = r.low[c];
    d.scale[c] = r.scale[c];
  }
  sg_u128 A, C;
  sg_pcg_jump_coeffs(inc, (sg_u128)r.tick_stride, A, C);
  d.inc_hi = r.inc_hi; d.inc_lo = r.inc_lo;
  d.a_hi = (uint64_t)(A >> 64); d.a_lo = (uint64_t)A;
  d.c_hi = (uint64_t)(C >> 64); d.c_lo = (uint64_t)C;
  return d;
}

static int check_rng(const SgActionRng& r) {
  if (r.offset[0] < 0 || r.offset[1] < 0 || r.tick_stride < 0) return set_msg("SgActionRng: negative offset / stride");
  if (!(r.inc_lo & 1)) return set_msg("SgActionRng: inc must be odd (not a PCG64 state)");
  return 0;
}

static int launch(const SgScene* sc, const SgParams* p, SgState* st, const SgInputs* in, int n_ticks,
                  int device, void* stream, int reset, const uint8_t* reset_mask = nullptr) {
  if (!sc || !p || !st) return set_msg("null argument");
  if (sc->n_slots < 1 || sc->n_slots > 1024) return set_msg("n_slots must be in 1..1024");
  if (sc->n_scenarios < 1) return set_msg("n_scenarios must be >= 1");
  SgScene view = *sc;  // (what the kernels get: the plane stride is always stated)
  if (view.plane_stride <= 0) {
    view.plane_stride = (int64_t)sc->n_scenarios * sc->n_slots;
    view.scenario_base = 0;
  } else {
    if (view.plane_stride < (int64_t)sc->n_scenarios * sc->n_slots || view.scenario_base < 0)
      return set_msg("scenario window: plane_stride smaller than the window / negative scenario_base");
    if (st->trace_cap > 0) return set_msg("traces are not supported on a scenario window");
  }
  sc = &view;
  cudaError_t err = cudaSetDevice(device);
  if (err != cudaSuccess) return set_err("cudaSetDevice", err);
  const bool ped = sc->route_off != nullptr && sc->n_route_pts > 0;
  const bool rss = (p->features & SG_FEAT_RSS) != 0;
  const uint32_t veh_bits = (1u << SG_KIND_VEHICLE), ok_bits = veh_bits | (1u << SG_KIND_EMPTY);
  // the ego_off_road terminal condition and the boundary forces live in the general kernel only
  const bool roads = (p->terminal & SG_TERM_EGO_OFF_ROAD) != 0;
  const bool veh_only = (sc->kind_mask & veh_bits) && !(sc->kind_mask & ~ok_bits) && !roads && !sc->veh_limits &&
                        !(sc->scene_flags & SG_SCENE_FLAT_BOXES);
  const bool grid_ok = ped && p->ped_distance_threshold > 0.0 && p->ped_distance_threshold < 1.0e6 &&
                       !(p->features & SG_FEAT_NO_GRID);
  GroupLayout L = make_layout(sc->n_slots, ped, rss, veh_only, grid_ok);
  if (L.grid && (size_t)L.bytes > 227 * 1024) L = make_layout(sc->n_slots, ped, rss, veh_only, false);
  const int threads = L.G <= SG_THREADS ? SG_THREADS : L.G;
  const bool big = threads > SG_THREADS;
  const int gpb = threads / L.G;
  const int blocks = (sc->n_scenarios + gpb - 1) / gpb;
  const size_t smem = (size_t)gpb * L.bytes;
  if (smem > 227 * 1024) return set_msg("scenario does not fit in shared memory");
  cudaStream_t s = (cudaStream_t)stream;
  if (reset) {
    err = sgi_launch_reset(rss, big, blocks, threads, smem, s, *sc, *p, *st, L, reset_mask);
    if (err != cudaSuccess) return set_err("sg_reset_kernel launch", err);
    return 0;
  }
  SgInputs none;
  memset(&none, 0, sizeof(none));
  const SgInputs inp = in ? *in : none;
  // replay-only scenes (every slot a BatchReplayEntity or ReplayTrajectoryAgent) rolled out for
  // several ticks: the tick-parallel kernel (sg_replay.cuh)
  const uint32_t replay_bits = (1u << SG_KIND_EMPTY) | (1u << SG_KIND_REPLAY) | (1u << SG_KIND_AGENT_REPLAY);
  const bool replay_only = sc->kind_mask != 0 && !(sc->kind_mask & ~replay_bits) &&
                           (sc->kind_mask & ~(1u << SG_KIND_EMPTY));
  if (replay_only && !roads && !rss && !ped && sc->n_slots <= 32 && st->trace_cap == 0 && !inp.step_done &&
      !inp.host_present && p->timestep > 0.0 && (n_ticks < 0 || n_ticks >= 8) &&
      !(p->features & SG_FEAT_SEQUENTIAL)) {
    err = sgi_launch_replay(s, *sc, *p, *st, n_ticks);
    if (err != cudaSuccess) return set_err("sg_replay_kernel launch", err);
    return 0;
  }
  // crowd scenes (more than 256 slots of pedestrians / replayed agents): the two-scenarios-per-SM kernel
  const uint32_t crowd_bits = (1u << SG_KIND_EMPTY) | (1u << SG_KIND_PEDESTRIAN) | (1u << SG_KIND_AGENT_REPLAY);
  if (grid_ok && !rss && !roads && sc->n_networks <= 0 && sc->n_slots > SG_THREADS && (sc->kind_mask & (1u << SG_KIND_PEDESTRIAN)) &&
      !(sc->kind_mask & ~crowd_bits) && st->trace_cap == 0 && !inp.host_present) {
    err = sgi_launch_crowd(s, *sc, *p, *st, inp, n_ticks);
    if (err != cudaSuccess) return set_err("sg_crowd_kernel launch", err);
    return 0;
  }
  const int act = inp.actions ? ACT_F64 : (inp.actions_f32 ? ACT_F32 : (inp.use_rng ? ACT_RNG : -1));
  SgRngDev rng;
  memset(&rng, 0, sizeof(rng));
  if (act == ACT_RNG) {
    const int rc = check_rng(inp.rng);
    if (rc) return rc;
    if (inp.rng_tick0 < 0) return set_msg("rng_tick0 must be >= 0");
    rng = make_rng_dev(inp.rng, inp.rng_tick0);
  }
  if (veh_only) {
    if (act < 0) return set_msg("vehicle scene needs an action source (table or rng)");
    if (act != ACT_F64 && !sgi_vehicle_lean(*p, *st))
      return set_msg("trace / pair-matrix rollouts of vehicle scenes take an fp64 action table "
                     "(materialise the rows with sg_fill_random_actions / widen the fp32 table)");
    err = rss ? sgi_launch_vehicle_rss1(sc->n_scenarios, s, *sc, *p, *st, inp, rng, act, n_ticks, L)
              : sgi_launch_vehicle_rss0(sc->n_scenarios, s, *sc, *p, *st, inp, rng, act, n_ticks, L);
  } else {
    err = sgi_launch_rollout(ped, rss, big, blocks, threads, smem, s, *sc, *p, *st, inp, rng, n_ticks, L);
  }
  if (err != cudaSuccess) return set_err("sg_rollout_kernel launch", err);
  return 0;
}

extern "C" {

int sg_abi_version(void) { return SG_ABI_VERSION; }

int64_t sg_sizeof(int which) {
  switch (which) {
    case 0: return sizeof(SgParams);
    case 1: return sizeof(SgScene);
    case 2: return sizeof(SgState);
    case 3: return sizeof(SgInputs);
    case 4: return sizeof(SgEvent);
    case 5: return sizeof(SgActionRng);
    case 6: return sizeof(SgHostResults);
    case 7: return sizeof(SgEnvSpec);
  }
  return -1;
}

const char* sg_last_error(void) { return g_err; }

void sg_default_params(SgParams* p) {
  memset(p, 0, sizeof(*p));
  p->timestep = 1.0 / 30.0;
  p->terminal = SG_TERM_MAX_LENGTH;
  p->features = SG_FEAT_COLLISIONS | SG_FEAT_EGO_METRICS;
  p->max_ticks = 1 << 20;
  p->veh_max_steer = 0.7;
  p->veh_max_accel = 5.0;
  p->veh_max_speed = NAN;
  p->ped_max_speed = 5.0;
  p->ped_distance_threshold = 1.0;
  p->sf_max_speed_factor = 1.3;
  p->sf_sight_weight = 0.5;
  p->sf_sight_weight_use = 1;
  p->sf_sight_angle = 200.0;
  p->sf_relaxation_time = 1.5;
  p->sf_ped_repulse_V = 1.0;
  p->sf_ped_repulse_sigma = 1.0;
  p->rss_response_time = 0.6;
  p->rss_min_long_accel = 1.2 * 9.81;
  p->rss_max_long_accel = 1.2 * 9.81;
  p->rss_min_safe_clearance = 0.1;
  p->pid_steer_Kp = 0.03054;
  p->pid_steer_Kd = 1.5709;
  p->pid_accel_Kp = 0.3753;
  p->pid_accel_Kd = 1.8970;
  p->pid_accel_Ki = 0.0204;
  p->sf_boundary_repulse_U = 10.0; /* pedestrian/social_force.py:26-29 */
  p->sf_boundary_repulse_R = 0.2;
  p->sf_imp_boundary_repulse_U = 2.0;
  p->sf_imp_boundary_repulse_R = 0.1;
}

int sg_reset(const SgScene* scene, const SgParams* params, SgState* state, int device, void* stream) {
  if (state && state->event_count) {
    cudaError_t err = cudaSetDevice(device);
    if (err != cudaSuccess) return set_err("cudaSetDevice", err);
    err = cudaMemsetAsync(state->event_count, 0, sizeof(int32_t), (cudaStream_t)stream);
    if (err != cudaSuccess) return set_err("cudaMemsetAsync", err);
  }
  return launch(scene, params, state, nullptr, 0, device, stream, 1);
}

int sg_rollout(const SgScene* scene, const SgParams* params, SgState* state, const SgInputs* inputs,
               int n_ticks, int device, void* stream) {
  return launch(scene, params, state, inputs, n_ticks, device, stream, 0);
}

int sg_reset_scenarios(const SgScene* scene, const SgParams* params, SgState* state, const uint8_t* mask,
                       int device, void* stream) {
  return launch(scene, params, state, nullptr, 0, device, stream, 1, mask);
}

// the checks sg_env_observe and sg_env_reward share; `view` gets the scene with its plane stride stated
static int check_env(const SgScene* sc, const SgParams* p, const SgState* st, const SgEnvSpec* e, SgScene* view) {
  if (!sc || !p || !st || !e) return set_msg("null argument");
  if (sc->n_slots < 1 || sc->n_slots > 1024) return set_msg("n_slots must be in 1..1024");
  if (sc->n_scenarios < 1) return set_msg("n_scenarios must be >= 1");
  if (sc->plane_stride > 0) return set_msg("sg_env_*: scenario windows are not supported");
  if (e->n_agents < 1 || e->n_agents > sc->n_slots) return set_msg("SgEnvSpec.n_agents must be in 1..n_slots");
  if (e->k_neighbours < 0 || e->k_neighbours > 32) return set_msg("SgEnvSpec.k_neighbours must be in 0..32");
  if (e->n_lookahead < 0 || e->n_lookahead > 8) return set_msg("SgEnvSpec.n_lookahead must be in 0..8");
  for (int k = 0; k < e->n_lookahead; ++k)
    if (!isfinite(e->lookahead[k])) return set_msg("SgEnvSpec.lookahead must be finite");
  if (!isfinite(e->radius)) return set_msg("SgEnvSpec.radius must be finite");
  if (!e->agent_slot || !e->snap_dist || !e->snap_collided || !e->snap_pair_ticks || !e->snap_rss)
    return set_msg("SgEnvSpec: agent_slot / snapshot buffers missing");
  *view = *sc;
  view->plane_stride = (int64_t)sc->n_scenarios * sc->n_slots;
  view->scenario_base = 0;
  return 0;
}

int sg_env_observe(const SgScene* scene, const SgParams* params, const SgState* state, const SgEnvSpec* spec,
                   const uint8_t* mask, float* obs, uint8_t* agent_mask, int device, void* stream) {
  SgScene view;
  int rc = check_env(scene, params, state, spec, &view);
  if (rc) return rc;
  if (!obs || !agent_mask) return set_msg("null argument");
  cudaError_t err = cudaSetDevice(device);
  if (err != cudaSuccess) return set_err("cudaSetDevice", err);
  err = sgi_launch_env_observe((cudaStream_t)stream, view, *state, *spec, mask, obs, agent_mask);
  if (err != cudaSuccess) return set_err("sg_env_observe_kernel launch", err);
  return 0;
}

int sg_env_reward(const SgScene* scene, const SgParams* params, const SgState* state, const SgEnvSpec* spec,
                  float* reward, float* terms, uint8_t* terminated, uint8_t* truncated, int device,
                  void* stream) {
  SgScene view;
  int rc = check_env(scene, params, state, spec, &view);
  if (rc) return rc;
  if (!reward || !terms || !terminated || !truncated) return set_msg("null argument");
  cudaError_t err = cudaSetDevice(device);
  if (err != cudaSuccess) return set_err("cudaSetDevice", err);
  err = sgi_launch_env_reward((cudaStream_t)stream, view, *params, *state, *spec, reward, terms, terminated,
                              truncated);
  if (err != cudaSuccess) return set_err("sg_env_reward_kernel launch", err);
  return 0;
}

int sg_fill_random_actions(const SgActionRng* rng, int tick0, int n_ticks, int64_t nm, double* out,
                           int device, void* stream) {
  if (!rng || (!out && n_ticks > 0 && nm > 0)) return set_msg("null argument");
  if (tick0 < 0 || n_ticks < 0 || nm < 0) return set_msg("negative size");
  const int rc = check_rng(*rng);
  if (rc) return rc;
  cudaError_t err = cudaSetDevice(device);
  if (err != cudaSuccess) return set_err("cudaSetDevice", err);
  err = sgi_launch_fill_actions((cudaStream_t)stream, make_rng_dev(*rng, tick0), n_ticks, nm, out);
  if (err != cudaSuccess) return set_err("sg_fill_actions_kernel launch", err);
  return 0;
}

int sg_entities_in_radius(const SgState* state, int n_scenarios, int n_slots, const double* x, const double* y,
                          const double* r, uint8_t* out, int device, void* stream) {
  if (!state || !x || !y || !r || !out) return set_msg("null argument");
  if (n_scenarios < 1 || n_slots < 1) return set_msg("empty batch");
  cudaError_t err = cudaSetDevice(device);
  if (err != cudaSuccess) return set_err("cudaSetDevice", err);
  err = sgi_launch_radius((cudaStream_t)stream, *state, n_scenarios, n_slots, x, y, r, out);
  if (err != cudaSuccess) return set_err("sg_radius_kernel launch", err);
  return 0;
}

int sg_build_union_x(const SgScene* scene, int device, void* stream) {
  if (!scene) return set_msg("null argument");
  if (scene->n_union_rows <= 0) return 0;
  if (!scene->union_off || !scene->union_t || !scene->union_x || !scene->traj_off || !scene->traj_rows || !scene->kind)
    return set_msg("sg_build_union_x: the scene lacks union_off / union_t / union_x / trajectories");
  cudaError_t err = cudaSetDevice(device);
  if (err != cudaSuccess) return set_err("cudaSetDevice", err);
  err = sgi_launch_union((cudaStream_t)stream, *scene, scene->n_union_rows);
  if (err != cudaSuccess) return set_err("sg_union_kernel launch", err);
  return 0;
}

int sg_test_trajectory(const double* rows, int64_t K, const double* t, int64_t n, int mode, double* pos,
                       uint8_t* ok, double* vel, int device, void* stream) {
  if (!rows || !t || !pos || !ok) return set_msg("null argument");
  if (K < 1 || K > 0x7fffffff || mode < 0 || mode > 2) return set_msg("bad trajectory length / mode");
  cudaError_t err = cudaSetDevice(device);
  if (err != cudaSuccess) return set_err("cudaSetDevice", err);
  err = sgi_launch_traj((cudaStream_t)stream, rows, (int)K, t, n, mode, pos, ok, vel);
  if (err != cudaSuccess) return set_err("sg_traj_kernel launch", err);
  return 0;
}

int sg_measure_fp64_peak(double* inst_per_s, int device, void* stream) {
  if (!inst_per_s) return set_msg("null argument");
  cudaError_t err = cudaSetDevice(device);
  if (err != cudaSuccess) return set_err("cudaSetDevice", err);
  err = sgi_measure_fp64((cudaStream_t)stream, inst_per_s);
  if (err != cudaSuccess) return set_err("sg_dfma_kernel", err);
  return 0;
}

int sg_test_box_pairs(const double* pose_a, const double* box_a, const double* pose_b,
                      const double* box_b, uint8_t* out, int64_t n, int device, void* stream) {
  cudaError_t err = cudaSetDevice(device);
  if (err != cudaSuccess) return set_err("cudaSetDevice", err);
  if (n <= 0) return 0;
  err = sgi_launch_box_pairs((cudaStream_t)stream, pose_a, box_a, pose_b, box_b, out, n);
  if (err != cudaSuccess) return set_err("sg_box_pairs_kernel launch", err);
  return 0;
}

int sg_future_collisions(const SgScene* scene, const double* t, const int32_t* slot, double horizon,
                         int n_samples, uint8_t* out, int device, void* stream) {
  if (!scene || !t || !out) return set_msg("null argument");
  if (n_samples < 1) return set_msg("n_samples must be >= 1");
  cudaError_t err = cudaSetDevice(device);
  if (err != cudaSuccess) return set_err("cudaSetDevice", err);
  SgScene view = *scene;
  if (view.plane_stride <= 0) view.plane_stride = (int64_t)scene->n_scenarios * scene->n_slots;
  err = sgi_launch_future((cudaStream_t)stream, view, t, slot, horizon, n_samples, out);
  if (err != cudaSuccess) return set_err("sg_future_kernel launch", err);
  return 0;
}

// ---- host-buffer path ------------------------------------------------------------------
// scenarios [n0, n1) of a scene laid out for the whole batch (SgScene.plane_stride / scenario_base)
static SgScene scene_window(const SgScene& s, int n0, int n1) {
  SgScene w = s;
  const int64_t M = s.n_slots, off = (int64_t)n0 * M;
  w.n_scenarios = n1 - n0;
  w.plane_stride = s.plane_stride > 0 ? s.plane_stride : (int64_t)s.n_scenarios * M;
  w.scenario_base = (s.plane_stride > 0 ? s.scenario_base : 0) + n0;
#define OFF(f, k) if (w.f) w.f += (k)
  OFF(kind, off); OFF(etype, off); OFF(box, off); OFF(traj_off, off); OFF(union_off, n0);
  OFF(t0, n0); OFF(length, n0); OFF(ego_slot, n0); OFF(first_slot, n0);
  OFF(ped_speed_desired, off); OFF(route_off, off); OFF(rn_of, n0); OFF(veh_limits, off);
#undef OFF
  return w;
}
static SgState state_window(const SgState& s, const SgParams& p, int n0, int M) {
  SgState w = s;
  const int64_t off = (int64_t)n0 * M, W = (M + 31) / 32;
#define OFF(f, k) if (w.f) w.f += (k)
  OFF(pose, off); OFF(vel, off); OFF(dist, off); OFF(present, off); OFF(speed, off); OFF(goal_idx, off);
  OFF(force, off); OFF(cur_own, off); OFF(collided, off); OFF(rss_state, off); OFF(rss_last, off);
  OFF(safe_dist, off); OFF(safe_ratio, off); OFF(pid_err, off);
  OFF(t, n0); OFF(prev_t, n0); OFF(tick, n0); OFF(done, n0); OFF(cur_union, n0);
  OFF(ego_avg_speed, n0); OFF(ego_avg_t, n0); OFF(ego_max_speed, n0); OFF(ego_dist, n0);
  OFF(first_coll_tick, n0); OFF(n_pair_ticks, n0); OFF(rss_flags, n0);
  OFF(ego_hits, (int64_t)n0 * W); OFF(first_coll_pair, 2 * (int64_t)n0);
  if (p.features & SG_FEAT_COLL_MATRIX) OFF(coll_mask, (int64_t)n0 * M * W);
#undef OFF
  return w;
}

// Host -> device copies of scenarios [n0, n1) of a scene (`shared`: also the arrays all scenarios share,
// the road networks).  With `do_copy` false only the bytes are counted.  Returns 0 or an error code.
// `part`: 0 = every array of scenarios [n0, n1); 1 = the per-slot / per-scenario arrays of the WHOLE batch and the
// control points / knot tables of [n0, n1); 2 = the control points / knot tables of [n0, n1) only.  (Upload-bound
// batches: the small arrays go up once with the first window instead of a dozen small copies per window.)
static int copy_scene_window(const SgScene* h, const SgScene* d, int n0, int n1, bool shared, bool do_copy,
                             cudaStream_t s, int64_t* bytes, int part = 0) {
  const int64_t N = h->n_scenarios, M = h->n_slots, NM = N * M;
  const int m0 = part == 1 ? 0 : n0, m1 = part == 1 ? (int)N : n1;  // the scenarios whose small arrays go up
  const int64_t o = (int64_t)m0 * M, cnt = part == 2 ? 0 : (int64_t)(m1 - m0) * M;
  const int ns = part == 2 ? 0 : m1 - m0;
  const int64_t bo = (int64_t)n0 * M, bcnt = (int64_t)(n1 - n0) * M;  // the slots whose control points go up
  int64_t total = 0;
  cudaError_t err = cudaSuccess;
  auto flat = [&](const void* src, const void* dst, int64_t first, int64_t n, int64_t esz) -> bool {
    if (!src || n <= 0) return true;
    total += n * esz;
    if (!do_copy) return true;
    if (!dst) { set_msg("device scene mirror is missing an array"); return false; }
    err = cudaMemcpyAsync((char*)dst + first * esz, (const char*)src + first * esz, (size_t)(n * esz),
                          cudaMemcpyHostToDevice, s);
    if (err != cudaSuccess) { set_err("cudaMemcpyAsync H2D scene", err); return false; }
    return true;
  };
  auto planes = [&](const void* src, const void* dst, int np, int64_t esz) -> bool {  // [np][N*M]
    if (!src || cnt <= 0) return true;
    total += (int64_t)np * cnt * esz;
    if (!do_copy) return true;
    if (!dst) { set_msg("device scene mirror is missing an array"); return false; }
    err = cudaMemcpy2DAsync((char*)dst + o * esz, (size_t)(NM * esz), (const char*)src + o * esz, (size_t)(NM * esz),
                            (size_t)(cnt * esz), (size_t)np, cudaMemcpyHostToDevice, s);
    if (err != cudaSuccess) { set_err("cudaMemcpy2DAsync H2D scene", err); return false; }
    return true;
  };
  bool ok = true;
  if (part != 2)
    ok = planes(h->kind, d->kind, 1, 1) && planes(h->etype, d->etype, 1, 1) && planes(h->box, d->box, 4, 8) &&
         flat(h->traj_off, d->traj_off, o, cnt + 1, 8) && planes(h->veh_limits, d->veh_limits, 4, 8) &&
         flat(h->union_off, d->union_off, m0, ns + 1, 8) && flat(h->t0, d->t0, m0, ns, 8) &&
         flat(h->length, d->length, m0, ns, 8) && flat(h->ego_slot, d->ego_slot, m0, ns, 4) &&
         flat(h->first_slot, d->first_slot, m0, ns, 4);
  if (ok && h->traj_off && h->traj_rows) {
    const int64_t r0 = h->traj_off[bo], r1 = h->traj_off[bo + bcnt];
    ok = flat(h->traj_rows, d->traj_rows, r0 * 7, (r1 - r0) * 7, 8);
  }
  if (ok && h->union_off && h->n_union_rows > 0) {
    const int64_t u0 = h->union_off[n0], u1 = h->union_off[n1];
    ok = flat(h->union_t, d->union_t, u0, u1 - u0, 8) && flat(h->union_x, d->union_x, u0 * 6 * M, (u1 - u0) * 6 * M, 8);
  }
  // (kind_mask: OR of 1 << kind over the slots, 0 = not stated) pedestrian rows are only read for pedestrians
  if (ok && (h->kind_mask == 0 || (h->kind_mask & (1u << SG_KIND_PEDESTRIAN)))) {
    if (part != 2)
      ok = planes(h->ped_speed_desired, d->ped_speed_desired, 1, 8) && flat(h->route_off, d->route_off, o, cnt + 1, 8);
    if (ok && h->route_off && h->route_xy) {
      const int64_t r0 = h->route_off[bo], r1 = h->route_off[bo + bcnt];
      ok = flat(h->route_xy, d->route_xy, r0 * 2, (r1 - r0) * 2, 8);
    }
  }
  if (ok && h->n_networks > 0 && part != 2) {
    ok = flat(h->rn_of, d->rn_of, m0, ns, 4);
    if (ok && shared)
      ok = flat(h->rn_poly_off, d->rn_poly_off, 0, 3 * (int64_t)h->n_networks + 1, 8) &&
           flat(h->rn_edge_off, d->rn_edge_off, 0, h->n_rn_polys + 1, 8) &&
           flat(h->rn_edges, d->rn_edges, 0, h->n_rn_edges * 4, 8) &&
           flat(h->rn_has_area, d->rn_has_area, 0, 3 * (int64_t)h->n_networks, 1);
  }
  if (bytes) *bytes = total;
  return ok ? 0 : (err != cudaSuccess ? -2 : -1);
}

int64_t sg_host_h2d_bytes(const SgScene* h, const SgInputs* in, int copy_static) {
  int64_t total = 0;
  if (copy_static) copy_scene_window(h, h, 0, h->n_scenarios, true, false, nullptr, &total);
  const int64_t nm = (int64_t)h->n_scenarios * h->n_slots;
  if (in && in->actions) total += (int64_t)in->n_action_ticks * 2 * nm * 8;
  else if (in && in->actions_f32) total += (int64_t)in->n_action_ticks * 2 * nm * 4;
  return total;
}

int64_t sg_host_d2h_bytes(const SgScene* h) {
  const int64_t N = h->n_scenarios;
  return N * (8 * 3 + 4 + 8 + 8 + 1 + 4 + 8) + 4;
}

// streams + events of the host-buffer path, one set per device (created on first use)
#define SG_HOST_MAX_WINDOWS 6
struct HostPathCtx {
  cudaStream_t copy_stream, aux_stream;
  cudaEvent_t ev_copy[2], ev_done, ev_win[SG_HOST_MAX_WINDOWS], ev_aux;
  bool ready;
};
static HostPathCtx g_host_ctx[64];

static int host_ctx(int device, HostPathCtx** out) {
  if (device < 0 || device >= 64) return set_msg("device index out of range");
  HostPathCtx& c = g_host_ctx[device];
  if (!c.ready) {  // (the caller has made `device` current)
    cudaError_t err = cudaStreamCreateWithFlags(&c.copy_stream, cudaStreamNonBlocking);
    if (err != cudaSuccess) return set_err("cudaStreamCreateWithFlags", err);
    err = cudaStreamCreateWithFlags(&c.aux_stream, cudaStreamNonBlocking);
    if (err != cudaSuccess) return set_err("cudaStreamCreateWithFlags", err);
    cudaEvent_t* evs[4 + SG_HOST_MAX_WINDOWS] = {&c.ev_copy[0], &c.ev_copy[1], &c.ev_done, &c.ev_aux};
    for (int q = 0; q < SG_HOST_MAX_WINDOWS; ++q) evs[4 + q] = &c.ev_win[q];
    for (int q = 0; q < 4 + SG_HOST_MAX_WINDOWS; ++q) {
      err = cudaEventCreateWithFlags(evs[q], cudaEventDisableTiming);
      if (err != cudaSuccess) return set_err("cudaEventCreateWithFlags", err);
    }
    c.ready = true;
  }
  *out = &c;
  return 0;
}

// How many windows a batch without an action table is uploaded and rolled out in: the first one small,
// so the rollout starts early, the upload of every later window hidden behind the rollout of the one
// before.  SG_HOST_WINDOWS=<n> (1 .. 4) overrides the choice (1: one upload, then one rollout).
// replay-only scenes: a rollout costs less than its upload (C2: 115 MB of control points against a 1 ms kernel)
static bool host_upload_bound(const SgScene* hs) {
  const uint32_t replay_bits = (1u << SG_KIND_EMPTY) | (1u << SG_KIND_REPLAY) | (1u << SG_KIND_AGENT_REPLAY);
  return hs->kind_mask != 0 && !(hs->kind_mask & ~replay_bits);
}
static int host_windows(const SgScene* hs, int64_t scene_bytes) {
  const char* env = getenv("SG_HOST_WINDOWS");
  int n = (scene_bytes >= (8 << 20) && hs->n_scenarios >= 64) ? (host_upload_bound(hs) ? 5 : (hs->n_scenarios >= 4096 ? 4 : 3)) : 1;
  if (env && env[0] >= '1' && env[0] <= '0' + SG_HOST_MAX_WINDOWS && !env[1]) n = env[0] - '0';
  if (n > hs->n_scenarios) n = hs->n_scenarios;
  return n < 1 ? 1 : n;
}

int sg_rollout_host(const SgScene* hs, const SgScene* ds, const SgParams* params, SgState* dst,
                    const SgInputs* hin, const SgInputs* din, SgHostResults* res, int copy_static,
                    int device, void* stream) {
  if (!hs || !ds || !params || !dst || !res) return set_msg("null argument");
  cudaError_t err = cudaSetDevice(device);
  if (err != cudaSuccess) return set_err("cudaSetDevice", err);
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t N = hs->n_scenarios, NM = N * hs->n_slots;
  const bool table64 = hin && hin->actions, table32 = hin && !hin->actions && hin->actions_f32;
  const bool build_union = copy_static && !hs->union_x && hs->n_union_rows > 0;  // knot times uploaded, rows built here
  int rc = 0;
#define SG_CK(call, what) do { err = (call); if (err != cudaSuccess) return set_err(what, err); } while (0)
  int64_t scene_bytes = 0;
  copy_scene_window(hs, ds, 0, (int)N, true, false, nullptr, &scene_bytes);
  const int nwin = (copy_static && !table64 && !table32 && dst->trace_cap <= 0 && hs->plane_stride <= 0)
                       ? host_windows(hs, scene_bytes) : 1;
  if (nwin > 1) {
    // Scenarios are independent: the batch goes up in windows on a copy stream, and every window is
    // reset and rolled out (alternating between two compute streams, so one window's last CTAs overlap
    // the next one's first) as soon as it has arrived.
    HostPathCtx* ctx = nullptr;
    rc = host_ctx(device, &ctx);
    if (rc) return rc;
    if (dst->event_count) SG_CK(cudaMemsetAsync(dst->event_count, 0, sizeof(int32_t), s), "cudaMemsetAsync");
    SG_CK(cudaEventRecord(ctx->ev_done, s), "cudaEventRecord");
    SG_CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_done, 0), "cudaStreamWaitEvent");
    SG_CK(cudaStreamWaitEvent(ctx->aux_stream, ctx->ev_done, 0), "cudaStreamWaitEvent");
    int bounds[SG_HOST_MAX_WINDOWS + 1];
    bounds[0] = 0;
    // Compute-bound batches: windows end at 1/32, 1/8, 1/2, 1 of the batch (four windows; three from 1/8 on when the
    // batch has fewer than 4096 scenarios: a first window of a few dozen one-scenario CTAs leaves the GPU idle), each four times the last --
    // the first rollout starts early and the uploads hide behind the rollouts.  Upload-bound batches (replay-only
    // scenes): what cannot hide is the LAST window's rollout, so the windows end at 1/8, 3/8, 5/8, 7/8, 1.
    const bool even = host_upload_bound(hs) && nwin >= 3;
    for (int w = 1; w <= nwin; ++w)
      bounds[w] = w == nwin ? (int)N
                            : even ? (int)(N * (2 * w - 1) / (2 * (nwin - 1))) : (int)(N >> (2 * (nwin - w) - 1));
    bool used_aux = false;
    for (int w = 0; w < nwin; ++w) {
      const int n0 = bounds[w], n1 = bounds[w + 1];
      if (n1 <= n0) continue;
      rc = copy_scene_window(hs, ds, n0, n1, w == 0, true, ctx->copy_stream, nullptr, even ? (w == 0 ? 1 : 2) : 0);
      if (rc) return rc;
      SG_CK(cudaEventRecord(ctx->ev_win[w], ctx->copy_stream), "cudaEventRecord");
      cudaStream_t cs = (w & 1) ? ctx->aux_stream : s;
      used_aux = used_aux || (w & 1);
      SG_CK(cudaStreamWaitEvent(cs, ctx->ev_win[w], 0), "cudaStreamWaitEvent");
      const SgScene sw = scene_window(*ds, n0, n1);
      SgState stw = state_window(*dst, *params, n0, hs->n_slots);
      if (build_union) {
        err = sgi_launch_union(cs, sw, hs->union_off[n1] - hs->union_off[n0]);
        if (err != cudaSuccess) return set_err("sg_union_kernel launch", err);
      }
      rc = launch(&sw, params, &stw, nullptr, 0, device, (void*)cs, 1);
      if (rc) return rc;
      rc = launch(&sw, params, &stw, hin && hin->use_rng ? hin : din, -1, device, (void*)cs, 0);
      if (rc) return rc;
    }
    if (used_aux) {
      SG_CK(cudaEventRecord(ctx->ev_aux, ctx->aux_stream), "cudaEventRecord");
      SG_CK(cudaStreamWaitEvent(s, ctx->ev_aux, 0), "cudaStreamWaitEvent");
    }
  } else {
    if (copy_static) {
      rc = copy_scene_window(hs, ds, 0, (int)N, true, true, s, nullptr);
      if (rc) return rc;
    }
    if (build_union) {
      rc = sg_build_union_x(ds, device, stream);
      if (rc) return rc;
    }
    rc = sg_reset(ds, params, dst, device, stream);
    if (rc) return rc;
    if (table64 || table32) {
      if (!din || (table64 ? !din->actions : !din->actions_f32)) return set_msg("device action buffer missing");
      // stream the action table in chunks of ticks: the copy of chunk c+1 overlaps the kernel
      // of chunk c (copies on a second stream, ordered with events)
      const int T = hin->n_action_ticks;
      const int chunk = T < 16 ? T : 16;
      const size_t esz = table64 ? 8 : 4;
      HostPathCtx* ctx = nullptr;
      rc = host_ctx(device, &ctx);
      if (rc) return rc;
      SG_CK(cudaEventRecord(ctx->ev_done, s), "cudaEventRecord");
      SG_CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_done, 0), "cudaStreamWaitEvent");
      int c = 0;
      for (int k0 = 0; k0 < T; k0 += chunk, ++c) {
        const int kt = (T - k0) < chunk ? (T - k0) : chunk;
        const size_t off = (size_t)k0 * 2 * NM;
        const char* src = table64 ? (const char*)hin->actions : (const char*)hin->actions_f32;
        char* dstp = table64 ? (char*)din->actions : (char*)din->actions_f32;
        SG_CK(cudaMemcpyAsync(dstp + off * esz, src + off * esz, (size_t)kt * 2 * NM * esz,
                              cudaMemcpyHostToDevice, ctx->copy_stream), "cudaMemcpyAsync H2D actions");
        SG_CK(cudaEventRecord(ctx->ev_copy[c & 1], ctx->copy_stream), "cudaEventRecord");
        SG_CK(cudaStreamWaitEvent(s, ctx->ev_copy[c & 1], 0), "cudaStreamWaitEvent");
        SgInputs part = *din;
        if (table64) { part.actions = din->actions + off; part.actions_f32 = nullptr; }
        else { part.actions = nullptr; part.actions_f32 = din->actions_f32 + off; }
        part.n_action_ticks = kt;
        rc = sg_rollout(ds, params, dst, &part, kt, device, stream);
        if (rc) return rc;
      }
    } else {  // no table to move (replay / pedestrians / device-side action source): one fused rollout
      rc = sg_rollout(ds, params, dst, hin && hin->use_rng ? hin : din, -1, device, stream);
      if (rc) return rc;
    }
  }
#undef SG_CK
#define BACK(field, bytes_)                                                                   \
  if (res->field) {                                                                           \
    err = cudaMemcpyAsync(res->field, dst->field, (size_t)(bytes_), cudaMemcpyDeviceToHost, s); \
    if (err != cudaSuccess) return set_err("cudaMemcpyAsync D2H " #field, err);               \
  }
  BACK(ego_avg_speed, N * 8);
  BACK(ego_max_speed, N * 8);
  BACK(ego_dist, N * 8);
  BACK(first_coll_tick, N * 4);
  BACK(first_coll_pair, N * 8);
  BACK(n_pair_ticks, N * 8);
  BACK(rss_flags, N);
  BACK(tick, N * 4);
  BACK(t, N * 8);
  BACK(event_count, 4);
#undef BACK
  return 0;
}

}  // extern "C"

