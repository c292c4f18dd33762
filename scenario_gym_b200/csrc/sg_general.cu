// sg_general.cu -- the general tick-loop kernel (replay / batch replay / vehicles / pedestrians /
// PID / host-driven slots) and the reset kernel.
#define SG_FLAT_BOXES 1  // boxes without area follow their own narrow-phase rules (sg_common.cuh)
#include "sg_common.cuh"
#include "sg_internal.h"
#include "sg_pcg.cuh"

// ---------------------------------------------------------------------------------
// General scenes: replay / batch replay / vehicles / pedestrians / host-driven slots.
// ---------------------------------------------------------------------------------
struct Ent {
  double pose[6], vel[6], dist, speed;
  bool present;
};

// VehicleAction row `row` of slot index i from the device-side action source (rare in this kernel:
// mixed scenes; the jump is recomputed per tick so the tick loop carries no generator state)
static __device__ __noinline__ double2 rng_action(SgRngDev rng, int row, int64_t i) {
  // advancing by `row` tick strides = applying x -> a x + c `row` times: composed by squaring
  sg_u128 am = 1, ap = 0, cm = sg_u128_make(rng.a_hi, rng.a_lo), cp = sg_u128_make(rng.c_hi, rng.c_lo);
  for (unsigned r = (unsigned)row; r > 0; r >>= 1) {
    if (r & 1) { am *= cm; ap = ap * cm + cp; }
    cp = (cm + 1) * cp;
    cm *= cm;
  }
  double2 out;
  sg_u128 q = am * sg_rng_slot_state(rng, 0, i) + ap;
  out.x = rng.low[0] + rng.scale[0] * sg_pcg_double((uint64_t)(q >> 64), (uint64_t)q);
  q = am * sg_rng_slot_state(rng, 1, i) + ap;
  out.y = rng.low[1] + rng.scale[1] * sg_pcg_double((uint64_t)(q >> 64), (uint64_t)q);
  return out;
}

template <bool PED, bool RSS, int MAXT>
__global__ void __launch_bounds__(MAXT, MAXT >= 1024 ? 1 : 2)
sg_rollout_kernel(SgScene sc, SgParams p, SgState st, SgInputs in, int n_ticks, GroupLayout L, SgRngDev rng) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int G = L.G, M = sc.n_slots, W = L.W;
  const int gpb = blockDim.x / G;  // scenario groups per CTA
  const int gl = threadIdx.x / G;
  const int s = threadIdx.x - gl * G;
  const int n = blockIdx.x * gpb + gl;
  if (gl >= gpb || n >= sc.n_scenarios) return;
  Grp c;
  setup_group(c, sc, L, smem, gl, s, n);

  const bool live = s < M;  // padding threads only take part in barriers
  const int64_t i = c.i, nm = c.nm;
  const int kind = live ? sc.kind[i] : SG_KIND_EMPTY;
  const int etype = live ? sc.etype[i] : 0;
  const int ego_slot = sc.ego_slot[n], first_slot = sc.first_slot[n];
  const bool need_coll = (p.features & SG_FEAT_COLLISIONS) ||
                         (p.terminal & (SG_TERM_COLLISION | SG_TERM_EGO_COLLISION));
  const bool feat_rss = RSS && (p.features & SG_FEAT_RSS);
  const bool matrix = (p.features & SG_FEAT_COLL_MATRIX) != 0;
  const bool exact_div = kind <= SG_KIND_AGENT_REPLAY || kind == SG_KIND_PID;  // IEEE quotients
  const RssConst KR = make_rss_const(p);

  double bl = 1;
  int orient_hint = 0;
  const double* rows = nullptr;
  int K = 0;
  if (kind != SG_KIND_EMPTY) {
    const double bw = sc.box[i];
    bl = sc.box[nm + i];
    c.boxp[s] = bw; c.boxp[G + s] = bl;
    c.boxp[2 * G + s] = sc.box[2 * nm + i]; c.boxp[3 * G + s] = sc.box[3 * nm + i];
    orient_hint = box_orientation_hint(bw, bl);
    const int64_t r0 = sc.traj_off[i];
    K = (int)(sc.traj_off[i + 1] - r0);
    rows = sc.traj_rows + r0 * 7;
  }
  const double traj_min_t = K ? __ldg(rows) : 0.0;
  const double traj_max_t = K ? __ldg(rows + (int64_t)(K - 1) * 7) : 0.0;
  const double rcp_bl = 1.0 / bl;
  double ox, oy;  // scenario origin for the fp32 bounds: the ego's first control point
  {
    const int64_t er = sc.traj_off[(int64_t)n * M + ego_slot];
    ox = __ldg(sc.traj_rows + er * 7 + 1);
    oy = __ldg(sc.traj_rows + er * 7 + 2);
  }
  const double sight_cos = PED ? cos(p.sf_sight_angle / 2 * M_PI / 180) : 0.0;
  const double length = sc.length[n];

  // ---- load the State rows ------------------------------------------------------------
  Ent e;
  double t = st.t[n], prev_t = st.prev_t[n];
  int tick = st.tick[n], cur_union = st.cur_union[n];
  bool done = st.done[n] != 0;
  int cur_own = 1, goal = 0;
  double force[2] = {0, 0}, sd[2] = {0, 0}, ratio[2] = {0, 0};
  uint8_t rss_state = 0, rss_last = SG_RSS_NONE, collided = 0;
  if (live) {
#pragma unroll
    for (int f = 0; f < 6; ++f) { e.pose[f] = st.pose[f * nm + i]; e.vel[f] = st.vel[f * nm + i]; }
    e.dist = st.dist[i];
    e.speed = st.speed[i];
    e.present = st.present[i] != 0;
    cur_own = st.cur_own[i];
    collided = st.collided[i];
    if (PED) { goal = st.goal_idx[i]; force[0] = st.force[i]; force[1] = st.force[nm + i]; }
    if (RSS) {
      rss_state = st.rss_state[i]; rss_last = st.rss_last[i];
      sd[0] = st.safe_dist[i]; sd[1] = st.safe_dist[nm + i];
      ratio[0] = st.safe_ratio[i]; ratio[1] = st.safe_ratio[nm + i];
    }
  } else {
#pragma unroll
    for (int f = 0; f < 6; ++f) { e.pose[f] = 0; e.vel[f] = 0; }
    e.dist = 0; e.speed = 0; e.present = false;
  }
  load_cold(st, c, n, s, W, ego_slot);
  if (RSS && s == ego_slot) publish_ego_box(c);
  // crowd scenarios (one CTA per scenario) bin their entities into a cell grid of the sensor radius
  const bool use_grid = PED && L.grid != 0;
  const double grid_cs = p.ped_distance_threshold * (1.0 + 1e-6), grid_inv_cs = 1.0 / grid_cs;
  GridPos gpos;
  gpos.ix = 0; gpos.iy = 0; gpos.large = false;
  if (PED) {  // the "old" state the pedestrians' sensors read in the first tick
    if (live) stage_ped_state(c, e.present, etype, e.pose[0], e.pose[1], e.vel[0], e.vel[1],
                              p.ped_distance_threshold, ox, oy);
    for (int q = s; q < 32; q += G) c.pednb[M + q] = make_float4(INFINITY, INFINITY, -INFINITY, -INFINITY);
    if (use_grid) gpos = grid_build(c, live && e.present, false, e.pose[0], e.pose[1], ox, oy, grid_cs, grid_inv_cs);
  }
  group_sync(c);

  int limit = n_ticks < 0 ? p.max_ticks : n_ticks;
  // only scenarios with VehicleController slots are bounded by the action rows of the call
  if ((in.actions || in.actions_f32 || in.use_rng) && limit > in.n_action_ticks) {
    if (kind == SG_KIND_VEHICLE) c.cold_i[COLD_HAS_VEH] = 1;  // (zeroed by load_cold before the barrier above)
    group_sync(c);
    if (c.cold_i[COLD_HAS_VEH]) limit = in.n_action_ticks;
  }
  int parity = 0;

  for (int k = 0; k < limit && (!done || in.step_done); ++k) {
    // ---------------- phase A: agents / batch replay produce the new poses ----------------
    const double next_t = t + p.timestep;  // scenario_gym.py:229
    double np_[6];
    bool newpres = false;
    double newspeed = e.speed;
    double ped_np[6], ped_speed = e.speed;
    if (PED)  // every lane calls: whole warps of a scenario share the neighbour terms
      pedestrian_step<PED>(sc, p, c, kind == SG_KIND_PEDESTRIAN && e.present, G >= 32, e.pose, e.vel, t,
                           prev_t, next_t, sight_cos, goal, force, ped_speed, ped_np, use_grid, ox, oy,
                           grid_inv_cs, tick);
    if (kind >= SG_KIND_AGENT_REPLAY) {  // scenario_gym.py:233-244
      if (e.present) {
        if (kind == SG_KIND_AGENT_REPLAY) {  // agent.py:125-128, extrapolate=(False, False)
          position_at_t(rows, K, next_t, EXT_CLAMP, cur_own, np_);
          newpres = true;
        } else if (kind == SG_KIND_VEHICLE || kind == SG_KIND_PID) {
          double accel, steer;
          double sh, ch;
          sincos(e.pose[3], &sh, &ch);
          if (kind == SG_KIND_PID) {
            // PIDAgent._step (agent.py:144-148) + PIDController._step (controller.py:205-258);
            // the three error terms stay in global memory (rare kind)
            double tgt[6];
            position_at_t(rows, K, next_t, EXT_CLAMP, cur_own, tgt);
            const double e0 = tgt[0] - e.pose[0], e1 = tgt[1] - e.pose[1];
            const double e_lon = ch * e0 + sh * e1, e_lat = -sh * e0 + ch * e1;
            double gain_adj;
            if (e.speed > 5.0 && e.speed <= 15) gain_adj = 1.0 - 0.9 * ((e.speed - 5.0)) / 10.0;
            else if (e.speed > 15) gain_adj = 0.1;
            else gain_adj = 1.0;
            const double sdt = t - prev_t;  // state.dt
            const double e_lat_D = (e_lat - st.pid_err[2 * nm + i]) / sdt;
            steer = (p.pid_steer_Kp * gain_adj) * e_lat + (p.pid_steer_Kd * gain_adj) * e_lat_D;
            const double e_lon_D = (e_lon - st.pid_err[i]) / sdt;
            const double e_lon_I = st.pid_err[nm + i] + e_lon * sdt;
            accel = fabs(e_lon) > 0.1
                        ? p.pid_accel_Kp * e_lon + p.pid_accel_Kd * e_lon_D + p.pid_accel_Ki * e_lon_I
                        : 0.0;
            st.pid_err[2 * nm + i] = e_lat;
            st.pid_err[i] = e_lon;
            st.pid_err[nm + i] = e_lon_I;
          } else {
            if (in.actions) {
              accel = __ldcs(in.actions + ((int64_t)k * 2 + 0) * nm + i);
              steer = __ldcs(in.actions + ((int64_t)k * 2 + 1) * nm + i);
            } else if (in.actions_f32) {  // fp32 policy outputs: widening is exact
              accel = (double)__ldcs(in.actions_f32 + ((int64_t)k * 2 + 0) * nm + i);
              steer = (double)__ldcs(in.actions_f32 + ((int64_t)k * 2 + 1) * nm + i);
            } else {
              const double2 a = rng_action(rng, k, i + (int64_t)sc.scenario_base * sc.n_slots);
              accel = a.x; steer = a.y;
            }
          }
          // VehicleController._step, controller.py:105-140 (limits per agent when the scene carries them)
          double max_steer = p.veh_max_steer, max_accel = p.veh_max_accel, max_speed = p.veh_max_speed;
          bool allow_reverse = p.veh_allow_reverse != 0;
          if (sc.veh_limits) {
            max_steer = sc.veh_limits[i]; max_accel = sc.veh_limits[nm + i];
            max_speed = sc.veh_limits[2 * nm + i]; allow_reverse = sc.veh_limits[3 * nm + i] != 0.0;
          }
          accel = np_clip(accel, -max_accel, max_accel);
          steer = np_clip(steer, -max_steer, max_steer);
          const double dt = next_t - t;
          const double dx = e.speed * ch, dy = e.speed * sh;
          const double dh = div_r(e.speed * tan(steer), bl, rcp_bl);
#pragma unroll
          for (int f = 0; f < 6; ++f) np_[f] = e.pose[f];
          np_[0] += dx * dt;
          np_[1] += dy * dt;
          np_[3] += dh * dt;
          double ns = e.speed + accel * dt;
          if (!allow_reverse) ns = fmax(0.0, ns);
          if (!isnan(max_speed)) ns = fmin(max_speed, ns);
          newspeed = ns;
          newpres = true;
        } else if (kind == SG_KIND_PEDESTRIAN) {
#pragma unroll
          for (int f = 0; f < 6; ++f) np_[f] = ped_np[f];
          newspeed = ped_speed;
          newpres = true;
        } else {  // SG_KIND_HOST
          if (in.host_present && in.host_present[i]) {
#pragma unroll
            for (int f = 0; f < 6; ++f) np_[f] = in.host_pose[f * nm + i];
            newpres = true;
          } else if (p.persist) {  // scenario_gym.py:238-239
#pragma unroll
            for (int f = 0; f < 6; ++f) np_[f] = e.pose[f];
            newpres = true;
          }
        }
      } else if (traj_min_t >= t) {  // :240-244 agent initialised at its start position
        position_at_t(rows, K, next_t, EXT_CLAMP, cur_own, np_);
        newpres = true;
      }
    } else if (kind == SG_KIND_REPLAY) {  // BatchReplayEntity.step, entity/batch.py:34-53
      const int64_t u0 = sc.union_off[n];
      const int UK = (int)(sc.union_off[n + 1] - u0);
      const double* ts = sc.union_t + u0;
      if (p.persist || K == 1 || (next_t >= traj_min_t && next_t <= traj_max_t)) {
        const double* X = sc.union_x + u0 * 6 * M;
        if (next_t < __ldg(ts)) {  // fill_value = (X[0], X[-1]), entity/batch.py:120-127
#pragma unroll
          for (int f = 0; f < 6; ++f) np_[f] = __ldg(X + f * M + s);
        } else if (next_t > __ldg(ts + UK - 1)) {
#pragma unroll
          for (int f = 0; f < 6; ++f) np_[f] = __ldg(X + ((int64_t)(UK - 1) * 6 + f) * M + s);
        } else {  // every thread advances the scenario's shared cursor identically
          cur_union = search_left_cursor(ts, 1, UK, next_t, cur_union);
          const double x_lo = __ldg(ts + cur_union - 1), x_hi = __ldg(ts + cur_union);
          const double w1 = (next_t - x_lo) / (x_hi - x_lo), w0 = (x_hi - next_t) / (x_hi - x_lo);
          const double* lo = X + (int64_t)(cur_union - 1) * 6 * M + s;
#pragma unroll
          for (int f = 0; f < 6; ++f) np_[f] = w1 * __ldg(lo + (6 + f) * M) + w0 * __ldg(lo + f * M);
        }
        newpres = true;
      }
    }
    // ---------------- State.step: update_poses / update_statistics (state.py:203-239) -------
    prev_t = t;
    t = next_t;
    tick += 1;
    const double dt = t - prev_t;
    if (newpres) {
      double prev[6];
      if (e.present) {
#pragma unroll
        for (int f = 0; f < 6; ++f) prev[f] = e.pose[f];
      } else {  // :219-222 newcomer: previous pose extrapolated from its trajectory
        int cur = 0;
        position_at_t(rows, K, prev_t, EXT_TRUE, cur, prev);
      }
      double d[6];
      if (exact_div) {
#pragma unroll
        for (int f = 0; f < 6; ++f) { d[f] = np_[f] - prev[f]; e.vel[f] = d[f] / dt; }
      } else {
        const double rdt = 1.0 / dt;
#pragma unroll
        for (int f = 0; f < 6; ++f) { d[f] = np_[f] - prev[f]; e.vel[f] = div_r(d[f], dt, rdt); }
      }
#pragma unroll
      for (int f = 0; f < 6; ++f) e.pose[f] = np_[f];
      e.dist += norm3(d[0], d[1], d[2]);
      e.speed = newspeed;
    }
    e.present = newpres;
    if (st.trace_cap > 0 && tick < st.trace_cap && live) {
      st.trace_present[(int64_t)tick * nm + i] = e.present;
#pragma unroll
      for (int f = 0; f < 6; ++f) st.trace_pose[((int64_t)tick * 6 + f) * nm + i] = e.pose[f];
      if (s == 0) st.trace_t[(int64_t)tick * sc.n_scenarios + n] = t;
    }
    double hs = 0, hc = 1;
    if (live) {
      if (need_coll || feat_rss) {
        if (e.present) sincos(e.pose[3], &hs, &hc);
        publish_box<RSS>(c, e.present, e.pose[0], e.pose[1], hc, hs, orient_hint, ox, oy);
      }
      if (matrix) {
        uint32_t* row = st.coll_mask + ((int64_t)n * M + s) * W;
        for (int w = 0; w < W; ++w) row[w] = 0;
      }
    }
    if (RSS && feat_rss && s == ego_slot)
      publish_ego(c, e.present, e.pose[0], e.pose[1], hc, hs, e.vel[0], e.vel[1]);
    group_sync(c);
    // ---------------- phase B1: callbacks (RSS) + broad phase -------------------------------
    if (live) {
      if (PED) stage_ped_state(c, e.present, etype, e.pose[0], e.pose[1], e.vel[0], e.vel[1],
                               p.ped_distance_threshold, ox, oy);
      if (RSS && feat_rss) {  // RSSDistances.__call__, callback.py:57-122
        rss_last = SG_RSS_NONE;
        if (t != 0.0 && s != ego_slot && e.present && c.egop[EGO_PRESENT] != 0.0) {
          double ro[4];
          rss_last = (uint8_t)rss_hazard(KR, c, e.pose[0], e.pose[1], e.vel[0], e.vel[1], rss_state, ro, 1);
          sd[0] = ro[0]; sd[1] = ro[1]; ratio[0] = ro[2]; ratio[1] = ro[3];
          const int found = (rss_state >> 2) & 3;  // RSS metric latch, rss.py:71-103
          if (found) atomicOr(&c.acc[parity * ACC_N + ACC_RSS], found == 2 ? 1 : 2);
        }
      }
      if (need_coll && e.present && !use_grid) broad_phase(c, parity);
      // ego_off_road (state/state.py:401-407): entities[0] absent, or not strictly inside the driveable surface
      if ((p.terminal & SG_TERM_EGO_OFF_ROAD) && s == first_slot &&
          !(e.present && surface_contains(sc, n, 0, e.pose[0], e.pose[1])))
        c.acc[parity * ACC_N + ACC_OFFROAD] = 1;
    }
    if (PED && use_grid) {  // bin the new positions: this tick's broad phase and the next tick's sensors
      gpos = grid_build(c, live && e.present, need_coll, e.pose[0], e.pose[1], ox, oy, grid_cs, grid_inv_cs);
      if (need_coll && live && e.present) broad_phase_grid(c, parity, gpos);
    }
    group_sync(c);
    done = finish_tick<false>(p, st, c, n + sc.scenario_base, s, W, G, ego_slot, first_slot, parity, tick, t, dt, length, live,
                       live && e.present, collided, e.vel[0], e.vel[1], e.vel[2], e.dist);
    parity ^= 1;
  }

  // ---------------- write the State rows back ----------------------------------------------
  if (live) {
#pragma unroll
    for (int f = 0; f < 6; ++f) { st.pose[f * nm + i] = e.pose[f]; st.vel[f * nm + i] = e.vel[f]; }
    st.dist[i] = e.dist;
    st.speed[i] = e.speed;
    st.present[i] = e.present;
    st.cur_own[i] = cur_own;
    st.collided[i] = collided;
    if (PED) { st.goal_idx[i] = goal; st.force[i] = force[0]; st.force[nm + i] = force[1]; }
    if (RSS) {
      st.rss_state[i] = rss_state; st.rss_last[i] = rss_last;
      st.safe_dist[i] = sd[0]; st.safe_dist[nm + i] = sd[1];
      st.safe_ratio[i] = ratio[0]; st.safe_ratio[nm + i] = ratio[1];
    }
  }
  if (s == 0) {
    st.t[n] = t; st.prev_t[n] = prev_t; st.tick[n] = tick; st.done[n] = done; st.cur_union[n] = cur_union;
  }
  store_cold(st, c, n, s, W, ego_slot);
}

// State.reset(t0) + Agent/Metric/StateCallback resets (reference state/state.py:106-143,
// controller.py:100-103, metrics/trajectory.py:13-18, metrics/rss/callback.py:44-55).
// mask != NULL: only the scenarios with mask[n] != 0 (a whole group leaves, so its barriers stay matched)
template <bool RSS, int MAXT>
__global__ void __launch_bounds__(MAXT, MAXT >= 1024 ? 1 : 2)
sg_reset_kernel(SgScene sc, SgParams p, SgState st, GroupLayout L, const uint8_t* __restrict__ mask) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int G = L.G, M = sc.n_slots, W = L.W;
  const int gpb = blockDim.x / G;
  const int gl = threadIdx.x / G;
  const int s = threadIdx.x - gl * G;
  const int n = blockIdx.x * gpb + gl;
  if (gl >= gpb || n >= sc.n_scenarios) return;
  if (mask && !mask[n]) return;
  Grp c;
  setup_group(c, sc, L, smem, gl, s, n);
  c.sorted = 0;  // no broad phase at reset
  const bool live = s < M;
  const int64_t i = c.i, nm = c.nm;
  const int kind = live ? sc.kind[i] : SG_KIND_EMPTY;
  const int ego_slot = sc.ego_slot[n];
  const double t = sc.t0[n];
  double pose[6] = {0, 0, 0, 0, 0, 0}, vel[6] = {0, 0, 0, 0, 0, 0};
  double speed = 0;
  int orient_hint = 0;
  bool present = false;
  if (kind != SG_KIND_EMPTY) {
    const double bw = sc.box[i], bl = sc.box[nm + i];
    c.boxp[s] = bw; c.boxp[G + s] = bl;
    c.boxp[2 * G + s] = sc.box[2 * nm + i]; c.boxp[3 * G + s] = sc.box[3 * nm + i];
    orient_hint = box_orientation_hint(bw, bl);
    const int64_t r0 = sc.traj_off[i];
    const int K = (int)(sc.traj_off[i + 1] - r0);
    const double* rows = sc.traj_rows + r0 * 7;
    const int mode = (K == 1) ? EXT_TRUE : (p.persist ? EXT_CLAMP : EXT_NONE);  // :123-129
    int cur = 0;
    present = position_at_t(rows, K, t, mode, cur, pose);
    if (present) velocity_at_t(rows, K, t, vel);  // :132
    else {
#pragma unroll
      for (int f = 0; f < 6; ++f) pose[f] = 0.0;
    }
    if (kind == SG_KIND_VEHICLE || kind == SG_KIND_PID) speed = norm2(vel[0], vel[1]);  // controller.py:100-103
  }
  uint8_t rss_state = 0, rss_last = SG_RSS_NONE;
  double sd[2] = {0.0, 0.0}, ratio[2] = {INFINITY, INFINITY};  // callback.py:51-55
  int rss_flags = 0;
  const bool feat_rss = RSS && (p.features & SG_FEAT_RSS);
  if (RSS && feat_rss) {  // update_callbacks() at reset, state.py:137-139
    const RssConst KR = make_rss_const(p);
    double ox, oy;
    {
      const int64_t er = sc.traj_off[(int64_t)n * M + ego_slot];
      ox = __ldg(sc.traj_rows + er * 7 + 1);
      oy = __ldg(sc.traj_rows + er * 7 + 2);
    }
    if (s == 0) c.acc[ACC_RSS] = 0;
    if (s == ego_slot) publish_ego_box(c);
    double hs = 0, hc = 1;
    if (live && present) sincos(pose[3], &hs, &hc);
    if (live) publish_box<RSS>(c, present, pose[0], pose[1], hc, hs, orient_hint, ox, oy);
    if (s == ego_slot) publish_ego(c, present, pose[0], pose[1], hc, hs, vel[0], vel[1]);
    group_sync(c);
    if (live && t != 0.0 && s != ego_slot && present && c.egop[EGO_PRESENT] != 0.0) {
      double ro[4];
      rss_last = (uint8_t)rss_hazard(KR, c, pose[0], pose[1], vel[0], vel[1], rss_state, ro, 1);
      sd[0] = ro[0]; sd[1] = ro[1]; ratio[0] = ro[2]; ratio[1] = ro[3];
      const int found = (rss_state >> 2) & 3;
      if (found) atomicOr(&c.acc[ACC_RSS], found == 2 ? 1 : 2);
    }
    group_sync(c);
    rss_flags = c.acc[ACC_RSS];
  }
  if (live) {
#pragma unroll
    for (int f = 0; f < 6; ++f) { st.pose[f * nm + i] = pose[f]; st.vel[f * nm + i] = vel[f]; }
    st.dist[i] = 0.0;
    st.speed[i] = speed;
    st.present[i] = present;
    st.cur_own[i] = 1;
    st.collided[i] = 0;
    st.goal_idx[i] = 0;
    st.force[i] = 0.0; st.force[nm + i] = 0.0;
    st.pid_err[i] = 0.0; st.pid_err[nm + i] = 0.0; st.pid_err[2 * nm + i] = 0.0;  // controller.py:198-203
    st.rss_state[i] = rss_state; st.rss_last[i] = rss_last;
    st.safe_dist[i] = sd[0]; st.safe_dist[nm + i] = sd[1];
    st.safe_ratio[i] = ratio[0]; st.safe_ratio[nm + i] = ratio[1];
    if (st.trace_cap > 0) {
      st.trace_present[i] = present;
#pragma unroll
      for (int f = 0; f < 6; ++f) st.trace_pose[f * nm + i] = pose[f];
    }
  }
  if (s == ego_slot) {  // Metric.reset, metrics/trajectory.py:13-18, 33-37
    const double sp = norm3(vel[0], vel[1], vel[2]);
    st.ego_avg_speed[n] = sp; st.ego_avg_t[n] = 0.0; st.ego_max_speed[n] = sp; st.ego_dist[n] = 0.0;
  }
  if (s == 0) {
    st.t[n] = t; st.prev_t[n] = t - 0.1;  // state.py:135
    st.tick[n] = 0; st.done[n] = 0; st.cur_union[n] = 1;
    st.first_coll_tick[n] = -1; st.first_coll_pair[2 * n] = -1; st.first_coll_pair[2 * n + 1] = -1;
    st.n_pair_ticks[n] = 0;
    st.rss_flags[n] = (uint8_t)rss_flags;
    if (st.trace_cap > 0) st.trace_t[n] = t;
  }
  if (s < W) st.ego_hits[(int64_t)n * W + s] = 0;
}

template <bool RSS>
static cudaError_t launch_reset_t(bool big, int blocks, int threads, size_t smem, cudaStream_t s,
                                const SgScene& sc, const SgParams& p, const SgState& st,
                                const GroupLayout& L, const uint8_t* mask) {
  auto kern = big ? sg_reset_kernel<RSS, 1024> : sg_reset_kernel<RSS, SG_THREADS>;
  if (smem > 48 * 1024) {
    cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return err;
  }
  kern<<<blocks, threads, smem, s>>>(sc, p, st, L, mask);
  return cudaGetLastError();
}

template <bool PED, bool RSS>
static cudaError_t launch_rollout_t(bool big, int blocks, int threads, size_t smem, cudaStream_t s,
                                  const SgScene& sc, const SgParams& p, const SgState& st,
                                  const SgInputs& in, const SgRngDev& rng, int n_ticks, const GroupLayout& L) {
  auto kern = big ? sg_rollout_kernel<PED, RSS, 1024> : sg_rollout_kernel<PED, RSS, SG_THREADS>;
  if (smem > 48 * 1024) {
    cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return err;
  }
  kern<<<blocks, threads, smem, s>>>(sc, p, st, in, n_ticks, L, rng);
  return cudaGetLastError();
}

cudaError_t sgi_launch_reset(bool rss, bool big, int blocks, int threads, size_t smem, cudaStream_t s,
                             const SgScene& sc, const SgParams& p, const SgState& st, const GroupLayout& L,
                             const uint8_t* mask) {
  return rss ? launch_reset_t<true>(big, blocks, threads, smem, s, sc, p, st, L, mask)
             : launch_reset_t<false>(big, blocks, threads, smem, s, sc, p, st, L, mask);
}

cudaError_t sgi_launch_rollout(bool ped, bool rss, bool big, int blocks, int threads, size_t smem,
                               cudaStream_t s, const SgScene& sc, const SgParams& p, const SgState& st,
                               const SgInputs& in, const SgRngDev& rng, int n_ticks, const GroupLayout& L) {
  if (ped && rss) return launch_rollout_t<true, true>(big, blocks, threads, smem, s, sc, p, st, in, rng, n_ticks, L);
  if (ped) return launch_rollout_t<true, false>(big, blocks, threads, smem, s, sc, p, st, in, rng, n_ticks, L);
  if (rss) return launch_rollout_t<false, true>(big, blocks, threads, smem, s, sc, p, st, in, rng, n_ticks, L);
  return launch_rollout_t<false, false>(big, blocks, threads, smem, s, sc, p, st, in, rng, n_ticks, L);
}
