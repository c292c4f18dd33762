/*
 * reset_oracle.c -- TEST INFRASTRUCTURE ONLY.
 *
 * Plain-C restatement of sg_reset_scenarios_init (include/sg_b200.h) with the prefix sgo_ and HOST pointers.  It
 * includes the environment oracle (oracle/sg_env_oracle.c, unchanged) and works in four steps:
 *   1. sgo_reset_scenarios on a copy of the scene whose t0 holds the start times;
 *   2. the perturbation of the flagged present slots;
 *   3. the reset's RSS fields cleared and rss_update run again on the perturbed start;
 *   4. the ego metrics recomputed from the perturbed velocity.
 * Built by tests/reset_oracle.py into a temporary directory with the oracle's flags: no FMA contraction.
 */
#include "sg_env_oracle.c"

/* the stream's first splitmix64 value for the key (seed, i, tick), the one noise2 starts from */
static uint64_t noise_key(uint64_t seed, int64_t i, int tick) {
  return splitmix64(seed ^ splitmix64((uint64_t)i * 0x9E3779B97F4A7C15ULL + (uint64_t)(unsigned)tick));
}
static double uniform(uint64_t seed, int64_t i, int tick) {
  return (double)(noise_key(seed, i, tick) >> 11) * (1.0 / 9007199254740992.0);
}
static int tick2(int64_t k) { return (int)(uint32_t)((uint64_t)k * 2u); }

/* u[j] = uniform(seed, i[j], tick) for j < n */
void sgr_uniform(uint64_t seed, const int64_t* i, int64_t n, int tick, double* u) {
  for (int64_t j = 0; j < n; ++j) u[j] = uniform(seed, i[j], tick);
}

int sgo_reset_scenarios_init(const SgScene* sc, const SgParams* p, SgState* st, const uint8_t* mask,
                             const SgResetInit* init, int device, void* stream) {
  if (!sc || !p || !st || !init) { snprintf(g_err, sizeof(g_err), "null argument"); return -1; }
  for (int c = 0; c < 4; ++c)
    if (!isfinite(init->sigma[c]) || init->sigma[c] < 0.0) {
      snprintf(g_err, sizeof(g_err), "sg_reset_scenarios_init: sigma must be finite and >= 0");
      return -1;
    }
  if (!init->counter) { snprintf(g_err, sizeof(g_err), "sg_reset_scenarios_init: counter missing"); return -1; }
  const int N = sc->n_scenarios, M = sc->n_slots;
  const int64_t nm = NM, base = sc->plane_stride > 0 ? sc->scenario_base : 0;
  const double* sg = init->sigma;
  /* 1. the reset at the start times */
  double* T = (double*)malloc(sizeof(double) * N);
  if (!T) { snprintf(g_err, sizeof(g_err), "out of memory"); return -1; }
  for (int n = 0; n < N; ++n) {
    if (init->t_start) T[n] = init->t_start[n];
    else if (init->start_window)
      T[n] = sc->t0[n] + uniform(init->seed, -1 - (base + n), tick2(init->counter[n])) * init->start_window[n];
    else T[n] = sc->t0[n];
  }
  SgScene at = *sc;
  at.t0 = T;
  const int32_t events = st->event_count[0];
  int rc = sgo_reset_scenarios(&at, p, st, mask, device, stream);
  st->event_count[0] = events;
  for (int n = 0; n < N && !rc; ++n) {
    if (mask && !mask[n]) continue;
    const int k2 = tick2(init->counter[n]);
    /* 2. the perturbation */
    for (int s = 0; s < M; ++s) {
      const int64_t i = IDX(n, s);
      if (!init->perturb || !init->perturb[i] || !st->present[i]) continue;
      double z01[2], z23[2];
      noise2(init->seed, (base + n) * M + s, k2, z01);
      noise2(init->seed, (base + n) * M + s, k2 + 1, z23);
      double *x = &st->pose[i], *y = &st->pose[nm + i], *h = &st->pose[3 * nm + i];
      double *vx = &st->vel[i], *vy = &st->vel[nm + i];
      const double v0 = norm2(*vx, *vy);
      double v = v0;
      if (sg[0] != 0.0 || sg[1] != 0.0) {
        const double c = cos(*h), sn = sin(*h), lon = sg[0] * z01[0], lat = sg[1] * z01[1];
        *x = *x + (c * lon - sn * lat);
        *y = *y + (sn * lon + c * lat);
      }
      double dh = 0.0;
      if (sg[2] != 0.0) {
        dh = sg[2] * z23[0];
        *h = *h + dh;
      }
      if (sg[2] != 0.0 || sg[3] != 0.0) {
        v = v0 + sg[3] * z23[1];
        v = v > 0.0 ? v : 0.0;
        if (v0 > 0.0) {
          const double cd = cos(dh), sd = sin(dh), f = v / v0, ux = *vx, uy = *vy;
          *vx = (cd * ux - sd * uy) * f;
          *vy = (sd * ux + cd * uy) * f;
        } else if (v > 0.0) {
          *vx = v * cos(*h);
          *vy = v * sin(*h);
        }
      }
      if (sc->kind[i] == SG_KIND_VEHICLE || sc->kind[i] == SG_KIND_PID) st->speed[i] = v;
    }
    /* 3. the RSS pass at reset on the perturbed start */
    if (p->features & SG_FEAT_RSS) {
      for (int s = 0; s < M; ++s) {
        const int64_t i = IDX(n, s);
        st->rss_state[i] = 0;
        st->safe_dist[i] = 0.0; st->safe_dist[nm + i] = 0.0;
        st->safe_ratio[i] = INFINITY; st->safe_ratio[nm + i] = INFINITY;
      }
      st->rss_flags[n] = 0;
      rss_update(&at, p, st, n);
    }
    /* 4. the ego metrics */
    const int64_t ei = IDX(n, sc->ego_slot[n]);
    const double sp = norm3(st->vel[ei], st->vel[nm + ei], st->vel[2 * nm + ei]);
    st->ego_avg_speed[n] = sp;
    st->ego_max_speed[n] = sp;
    if (st->trace_cap > 0) record_trace(&at, st, n);
  }
  free(T);
  return rc;
}
