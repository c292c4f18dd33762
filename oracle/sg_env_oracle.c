/*
 * sg_env_oracle.c -- TEST INFRASTRUCTURE ONLY.
 *
 * Plain-C restatement of the closed-loop environment's entry points (sg_reset_scenarios,
 * sg_env_observe, sg_env_reward; semantics in include/sg_b200.h, SgEnvSpec) with the prefix sgo_ and
 * HOST pointers.  It includes the oracle (sg_oracle.c) to reuse its restatements -- position_at_t,
 * polygon_side / surface_contains, sgo_reset -- and is built into its own library,
 * oracle/_build/libsg_env_oracle.so, which therefore exports every sgo_ entry point
 * (oracle/env_runner.py).  Build flags as oracle/Makefile: no FMA contraction.
 */
#define sgo_sizeof sgo_sizeof_base
#include "sg_oracle.c"
#undef sgo_sizeof

int64_t sgo_sizeof(int which) { return which == 7 ? (int64_t)sizeof(SgEnvSpec) : sgo_sizeof_base(which); }

/* ---- sg_reset_scenarios: sgo_reset, with every field of the scenarios outside the mask (and the event
   count) put back as it was.  A field is `planes` planes of N * per elements of `esz` bytes; scenario n
   owns elements [n * per, (n + 1) * per) of each plane. */
typedef struct { void* p; size_t esz; int planes; int64_t per; } EnvField;

int sgo_reset_scenarios(const SgScene* sc, const SgParams* p, SgState* st, const uint8_t* mask, int device,
                        void* stream) {
  if (!mask) return sgo_reset(sc, p, st, device, stream);
  const int N = sc->n_scenarios;
  const int64_t M = sc->n_slots, W = (M + 31) / 32;
  EnvField f[40];
  int nf = 0;
#define FIELD(ptr, planes_, per_) f[nf++] = (EnvField){(void*)(ptr), sizeof(*(ptr)), (planes_), (per_)}
  FIELD(st->pose, 6, M); FIELD(st->vel, 6, M); FIELD(st->dist, 1, M); FIELD(st->present, 1, M);
  FIELD(st->t, 1, 1); FIELD(st->prev_t, 1, 1); FIELD(st->tick, 1, 1); FIELD(st->done, 1, 1);
  FIELD(st->speed, 1, M); FIELD(st->goal_idx, 1, M); FIELD(st->force, 2, M); FIELD(st->cur_own, 1, M);
  FIELD(st->cur_union, 1, 1); FIELD(st->ego_avg_speed, 1, 1); FIELD(st->ego_avg_t, 1, 1);
  FIELD(st->ego_max_speed, 1, 1); FIELD(st->ego_dist, 1, 1); FIELD(st->ego_hits, 1, W);
  FIELD(st->collided, 1, M); FIELD(st->first_coll_tick, 1, 1); FIELD(st->first_coll_pair, 1, 2);
  FIELD(st->n_pair_ticks, 1, 1); FIELD(st->rss_state, 1, M); FIELD(st->rss_last, 1, M);
  FIELD(st->safe_dist, 2, M); FIELD(st->safe_ratio, 2, M); FIELD(st->rss_flags, 1, 1); FIELD(st->pid_err, 3, M);
  if (st->trace_cap > 0) { /* (the reset writes trace row 0) */
    FIELD(st->trace_pose, 6, M); FIELD(st->trace_present, 1, M); FIELD(st->trace_t, 1, 1);
  }
#undef FIELD
  void* saved[40];
  int rc = 0;
  for (int k = 0; k < nf; ++k) {
    const size_t bytes = (size_t)f[k].planes * N * f[k].per * f[k].esz;
    saved[k] = malloc(bytes);
    if (!saved[k]) { rc = -1; nf = k; snprintf(g_err, sizeof(g_err), "out of memory"); break; }
    memcpy(saved[k], f[k].p, bytes);
  }
  const int32_t events = st->event_count[0];
  if (!rc) rc = sgo_reset(sc, p, st, device, stream);
  st->event_count[0] = events;
  for (int k = 0; k < nf; ++k) {
    const size_t row = (size_t)f[k].per * f[k].esz, plane = (size_t)N * row;
    if (!rc)
      for (int q = 0; q < f[k].planes; ++q)
        for (int n = 0; n < N; ++n)
          if (!mask[n])
            memcpy((char*)f[k].p + q * plane + n * row, (const char*)saved[k] + q * plane + n * row, row);
    free(saved[k]);
  }
  return rc;
}

/* squared distance from (px, py) to the closest point on the rings of polygons [q0, q1)
   (GEOS LineSegment::closestPoint, as in surface_nearest) */
static double ring_dist2(const SgScene* sc, int64_t q0, int64_t q1, double px, double py) {
  double best = INFINITY;
  for (int64_t e = sc->rn_edge_off[q0]; e < sc->rn_edge_off[q1]; ++e) {
    const double* E = sc->rn_edges + 4 * e;
    double ax = E[0], ay = E[1], bx = E[2], by = E[3];
    double dx = bx - ax, dy = by - ay, len2 = dx * dx + dy * dy, cx = ax, cy = ay;
    if (len2 > 0.0) {
      double fr = ((px - ax) * dx + (py - ay) * dy) / len2;
      if (fr > 0.0 && fr < 1.0) { cx = ax + fr * dx; cy = ay + fr * dy; }
      else {
        double da = (px - ax) * (px - ax) + (py - ay) * (py - ay);
        double db = (px - bx) * (px - bx) + (py - by) * (py - by);
        if (db < da) { cx = bx; cy = by; }
      }
    }
    double d2 = (px - cx) * (px - cx) + (py - cy) * (py - cy);
    if (d2 < best) best = d2;
  }
  return best;
}

/* ---- closed-loop environment (sg_env_observe / sg_env_reward; semantics in include/sg_b200.h) ---- */
static int env_check(const SgScene* sc, const SgEnvSpec* e) {
  if (e->n_agents < 1 || e->n_agents > sc->n_slots) { snprintf(g_err, sizeof(g_err), "SgEnvSpec.n_agents must be in 1..n_slots"); return -1; }
  if (e->k_neighbours < 0 || e->k_neighbours > 32) { snprintf(g_err, sizeof(g_err), "SgEnvSpec.k_neighbours must be in 0..32"); return -1; }
  if (e->n_lookahead < 0 || e->n_lookahead > 8) { snprintf(g_err, sizeof(g_err), "SgEnvSpec.n_lookahead must be in 0..8"); return -1; }
  return 0;
}

int sgo_env_observe(const SgScene* sc, const SgParams* p, const SgState* st, const SgEnvSpec* e,
                    const uint8_t* mask, float* obs, uint8_t* agent_mask, int device, void* stream) {
  (void)p; (void)device; (void)stream;
  int rc = env_check(sc, e);
  if (rc) return rc;
  const int64_t nm = NM;
  const int M = sc->n_slots, A = e->n_agents, K = e->k_neighbours, L = e->n_lookahead;
  const int F = 4 + 3 * L + 10 * K + (e->road ? 2 : 0);
  for (int n = 0; n < sc->n_scenarios; ++n) {
    if (mask && !mask[n]) continue;
    e->snap_pair_ticks[n] = st->n_pair_ticks[n];
    e->snap_rss[n] = st->rss_flags[n];
    const double t = st->t[n];
    for (int a = 0; a < A; ++a) {
      const int64_t ia = (int64_t)n * A + a;
      const int slot = e->agent_slot[ia];
      const int real = slot >= 0 && slot < M;
      const int64_t i = IDX(n, real ? slot : 0);
      const int here = real && st->present[i];
      agent_mask[ia] = (uint8_t)here;
      e->snap_dist[ia] = real ? st->dist[i] : 0.0;
      e->snap_collided[ia] = real ? st->collided[i] : 0;
      float* row = obs + ia * F;
      for (int f = 0; f < F; ++f) row[f] = 0.0f;
      if (!here) continue;
      const double x = st->pose[i], y = st->pose[nm + i], h = st->pose[3 * nm + i];
      const double vx = st->vel[i], vy = st->vel[nm + i];
      const double c = cos(h), s = sin(h);
      int f = 0;
      row[f++] = (float)st->speed[i];
      row[f++] = (float)(c * vx + s * vy);
      row[f++] = (float)(-s * vx + c * vy);
      row[f++] = (float)st->vel[3 * nm + i];
      int64_t Kt;
      const double* rows = slot_rows(sc, i, &Kt);
      for (int l = 0; l < L; ++l) {
        double q[6] = {x, y, 0.0, h, 0.0, 0.0};
        if (Kt > 0) position_at_t(rows, Kt, t + e->lookahead[l], EXT_CLAMP, q);
        const double dx = q[0] - x, dy = q[1] - y;
        row[f++] = (float)(c * dx + s * dy);
        row[f++] = (float)(-s * dx + c * dy);
        row[f++] = (float)remainder(q[3] - h, 2.0 * M_PI);
      }
      /* the K smallest (d2, slot), by selection: repeatedly the smallest pair above the last one taken */
      double last_d = -INFINITY;
      int last_j = -1;
      for (int q = 0; q < K; ++q, f += 10) {
        int bj = -1;
        double bdist = 0.0;
        for (int j = 0; j < M; ++j) {
          const int64_t jg = IDX(n, j);
          if (j == slot || !st->present[jg]) continue;
          const double dx = st->pose[jg] - x, dy = st->pose[nm + jg] - y, d2 = dx * dx + dy * dy;
          if (e->radius > 0.0 && !(d2 < e->radius * e->radius)) continue;
          if (d2 < last_d || (d2 == last_d && j <= last_j)) continue;
          if (bj < 0 || d2 < bdist || (d2 == bdist && j < bj)) { bj = j; bdist = d2; }
        }
        if (bj < 0) continue; /* zero row */
        last_d = bdist; last_j = bj;
        const int64_t jg = IDX(n, bj);
        const double dx = st->pose[jg] - x, dy = st->pose[nm + jg] - y;
        const double dvx = st->vel[jg] - vx, dvy = st->vel[nm + jg] - vy;
        const double dh = st->pose[3 * nm + jg] - h;
        float* nb = row + f;
        nb[0] = (float)(c * dx + s * dy);
        nb[1] = (float)(-s * dx + c * dy);
        nb[2] = (float)cos(dh);
        nb[3] = (float)sin(dh);
        nb[4] = (float)(c * dvx + s * dvy);
        nb[5] = (float)(-s * dvx + c * dvy);
        nb[6] = (float)sc->box[jg];
        nb[7] = (float)sc->box[nm + jg];
        nb[8] = sc->etype[jg] == SG_ETYPE_PEDESTRIAN ? 1.0f : 0.0f;
        nb[9] = 1.0f;
      }
      if (e->road && surface_has_area(sc, n, 0)) {
        const int r = surface_network(sc, n);
        row[f] = surface_contains(sc, n, 0, x, y) ? 1.0f : 0.0f;
        row[f + 1] = (float)sqrt(ring_dist2(sc, sc->rn_poly_off[3 * r], sc->rn_poly_off[3 * r + 1], x, y));
      }
    }
  }
  return 0;
}

int sgo_env_reward(const SgScene* sc, const SgParams* p, const SgState* st, const SgEnvSpec* e, float* reward,
                   float* terms, uint8_t* terminated, uint8_t* truncated, int device, void* stream) {
  (void)device; (void)stream;
  int rc = env_check(sc, e);
  if (rc) return rc;
  const int64_t nm = NM;
  const int M = sc->n_slots, A = e->n_agents;
  for (int n = 0; n < sc->n_scenarios; ++n) {
    for (int a = 0; a < A; ++a) {
      const int64_t ia = (int64_t)n * A + a;
      const int slot = e->agent_slot[ia];
      double term[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
      if (slot >= 0 && slot < M && st->present[IDX(n, slot)]) {
        const int64_t i = IDX(n, slot);
        const double x = st->pose[i], y = st->pose[nm + i];
        term[0] = st->dist[i] - e->snap_dist[ia];                       /* progress */
        term[1] = (st->collided[i] && !e->snap_collided[ia]) ? 1.0 : 0.0; /* collision */
        term[2] = (surface_has_area(sc, n, 0) && !surface_contains(sc, n, 0, x, y)) ? 1.0 : 0.0;
        int64_t Kt;
        const double* rows = slot_rows(sc, i, &Kt);
        if (Kt > 0) {
          double q[6];
          position_at_t(rows, Kt, st->t[n], EXT_CLAMP, q);
          const double dx = x - q[0], dy = y - q[1];
          term[3] = -sqrt(dx * dx + dy * dy);                           /* tracking */
        }
        term[4] = (slot == sc->ego_slot[n] && (st->rss_flags[n] & ~e->snap_rss[n])) ? 1.0 : 0.0;
      }
      double r = 0.0;
      for (int k = 0; k < 5; ++k) {
        r += e->weights[k] * term[k];
        terms[ia * 5 + k] = (float)term[k];
      }
      reward[ia] = (float)r;
    }
    uint8_t te = 0, tr = 0;
    if (st->done[n]) { /* the terminal conditions of this tick (state/state.py:397-408), from the state */
      const int64_t fi = IDX(n, sc->first_slot[n]);
      int hit = 0;
      if ((p->terminal & SG_TERM_COLLISION) && st->n_pair_ticks[n] > e->snap_pair_ticks[n]) hit = 1;
      if ((p->terminal & SG_TERM_EGO_COLLISION) && st->collided[fi]) hit = 1;
      if ((p->terminal & SG_TERM_EGO_OFF_ROAD) &&
          !(st->present[fi] && surface_contains(sc, n, 0, st->pose[fi], st->pose[nm + fi])))
        hit = 1;
      te = (uint8_t)hit;
      tr = (uint8_t)!hit;
    }
    terminated[n] = te;
    truncated[n] = tr;
  }
  return 0;
}
