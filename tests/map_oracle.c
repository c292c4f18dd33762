/*
 * map_oracle.c -- TEST INFRASTRUCTURE ONLY.
 *
 * Plain-C restatement of the map block of sg_env_observe (semantics in include/sg_b200.h, SgEnvSpec):
 * sgo_env_observe_map builds full rows -- the environment oracle's row, then the map block by brute force over
 * every edge of the scenario's network table (the culling grid is not read), then the lidar readings.  It
 * includes tests/lidar_oracle.c unchanged (which includes oracle/sg_env_oracle.c), so this library exports
 * every sgo_ entry point too.  Built by tests/map_oracle.py into a temporary directory with the oracle's flags:
 * no FMA contraction.
 */
#include "lidar_oracle.c"

/* the distance of include/sg_b200.h in its operation order: d2, and the nearest point in *qx, *qy */
static double map_d2(const double* g, double x, double y, double* qx, double* qy) {
  const double dx = g[2] - g[0], dy = g[3] - g[1], wx = x - g[0], wy = y - g[1];
  const double L2 = dx * dx + dy * dy;
  double t = L2 > 0.0 ? (wx * dx + wy * dy) / L2 : 0.0;
  t = t < 0.0 ? 0.0 : (t > 1.0 ? 1.0 : t);
  *qx = g[0] + t * dx;
  *qy = g[1] + t * dy;
  return (*qx - x) * (*qx - x) + (*qy - y) * (*qy - y);
}

/* the 10 * Km map columns of the agent at slot `slot` of scenario n (zeros where nothing is selected) */
static void map_row(const SgScene* sc, const SgState* st, const SgEnvSpec* e, int n, int slot, float* out) {
  const int64_t nm = NM;
  const int Km = e->map_edges;
  const int64_t i = IDX(n, slot);
  const double x = st->pose[i], y = st->pose[nm + i], c = cos(st->pose[3 * nm + i]), s = sin(st->pose[3 * nm + i]);
  for (int k = 0; k < 10 * Km; ++k) out[k] = 0.0f;
  const int r = sc->rn_of ? sc->rn_of[n] : -1;
  if (r < 0) return;
  const int64_t row0 = e->map_off[r], E = e->map_off[r + 1] - row0;
  double bd[32];
  int64_t be[32];
  int cnt = 0;
  const double r2 = e->map_radius * e->map_radius;
  for (int64_t ed = 0; ed < E; ++ed) {  /* edges in ascending e: a later equal d2 never displaces an earlier one */
    double qx, qy;
    const double d2 = map_d2(e->map_seg + 4 * (row0 + ed), x, y, &qx, &qy);
    if (!(d2 < r2)) continue;
    int pos = cnt;
    while (pos > 0 && d2 < bd[pos - 1]) --pos;
    if (pos >= Km) continue;
    for (int q = (cnt < Km ? cnt : Km - 1); q > pos; --q) { bd[q] = bd[q - 1]; be[q] = be[q - 1]; }
    bd[pos] = d2;
    be[pos] = ed;
    if (cnt < Km) ++cnt;
  }
  for (int q = 0; q < cnt; ++q) {
    const double* g = e->map_seg + 4 * (row0 + be[q]);
    double qx, qy;
    map_d2(g, x, y, &qx, &qy);
    const double p[3][2] = {{qx - x, qy - y}, {g[0] - x, g[1] - y}, {g[2] - x, g[3] - y}};
    float* m = out + 10 * q;
    for (int k = 0; k < 3; ++k) {
      m[2 * k] = (float)(c * p[k][0] + s * p[k][1]);
      m[2 * k + 1] = (float)(-s * p[k][0] + c * p[k][1]);
    }
    const unsigned fl = e->map_flags[row0 + be[q]];
    for (int k = 0; k < 3; ++k) m[6 + k] = ((fl >> k) & 1u) ? 1.0f : 0.0f;
    m[9] = 1.0f;
  }
}

/* sgo_env_observe with rows of F = F0 + 10 * Km + R floats: the oracle's row, the map block, the lidar */
int sgo_env_observe_map(const SgScene* sc, const SgParams* p, const SgState* st, const SgEnvSpec* e,
                        const uint8_t* mask, float* obs, uint8_t* agent_mask, int device, void* stream) {
  const int Km = e->map_edges, R = e->n_rays;
  if (Km < 0 || Km > 32) { snprintf(g_err, sizeof(g_err), "SgEnvSpec.map_edges must be in 0..32"); return -1; }
  if (R < 0 || R > 256) { snprintf(g_err, sizeof(g_err), "SgEnvSpec.n_rays must be in 0..256"); return -1; }
  if (Km > 0 && (!isfinite(e->map_radius) || !(e->map_radius > 0.0) || e->map_networks != sc->n_networks ||
                 (sc->n_networks > 0 && (!e->map_off || !e->map_seg || !e->map_flags)))) {
    snprintf(g_err, sizeof(g_err), "SgEnvSpec: map_radius must be finite and > 0, map_networks the scene's and "
             "the map table given when map_edges > 0");
    return -1;
  }
  if (R > 0 && (!isfinite(e->ray_range) || !(e->ray_range > 0.0) || !e->ray_dir)) {
    snprintf(g_err, sizeof(g_err), "SgEnvSpec.ray_range must be finite and > 0 (and ray_dir given) when n_rays > 0");
    return -1;
  }
  const int N = sc->n_scenarios, A = e->n_agents;
  const int F0 = 4 + 3 * e->n_lookahead + 10 * e->k_neighbours + (e->road ? 2 : 0), F = F0 + 10 * Km + R;
  float* base = (float*)calloc((size_t)N * A * F0 + 1, sizeof(float));
  if (!base) { snprintf(g_err, sizeof(g_err), "out of memory"); return -1; }
  const int rc = sgo_env_observe(sc, p, st, e, mask, base, agent_mask, device, stream);
  if (!rc) {
    for (int n = 0; n < N; ++n) {
      if (mask && !mask[n]) continue;
      for (int a = 0; a < A; ++a) {
        const int64_t ia = (int64_t)n * A + a;
        float* row = obs + ia * F;
        memcpy(row, base + ia * F0, (size_t)F0 * sizeof(float));
        for (int k = F0; k < F; ++k) row[k] = 0.0f;
        if (!agent_mask[ia]) continue;
        if (Km > 0) map_row(sc, st, e, n, e->agent_slot[ia], row + F0);
        if (R > 0) lidar_row(sc, st, e, n, e->agent_slot[ia], row + F0 + 10 * Km);
      }
    }
  }
  free(base);
  return rc;
}
