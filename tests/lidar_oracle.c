/*
 * lidar_oracle.c -- TEST INFRASTRUCTURE ONLY.
 *
 * Plain-C restatement of the lidar block of sg_env_observe (semantics in include/sg_b200.h, SgEnvSpec):
 * sgo_env_observe_lidar is the environment oracle's sgo_env_observe (oracle/sg_env_oracle.c, included
 * unchanged, so this library exports every sgo_ entry point too) with the R lidar readings appended to each
 * row, every ray tested against every other present slot.  Built by tests/lidar_oracle.py into a temporary
 * directory with the oracle's flags: no FMA contraction.
 */
#include "sg_env_oracle.c"

/* the slab test of include/sg_b200.h in its operation order; 1 with the hit distance in *t */
static int lidar_ray_box(double px, double py, double ux, double uy, double cj, double sj, double hl, double hw,
                         double* t) {
  const double o[2] = {cj * px + sj * py, -sj * px + cj * py};
  const double d[2] = {cj * ux + sj * uy, -sj * ux + cj * uy};
  const double ext[2] = {hl, hw};
  double enter = -INFINITY, exit = INFINITY;
  for (int ax = 0; ax < 2; ++ax) {
    if (d[ax] != 0.0) {
      const double t1 = (-ext[ax] - o[ax]) / d[ax], t2 = (ext[ax] - o[ax]) / d[ax];
      const double lo = t1 < t2 ? t1 : t2, hi = t1 < t2 ? t2 : t1;
      if (lo > enter) enter = lo;
      if (hi < exit) exit = hi;
    } else if (fabs(o[ax]) > ext[ax]) {
      return 0;
    }
  }
  if (!(exit >= enter && exit >= 0.0)) return 0;
  *t = enter > 0.0 ? enter : 0.0;
  return 1;
}

/* the R readings of the agent at slot `slot` of scenario n */
static void lidar_row(const SgScene* sc, const SgState* st, const SgEnvSpec* e, int n, int slot, float* out) {
  const int64_t nm = NM;
  const int M = sc->n_slots, R = e->n_rays;
  const int64_t i = IDX(n, slot);
  const double x = st->pose[i], y = st->pose[nm + i], c = cos(st->pose[3 * nm + i]), s = sin(st->pose[3 * nm + i]);
  double best[256], ux[256], uy[256];
  for (int k = 0; k < R; ++k) {
    const double ex = e->ray_dir[2 * k], ey = e->ray_dir[2 * k + 1];
    ux[k] = c * ex - s * ey;
    uy[k] = s * ex + c * ey;
    best[k] = e->ray_range;
  }
  for (int j = 0; j < M; ++j) {
    const int64_t g = IDX(n, j);
    if (j == slot || !st->present[g]) continue;
    const double hj = st->pose[3 * nm + g], cj = cos(hj), sj = sin(hj);
    const double bcx = sc->box[2 * nm + g], bcy = sc->box[3 * nm + g];
    const double X = st->pose[g] + (bcx * cj - bcy * sj), Y = st->pose[nm + g] + (bcx * sj + bcy * cj);
    const double hl = 0.5 * sc->box[nm + g], hw = 0.5 * sc->box[g];
    for (int k = 0; k < R; ++k) {
      double t;
      if (lidar_ray_box(x - X, y - Y, ux[k], uy[k], cj, sj, hl, hw, &t) && t < best[k]) best[k] = t;
    }
  }
  for (int k = 0; k < R; ++k) out[k] = (float)best[k];
}

/* sgo_env_observe with rows of F = F0 + n_rays floats: the first F0 are the oracle's row, then the lidar */
int sgo_env_observe_lidar(const SgScene* sc, const SgParams* p, const SgState* st, const SgEnvSpec* e,
                          const uint8_t* mask, float* obs, uint8_t* agent_mask, int device, void* stream) {
  const int R = e->n_rays;
  if (R < 0 || R > 256) { snprintf(g_err, sizeof(g_err), "SgEnvSpec.n_rays must be in 0..256"); return -1; }
  if (R == 0) return sgo_env_observe(sc, p, st, e, mask, obs, agent_mask, device, stream);
  if (!isfinite(e->ray_range) || !(e->ray_range > 0.0) || !e->ray_dir) {
    snprintf(g_err, sizeof(g_err), "SgEnvSpec.ray_range must be finite and > 0 (and ray_dir given) when n_rays > 0");
    return -1;
  }
  const int N = sc->n_scenarios, A = e->n_agents;
  const int F0 = 4 + 3 * e->n_lookahead + 10 * e->k_neighbours + (e->road ? 2 : 0), F = F0 + R;
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
        for (int k = 0; k < R; ++k) row[F0 + k] = 0.0f;
        if (agent_mask[ia]) lidar_row(sc, st, e, n, e->agent_slot[ia], row + F0);
      }
    }
  }
  free(base);
  return rc;
}
