/*
 * raster_oracle.c -- TEST INFRASTRUCTURE ONLY.
 *
 * Plain-C restatement of sg_env_raster (semantics in include/sg_b200.h, SgRasterSpec), by brute force: every
 * pixel of a surface channel walks every polygon of the surface and every edge of the polygon, every pixel of a
 * box channel every other present slot.  Nothing is culled and SgRasterSpec.poly_box / margin are not read.  It
 * includes oracle/sg_env_oracle.c unchanged (which includes oracle/sg_oracle.c), so this library exports every
 * sgo_ entry point too, and a wrapper of the oracle's surface_contains.  Built by tests/raster_oracle.py into a
 * temporary directory with the oracle's flags: no FMA contraction.
 */
#include "sg_env_oracle.c"

/* the raster of the agent at slot `slot` of scenario n: img [5][S][S] */
static void raster_agent(const SgScene* sc, const SgState* st, const SgRasterSpec* r, int n, int slot,
                         uint8_t* img) {
  const int64_t nm = NM, M = sc->n_slots;
  const int S = r->size;
  const double h = 0.5 * r->resolution;
  const int64_t i = IDX(n, slot);
  const double x = st->pose[i], y = st->pose[nm + i], c = cos(st->pose[3 * nm + i]), s = sin(st->pose[3 * nm + i]);
  const int rn = (sc->rn_of && sc->n_networks > 0) ? sc->rn_of[n] : -1;
  for (int pi = 0; pi < S; ++pi) {
    const double pu = r->ahead + (double)(S - 1 - 2 * pi) * h;
    for (int pj = 0; pj < S; ++pj) {
      const double pv = (double)(S - 1 - 2 * pj) * h;
      for (int k = 0; k < 3 && rn >= 0; ++k) {
        int in = 0;
        for (int64_t q = sc->rn_poly_off[3 * rn + k]; q < sc->rn_poly_off[3 * rn + k + 1] && !in; ++q) {
          int odd = 0;
          for (int64_t e = sc->rn_edge_off[q]; e < sc->rn_edge_off[q + 1]; ++e) {
            const double* E = sc->rn_edges + 4 * e;
            const double adx = E[0] - x, ady = E[1] - y, bdx = E[2] - x, bdy = E[3] - y;
            const double au = c * adx + s * ady, av = -s * adx + c * ady;
            const double bu = c * bdx + s * bdy, bv = -s * bdx + c * bdy;
            if ((au > pu) != (bu > pu)) {
              const double vc = av + ((pu - au) * (bv - av)) / (bu - au);
              if (vc > pv) odd ^= 1;
            }
          }
          in = odd;
        }
        img[((int64_t)k * S + pi) * S + pj] = (uint8_t)in;
      }
      const double Px = x + (c * pu - s * pv), Py = y + (s * pu + c * pv);
      for (int j = 0; j < M; ++j) {
        const int64_t b = IDX(n, j);
        if (j == slot || !st->present[b]) continue;
        const double cj = cos(st->pose[3 * nm + b]), sj = sin(st->pose[3 * nm + b]);
        const double bcx = sc->box[2 * nm + b], bcy = sc->box[3 * nm + b];
        const double hl = 0.5 * sc->box[nm + b], hw = 0.5 * sc->box[b];
        const double X = st->pose[b] + (bcx * cj - bcy * sj), Y = st->pose[nm + b] + (bcx * sj + bcy * cj);
        const double px = Px - X, py = Py - Y;
        const double ox = cj * px + sj * py, oy = -sj * px + cj * py;
        if (fabs(ox) <= hl && fabs(oy) <= hw) {
          const int ch = sc->etype[b] == SG_ETYPE_PEDESTRIAN ? 4 : 3;
          img[((int64_t)ch * S + pi) * S + pj] = 1;
        }
      }
    }
  }
}

/* sg_env_raster on host buffers: out [N][A][5][S][S]; scenarios with mask[n] == 0 are not written */
int sgo_env_raster_brute(const SgScene* sc, const SgParams* p, const SgState* st, const SgEnvSpec* e,
                         const SgRasterSpec* r, const uint8_t* mask, uint8_t* out) {
  (void)p;
  if (!sc || !st || !e || !r || !out) { snprintf(g_err, sizeof(g_err), "null argument"); return -1; }
  if (r->size < 32 || r->size > 256 || r->size % 32 != 0) {
    snprintf(g_err, sizeof(g_err), "SgRasterSpec.size must be a multiple of 32 in 32..256");
    return -1;
  }
  if (!isfinite(r->resolution) || !(r->resolution > 0.0) || !isfinite(r->ahead)) {
    snprintf(g_err, sizeof(g_err), "SgRasterSpec.resolution must be finite and > 0, ahead finite");
    return -1;
  }
  const int N = sc->n_scenarios, A = e->n_agents, M = sc->n_slots;
  const int64_t per = 5 * (int64_t)r->size * r->size;
  for (int n = 0; n < N; ++n) {
    if (mask && !mask[n]) continue;
    for (int a = 0; a < A; ++a) {
      uint8_t* img = out + ((int64_t)n * A + a) * per;
      memset(img, 0, (size_t)per);
      const int slot = e->agent_slot[(int64_t)n * A + a];
      if (slot < 0 || slot >= M || !st->present[IDX(n, slot)]) continue;
      raster_agent(sc, st, r, n, slot, img);
    }
  }
  return 0;
}

/* the oracle's surface_contains (strict containment, exact orientation signs) at points (px[q], py[q]) */
int sgo_test_surface_contains(const SgScene* sc, int n, int k, const double* px, const double* py, int64_t count,
                              uint8_t* out) {
  for (int64_t q = 0; q < count; ++q) out[q] = (uint8_t)surface_contains(sc, n, k, px[q], py[q]);
  return 0;
}
