// sg_env.cu -- the closed-loop environment's device side (sg_env_observe / sg_env_reward): per-agent
// observations in the agent's frame, reward terms and terminated / truncated flags, recomputed from the
// State planes the tick kernels leave behind (which therefore need no change).
#include "sg_device.cuh"
#include "sg_internal.h"

#include <limits.h>

#define SG_ENV_TERMS 5

// sg_env_observe: one CTA per scenario.  The present slots' x, y, h, vx, vy are staged in shared memory;
// then one thread per agent keeps the KCAP smallest (d2, slot) candidates in a register-resident sorted
// list (an unrolled insertion, so the list never leaves registers) and writes its row.
template <int KCAP>
__global__ void __launch_bounds__(256)
sg_env_observe_kernel(SgScene sc, SgState st, SgEnvSpec e, const uint8_t* __restrict__ mask,
                      float* __restrict__ obs, uint8_t* __restrict__ agent_mask, int F) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int n = blockIdx.x;
  if (mask && !mask[n]) return;
  const int M = sc.n_slots, A = e.n_agents, K = e.k_neighbours, L = e.n_lookahead;
  const int64_t nm = sc.plane_stride, base = (int64_t)n * M;
  double* sx = (double*)smem;
  double* sy = sx + M;
  double* sh = sy + M;
  double* svx = sh + M;
  double* svy = svx + M;
  uint8_t* sp = (uint8_t*)(svy + M);
  for (int j = threadIdx.x; j < M; j += blockDim.x) {
    const int64_t i = base + j;
    sp[j] = st.present[i];
    sx[j] = st.pose[i]; sy[j] = st.pose[nm + i]; sh[j] = st.pose[3 * nm + i];
    svx[j] = st.vel[i]; svy[j] = st.vel[nm + i];
  }
  if (threadIdx.x == 0) {
    e.snap_pair_ticks[n] = st.n_pair_ticks[n];
    e.snap_rss[n] = st.rss_flags[n];
  }
  __syncthreads();
  const double t = st.t[n];
  const double r2 = e.radius * e.radius;
  const bool cut = e.radius > 0.0;
  for (int a = threadIdx.x; a < A; a += blockDim.x) {
    const int64_t ia = (int64_t)n * A + a;
    const int slot = e.agent_slot[ia];
    const bool real = slot >= 0 && slot < M;
    const int64_t i = base + (real ? slot : 0);
    const bool here = real && sp[slot];
    agent_mask[ia] = here ? 1 : 0;
    e.snap_dist[ia] = real ? st.dist[i] : 0.0;
    e.snap_collided[ia] = real ? st.collided[i] : 0;
    float* row = obs + ia * F;
    if (!here) {
      for (int f = 0; f < F; ++f) row[f] = 0.0f;
      continue;
    }
    const double x = sx[slot], y = sy[slot], h = sh[slot], vx = svx[slot], vy = svy[slot];
    double s, c;
    sincos(h, &s, &c);
    int f = 0;
    row[f++] = (float)st.speed[i];
    row[f++] = (float)(c * vx + s * vy);
    row[f++] = (float)(-s * vx + c * vy);
    row[f++] = (float)st.vel[3 * nm + i];
    // target: the agent's own trajectory ahead of it, clamped at its ends
    const int64_t r0 = sc.traj_off[i];
    const int Kt = (int)(sc.traj_off[i + 1] - r0);
    for (int l = 0; l < L; ++l) {
      double q[6] = {x, y, 0.0, h, 0.0, 0.0};
      int cur = 0;
      if (Kt > 0) position_at_t(sc.traj_rows + r0 * 7, Kt, t + e.lookahead[l], EXT_CLAMP, cur, q);
      const double dx = q[0] - x, dy = q[1] - y;
      row[f++] = (float)(c * dx + s * dy);
      row[f++] = (float)(-s * dx + c * dy);
      row[f++] = (float)remainder(q[3] - h, 2.0 * M_PI);
    }
    // neighbours: the K smallest (d2, slot) among the other present slots inside the radius
    double bd[KCAP];
    int bs[KCAP];
#pragma unroll
    for (int q = 0; q < KCAP; ++q) { bd[q] = INFINITY; bs[q] = INT_MAX; }
    for (int j = 0; j < M; ++j) {
      if (j == slot || !sp[j]) continue;
      const double dx = sx[j] - x, dy = sy[j] - y, d2 = dx * dx + dy * dy;
      if (cut && !(d2 < r2)) continue;
      if (!(d2 < bd[KCAP - 1] || (d2 == bd[KCAP - 1] && j < bs[KCAP - 1]))) continue;
      double cd = d2;
      int cj = j;
#pragma unroll
      for (int q = 0; q < KCAP; ++q) {
        const bool lt = cd < bd[q] || (cd == bd[q] && cj < bs[q]);
        const double td = bd[q];
        const int tj = bs[q];
        bd[q] = lt ? cd : td; bs[q] = lt ? cj : tj;
        cd = lt ? td : cd; cj = lt ? tj : cj;
      }
    }
#pragma unroll
    for (int q = 0; q < KCAP; ++q) {
      if (q >= K) break;
      float* nb = row + f + 10 * q;
      const int j = bs[q];
      if (j == INT_MAX) {
#pragma unroll
        for (int k = 0; k < 10; ++k) nb[k] = 0.0f;
        continue;
      }
      const int64_t jg = base + j;
      const double dx = sx[j] - x, dy = sy[j] - y;
      const double dvx = svx[j] - vx, dvy = svy[j] - vy;
      double sj, cj;
      sincos(sh[j] - h, &sj, &cj);
      nb[0] = (float)(c * dx + s * dy);
      nb[1] = (float)(-s * dx + c * dy);
      nb[2] = (float)cj;
      nb[3] = (float)sj;
      nb[4] = (float)(c * dvx + s * dvy);
      nb[5] = (float)(-s * dvx + c * dvy);
      nb[6] = (float)sc.box[jg];
      nb[7] = (float)sc.box[nm + jg];
      nb[8] = sc.etype[jg] == SG_ETYPE_PEDESTRIAN ? 1.0f : 0.0f;
      nb[9] = 1.0f;
    }
    f += 10 * K;
    if (e.road) {
      float inside = 0.0f, dist = 0.0f;
      if (surface_has_area(sc, n, 0)) {
        inside = surface_contains(sc, n, 0, x, y) ? 1.0f : 0.0f;
        const int r = sc.rn_of[n];
        double d2;
        ring_nearest(sc, sc.rn_poly_off[3 * r], sc.rn_poly_off[3 * r + 1], x, y, d2);
        dist = (float)sqrt(d2);
      }
      row[f++] = inside;
      row[f++] = dist;
    }
  }
}

// sg_env_reward: one thread per (scenario, agent); agent 0's thread also decides the scenario's flags
__global__ void sg_env_reward_kernel(SgScene sc, SgParams p, SgState st, SgEnvSpec e, float* __restrict__ reward,
                                     float* __restrict__ terms, uint8_t* __restrict__ terminated,
                                     uint8_t* __restrict__ truncated) {
  const int64_t ia = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int A = e.n_agents, M = sc.n_slots;
  if (ia >= (int64_t)sc.n_scenarios * A) return;
  const int n = (int)(ia / A), a = (int)(ia - (int64_t)n * A);
  const int64_t nm = sc.plane_stride;
  const int slot = e.agent_slot[ia];
  double term[SG_ENV_TERMS] = {0.0, 0.0, 0.0, 0.0, 0.0};
  if (slot >= 0 && slot < M && st.present[(int64_t)n * M + slot]) {
    const int64_t i = (int64_t)n * M + slot;
    const double x = st.pose[i], y = st.pose[nm + i];
    term[0] = st.dist[i] - e.snap_dist[ia];
    term[1] = (st.collided[i] && !e.snap_collided[ia]) ? 1.0 : 0.0;
    term[2] = (surface_has_area(sc, n, 0) && !surface_contains(sc, n, 0, x, y)) ? 1.0 : 0.0;
    const int64_t r0 = sc.traj_off[i];
    const int Kt = (int)(sc.traj_off[i + 1] - r0);
    if (Kt > 0) {
      double q[6];
      int cur = 0;
      position_at_t(sc.traj_rows + r0 * 7, Kt, st.t[n], EXT_CLAMP, cur, q);
      const double dx = x - q[0], dy = y - q[1];
      term[3] = -sqrt(dx * dx + dy * dy);
    }
    term[4] = (slot == sc.ego_slot[n] && (st.rss_flags[n] & ~e.snap_rss[n])) ? 1.0 : 0.0;
  }
  double r = 0.0;
#pragma unroll
  for (int k = 0; k < SG_ENV_TERMS; ++k) {
    r += e.weights[k] * term[k];
    terms[ia * SG_ENV_TERMS + k] = (float)term[k];
  }
  reward[ia] = (float)r;
  if (a == 0) {
    uint8_t te = 0, tr = 0;
    if (st.done[n]) {  // the conditions finish_tick tested at this tick, from the state it left
      const int64_t fi = (int64_t)n * M + sc.first_slot[n];
      bool hit = false;
      if ((p.terminal & SG_TERM_COLLISION) && st.n_pair_ticks[n] > e.snap_pair_ticks[n]) hit = true;
      if ((p.terminal & SG_TERM_EGO_COLLISION) && st.collided[fi]) hit = true;
      if ((p.terminal & SG_TERM_EGO_OFF_ROAD) &&
          !(st.present[fi] && surface_contains(sc, n, 0, st.pose[fi], st.pose[nm + fi])))
        hit = true;
      te = hit ? 1 : 0;
      tr = hit ? 0 : 1;
    }
    terminated[n] = te;
    truncated[n] = tr;
  }
}

// ---- lidar block of sg_env_observe (semantics in include/sg_b200.h, SgEnvSpec) ----
#define SG_LIDAR_THREADS 256
#define SG_LIDAR_MIN_BYTES (48 * 1024)  // shared memory for a chunk's per-ray minima: 48 agents at R = 256

// one axis of the slab test: the ray parameters [lo, hi] inside |o + t d| <= e; false: never inside
static __device__ __forceinline__ bool lidar_slab(double o, double d, double e, double& lo, double& hi) {
  if (d != 0.0) {
    const double t1 = (-e - o) / d, t2 = (e - o) / d;
    lo = t1 < t2 ? t1 : t2;
    hi = t1 < t2 ? t2 : t1;
    return true;
  }
  lo = -INFINITY;
  hi = INFINITY;
  return !(fabs(o) > e);
}

// the ray p + t u (p relative to the box centre, world frame) against the closed box (cj, sj, hl, hw):
// true with the hit distance in `t`
static __device__ __forceinline__ bool lidar_ray_box(double px, double py, double ux, double uy, double cj,
                                                     double sj, double hl, double hw, double& t) {
  const double ox = cj * px + sj * py, oy = -sj * px + cj * py;
  const double dx = cj * ux + sj * uy, dy = -sj * ux + cj * uy;
  double lx, hx, ly, hy;
  if (!lidar_slab(ox, dx, hl, lx, hx) || !lidar_slab(oy, dy, hw, ly, hy)) return false;
  const double enter = lx > ly ? lx : ly, exit = hx < hy ? hx : hy;
  if (!(exit >= enter && exit >= 0.0)) return false;
  t = enter > 0.0 ? enter : 0.0;
  return true;
}

// sg_env_lidar_kernel: one CTA per (scenario, chunk of `chunk` agents).  The present slots' boxes (centre,
// cos / sin, half extents, circumscribed radius) are staged in shared memory in fp64, and so are the chunk
// agents' poses.  The readings are kept per (agent, ray) in shared memory as the bit patterns of fp32
// distances: non-negative floats order like their bits and rounding is monotone, so a 32-bit atomicMin of
// the rounded hit distances leaves the rounded minimum, whatever order the hits arrive in.
//   default          one thread per (agent, slot) pair; the pair is culled by the box's circumscribed circle
//                    (beyond the range: skipped; origin inside: every ray; otherwise the rays within the
//                    circle's angular half-width, from fp32 atan2 / asin, one ray of margin either side,
//                    modulo R).  Culling only chooses which rays are tested: the fp64 slab test decides hits.
//   SG_LIDAR_BRUTE   one thread per (agent, ray), every slot tested (the variant the culled form was
//                    measured against, DESIGN.md section 6b).
// Each agent's R readings are then stored to columns [F - R, F) of its row, contiguous across the threads.
__global__ void __launch_bounds__(SG_LIDAR_THREADS)
sg_env_lidar_kernel(SgScene sc, SgState st, SgEnvSpec e, const uint8_t* __restrict__ mask,
                    float* __restrict__ obs, int F, int chunk, int n_chunks) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int n = blockIdx.x / n_chunks;
  const int a0 = (blockIdx.x - n * n_chunks) * chunk;
  if (mask && !mask[n]) return;
  const int M = sc.n_slots, A = e.n_agents, R = e.n_rays;
  const int na = min(chunk, A - a0);
  const int64_t nm = sc.plane_stride, base = (int64_t)n * M;
  double* bx = (double*)smem;  // box centres, cos / sin, half extents, circumscribed radius
  double* by = bx + M;
  double* bc = by + M;
  double* bs = bc + M;
  double* bl = bs + M;
  double* bw = bl + M;
  double* br = bw + M;
  double* ax = br + M;  // agents: origin, cos / sin of the heading
  double* ay = ax + chunk;
  double* ac = ay + chunk;
  double* as = ac + chunk;
  unsigned* best = (unsigned*)(as + chunk);  // [chunk][R]
  int* aslot = (int*)(best + chunk * R);     // the agent's slot, -1: absent / padding
  uint8_t* bp = (uint8_t*)(aslot + chunk);   // slot present
  for (int j = threadIdx.x; j < M; j += blockDim.x) {
    const int64_t i = base + j;
    const uint8_t p = st.present[i];
    bp[j] = p;
    if (!p) continue;
    double s, c;
    sincos(st.pose[3 * nm + i], &s, &c);
    const double bcx = sc.box[2 * nm + i], bcy = sc.box[3 * nm + i];
    const double hl = 0.5 * sc.box[nm + i], hw = 0.5 * sc.box[i];
    bx[j] = st.pose[i] + (bcx * c - bcy * s);
    by[j] = st.pose[nm + i] + (bcx * s + bcy * c);
    bc[j] = c;
    bs[j] = s;
    bl[j] = hl;
    bw[j] = hw;
    br[j] = sqrt(hl * hl + hw * hw);
  }
  for (int q = threadIdx.x; q < na; q += blockDim.x) {
    const int slot = e.agent_slot[(int64_t)n * A + a0 + q];
    const bool here = slot >= 0 && slot < M && st.present[base + slot];
    aslot[q] = here ? slot : -1;
    if (!here) continue;
    const int64_t i = base + slot;
    double s, c;
    sincos(st.pose[3 * nm + i], &s, &c);
    ax[q] = st.pose[i];
    ay[q] = st.pose[nm + i];
    ac[q] = c;
    as[q] = s;
  }
  const double range = e.ray_range;
  const unsigned range_bits = __float_as_uint((float)range);
  for (int q = threadIdx.x; q < na * R; q += blockDim.x) best[q] = range_bits;
  __syncthreads();
#ifndef SG_LIDAR_BRUTE
  const float rays_per_rad = (float)R * (float)(0.5 / M_PI);
  for (int q = threadIdx.x; q < na * M; q += blockDim.x) {
    const int a = q / M, j = q - a * M;
    const int slot = aslot[a];
    if (slot < 0 || j == slot || !bp[j]) continue;
    const double x = ax[a], y = ay[a], c = ac[a], s = as[a];
    const double gx = bx[j] - x, gy = by[j] - y, rc = br[j];
    const double D = sqrt(gx * gx + gy * gy);
    if (D - rc > range + 1e-6 * (1.0 + range)) continue;  // every point of the box lies beyond the range
    int k0 = 0, nk = R;
    if (D > rc * (1.0 + 1e-6) + 1e-9) {  // origin outside the circle: the rays within its angular half-width
      const float phi = atan2f((float)(-s * gx + c * gy), (float)(c * gx + s * gy));
      const float alpha = asinf(fminf(1.0f, (float)(rc / D)));
      const int lo = (int)floorf((phi - alpha) * rays_per_rad) - 1;
      const int hi = (int)ceilf((phi + alpha) * rays_per_rad) + 1;
      if (hi - lo + 1 < R) {
        k0 = lo;
        nk = hi - lo + 1;
      }
    }
    const double px = x - bx[j], py = y - by[j], cj = bc[j], sj = bs[j], hl = bl[j], hw = bw[j];
    unsigned* row = best + a * R;
    for (int kk = 0; kk < nk; ++kk) {
      int k = (k0 + kk) % R;
      if (k < 0) k += R;
      const double ex = e.ray_dir[2 * k], ey = e.ray_dir[2 * k + 1];
      const double ux = c * ex - s * ey, uy = s * ex + c * ey;
      double t;
      if (lidar_ray_box(px, py, ux, uy, cj, sj, hl, hw, t) && t < range) atomicMin(row + k, __float_as_uint((float)t));
    }
  }
#else
  for (int q = threadIdx.x; q < na * R; q += blockDim.x) {
    const int a = q / R, k = q - a * R;
    const int slot = aslot[a];
    if (slot < 0) continue;
    const double x = ax[a], y = ay[a], c = ac[a], s = as[a];
    const double ex = e.ray_dir[2 * k], ey = e.ray_dir[2 * k + 1];
    const double ux = c * ex - s * ey, uy = s * ex + c * ey;
    double m = range;
    for (int j = 0; j < M; ++j) {
      if (j == slot || !bp[j]) continue;
      double t;
      if (lidar_ray_box(x - bx[j], y - by[j], ux, uy, bc[j], bs[j], bl[j], bw[j], t) && t < m) m = t;
    }
    best[q] = __float_as_uint((float)m);
  }
#endif
  __syncthreads();
  for (int q = threadIdx.x; q < na * R; q += blockDim.x) {
    const int a = q / R, k = q - a * R;
    if (aslot[a] < 0) continue;  // (the observe kernel zero-filled the row)
    obs[((int64_t)n * A + a0 + a) * F + (F - R) + k] = __uint_as_float(best[q]);
  }
}

static cudaError_t launch_lidar(cudaStream_t s, const SgScene& sc, const SgState& st, const SgEnvSpec& e,
                                const uint8_t* mask, float* obs, int F) {
  const int M = sc.n_slots, A = e.n_agents, R = e.n_rays;
  const int chunk = min(A, SG_LIDAR_MIN_BYTES / (4 * R));
  const int n_chunks = (A + chunk - 1) / chunk;
  // 7 doubles + a presence byte per slot, 4 doubles + a slot number + R minima per agent of the chunk
  const size_t smem = (size_t)M * (7 * sizeof(double) + 1) + (size_t)chunk * (4 * sizeof(double) + 4 + 4 * R);
  if (smem > 48 * 1024) {  // at most 57 KB of boxes (M = 1024) + 48 KB of minima + 1.7 KB of agents
    const cudaError_t err =
        cudaFuncSetAttribute(sg_env_lidar_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return err;
  }
  sg_env_lidar_kernel<<<(unsigned)((int64_t)sc.n_scenarios * n_chunks), SG_LIDAR_THREADS, smem, s>>>(
      sc, st, e, mask, obs, F, chunk, n_chunks);
  return cudaGetLastError();
}

template <int KCAP>
static cudaError_t launch_observe_t(cudaStream_t s, const SgScene& sc, const SgState& st, const SgEnvSpec& e,
                                    const uint8_t* mask, float* obs, uint8_t* agent_mask, int F) {
  const int M = sc.n_slots;
  const int threads = M >= 256 ? 256 : ((M + 31) / 32) * 32;
  const size_t smem = (size_t)M * (5 * sizeof(double) + 1);  // at most 42 KB (M <= 1024)
  sg_env_observe_kernel<KCAP><<<sc.n_scenarios, threads, smem, s>>>(sc, st, e, mask, obs, agent_mask, F);
  return cudaGetLastError();
}

cudaError_t sgi_launch_env_observe(cudaStream_t s, const SgScene& sc, const SgState& st, const SgEnvSpec& e,
                                   const uint8_t* mask, float* obs, uint8_t* agent_mask) {
  const int F = 4 + 3 * e.n_lookahead + 10 * e.k_neighbours + (e.road ? 2 : 0) + e.n_rays;
  cudaError_t err;
  if (e.k_neighbours <= 8) err = launch_observe_t<8>(s, sc, st, e, mask, obs, agent_mask, F);
  else if (e.k_neighbours <= 16) err = launch_observe_t<16>(s, sc, st, e, mask, obs, agent_mask, F);
  else err = launch_observe_t<32>(s, sc, st, e, mask, obs, agent_mask, F);
  if (err != cudaSuccess || e.n_rays <= 0) return err;
  return launch_lidar(s, sc, st, e, mask, obs, F);  // (after the row prefix and the zero rows, same stream)
}

cudaError_t sgi_launch_env_reward(cudaStream_t s, const SgScene& sc, const SgParams& p, const SgState& st,
                                  const SgEnvSpec& e, float* reward, float* terms, uint8_t* terminated,
                                  uint8_t* truncated) {
  const int64_t n = (int64_t)sc.n_scenarios * e.n_agents;
  sg_env_reward_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(sc, p, st, e, reward, terms, terminated,
                                                                  truncated);
  return cudaGetLastError();
}
