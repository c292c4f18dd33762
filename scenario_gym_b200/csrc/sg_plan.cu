// sg_plan.cu -- the device side of sg_plan_sample / sg_plan_update (MPPI over the branch action tables; semantics
// in include/sg_b200.h).  Both kernels map threadIdx.x / blockIdx.x to the agents (n, a) of one (branch, tick) or
// one tick, so a warp's table accesses table_b[h][c][n*M + s] and mean accesses mu[n][h][a][c] are consecutive.
#include <stdint.h>

#include "sg_device.cuh"
#include "sg_internal.h"

#define SG_PLAN_THREADS 256
#define SG_PLAN_MAX_GRID_Y 65535

template <typename T>
__global__ void __launch_bounds__(SG_PLAN_THREADS)
sg_plan_sample_kernel(const int32_t* __restrict__ agent_slot, int64_t NA, int A, int M, int64_t NM, int B, int H,
                      uint64_t seed, int k, double sigma0, double sigma1, double* __restrict__ mu,
                      const uint8_t* __restrict__ reset, T* __restrict__ table) {
  const int64_t na = (int64_t)blockIdx.x * SG_PLAN_THREADS + threadIdx.x;
  if (na >= NA) return;
  const int s = agent_slot[na];
  if (s < 0) return;
  const int64_t n = na / A, a = na - n * A;
  const bool zero = reset && reset[n];
  for (int bh = blockIdx.y; bh < B * H; bh += gridDim.y) {
    const int b = bh / H, h = bh - b * H;
    double* const m = mu + ((n * H + h) * A + a) * 2;
    double m0 = 0.0, m1 = 0.0;
    if (zero) {
      if (b == 0) m[0] = m[1] = 0.0;  // (every thread of this scenario reads 0 instead of m: no race)
    } else {
      m0 = m[0];
      m1 = m[1];
    }
    double v0 = m0, v1 = m1;
    if (b > 0) {
      const double2 z = sg_noise2(seed, ((na * B + b) * H + h), k);
      v0 = m0 + sigma0 * z.x;
      v1 = m1 + sigma1 * z.y;
    }
    T* const row = table + (int64_t)bh * 2 * NM + n * M + s;
    row[0] = (T)v0;
    row[NM] = (T)v1;
  }
}

template <typename T>
__global__ void __launch_bounds__(SG_PLAN_THREADS)
sg_plan_update_kernel(const int32_t* __restrict__ agent_slot, int64_t NA, int A, int M, int64_t NM, int B, int H,
                      double lambda, const float* __restrict__ reward, const T* __restrict__ table,
                      const double* __restrict__ mu_in, double* __restrict__ mu_out, int finish,
                      float* __restrict__ action, int32_t* __restrict__ best_branch, float* __restrict__ best_reward) {
  const int64_t na = (int64_t)blockIdx.x * SG_PLAN_THREADS + threadIdx.x;
  if (na >= NA) return;
  const int s = agent_slot[na];
  if (s < 0) return;
  const int64_t n = na / A, a = na - n * A;
  float rmax = reward[na];
  int best = 0;
  for (int b = 1; b < B; ++b) {
    const float r = reward[(int64_t)b * NA + na];
    if (r > rmax) {
      rmax = r;
      best = b;
    }
  }
  for (int h = blockIdx.y; h < H; h += gridDim.y) {
    const double* const m = mu_in + ((n * H + h) * A + a) * 2;
    const double m0 = m[0], m1 = m[1];
    double wsum = 0.0, acc0 = 0.0, acc1 = 0.0;
#pragma unroll 1
    for (int b = 0; b < B; ++b) {
      const double w = exp(((double)reward[(int64_t)b * NA + na] - (double)rmax) / lambda);
      const T* const row = table + ((int64_t)b * H + h) * 2 * NM + n * M + s;
      wsum += w;
      acc0 += w * ((double)row[0] - m0);
      acc1 += w * ((double)row[NM] - m1);
    }
    const double u0 = m0 + acc0 / wsum, u1 = m1 + acc1 / wsum;
    if (!finish) {
      double* const o = mu_out + ((n * H + h) * A + a) * 2;
      o[0] = u0;
      o[1] = u1;
      continue;
    }
    if (h == 0) {
      action[na * 2] = (float)u0;
      action[na * 2 + 1] = (float)u1;
    } else {
      double* const o = mu_out + ((n * H + h - 1) * A + a) * 2;
      o[0] = u0;
      o[1] = u1;
    }
    if (h == H - 1) {
      double* const o = mu_out + ((n * H + h) * A + a) * 2;
      o[0] = o[1] = 0.0;
    }
  }
  if (blockIdx.y == 0) {
    best_branch[na] = best;
    best_reward[na] = rmax;
  }
}

static dim3 plan_grid(int64_t NA, int64_t rows) {
  return dim3((unsigned)((NA + SG_PLAN_THREADS - 1) / SG_PLAN_THREADS),
              (unsigned)(rows < SG_PLAN_MAX_GRID_Y ? rows : SG_PLAN_MAX_GRID_Y));
}

cudaError_t sgi_launch_plan_sample(cudaStream_t s, const SgEnvSpec& e, int N, int M, int B, int H, uint64_t seed,
                                   int k, const double sigma[2], double* mu, const uint8_t* reset, void* table,
                                   bool table_f64) {
  const int64_t NA = (int64_t)N * e.n_agents, NM = (int64_t)N * M;
  const dim3 grid = plan_grid(NA, (int64_t)B * H);
  if (table_f64)
    sg_plan_sample_kernel<double><<<grid, SG_PLAN_THREADS, 0, s>>>(e.agent_slot, NA, e.n_agents, M, NM, B, H, seed,
                                                                   k, sigma[0], sigma[1], mu, reset, (double*)table);
  else
    sg_plan_sample_kernel<float><<<grid, SG_PLAN_THREADS, 0, s>>>(e.agent_slot, NA, e.n_agents, M, NM, B, H, seed,
                                                                  k, sigma[0], sigma[1], mu, reset, (float*)table);
  return cudaGetLastError();
}

cudaError_t sgi_launch_plan_update(cudaStream_t s, const SgEnvSpec& e, int N, int M, int B, int H, double lambda,
                                   const float* reward, const void* table, bool table_f64, const double* mu_in,
                                   double* mu_out, bool finish, float* action, int32_t* best_branch,
                                   float* best_reward) {
  const int64_t NA = (int64_t)N * e.n_agents, NM = (int64_t)N * M;
  const dim3 grid = plan_grid(NA, H);
  if (table_f64)
    sg_plan_update_kernel<double><<<grid, SG_PLAN_THREADS, 0, s>>>(
        e.agent_slot, NA, e.n_agents, M, NM, B, H, lambda, reward, (const double*)table, mu_in, mu_out, finish,
        action, best_branch, best_reward);
  else
    sg_plan_update_kernel<float><<<grid, SG_PLAN_THREADS, 0, s>>>(
        e.agent_slot, NA, e.n_agents, M, NM, B, H, lambda, reward, (const float*)table, mu_in, mu_out, finish,
        action, best_branch, best_reward);
  return cudaGetLastError();
}
