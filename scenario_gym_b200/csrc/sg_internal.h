// sg_internal.h -- host-side launchers of the kernels, one translation unit per kernel family
// (compiled in parallel; no relocatable device code).
#pragma once
#include <cuda_runtime.h>

#include "../../include/sg_b200.h"
#include "sg_layout.h"
#include "sg_pcg.cuh"

// mask: [N] scenarios to reset (NULL: all); init: the start times / perturbation of sg_reset_scenarios_init
// (NULL: the reset at t0, sg_reset_scenarios)
cudaError_t sgi_launch_reset(bool rss, bool big, int blocks, int threads, size_t smem, cudaStream_t s,
                             const SgScene& sc, const SgParams& p, const SgState& st, const GroupLayout& L,
                             const uint8_t* mask, const SgResetInit* init);
cudaError_t sgi_launch_rollout(bool ped, bool rss, bool big, int blocks, int threads, size_t smem,
                               cudaStream_t s, const SgScene& sc, const SgParams& p, const SgState& st,
                               const SgInputs& in, const SgRngDev& rng, int n_ticks, const GroupLayout& L);
// where the VehicleAction rows come from
enum { ACT_F64 = 0, ACT_RNG = 1, ACT_F32 = 2 };

// vehicle-only scenes; act: 0 fp64 table, 1 device PCG64 stream (rng), 2 fp32 table.  The lean
// variants (collisions on, no trace, no pair matrix) exist for every action source, the others for
// the fp64 table only.
static inline bool sgi_vehicle_lean(const SgParams& p, const SgState& st) {
  const bool need_coll = (p.features & SG_FEAT_COLLISIONS) ||
                         (p.terminal & (SG_TERM_COLLISION | SG_TERM_EGO_COLLISION));
  return need_coll && st.trace_cap <= 0 && !(p.features & SG_FEAT_COLL_MATRIX);
}
cudaError_t sgi_launch_vehicle_rss0(int n_scen, cudaStream_t s, const SgScene& sc, const SgParams& p,
                                    const SgState& st, const SgInputs& in, const SgRngDev& rng, int act,
                                    int n_ticks, const GroupLayout& L);
cudaError_t sgi_launch_vehicle_rss1(int n_scen, cudaStream_t s, const SgScene& sc, const SgParams& p,
                                    const SgState& st, const SgInputs& in, const SgRngDev& rng, int act,
                                    int n_ticks, const GroupLayout& L);
cudaError_t sgi_launch_fill_actions(cudaStream_t s, const SgRngDev& rng, int n_ticks, int64_t nm, double* out);
cudaError_t sgi_launch_replay(cudaStream_t s, const SgScene& sc, const SgParams& p, const SgState& st,
                              int n_ticks);
cudaError_t sgi_launch_box_pairs(cudaStream_t s, const double* pa, const double* ba, const double* pb,
                                 const double* bb, uint8_t* out, int64_t n);
cudaError_t sgi_launch_future(cudaStream_t s, const SgScene& sc, const double* t, const int32_t* slot,
                              double horizon, int n_samples, uint8_t* out);
cudaError_t sgi_measure_fp64(cudaStream_t s, double* inst_per_s);
cudaError_t sgi_launch_crowd(cudaStream_t s, const SgScene& sc, const SgParams& p, const SgState& st,
                             const SgInputs& in, int n_ticks);
cudaError_t sgi_launch_radius(cudaStream_t s, const SgState& st, int n_scen, int M, const double* x, const double* y,
                              const double* r, uint8_t* out);
// rows: an upper bound of the union rows of the scene's scenarios (a window holds fewer than n_union_rows)
cudaError_t sgi_launch_union(cudaStream_t s, const SgScene& sc, int64_t rows);
// closed-loop environment (sg_env.cu); `sc` has its plane stride stated
cudaError_t sgi_launch_env_observe(cudaStream_t s, const SgScene& sc, const SgState& st, const SgEnvSpec& e,
                                   const uint8_t* mask, float* obs, uint8_t* agent_mask);
cudaError_t sgi_launch_env_reward(cudaStream_t s, const SgScene& sc, const SgParams& p, const SgState& st,
                                  const SgEnvSpec& e, float* reward, float* terms, uint8_t* terminated,
                                  uint8_t* truncated);
// sg_env_raster (sg_raster.cu); `sc` has its plane stride stated, the arguments are checked
cudaError_t sgi_launch_env_raster(cudaStream_t s, const SgScene& sc, const SgState& st, const SgEnvSpec& e,
                                  const SgRasterSpec& r, const uint8_t* mask, uint8_t* out);
// sg_fork_state (sg_fork.cu); `sc` has its plane stride stated, the arguments are checked
cudaError_t sgi_launch_fork(cudaStream_t s, const SgScene& sc, const SgState& src, SgState* const* dst, int n_dst,
                            const SgEnvSpec* src_spec, SgEnvSpec* const* dst_spec);
// sg_plan_sample / sg_plan_update (sg_plan.cu); the arguments are checked
cudaError_t sgi_launch_plan_sample(cudaStream_t s, const SgEnvSpec& e, int N, int M, int B, int H, uint64_t seed,
                                   int k, const double sigma[2], double* mu, const uint8_t* reset, void* table,
                                   bool table_f64);
cudaError_t sgi_launch_plan_update(cudaStream_t s, const SgEnvSpec& e, int N, int M, int B, int H, double lambda,
                                   const float* reward, const void* table, bool table_f64, const double* mu_in,
                                   double* mu_out, bool finish, float* action, int32_t* best_branch,
                                   float* best_reward);
cudaError_t sgi_launch_traj(cudaStream_t s, const double* rows, int K, const double* t, int64_t n, int mode,
                            double* pos, uint8_t* ok, double* vel);
