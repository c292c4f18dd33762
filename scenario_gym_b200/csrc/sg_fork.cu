// sg_fork.cu -- sg_fork_state's device side: one launch copies every field of an SgState (and optionally the
// snapshot arrays of an SgEnvSpec) into up to SG_FORK_MAX_DST destination states.
#include <stdint.h>
#include <string.h>

#include "sg_internal.h"

#define SG_FORK_MAX_FIELDS 40
#define SG_FORK_MAX_DST 64
#define SG_FORK_THREADS 256
#define SG_FORK_UPT 4  // copy units per thread: their loads are all issued before the stores

// one field: `planes` planes of plane_bytes bytes, `stride` bytes apart in the source and in every destination.
// A plane is copied as nvec 16-byte vectors (when the source and every destination are 16-byte aligned) followed
// by scalar elements of es bytes; `units` = vectors + scalar elements of one plane.
struct SgForkField {
  const unsigned char* src;  // NULL: the destinations are zero-filled
  int64_t plane_bytes, stride, nvec, units;
  int64_t block0;  // first CTA of the field
  int32_t planes, es;
};

// passed by value as the kernel parameter (~22 KB; a parameter block of up to 32 KB needs CUDA 12.1 and sm_70+)
struct SgForkTable {
  int32_t n_fields, n_dst;
  SgForkField f[SG_FORK_MAX_FIELDS];
  unsigned char* dst[SG_FORK_MAX_FIELDS][SG_FORK_MAX_DST];  // NULL: that destination skips the field
};

// Every CTA copies SG_FORK_THREADS * SG_FORK_UPT consecutive units of one field (the fields own consecutive
// ranges of CTAs, in proportion to their sizes): each unit is read once and stored to all n_dst destinations.
__global__ void __launch_bounds__(SG_FORK_THREADS) sg_fork_kernel(const __grid_constant__ SgForkTable t) {
  int f = 0;
  while (f + 1 < t.n_fields && (int64_t)blockIdx.x >= t.f[f + 1].block0) ++f;
  const SgForkField& F = t.f[f];
  const int64_t total = F.units * F.planes;
  const int64_t u0 = ((int64_t)blockIdx.x - F.block0) * (SG_FORK_THREADS * SG_FORK_UPT) + threadIdx.x;
  uint4 v[SG_FORK_UPT];
  int64_t off[SG_FORK_UPT];
  int kind[SG_FORK_UPT];  // 0: none, 16: vector, else the element size
#pragma unroll
  for (int k = 0; k < SG_FORK_UPT; ++k) {
    const int64_t u = u0 + k * SG_FORK_THREADS;
    kind[k] = 0;
    v[k] = make_uint4(0u, 0u, 0u, 0u);
    if (u >= total) continue;
    int64_t pl = 0, w = u;
    if (F.planes > 1) {
      pl = u / F.units;
      w = u - pl * F.units;
    }
    if (w < F.nvec) {
      off[k] = pl * F.stride + w * 16;
      kind[k] = 16;
      if (F.src) v[k] = *(const uint4*)(F.src + off[k]);
    } else {
      off[k] = pl * F.stride + F.nvec * 16 + (w - F.nvec) * F.es;
      kind[k] = F.es;
      if (F.src) {
        if (F.es == 8) {
          const unsigned long long q = *(const unsigned long long*)(F.src + off[k]);
          v[k].x = (unsigned)q;
          v[k].y = (unsigned)(q >> 32);
        } else if (F.es == 4) {
          v[k].x = *(const unsigned*)(F.src + off[k]);
        } else {
          v[k].x = F.src[off[k]];
        }
      }
    }
  }
  for (int d = 0; d < t.n_dst; ++d) {
    unsigned char* const base = t.dst[f][d];
    if (!base) continue;
#pragma unroll
    for (int k = 0; k < SG_FORK_UPT; ++k) {
      unsigned char* p = base + off[k];
      if (kind[k] == 16) *(uint4*)p = v[k];
      else if (kind[k] == 8) *(unsigned long long*)p = (unsigned long long)v[k].x | ((unsigned long long)v[k].y << 32);
      else if (kind[k] == 4) *(unsigned*)p = v[k].x;
      else if (kind[k] == 1) *p = (unsigned char)v[k].x;
    }
  }
}

namespace {

struct Builder {
  SgForkTable t;
  int64_t blocks = 0;
  bool overflow = false;

  // planes x elems elements of es bytes, planes `stride` elements apart
  void add(const void* src, void* const* dst, int n_dst, int es, int planes, int64_t elems, int64_t stride) {
    if (t.n_fields >= SG_FORK_MAX_FIELDS) {
      overflow = true;
      return;
    }
    if (planes > 1 && stride == elems) {  // contiguous planes: one plane
      elems *= planes;
      planes = 1;
    }
    SgForkField& F = t.f[t.n_fields];
    F.src = (const unsigned char*)src;
    F.es = es;
    F.planes = planes;
    F.plane_bytes = elems * es;
    F.stride = stride * es;
    bool aligned = ((uintptr_t)src & 15) == 0 && (planes == 1 || (F.stride & 15) == 0);
    for (int d = 0; d < n_dst; ++d) {
      t.dst[t.n_fields][d] = (unsigned char*)dst[d];
      if (dst[d]) aligned = aligned && ((uintptr_t)dst[d] & 15) == 0;
    }
    F.nvec = aligned ? F.plane_bytes / 16 : 0;
    F.units = F.nvec + (F.plane_bytes - F.nvec * 16) / es;
    F.block0 = blocks;
    const int64_t per_cta = SG_FORK_THREADS * SG_FORK_UPT;
    blocks += (F.units * planes + per_cta - 1) / per_cta;
    ++t.n_fields;
  }
};

}  // namespace

// `sc` has its plane stride stated; the arguments were checked by sg_fork_state
cudaError_t sgi_launch_fork(cudaStream_t s, const SgScene& sc, const SgState& src, SgState* const* dst, int n_dst,
                            const SgEnvSpec* src_spec, SgEnvSpec* const* dst_spec) {
  const int64_t N = sc.n_scenarios, M = sc.n_slots, NM = N * M, W = (M + 31) / 32, ps = sc.plane_stride;
  for (int d0 = 0; d0 < n_dst; d0 += SG_FORK_MAX_DST) {
    const int nd = n_dst - d0 < SG_FORK_MAX_DST ? n_dst - d0 : SG_FORK_MAX_DST;
    static thread_local Builder b;  // (22 KB: kept off the stack)
    memset(&b.t, 0, sizeof(b.t));
    b.blocks = 0;
    b.overflow = false;
    b.t.n_dst = nd;
    void* dp[SG_FORK_MAX_DST];
#define SG_FORK_FIELD(name, planes, elems, stride)                                            \
  do {                                                                                        \
    for (int d = 0; d < nd; ++d) dp[d] = (void*)dst[d0 + d]->name;                            \
    b.add(src.name, dp, nd, (int)sizeof(*src.name), planes, elems, stride);                   \
  } while (0)
    // per-slot planes: [C][N*M], planes plane_stride apart
    SG_FORK_FIELD(pose, 6, NM, ps);
    SG_FORK_FIELD(vel, 6, NM, ps);
    SG_FORK_FIELD(force, 2, NM, ps);
    SG_FORK_FIELD(safe_dist, 2, NM, ps);
    SG_FORK_FIELD(safe_ratio, 2, NM, ps);
    SG_FORK_FIELD(pid_err, 3, NM, ps);
    SG_FORK_FIELD(dist, 1, NM, ps);
    SG_FORK_FIELD(speed, 1, NM, ps);
    SG_FORK_FIELD(goal_idx, 1, NM, ps);
    SG_FORK_FIELD(cur_own, 1, NM, ps);
    SG_FORK_FIELD(present, 1, NM, ps);
    SG_FORK_FIELD(collided, 1, NM, ps);
    SG_FORK_FIELD(rss_state, 1, NM, ps);
    SG_FORK_FIELD(rss_last, 1, NM, ps);
    // per-scenario fields
    SG_FORK_FIELD(t, 1, N, N);
    SG_FORK_FIELD(prev_t, 1, N, N);
    SG_FORK_FIELD(ego_avg_speed, 1, N, N);
    SG_FORK_FIELD(ego_avg_t, 1, N, N);
    SG_FORK_FIELD(ego_max_speed, 1, N, N);
    SG_FORK_FIELD(ego_dist, 1, N, N);
    SG_FORK_FIELD(n_pair_ticks, 1, N, N);
    SG_FORK_FIELD(tick, 1, N, N);
    SG_FORK_FIELD(cur_union, 1, N, N);
    SG_FORK_FIELD(first_coll_tick, 1, N, N);
    SG_FORK_FIELD(first_coll_pair, 1, 2 * N, 2 * N);
    SG_FORK_FIELD(ego_hits, 1, N * W, N * W);
    SG_FORK_FIELD(done, 1, N, N);
    SG_FORK_FIELD(rss_flags, 1, N, N);
    if (src.coll_mask) SG_FORK_FIELD(coll_mask, 1, NM * W, NM * W);  // (NULL destinations skip it)
#undef SG_FORK_FIELD
    for (int d = 0; d < nd; ++d) dp[d] = (void*)dst[d0 + d]->event_count;
    b.add(nullptr, dp, nd, 4, 1, 1, 1);  // event_count = 0
    if (src_spec) {
      const int64_t NA = N * src_spec->n_agents;
#define SG_FORK_SNAP(name, elems)                                                             \
  do {                                                                                        \
    for (int d = 0; d < nd; ++d) dp[d] = (void*)dst_spec[d0 + d]->name;                       \
    b.add(src_spec->name, dp, nd, (int)sizeof(*src_spec->name), 1, elems, elems);             \
  } while (0)
      SG_FORK_SNAP(snap_dist, NA);
      SG_FORK_SNAP(snap_pair_ticks, N);
      SG_FORK_SNAP(snap_collided, NA);
      SG_FORK_SNAP(snap_rss, N);
#undef SG_FORK_SNAP
    }
    if (b.overflow) return cudaErrorInvalidValue;
    if (b.blocks > 0x7fffffff) return cudaErrorInvalidConfiguration;
    sg_fork_kernel<<<(unsigned)b.blocks, SG_FORK_THREADS, 0, s>>>(b.t);
    const cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return err;
  }
  return cudaSuccess;
}
