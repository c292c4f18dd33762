// sg_raster.cu -- bird's-eye rasters of the closed-loop environment's agents (sg_env_raster; semantics and the
// culling conditions in include/sg_b200.h, SgRasterSpec).
#include "sg_device.cuh"
#include "sg_internal.h"

#define SG_RASTER_WARPS 4

// the column of pixel j: pv_j = (S - 1 - 2j) * h
template <int S>
static __device__ __forceinline__ double raster_pv(int j, double h) {
  return (double)(S - 1 - 2 * j) * h;
}

// the first j with vc > pv_j (S when there is none): pv_j decreases with j, so the toggled set is the suffix
// [j0, S).  The floor (with 1 / h, not a division) gives j0 to within a pixel; the exact comparisons settle it.
template <int S>
static __device__ __forceinline__ int raster_suffix(double vc, double h, double inv_h) {
  double f = floor(0.5 * ((double)(S - 1) - vc * inv_h)) + 1.0;
  f = f < 0.0 ? 0.0 : (f > (double)S ? (double)S : f);
  int j0 = (int)f;
  while (j0 > 0 && vc > raster_pv<S>(j0 - 1, h)) --j0;
  while (j0 < S && !(vc > raster_pv<S>(j0, h))) ++j0;
  return j0;
}

// four bits -> four bytes of 0 / 1 (little endian: bit k -> byte k)
static __device__ __forceinline__ unsigned raster_spread4(unsigned b) { return ((b & 15u) * 0x00204081u) & 0x01010101u; }

// sg_env_raster_kernel: one warp per (scenario, agent), SG_RASTER_WARPS agents of one scenario per block.  The
// block first stages every present slot's box (centre, axes, half extents, circumscribed radius, channel) in
// shared memory; each warp compacts the boxes whose circle can reach its raster into a list (ballots).  Lane l
// then scan-converts rows l, l + 32, ...: for each row it walks the polygons of the three surfaces, 32 bounding
// boxes per ballot, and for each candidate polygon XOR-accumulates the suffix masks {j : vc > pv_j} of the edges
// crossing the row, then ORs the polygon's mask into the surface's; the boxes are tested pixel by pixel within
// the span of their circle on the row.  The row's five channels leave as 16-byte stores.  Compiled with
// -DSG_RASTER_BRUTE every polygon and every box is tested at every pixel (the form the culled one was measured
// against, DESIGN.md section 6b).
template <int W>
__global__ void __launch_bounds__(SG_RASTER_WARPS * 32)
sg_env_raster_kernel(SgScene sc, SgState st, SgEnvSpec e, SgRasterSpec rs, const uint8_t* __restrict__ mask,
                     uint8_t* __restrict__ out, int chunks) {
  constexpr int S = 32 * W;
  extern __shared__ __align__(16) unsigned char smem[];
  const int n = blockIdx.x / chunks;
  if (mask && !mask[n]) return;
  const int M = sc.n_slots, A = e.n_agents, nw = blockDim.x >> 5;
  const int a0 = (blockIdx.x - n * chunks) * nw;
  const int64_t nm = sc.plane_stride, base = (int64_t)n * M;
  double* bx = (double*)smem;  // box centres, cos / sin, half extents, circumscribed radius
  double* by = bx + M;
  double* bc = by + M;
  double* bs = bc + M;
  double* bl = bs + M;
  double* bw = bl + M;
  double* br = bw + M;
  uint16_t* cand = (uint16_t*)(br + M);       // [nw][M] the warps' candidate boxes
  uint8_t* bk = (uint8_t*)(cand + nw * M);    // 0 absent, 1 channel 3, 2 channel 4 (pedestrian)
  for (int j = threadIdx.x; j < M; j += blockDim.x) {
    const int64_t i = base + j;
    const uint8_t p = st.present[i];
    bk[j] = p ? (sc.etype[i] == SG_ETYPE_PEDESTRIAN ? 2 : 1) : 0;
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
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int a = a0 + warp;
  if (a >= A) return;
  const int64_t ia = (int64_t)n * A + a;
  const int slot = e.agent_slot[ia];
  const bool here = slot >= 0 && slot < M && bk[slot] != 0;
  const double h = 0.5 * rs.resolution, inv_h = 1.0 / h, ahead = rs.ahead;
  const double D = 1.4142135623730951 * ((double)S * h);  // the raster's half-diagonal
  double x = 0.0, y = 0.0, c = 1.0, s = 0.0;
  if (here) {
    x = st.pose[base + slot];
    y = st.pose[nm + base + slot];
    sincos(st.pose[3 * nm + base + slot], &s, &c);
  }
  const double cx = x + c * ahead, cy = y + s * ahead;  // the raster's world centre
  const double big = fmax(fabs(x), fabs(y));
  // the boxes that can reach the raster, in slot order
  uint16_t* mine = cand + warp * M;
  int nb = 0;
  if (here) {
    for (int j0 = 0; j0 < M; j0 += 32) {
      const int j = j0 + lane;
      bool ok = j < M && j != slot && bk[j] != 0;
#ifndef SG_RASTER_BRUTE
      if (ok) {
        const double mb = 1e-9 * (1.0 + fmax(big, fmax(fabs(bx[j]), fabs(by[j]))) + D);
        const double reach = D + br[j] + mb;
        ok = fabs(bx[j] - cx) <= reach && fabs(by[j] - cy) <= reach;
      }
#endif
      const unsigned bal = __ballot_sync(0xffffffffu, ok);
      if (ok) mine[nb + __popc(bal & ((1u << lane) - 1u))] = (uint16_t)j;
      nb += __popc(bal);
    }
    __syncwarp();
  }
  const int r = (here && sc.rn_of && sc.n_networks > 0) ? sc.rn_of[n] : -1;
#ifndef SG_RASTER_BRUTE
  const double pm_lo_x = cx - D - rs.margin, pm_hi_x = cx + D + rs.margin;
  const double pm_lo_y = cy - D - rs.margin, pm_hi_y = cy + D + rs.margin;
#endif
  uint8_t* img = out + ia * (int64_t)(5 * S * S);
#pragma unroll 1
  for (int pass = 0; pass < W; ++pass) {
    const int i = pass * 32 + lane;
    const double pu = ahead + (double)(S - 1 - 2 * i) * h;
    unsigned surf[3][W], veh[W], ped[W];
#pragma unroll
    for (int w = 0; w < W; ++w) { surf[0][w] = surf[1][w] = surf[2][w] = veh[w] = ped[w] = 0u; }
    if (r >= 0) {
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const int64_t q0 = sc.rn_poly_off[3 * r + k], q1 = sc.rn_poly_off[3 * r + k + 1];
        for (int64_t qb = q0; qb < q1; qb += 32) {
          const int64_t ql = qb + lane;
          bool ok = ql < q1;
#ifndef SG_RASTER_BRUTE
          if (ok) {
            const double* b = rs.poly_box + 4 * ql;
            ok = b[0] <= pm_hi_x && b[2] >= pm_lo_x && b[1] <= pm_hi_y && b[3] >= pm_lo_y;
          }
#endif
          unsigned bal = __ballot_sync(0xffffffffu, ok);
          while (bal) {
            const int64_t q = qb + (__ffs(bal) - 1);
            bal &= bal - 1u;
            unsigned pm[W];
#pragma unroll
            for (int w = 0; w < W; ++w) pm[w] = 0u;
            const int64_t e1 = sc.rn_edge_off[q + 1];
            // the previous edge's end in both frames: a ring's next edge starts where it ended, so its start is
            // transformed once (the same bits give the same result)
            long long px = 0x7ff8dead00000000ll, py = px;
            double pbu = 0.0, pbv = 0.0;
            for (int64_t ed = sc.rn_edge_off[q]; ed < e1; ++ed) {
              const double2 p0 = reinterpret_cast<const double2*>(sc.rn_edges)[2 * ed];
              const double2 p1 = reinterpret_cast<const double2*>(sc.rn_edges)[2 * ed + 1];
              double au, av;
              if (__double_as_longlong(p0.x) == px && __double_as_longlong(p0.y) == py) {
                au = pbu;
                av = pbv;
              } else {
                const double dx = p0.x - x, dy = p0.y - y;
                au = c * dx + s * dy;
                av = -s * dx + c * dy;
              }
              const double dx = p1.x - x, dy = p1.y - y;
              const double bu = c * dx + s * dy, bv = -s * dx + c * dy;
              px = __double_as_longlong(p1.x);
              py = __double_as_longlong(p1.y);
              pbu = bu;
              pbv = bv;
              if ((au > pu) != (bu > pu)) {
                const double vc = av + ((pu - au) * (bv - av)) / (bu - au);
                const int j0 = raster_suffix<S>(vc, h, inv_h);
#pragma unroll
                for (int w = 0; w < W; ++w) {
                  const int lo = 32 * w;
                  pm[w] ^= j0 <= lo ? 0xffffffffu : (j0 >= lo + 32 ? 0u : (0xffffffffu << (j0 - lo)));
                }
              }
            }
#pragma unroll
            for (int w = 0; w < W; ++w) surf[k][w] |= pm[w];
          }
        }
      }
    }
    for (int q = 0; q < nb; ++q) {
      const int j = mine[q];
      const double X = bx[j], Y = by[j], cj = bc[j], sj = bs[j], hl = bl[j], hw = bw[j];
      int jlo = 0, jhi = S - 1;
#ifndef SG_RASTER_BRUTE
      // the row's pixels near the box's circle, one pixel of slack either side; the exact test decides
      const double mb = 1e-9 * (1.0 + fmax(big, fmax(fabs(X), fabs(Y))) + D);
      const double R = br[j] + mb;
      const double gx = X - x, gy = Y - y;
      const double du = (c * gx + s * gy) - pu, bv = -s * gx + c * gy;
      if (fabs(du) > R) continue;
      const double half = sqrt(fmax(0.0, R * R - du * du)) + mb;
      double flo = floor(0.5 * ((double)(S - 1) - (bv + half) * inv_h)) - 1.0;
      double fhi = ceil(0.5 * ((double)(S - 1) - (bv - half) * inv_h)) + 1.0;
      flo = flo < 0.0 ? 0.0 : flo;
      fhi = fhi > (double)(S - 1) ? (double)(S - 1) : fhi;
      if (flo > fhi) continue;
      jlo = (int)flo;
      jhi = (int)fhi;
#endif
      const bool is_ped = bk[j] == 2;
#pragma unroll
      for (int w = 0; w < W; ++w) {
        const int lo = max(jlo, 32 * w), hi = min(jhi, 32 * w + 31);
        unsigned bits = 0u;
        for (int jj = lo; jj <= hi; ++jj) {
          const double pv = raster_pv<S>(jj, h);
          const double Px = x + (c * pu - s * pv), Py = y + (s * pu + c * pv);
          const double qx = Px - X, qy = Py - Y;
          const double ox = cj * qx + sj * qy, oy = -sj * qx + cj * qy;
          if (fabs(ox) <= hl && fabs(oy) <= hw) bits |= 1u << (jj - 32 * w);
        }
        if (is_ped) ped[w] |= bits;
        else veh[w] |= bits;
      }
    }
    uint8_t* row = img + (int64_t)i * S;
#pragma unroll
    for (int ch = 0; ch < 5; ++ch) {
      uint4* dst = reinterpret_cast<uint4*>(row + (int64_t)ch * S * S);
#pragma unroll
      for (int w = 0; w < W; ++w) {
        const unsigned b = ch < 3 ? surf[ch][w] : (ch == 3 ? veh[w] : ped[w]);
        dst[2 * w] = make_uint4(raster_spread4(b), raster_spread4(b >> 4), raster_spread4(b >> 8),
                                raster_spread4(b >> 12));
        dst[2 * w + 1] = make_uint4(raster_spread4(b >> 16), raster_spread4(b >> 20), raster_spread4(b >> 24),
                                    raster_spread4(b >> 28));
      }
    }
  }
}

template <int W>
static cudaError_t launch_raster_t(cudaStream_t s, const SgScene& sc, const SgState& st, const SgEnvSpec& e,
                                   const SgRasterSpec& r, const uint8_t* mask, uint8_t* out) {
  const int M = sc.n_slots, A = e.n_agents;
  const int nw = A < SG_RASTER_WARPS ? A : SG_RASTER_WARPS;
  const int chunks = (A + nw - 1) / nw;
  // 7 doubles + a channel byte per slot, a candidate list of M slot numbers per warp: at most 68 KB (M = 1024)
  const size_t smem = (size_t)M * (7 * sizeof(double) + 1 + 2 * nw);
  if (smem > 48 * 1024) {
    const cudaError_t err =
        cudaFuncSetAttribute(sg_env_raster_kernel<W>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return err;
  }
  sg_env_raster_kernel<W><<<(unsigned)((int64_t)sc.n_scenarios * chunks), 32 * nw, smem, s>>>(sc, st, e, r, mask,
                                                                                                out, chunks);
  return cudaGetLastError();
}

cudaError_t sgi_launch_env_raster(cudaStream_t s, const SgScene& sc, const SgState& st, const SgEnvSpec& e,
                                  const SgRasterSpec& r, const uint8_t* mask, uint8_t* out) {
  switch (r.size / 32) {
    case 1: return launch_raster_t<1>(s, sc, st, e, r, mask, out);
    case 2: return launch_raster_t<2>(s, sc, st, e, r, mask, out);
    case 3: return launch_raster_t<3>(s, sc, st, e, r, mask, out);
    case 4: return launch_raster_t<4>(s, sc, st, e, r, mask, out);
    case 5: return launch_raster_t<5>(s, sc, st, e, r, mask, out);
    case 6: return launch_raster_t<6>(s, sc, st, e, r, mask, out);
    case 7: return launch_raster_t<7>(s, sc, st, e, r, mask, out);
    default: return launch_raster_t<8>(s, sc, st, e, r, mask, out);
  }
}
