// sg_device.cuh -- device-side building blocks of the rollout engine (sm_100a).
//
// Everything is fp64 and keeps the reference's operation order; the translation unit
// is compiled with -fmad=false so a*b+c is never contracted (numpy has no FMA on this
// path).  fma() is used explicitly only inside the exact-arithmetic predicates, where
// it is an error-free transformation, not an approximation.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/sg_b200.h"

#define SG_DEV __device__ __forceinline__

// ----------------------------------------------------------------------------------
// Linear interpolation with scipy's interp1d._call_linear operation order (third-party
// arithmetic reached from reference trajectory.py:178-184, entity/batch.py:99-127):
//   w1 = (t - x_lo) / (x_hi - x_lo);  w0 = (x_hi - t) / (x_hi - x_lo);  y = w1*y_hi + w0*y_lo
// ----------------------------------------------------------------------------------
enum { EXT_NONE = 0, EXT_CLAMP = 1, EXT_TRUE = 2 };

// first index i in [0, K) with x[i*stride] >= t (numpy searchsorted side='left')
SG_DEV int search_left(const double* __restrict__ x, int stride, int K, double t) {
  int lo = 0, hi = K;
  while (lo < hi) {
    int mid = (lo + hi) >> 1;
    if (__ldg(x + (int64_t)mid * stride) < t) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// Monotone cursor version: `cur` is the previous clipped index (in [1, K-1]); the tick
// times only grow, so the control-point search is O(1) amortised.  Falls back to a
// binary search when t moved backwards.
SG_DEV int search_left_cursor(const double* __restrict__ x, int stride, int K, double t, int cur) {
  if (cur < 1 || cur > K - 1 || __ldg(x + (int64_t)(cur - 1) * stride) >= t) {
    int i = search_left(x, stride, K, t);
    return min(max(i, 1), K - 1);
  }
  while (cur < K - 1 && __ldg(x + (int64_t)cur * stride) < t) ++cur;
  return cur;
}

// Trajectory.position_at_t for scalar t (reference trajectory.py:142-197) on the slot's
// own control points rows[K][7].  Returns false when the reference returns None.
SG_DEV bool position_at_t(const double* __restrict__ rows, int K, double t, int mode, int& cur,
                          double out[6]) {
  const double min_t = __ldg(rows), max_t = __ldg(rows + (int64_t)(K - 1) * 7);
  if (mode == EXT_NONE && (t < min_t || t > max_t)) return false;  // :191-192
  if (mode != EXT_TRUE && t < min_t) {                               // :193-194
#pragma unroll
    for (int f = 0; f < 6; ++f) out[f] = __ldg(rows + 1 + f);
    return true;
  }
  if (mode != EXT_TRUE && t > max_t) {  // :195-196
#pragma unroll
    for (int f = 0; f < 6; ++f) out[f] = __ldg(rows + (int64_t)(K - 1) * 7 + 1 + f);
    return true;
  }
  if (K == 1) {  // :175-177 single control point duplicated at t + 1e-3
    const double x_lo = min_t, x_hi = min_t + 1e-3;
    const double w1 = (t - x_lo) / (x_hi - x_lo), w0 = (x_hi - t) / (x_hi - x_lo);
#pragma unroll
    for (int f = 0; f < 6; ++f) {
      const double y = __ldg(rows + 1 + f);
      out[f] = w1 * y + w0 * y;
    }
    return true;
  }
  cur = search_left_cursor(rows, 7, K, t, cur);
  const double* lo = rows + (int64_t)(cur - 1) * 7;
  const double* hi = lo + 7;
  const double x_lo = __ldg(lo), x_hi = __ldg(hi);
  const double w1 = (t - x_lo) / (x_hi - x_lo), w0 = (x_hi - t) / (x_hi - x_lo);
#pragma unroll
  for (int f = 0; f < 6; ++f) out[f] = w1 * __ldg(hi + 1 + f) + w0 * __ldg(lo + 1 + f);
  return true;
}

// Trajectory.velocity_at_t (reference trajectory.py:243-273), eps = 1e-4
SG_DEV void velocity_at_t(const double* __restrict__ rows, int K, double t, double out[6]) {
  const double eps = 1e-4;
  const double min_t = __ldg(rows), max_t = __ldg(rows + (int64_t)(K - 1) * 7);
  const bool inside = (min_t <= t) && (t <= max_t);
  double a[6], b[6];
  int c0 = 0, c1 = 0;
  position_at_t(rows, K, t + eps / 2, EXT_TRUE, c0, a);
  position_at_t(rows, K, t - eps / 2, EXT_TRUE, c1, b);
#pragma unroll
  for (int f = 0; f < 6; ++f) out[f] = inside ? (a[f] - b[f]) / eps : 0.0;
}

// ----------------------------------------------------------------------------------
// Exact orientation sign (GEOS decides `intersects` with robust orientation predicates;
// Shapely call sites: reference utils.py:51-62, metrics/rss/callback.py:191-196,317-328).
// Static filter with Shewchuk's bound, exact expansion arithmetic behind it.
// ----------------------------------------------------------------------------------
SG_DEV void two_sum(double a, double b, double& s, double& e) {
  s = __dadd_rn(a, b);
  const double bv = __dsub_rn(s, a), av = __dsub_rn(s, bv);
  e = __dadd_rn(__dsub_rn(a, av), __dsub_rn(b, bv));
}
SG_DEV void two_prod(double a, double b, double& p, double& e) {
  p = __dmul_rn(a, b);
  e = __fma_rn(a, b, -p);
}

static __device__ __noinline__ int orient_exact(double ax, double ay, double bx, double by, double cx,
                                         double cy) {
  double d[4][2];
  two_sum(ax, -cx, d[0][0], d[0][1]);
  two_sum(by, -cy, d[1][0], d[1][1]);
  two_sum(ay, -cy, d[2][0], d[2][1]);
  two_sum(bx, -cx, d[3][0], d[3][1]);
  double h[20];
  int n = 0;
  auto grow = [&](double b) {  // Shewchuk grow-expansion
    double q = b;
    for (int i = 0; i < n; ++i) {
      double s, e;
      two_sum(q, h[i], s, e);
      h[i] = e;
      q = s;
    }
    h[n++] = q;
  };
  for (int i = 0; i < 2; ++i)
    for (int j = 0; j < 2; ++j) {
      double p, e;
      two_prod(d[0][i], d[1][j], p, e);
      grow(e);
      grow(p);
      two_prod(d[2][i], d[3][j], p, e);
      grow(-e);
      grow(-p);
    }
  for (int i = n - 1; i >= 0; --i) {
    if (h[i] > 0) return 1;
    if (h[i] < 0) return -1;
  }
  return 0;
}

SG_DEV int orient_sign(double ax, double ay, double bx, double by, double cx, double cy) {
  const double errbound = (3.0 + 16.0 * 1.1102230246251565e-16) * 1.1102230246251565e-16;
  const double l = (ax - cx) * (by - cy), r = (ay - cy) * (bx - cx);
  const double det = l - r;
  if (fabs(det) > errbound * (fabs(l) + fabs(r))) return det > 0 ? 1 : -1;
  return orient_exact(ax, ay, bx, by, cx, cy);
}

// The exact quad predicates run on the rare path (AABB survivors, RSS boundary cases) with few
// active lanes.  They are out of line, keep the quad in registers (loaded once with ld.shared
// from the group's staged corners) and walk the edges by rotating the corner registers, so the
// orientation predicate is instantiated only four times per routine.
struct Quad {
  double x0, y0, x1, y1, x2, y2, x3, y3;
};
SG_DEV void rotate(Quad& q) {  // corner k <- corner k+1
  const double tx = q.x0, ty = q.y0;
  q.x0 = q.x1; q.y0 = q.y1; q.x1 = q.x2; q.y1 = q.y2; q.x2 = q.x3; q.y2 = q.y3; q.x3 = tx; q.y3 = ty;
}
// Only used inside out-of-line helpers that do not store to shared memory themselves (the call is
// the ordering point), so the loads may be scheduled freely: not volatile.
SG_DEV double lds_f64(unsigned addr) {
  double v;
  asm("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
  return v;
}
// corner k of a staged quad sits at shared address base + (2k)*stride (x) and base + (2k+1)*stride (y)
SG_DEV Quad load_quad_shared(unsigned base, unsigned stride) {
  Quad q;
  q.x0 = lds_f64(base); q.y0 = lds_f64(base + stride);
  q.x1 = lds_f64(base + 2 * stride); q.y1 = lds_f64(base + 3 * stride);
  q.x2 = lds_f64(base + 4 * stride); q.y2 = lds_f64(base + 5 * stride);
  q.x3 = lds_f64(base + 6 * stride); q.y3 = lds_f64(base + 7 * stride);
  return q;
}
SG_DEV Quad quad_from_array(const double* p) {
  Quad q = {p[0], p[1], p[2], p[3], p[4], p[5], p[6], p[7]};
  return q;
}

// ring orientation of a convex quad: +1 ccw, -1 cw, 0 degenerate
SG_DEV int quad_orientation(const Quad& q) {
  int s = orient_sign(q.x0, q.y0, q.x1, q.y1, q.x2, q.y2);
  if (s == 0) s = orient_sign(q.x1, q.y1, q.x2, q.y2, q.x3, q.y3);
  return s;
}

// are all four corners of b strictly outside edge (corner 0 -> corner 1) of a (orientation o)?
// A quad without area (o == 0: a segment or a point) has no inside: its edge separates when b lies
// strictly on one side of it, whichever side.
SG_DEV bool edge01_separates(const Quad& a, int o, const Quad& b) {
  const int s0 = orient_sign(a.x0, a.y0, a.x1, a.y1, b.x0, b.y0);
  if (o != 0 ? s0 * o >= 0 : s0 == 0) return false;
  const int want = o != 0 ? -o : s0;
  return orient_sign(a.x0, a.y0, a.x1, a.y1, b.x1, b.y1) == want &&
         orient_sign(a.x0, a.y0, a.x1, a.y1, b.x2, b.y2) == want &&
         orient_sign(a.x0, a.y0, a.x1, a.y1, b.x3, b.y3) == want;
}

// closed segments (a, b) and (c, d) share a point (exact)
SG_DEV bool on_segment(double ax, double ay, double bx, double by, double px, double py) {
  return orient_sign(ax, ay, bx, by, px, py) == 0 && fmin(ax, bx) <= px && px <= fmax(ax, bx) &&
         fmin(ay, by) <= py && py <= fmax(ay, by);
}
SG_DEV bool segments_meet(double ax, double ay, double bx, double by, double cx, double cy, double dx, double dy) {
  const int o1 = orient_sign(ax, ay, bx, by, cx, cy), o2 = orient_sign(ax, ay, bx, by, dx, dy);
  const int o3 = orient_sign(cx, cy, dx, dy, ax, ay), o4 = orient_sign(cx, cy, dx, dy, bx, by);
  if (o1 * o2 < 0 && o3 * o4 < 0) return true;
  return on_segment(ax, ay, bx, by, cx, cy) || on_segment(ax, ay, bx, by, dx, dy) ||
         on_segment(cx, cy, dx, dy, ax, ay) || on_segment(cx, cy, dx, dy, bx, by);
}
// two quads without area (segments / points): they meet iff their rings do
static __device__ __noinline__ bool flat_quads_meet(Quad a, Quad b) {
#pragma unroll 1
  for (int i = 0; i < 4; ++i) {
#pragma unroll 1
    for (int j = 0; j < 4; ++j) {
      if (segments_meet(a.x0, a.y0, a.x1, a.y1, b.x0, b.y0, b.x1, b.y1)) return true;
      rotate(b);
    }
    rotate(a);
  }
  return false;
}

// closed-set intersection of two convex quads (touching counts, as GEOS `intersects`):
// disjoint iff some edge of either has all four corners of the other strictly outside
static __device__ __noinline__ bool quads_intersect(Quad a, int oa, Quad b, int ob) {
  if (oa == 0 && ob == 0) return flat_quads_meet(a, b);
#pragma unroll 1
  for (int pass = 0; pass < 2; ++pass) {
#pragma unroll 1
    for (int k = 0; k < 4; ++k) {
      if (edge01_separates(a, oa, b)) return false;
      rotate(a);
    }
    const Quad t = a; a = b; b = t;
    const int to = oa; oa = ob; ob = to;
  }
  return true;
}

// closed-set intersection of a convex quad and the segment (x0, y0)-(x1, y1)
static __device__ __noinline__ bool quad_intersects_segment(Quad q, int o, double x0, double y0, double x1,
                                                     double y1) {
  int pos = 0, neg = 0;
#pragma unroll 1
  for (int k = 0; k < 4; ++k) {
    if (orient_sign(q.x0, q.y0, q.x1, q.y1, x0, y0) * o < 0 &&
        orient_sign(q.x0, q.y0, q.x1, q.y1, x1, y1) * o < 0)
      return false;  // both end points strictly outside this edge
    const int sg = orient_sign(x0, y0, x1, y1, q.x0, q.y0);
    pos += sg > 0;
    neg += sg < 0;
    rotate(q);
  }
  return !(pos == 4 || neg == 4);  // corners strictly on one side of the segment's line
}

// Entity.get_bounding_box_points (reference entity/base.py:100-138)
SG_DEV void box_points(double x, double y, double h, double W, double L, double cx, double cy,
                       double out[8]) {
  double s, c;
  sincos(h, &s, &c);
  const double hx0 = cx - 0.5 * L, hx1 = cx + 0.5 * L;
  const double hy0 = cy + 0.5 * W, hy1 = cy - 0.5 * W;
  const double px[4] = {hx0, hx1, hx1, hx0};
  const double py[4] = {hy0, hy0, hy1, hy1};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    out[2 * i] = x + (px[i] * c + py[i] * -s);
    out[2 * i + 1] = y + (px[i] * s + py[i] * c);
  }
}

SG_DEV double norm2(double a, double b) { return sqrt(a * a + b * b); }
SG_DEV double norm3(double a, double b, double c) { return sqrt(a * a + b * b + c * c); }
SG_DEV double dot2(double a0, double a1, double b0, double b1) { return a0 * b0 + a1 * b1; }
SG_DEV double py_max(double a, double b) { return b > a ? b : a; }
SG_DEV double py_min(double a, double b) { return b < a ? b : a; }
SG_DEV double np_sign(double v) { return v > 0 ? 1.0 : (v < 0 ? -1.0 : (v == 0 ? 0.0 : NAN)); }
SG_DEV double np_clip(double v, double lo, double hi) { return fmin(fmax(v, lo), hi); }

// ----------------------------------------------------------------------------------
// RSS (reference metrics/rss/callback.py, rss_utils.py)
// ----------------------------------------------------------------------------------
SG_DEV void inverse_direction(const double v[2], double out[2]) {  // rss_utils.py:7-21
  const double n = norm2(v[1], v[0]);
  out[0] = v[1] / n;
  out[1] = -v[0] / n;
}

// ----------------------------------------------------------------------------------
// pedestrians
// ----------------------------------------------------------------------------------
// LineString(route).project(Point) (GEOS LengthIndexedLine semantics; reference
// pedestrian/agent.py:61)
SG_DEV double route_project(const double* __restrict__ xy, int R, double px, double py) {
  double best_d = INFINITY, best_s = 0.0, s0 = 0.0;
  for (int i = 0; i + 1 < R; ++i) {
    const double ax = __ldg(xy + 2 * i), ay = __ldg(xy + 2 * i + 1);
    const double bx = __ldg(xy + 2 * i + 2), by = __ldg(xy + 2 * i + 3);
    const double dx = bx - ax, dy = by - ay, seg2 = dx * dx + dy * dy, seglen = sqrt(seg2);
    const double r = seg2 == 0.0 ? 0.0 : ((px - ax) * dx + (py - ay) * dy) / seg2;
    double qx, qy, sl;
    if (r <= 0.0) { qx = ax; qy = ay; sl = 0.0; }
    else if (r >= 1.0) { qx = bx; qy = by; sl = seglen; }
    else { qx = ax + r * dx; qy = ay + r * dy; sl = r * seglen; }
    const double d = hypot(px - qx, py - qy);
    if (d < best_d) { best_d = d; best_s = s0 + sl; }
    s0 += seglen;
  }
  return best_s;
}

// ----------------------------------------------------------------------------------
// Road-network surfaces as polygon soups (SgScene.rn_*; reference road_network/road_network.py:
// 306-328 builds them with shapely's unary_union).  Restated semantics: a point is contained in a
// surface iff it is strictly inside one of its polygons (crossing parity over all rings of the
// polygon, decided with exact orientation signs; a point on a ring is on the boundary), and the
// nearest point of a surface to a point outside it is the nearest point on the polygons' rings.
// Knife-edge cases that GEOS' dissolved union would decide differently (points exactly on an edge
// shared by two polygons) are unpinned -- see DESIGN.md.
// ----------------------------------------------------------------------------------
// +1 strictly inside, 0 on the boundary, -1 outside
static __device__ __noinline__ int polygon_side(const double* __restrict__ edges, int64_t e0, int64_t e1, double px,
                                                double py) {
  bool inside = false;
  for (int64_t e = e0; e < e1; ++e) {
    const double ax = __ldg(edges + 4 * e), ay = __ldg(edges + 4 * e + 1);
    const double bx = __ldg(edges + 4 * e + 2), by = __ldg(edges + 4 * e + 3);
    const bool straddles = (ay > py) != (by > py);
    const bool in_box = px >= fmin(ax, bx) && px <= fmax(ax, bx) && py >= fmin(ay, by) && py <= fmax(ay, by);
    if (!straddles && !in_box) continue;
    const int o = orient_sign(ax, ay, bx, by, px, py);
    if (o == 0 && in_box) return 0;
    if (straddles && ((o > 0) == (by > ay))) inside = !inside;
  }
  return inside ? 1 : -1;
}

SG_DEV bool surface_has_area(const SgScene& sc, int n, int k) {
  if (!sc.rn_of || sc.n_networks <= 0) return false;
  const int r = sc.rn_of[n];
  return r >= 0 && sc.rn_has_area[3 * r + k] != 0;
}

// shapely: surface.contains(Point(px, py))
static __device__ __noinline__ bool surface_contains(const SgScene sc, int n, int k, double px, double py) {
  if (!sc.rn_of || sc.n_networks <= 0) return false;
  const int r = sc.rn_of[n];
  if (r < 0) return false;
  for (int64_t q = sc.rn_poly_off[3 * r + k]; q < sc.rn_poly_off[3 * r + k + 1]; ++q)
    if (polygon_side(sc.rn_edges, sc.rn_edge_off[q], sc.rn_edge_off[q + 1], px, py) > 0) return true;
  return false;
}

// The closest point to (px, py) on the rings of polygons [q0, q1) (GEOS LineSegment::closestPoint:
// projection factor r = ((p - a).(b - a)) / |b - a|^2, the projection for 0 < r < 1, else the closer end
// point); best_d2 gets its squared distance.  No ring: (px, py) and INFINITY.
SG_DEV double2 ring_nearest(const SgScene& sc, int64_t q0, int64_t q1, double px, double py, double& best_d2) {
  double2 best = make_double2(px, py);
  best_d2 = INFINITY;
  for (int64_t e = sc.rn_edge_off[q0]; e < sc.rn_edge_off[q1]; ++e) {
    const double ax = __ldg(sc.rn_edges + 4 * e), ay = __ldg(sc.rn_edges + 4 * e + 1);
    const double bx = __ldg(sc.rn_edges + 4 * e + 2), by = __ldg(sc.rn_edges + 4 * e + 3);
    const double dx = bx - ax, dy = by - ay, len2 = dx * dx + dy * dy;
    double cx = ax, cy = ay;
    if (len2 > 0.0) {
      const double f = ((px - ax) * dx + (py - ay) * dy) / len2;
      if (f > 0.0 && f < 1.0) { cx = ax + f * dx; cy = ay + f * dy; }
      else {
        const double da = (px - ax) * (px - ax) + (py - ay) * (py - ay);
        const double db = (px - bx) * (px - bx) + (py - by) * (py - by);
        if (db < da) { cx = bx; cy = by; }
      }
    }
    const double d2 = (px - cx) * (px - cx) + (py - cy) * (py - cy);
    if (d2 < best_d2) { best_d2 = d2; best = make_double2(cx, cy); }
  }
  return best;
}

// shapely.ops.nearest_points(surface, Point(px, py))[0]: the point itself when it lies in the
// (closed) surface, else the closest point on a ring
static __device__ __noinline__ double2 surface_nearest(const SgScene sc, int n, int k, double px, double py) {
  const int r = sc.rn_of[n];
  const int64_t q0 = sc.rn_poly_off[3 * r + k], q1 = sc.rn_poly_off[3 * r + k + 1];
  for (int64_t q = q0; q < q1; ++q)
    if (polygon_side(sc.rn_edges, sc.rn_edge_off[q], sc.rn_edge_off[q + 1], px, py) >= 0)
      return make_double2(px, py);
  double d2;
  return ring_nearest(sc, q0, q1, px, py, d2);
}

// SocialForce._force_boundary (pedestrian/social_force.py:190-211) for surface k
SG_DEV void boundary_force(const SgScene& sc, int n, int k, double px, double py, double U, double R, double out[2]) {
  const double2 c = surface_nearest(sc, n, k, px, py);
  const double r0 = px - c.x, r1 = py - c.y;
  const double rn = sqrt(r0 * r0 + r1 * r1);
  const double u0 = r0 / (rn + 0.0000000001), u1 = r1 / (rn + 0.0000000001);
  const double ex = exp(-rn / R);
  out[0] = U / R * u0 * ex;
  out[1] = U / R * u1 * ex;
}

// ----------------------------------------------------------------------------------
// SocialForce noise (SgParams.sf_std_*): two independent N(0, 1) values as a pure function of
// (seed, slot index, tick) -- splitmix64 of the counter, Box-Muller on the two 53-bit uniforms.
// Engine-defined (the reference draws from numpy's global generator: not reproducible by design).
// ----------------------------------------------------------------------------------
SG_DEV uint64_t sg_splitmix64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ULL;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  return z ^ (z >> 31);
}
// the stream's first splitmix64 value for the key (seed, i, tick)
SG_DEV uint64_t sg_noise_key(uint64_t seed, int64_t i, int tick) {
  return sg_splitmix64(seed ^ sg_splitmix64((uint64_t)i * 0x9E3779B97F4A7C15ULL + (uint64_t)(unsigned)tick));
}
static __device__ __noinline__ double2 sg_noise2(uint64_t seed, int64_t i, int tick) {
  const uint64_t a = sg_noise_key(seed, i, tick);
  const uint64_t b = sg_splitmix64(a);
  const double u1 = ((double)(a >> 11) + 1.0) * (1.0 / 9007199254740992.0);  // (0, 1]
  const double u2 = (double)(b >> 11) * (1.0 / 9007199254740992.0);          // [0, 1)
  const double r = sqrt(-2.0 * log(u1));
  double sn, cs;
  sincos(2.0 * M_PI * u2, &sn, &cs);
  return make_double2(r * cs, r * sn);
}
// a uniform in [0, 1) from the same key: (a >> 11) * 2^-53, a the value sg_noise2 starts from
SG_DEV double sg_uniform(uint64_t seed, int64_t i, int tick) {
  return (double)(sg_noise_key(seed, i, tick) >> 11) * (1.0 / 9007199254740992.0);
}
