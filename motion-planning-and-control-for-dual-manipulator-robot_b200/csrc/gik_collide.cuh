// gik_collide.cuh -- convex-pair intersection for the batched collision(q) / distanceToObstacle(q) kernels.
// Compiles for the device (nvcc) and, for the CPU unit tests under tests/hostsim only, as plain C++17.
//
// Reference semantics (tools.py:25-51): hpp-fcl tests every collision pair of boxes / spheres / cylinders (and the
// cube mesh, here its solid box) for intersection; `collision` is "any pair intersects", `distanceToObstacle` the
// minimum pair distance.  All shapes are convex, so one boolean GJK over support mappings covers every pair type;
// "distance >= m" is decided as "shape A inflated by m does not intersect shape B" (no distance sub-algorithm).
#pragma once
#include "gik_core.cuh"

#ifndef GIK_MAX_GEOMS
#define GIK_MAX_GEOMS 64
#endif

namespace gik {

enum { GEOM_BOX = 0, GEOM_SPHERE = 1, GEOM_CYLINDER = 2 };

template <typename T> struct V3 { T x, y, z; };
template <typename T> GIK_HD V3<T> operator+(V3<T> a, V3<T> b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
template <typename T> GIK_HD V3<T> operator-(V3<T> a, V3<T> b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
template <typename T> GIK_HD V3<T> operator-(V3<T> a) { return {-a.x, -a.y, -a.z}; }
template <typename T> GIK_HD V3<T> operator*(T s, V3<T> a) { return {s * a.x, s * a.y, s * a.z}; }
template <typename T> GIK_HD T dot(V3<T> a, V3<T> b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
template <typename T> GIK_HD V3<T> cross(V3<T> a, V3<T> b) {
  return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};
}
// (a x b) x c
template <typename T> GIK_HD V3<T> triple(V3<T> a, V3<T> b, V3<T> c) { return cross(cross(a, b), c); }

// A placed convex shape: world rotation (row-major), world position, type and size
// (box: half extents | sphere: radius | cylinder: radius, half length along local z).
template <typename T>
struct Shape {
  T R[9];
  V3<T> p;
  T s0, s1, s2;
  int type;
};

// support point of the shape in world direction d (farthest point along d)
template <typename T>
GIK_HD V3<T> support(const Shape<T>& S, V3<T> d) {
  const V3<T> l = {S.R[0] * d.x + S.R[3] * d.y + S.R[6] * d.z, S.R[1] * d.x + S.R[4] * d.y + S.R[7] * d.z,
                   S.R[2] * d.x + S.R[5] * d.y + S.R[8] * d.z};   // R^T d
  V3<T> s;
  if (S.type == GEOM_BOX) {
    s = {l.x >= T(0) ? S.s0 : -S.s0, l.y >= T(0) ? S.s1 : -S.s1, l.z >= T(0) ? S.s2 : -S.s2};
  } else if (S.type == GEOM_SPHERE) {
    const T n2 = dot(l, l);
    const T k = n2 > T(0) ? S.s0 * rsqrt_(n2) : T(0);
    s = {k * l.x, k * l.y, k * l.z};
  } else {
    const T r2 = l.x * l.x + l.y * l.y;
    const T k = r2 > T(1e-30) ? S.s0 * rsqrt_(r2) : T(0);
    s = {k * l.x, k * l.y, l.z >= T(0) ? S.s1 : -S.s1};
  }
  return {S.p.x + S.R[0] * s.x + S.R[1] * s.y + S.R[2] * s.z, S.p.y + S.R[3] * s.x + S.R[4] * s.y + S.R[5] * s.z,
          S.p.z + S.R[6] * s.x + S.R[7] * s.y + S.R[8] * s.z};
}

// support of the Minkowski difference (A inflated by `margin`) - B
template <typename T>
GIK_HD V3<T> support_diff(const Shape<T>& A, const Shape<T>& B, V3<T> d, T margin) {
  V3<T> s = support(A, d) - support(B, -d);
  if (margin > T(0)) {
    const T n2 = dot(d, d);
    if (n2 > T(0)) s = s + (margin * rsqrt_(n2)) * d;
  }
  return s;
}

// radius of the bounding sphere centred at the shape's position
template <typename T>
GIK_HD T bound_radius(int type, T s0, T s1, T s2) {
  if (type == GEOM_BOX) return sqrt_(s0 * s0 + s1 * s1 + s2 * s2);
  if (type == GEOM_SPHERE) return s0;
  return sqrt_(s0 * s0 + s1 * s1);
}

// Boolean GJK: does (A inflated by margin) intersect B?  Simplex points are kept newest-first (a, b, c, d).
// Touching (origin on the simplex boundary within round-off) and an exhausted iteration budget count as intersecting.
template <typename T>
GIK_HD bool gjk_intersect(const Shape<T>& A, const Shape<T>& B, T margin) {
  const T kTiny = sizeof(T) == 4 ? T(1e-14) : T(1e-28);   // squared-length floor of a search direction
  V3<T> dir = B.p - A.p;
  if (dot(dir, dir) < kTiny) dir = {T(1), T(0), T(0)};
  V3<T> a = support_diff(A, B, dir, margin), b = a, c = a, d = a;
  int n = 1;
  dir = -a;
  for (int iter = 0; iter < 48; ++iter) {
    if (dot(dir, dir) < kTiny) return true;                 // origin lies on the current simplex
    const V3<T> w = support_diff(A, B, dir, margin);
    if (dot(w, dir) < T(0)) return false;                   // the difference does not reach past the origin along dir
    d = c; c = b; b = a; a = w; ++n;                        // push front
    const V3<T> ao = -a;
    if (n == 2) {
      const V3<T> ab = b - a;
      if (dot(ab, ao) > T(0)) dir = triple(ab, ao, ab);
      else { n = 1; dir = ao; }
      continue;
    }
    if (n == 4) {
      const V3<T> ab = b - a, ac = c - a, ad = d - a;
      const V3<T> abc = cross(ab, ac), acd = cross(ac, ad), adb = cross(ad, ab);
      if (dot(abc, ao) > T(0)) { n = 3; }                                   // keep (a, b, c)
      else if (dot(acd, ao) > T(0)) { b = c; c = d; n = 3; }                // (a, c, d)
      else if (dot(adb, ao) > T(0)) { const V3<T> t = b; b = d; c = t; n = 3; }   // (a, d, b)
      else return true;                                                     // origin inside the tetrahedron
    }
    // n == 3: triangle (a, b, c)
    {
      const V3<T> ab = b - a, ac = c - a;
      const V3<T> abc = cross(ab, ac);
      bool edge_ab = false;
      if (dot(cross(abc, ac), ao) > T(0)) {
        if (dot(ac, ao) > T(0)) { b = c; n = 2; dir = triple(ac, ao, ac); }
        else edge_ab = true;
      } else if (dot(cross(ab, abc), ao) > T(0)) {
        edge_ab = true;
      } else {
        const T h = dot(abc, ao);
        if (h > T(0)) dir = abc;
        else if (h < T(0)) { const V3<T> t = b; b = c; c = t; dir = -abc; }
        else return true;                                                   // origin in the triangle's plane, inside
      }
      if (edge_ab) {
        if (dot(ab, ao) > T(0)) { n = 2; dir = triple(ab, ao, ab); }
        else { n = 1; dir = ao; }
      }
    }
  }
  return true;
}

// ---------------------------------------------------------------------------------------------------------------
// Generic forward kinematics of the whole tree (pin.updateGeometryPlacements needs every joint, head included):
// oMi[i] = oMi[parent] * jointPlacement[i] * Rot(axis_i, q_i).  M is stored as 12 values (R row-major, p).
// ---------------------------------------------------------------------------------------------------------------
template <typename T>
struct TreeConst {
  int32_t nq;
  int32_t max_depth;               // depth of the deepest joint (root joints have depth 0)
  int32_t parent[GIK_MAX_NQ];
  int32_t depth[GIK_MAX_NQ];
  int32_t axis[GIK_MAX_NQ];
  T jR[GIK_MAX_NQ][9];
  T jp[GIK_MAX_NQ][3];
};

template <typename T>
GIK_HD void se3_mul12(const T* A, const T* B, T* C) {   // C = A * B
#pragma unroll
  for (int r = 0; r < 3; ++r) {
#pragma unroll
    for (int c = 0; c < 3; ++c) C[3 * r + c] = A[3 * r] * B[c] + A[3 * r + 1] * B[3 + c] + A[3 * r + 2] * B[6 + c];
    C[9 + r] = A[9 + r] + A[3 * r] * B[9] + A[3 * r + 1] * B[10] + A[3 * r + 2] * B[11];
  }
}

// world placement of joint i given its parent's (par = nullptr for the universe) and q_i
template <typename T>
GIK_HD void joint_placement(const TreeConst<T>& tc, int i, const T* par, T qi, T* out) {
  T L[12], s, c;
  sincos_<false>(qi, s, c);
  const int ax = tc.axis[i], I = (ax + 1) % 3, J = (ax + 2) % 3;
  // jointPlacement * Rot(axis, q): columns I, J of jR are rotated
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const T bi = tc.jR[i][3 * r + I], bj = tc.jR[i][3 * r + J];
    L[3 * r + ax] = tc.jR[i][3 * r + ax];
    L[3 * r + I] = c * bi + s * bj;
    L[3 * r + J] = -s * bi + c * bj;
    L[9 + r] = tc.jp[i][r];
  }
  if (par) se3_mul12(par, L, out);
  else {
#pragma unroll
    for (int k = 0; k < 12; ++k) out[k] = L[k];
  }
}

template <typename T>
struct DevGeom { T R[9], p[3], s0, s1, s2, bound; int32_t type, joint; };

template <typename T>
struct DevScene {
  TreeConst<T> tree;
  int32_t n_geoms, cube_geom;
  DevGeom<T> g[GIK_MAX_GEOMS];
};

template <typename T>
GIK_HD Shape<T> make_shape(const DevGeom<T>& g, const T* M) {
  Shape<T> S;
#pragma unroll
  for (int k = 0; k < 9; ++k) S.R[k] = M[k];
  S.p = {M[9], M[10], M[11]};
  S.s0 = g.s0; S.s1 = g.s1; S.s2 = g.s2; S.type = g.type;
  return S;
}

// World placement of geometry g: oMi[joint] * placement (pin.updateGeometryPlacements).  The cube takes the problem's
// pose cube[k * ld + i], k < 12 (cube = nullptr: the scene's own).  oMi = nullptr (no configuration): every geometry
// keeps its placement in its joint's frame.
template <typename T>
GIK_HD void place_geom(const DevScene<T>* sc, int g, const T* cube, int64_t ld, int64_t i, const T (*oMi)[12], T* out) {
  const DevGeom<T>& G = sc->g[g];
  T P[12];
  if (g == sc->cube_geom && cube) {
#pragma unroll
    for (int k = 0; k < 12; ++k) P[k] = cube[k * ld + i];
  } else {
#pragma unroll
    for (int k = 0; k < 9; ++k) P[k] = G.R[k];
    P[9] = G.p[0]; P[10] = G.p[1]; P[11] = G.p[2];
  }
  if (G.joint >= 0 && oMi) se3_mul12(&oMi[G.joint][0], P, out);
  else {
#pragma unroll
    for (int k = 0; k < 12; ++k) out[k] = P[k];
  }
}

// The shape ERODED by `shrink` (the points whose shrink-ball lies inside it): box -> smaller box, sphere -> smaller
// sphere, cylinder -> thinner and shorter cylinder.  Returns false when nothing is left.
template <typename T>
GIK_HD bool erode_shape(Shape<T>& S, T shrink) {
  S.s0 -= shrink;
  if (S.type != GEOM_SPHERE) S.s1 -= shrink;
  if (S.type == GEOM_BOX) S.s2 -= shrink;
  return S.s0 > T(0) && (S.type == GEOM_SPHERE || S.s1 > T(0)) && (S.type != GEOM_BOX || S.s2 > T(0));
}

// smallest half extent of a shape: how much erosion it survives
template <typename T>
GIK_HD T min_extent(const Shape<T>& S) {
  if (S.type == GEOM_SPHERE) return S.s0;
  if (S.type == GEOM_BOX) return min_(S.s0, min_(S.s1, S.s2));
  return min_(S.s0, S.s1);
}

// Narrow phase of one pair.  margin >= 0: does (A inflated by margin) intersect B  (collision: 0; clearance: the
// threshold).  margin < 0: does the THICKER of the two solids, eroded by |margin|, still intersect the other one -- a
// PERSISTENT collision: a point x of that intersection has its |margin|-ball inside the eroded solid's original, so the
// two solids keep intersecting under any relative displacement of their points of at most |margin| (used to settle the
// reference's keep-descending-while-colliding tail without testing every iterate, gik_collide_impl.cuh).
template <typename T>
GIK_HD bool narrow_hits(const DevGeom<T>& ga, const T* Ma, const DevGeom<T>& gb, const T* Mb, T margin) {
  Shape<T> A = make_shape(ga, Ma), B = make_shape(gb, Mb);
  if (margin < T(0)) {
    const bool a_thicker = min_extent(A) >= min_extent(B);
    if (!erode_shape(a_thicker ? A : B, -margin)) return false;
    return gjk_intersect(A, B, T(0));
  }
  return gjk_intersect(A, B, margin);
}

// pair (a, b) with world placements Ma, Mb: bounding spheres, then GJK
template <typename T>
GIK_HD bool pair_hits(const DevGeom<T>& ga, const T* Ma, const DevGeom<T>& gb, const T* Mb, T margin) {
  const T dx = Ma[9] - Mb[9], dy = Ma[10] - Mb[10], dz = Ma[11] - Mb[11];
  const T reach = ga.bound + gb.bound + max_(margin, T(0));
  if (dx * dx + dy * dy + dz * dz > reach * reach) return false;
  return narrow_hits(ga, Ma, gb, Mb, margin);
}

}  // namespace gik
