// gik_table.h -- host side: validate a gik_table_t (the flattened pinocchio model, include/gik.h) and derive
// the constants of the compiled fast path (gik::DevTable<T>).  Plain C++17, no CUDA.
#pragma once
#include <math.h>
#include <string.h>

#include "../../include/gik.h"
#include "gik_core.cuh"
#include "gik_collide.cuh"

namespace gik {

inline bool is_identity3(const double* R, double tol = 1e-12) {
  for (int i = 0; i < 9; ++i)
    if (fabs(R[i] - ((i % 4 == 0) ? 1.0 : 0.0)) > tol) return false;
  return true;
}

// Limits are rounded INWARD when narrowed to T, so a clamped fp32 q never violates the fp64 limits
// (tools.jointlimitsviolated, tools.py:17-19, tests q against the double-precision limits).
template <typename T> inline T narrow_lo(double x) {
  T v = (T)x;
  if ((double)v < x) v = (T)nextafter(v, (T)INFINITY);
  return v;
}
template <typename T> inline T narrow_hi(double x) {
  T v = (T)x;
  if ((double)v > x) v = (T)nextafter(v, (T)-INFINITY);
  return v;
}

// Generic checks: a tree of 1-dof revolute joints with parents listed first.
inline int validate_table(const gik_table_t& t) {
  if (t.nq < 1 || t.nq > GIK_MAX_NQ) return GIK_E_MODEL;
  for (int i = 0; i < t.nq; ++i) {
    if (t.parent[i] < -1 || t.parent[i] >= i) return GIK_E_MODEL;
    if (t.axis[i] < 0 || t.axis[i] > 2) return GIK_E_MODEL;
    if (!(t.lower[i] <= t.upper[i])) return GIK_E_MODEL;
  }
  for (int h = 0; h < 2; ++h)
    if (t.hand_joint[h] < 0 || t.hand_joint[h] >= t.nq) return GIK_E_MODEL;
  return GIK_OK;
}

// Fast-path structure: both hands hang off 6-joint arms (axes z y y x y z, translation-only joint
// placements) that share exactly one root joint (axis z, parent = universe).
template <typename T>
inline int build_dev_table(const gik_table_t& t, DevTable<T>& d) {
  int rc = validate_table(t);
  if (rc != GIK_OK) return rc;
  memset(&d, 0, sizeof(d));
  int chain[2][7];
  for (int h = 0; h < 2; ++h) {
    int k = t.hand_joint[h];
    for (int c = 6; c >= 0; --c) {
      if (k < 0) return GIK_E_TOPOLOGY;
      chain[h][c] = k;
      k = t.parent[k];
    }
    if (k != -1) return GIK_E_TOPOLOGY;  // chain longer than 7
    for (int c = 0; c < 7; ++c) {
      const int j = chain[h][c];
      if (t.axis[j] != chain_axis(c)) return GIK_E_TOPOLOGY;
      if (!is_identity3(t.joint_R[j])) return GIK_E_TOPOLOGY;
    }
  }
  if (chain[0][0] != chain[1][0]) return GIK_E_TOPOLOGY;
  for (int a = 1; a < 7; ++a)
    for (int b = 1; b < 7; ++b)
      if (chain[0][a] == chain[1][b]) return GIK_E_TOPOLOGY;

  d.nq = t.nq;
  bool active[GIK_MAX_NQ] = {false};
  for (int h = 0; h < 2; ++h) {
    ArmConst<T>& ac = d.arm[h];
    for (int c = 0; c < 7; ++c) {
      const int j = chain[h][c];
      for (int i = 0; i < 3; ++i) ac.t[c][i] = (T)t.joint_p[j][i];
      const int slot = (c == 0) ? 0 : h * 6 + c;
      d.act_q[slot] = j;
      d.lo[slot] = narrow_lo<T>(t.lower[j]);
      d.hi[slot] = narrow_hi<T>(t.upper[j]);
      active[j] = true;
    }
    // inverse of the hand frame offset: (R, p)^-1 = (R^T, -R^T p)
    const double* R = t.hand_R[h];
    const double* p = t.hand_p[h];
    for (int r = 0; r < 3; ++r) {
      for (int c = 0; c < 3; ++c) ac.finv_R[3 * r + c] = (T)R[3 * c + r];
      ac.finv_p[r] = (T)(-(R[r] * p[0] + R[3 + r] * p[1] + R[6 + r] * p[2]));
    }
    {  // constant LOCAL Jacobian column of the tip joint: linear part = finv_p x finv_R[:, axis]
      const int ax = chain_axis(6);
      double fi_R[9], fi_p[3];
      for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 3; ++c) fi_R[3 * r + c] = R[3 * c + r];
        fi_p[r] = -(R[r] * p[0] + R[3 + r] * p[1] + R[6 + r] * p[2]);
      }
      const double av[3] = {fi_R[ax], fi_R[3 + ax], fi_R[6 + ax]};
      ac.tip_lin[0] = (T)(fi_p[1] * av[2] - fi_p[2] * av[1]);
      ac.tip_lin[1] = (T)(fi_p[2] * av[0] - fi_p[0] * av[2]);
      ac.tip_lin[2] = (T)(fi_p[0] * av[1] - fi_p[1] * av[0]);
      // the tip column as the kernels see it (rounded to T), and its outer product
      const double col[6] = {(double)ac.tip_lin[0], (double)ac.tip_lin[1], (double)ac.tip_lin[2],
                             (double)(T)av[0], (double)(T)av[1], (double)(T)av[2]};
      for (int i = 0; i < 6; ++i)
        for (int j = 0; j <= i; ++j) ac.g6[i * (i + 1) / 2 + j] = (T)(col[i] * col[j]);
      // wrist centre in the hand frame: the tip joint's origin moved back along the tip axis by its own placement
      // (t[6] = (0, 0, z) on spherical-wrist tables; unused otherwise)
      const double tz = t.joint_p[chain[h][6]][2];
      for (int i = 0; i < 3; ++i) ac.rw[i] = (T)(fi_p[i] - tz * av[i]);
    }
    ac.tip_psi = (T)atan2(R[1], R[0]);       // finv_R = R^T = Rot(z, psi) when the hand frame is tip-aligned (kTipZ below)
    for (int i = 0; i < 9; ++i) ac.hook_R[i] = (T)t.hook_R[h][i];
    for (int i = 0; i < 3; ++i) ac.hook_p[i] = (T)t.hook_p[h][i];
  }
  d.tzero = 0;
  for (int c = 0; c < 7; ++c)
    for (int i = 0; i < 3; ++i)
      if (t.joint_p[chain[0][c]][i] == 0.0 && t.joint_p[chain[1][c]][i] == 0.0) d.tzero |= 1u << (3 * c + i);
  {  // tip-aligned hand frames: both hand rotations are rotations about z, the tip joint's axis
    static_assert(chain_axis(6) == 2, "kTipZ assumes a z tip axis");
    bool tipz = true;
    for (int h = 0; h < 2; ++h) {
      const double* R = t.hand_R[h];
      tipz = tipz && R[2] == 0.0 && R[5] == 0.0 && R[6] == 0.0 && R[7] == 0.0 && R[8] == 1.0 &&
             fabs(R[0] - R[4]) < 1e-12 && fabs(R[1] + R[3]) < 1e-12 && fabs(R[0] * R[0] + R[1] * R[1] - 1.0) < 1e-12;
    }
    if (tipz) d.tzero |= kTipZ;
  }
  for (int j = 0; j < t.nq; ++j) {
    d.qlo[j] = narrow_lo<T>(t.lower[j]);
    d.qhi[j] = narrow_hi<T>(t.upper[j]);
    if (!active[j]) d.passive_q[d.n_passive++] = j;
  }
  return GIK_OK;
}

// (left, right)-packed constants for the fp32 packed lane kernel
inline void build_packed_table(const DevTable<float>& d, PackedTable& p) {
  const ArmConst<float>&L = d.arm[0], &R = d.arm[1];
  for (int k = 0; k < 7; ++k)
    for (int i = 0; i < 3; ++i) p.arm.t[k][i] = F2(L.t[k][i], R.t[k][i]);
  for (int i = 0; i < 9; ++i) { p.arm.finv_R[i] = F2(L.finv_R[i], R.finv_R[i]); p.arm.hook_R[i] = F2(L.hook_R[i], R.hook_R[i]); }
  for (int i = 0; i < 21; ++i) p.arm.g6[i] = F2(L.g6[i], R.g6[i]);
  for (int i = 0; i < 3; ++i) {
    p.arm.finv_p[i] = F2(L.finv_p[i], R.finv_p[i]);
    p.arm.tip_lin[i] = F2(L.tip_lin[i], R.tip_lin[i]);
    p.arm.hook_p[i] = F2(L.hook_p[i], R.hook_p[i]);
    p.arm.rw[i] = F2(L.rw[i], R.rw[i]);
  }
  p.arm.tip_psi = F2(L.tip_psi, R.tip_psi);
  for (int k = 0; k < 6; ++k) { p.lo[k] = F2(d.lo[1 + k], d.lo[7 + k]); p.hi[k] = F2(d.hi[1 + k], d.hi[7 + k]); }
  p.lo0 = d.lo[0]; p.hi0 = d.hi[0];
}

// ---- collision scene (gik_scene_t -> DevScene<T>) ----
inline int validate_scene(const gik_table_t& t, const gik_scene_t& s) {
  if (s.n_geoms < 1 || s.n_geoms > GIK_MAX_GEOMS || s.n_pairs < 0 || s.n_pairs > GIK_MAX_PAIRS) return GIK_E_SIZE;
  for (int g = 0; g < s.n_geoms; ++g) {
    if (s.geoms[g].type < 0 || s.geoms[g].type > 2 || s.geoms[g].joint < -1 || s.geoms[g].joint >= t.nq) return GIK_E_MODEL;
    if (!(s.geoms[g].size[0] > 0.0)) return GIK_E_MODEL;
  }
  for (int k = 0; k < s.n_pairs; ++k)
    if (s.pair_a[k] >= s.n_geoms || s.pair_b[k] >= s.n_geoms) return GIK_E_MODEL;
  const int special[3] = {s.cube_geom, s.table_geom, s.obstacle_geom};
  for (int k = 0; k < 3; ++k)
    if (special[k] < -1 || special[k] >= s.n_geoms) return GIK_E_MODEL;
  return GIK_OK;
}


template <typename T>
inline void fill_dev_scene(const gik_table_t& t, const gik_scene_t& s, DevScene<T>& d) {
  memset(&d, 0, sizeof(d));
  d.tree.nq = t.nq;
  for (int i = 0; i < t.nq; ++i) {
    d.tree.parent[i] = t.parent[i];
    d.tree.depth[i] = t.parent[i] < 0 ? 0 : d.tree.depth[t.parent[i]] + 1;     // parents are listed first
    if (d.tree.depth[i] > d.tree.max_depth) d.tree.max_depth = d.tree.depth[i];
    d.tree.axis[i] = t.axis[i];
    for (int k = 0; k < 9; ++k) d.tree.jR[i][k] = (T)t.joint_R[i][k];
    for (int k = 0; k < 3; ++k) d.tree.jp[i][k] = (T)t.joint_p[i][k];
  }
  d.n_geoms = s.n_geoms;
  d.cube_geom = s.cube_geom;
  for (int g = 0; g < s.n_geoms; ++g) {
    DevGeom<T>& G = d.g[g];
    for (int k = 0; k < 9; ++k) G.R[k] = (T)s.geoms[g].R[k];
    for (int k = 0; k < 3; ++k) G.p[k] = (T)s.geoms[g].p[k];
    G.s0 = (T)s.geoms[g].size[0]; G.s1 = (T)s.geoms[g].size[1]; G.s2 = (T)s.geoms[g].size[2];
    G.type = s.geoms[g].type; G.joint = s.geoms[g].joint;
    const double a = s.geoms[g].size[0], b = s.geoms[g].size[1], c = s.geoms[g].size[2];
    const double r = G.type == GIK_GEOM_BOX ? sqrt(a * a + b * b + c * c) : G.type == GIK_GEOM_SPHERE ? a : sqrt(a * a + b * b);
    G.bound = (T)(r * (1.0 + 1e-6));
  }
}

// ---- the pair lists of a scene: each collision query scans one of them ----
enum PairList {
  kListAll = 0,    // every pair of the scene: collision(q)
  kListEnv = 1,    // the pairs whose second geometry is the table or the obstacle: distanceToObstacle, clearance
  kListCube = 2,   // the cube against the table and the obstacle: the cube-only test
  kListTraj = 3,   // the trajectory check's pairs (gik_traj.cuh)
  kNumPairLists = 4
};
constexpr int kPairListCap = GIK_MAX_PAIRS + 2;   // kListTraj: at most every pair plus the cube's two own pairs

struct PairLists {
  uint8_t pairs[kNumPairLists][2][kPairListCap];   // pair k of list l: (pairs[l][0][k], pairs[l][1][k])
  int32_t n[kNumPairLists];
};

// The scene must have passed validate_scene.
inline void build_pair_lists(const gik_table_t& t, const gik_scene_t& s, PairLists& L) {
  memset(&L, 0, sizeof(L));
  auto add = [&](int l, int a, int b) {
    L.pairs[l][0][L.n[l]] = (uint8_t)a;
    L.pairs[l][1][L.n[l]++] = (uint8_t)b;
  };
  for (int k = 0; k < s.n_pairs; ++k) {
    const int a = s.pair_a[k], b = s.pair_b[k];
    add(kListAll, a, b);
    if (b == s.table_geom || b == s.obstacle_geom) add(kListEnv, a, b);          // tools.py:42
  }
  const int env[2] = {s.table_geom, s.obstacle_geom};                            // setup_pinocchio.py:66-70
  for (int e : env)
    if (e >= 0 && s.cube_geom >= 0) add(kListCube, e, s.cube_geom);
  // kListTraj: kListAll without the pairs of the cube with a geometry on either hand joint -- the grasp error judges
  // that contact, GJK would only measure the millimetre between the fingers and the cube -- plus the pairs of kListCube
  // that kListAll lacks
  auto on_hand = [&](int g) { return s.geoms[g].joint == t.hand_joint[0] || s.geoms[g].joint == t.hand_joint[1]; };
  for (int k = 0; k < L.n[kListAll]; ++k) {
    const int a = L.pairs[kListAll][0][k], b = L.pairs[kListAll][1][k];
    if ((a == s.cube_geom && on_hand(b)) || (b == s.cube_geom && on_hand(a))) continue;
    add(kListTraj, a, b);
  }
  for (int k = 0; k < L.n[kListCube]; ++k) {
    const int a = L.pairs[kListCube][0][k], b = L.pairs[kListCube][1][k];
    const uint8_t* ta = L.pairs[kListTraj][0];
    const uint8_t* tb = L.pairs[kListTraj][1];
    bool listed = false;
    for (int j = 0; j < L.n[kListTraj] && !listed; ++j) listed = (ta[j] == a && tb[j] == b) || (ta[j] == b && tb[j] == a);
    if (!listed) add(kListTraj, a, b);
  }
}

}  // namespace gik
