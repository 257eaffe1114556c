// hostsim.cpp -- TEST INFRASTRUCTURE.  Compiles the device arithmetic of csrc/gik_core.cuh as plain C++ so the
// `-m "not gpu"` tests can check the kernel math (fp32 and fp64) against the oracle without a GPU.  It is not
// part of the product: the package never loads this library and there is no CPU fallback.
// Same SoA layouts as include/gik.h, host pointers.
#include <stdint.h>
#include <stdlib.h>

#include "../../motion-planning-and-control-for-dual-manipulator-robot_b200/csrc/gik_table.h"

using namespace gik;

template <typename T>
static int fk_impl(const gik_table_t* tab, int64_t n, const T* q, T* frames) {
  DevTable<T> d;
  int rc = build_dev_table<T>(*tab, d);
  if (rc) return rc;
  for (int64_t i = 0; i < n; ++i) {
    T qa[kActive], fr[2][12];
    for (int a = 0; a < kActive; ++a) qa[a] = q[(int64_t)d.act_q[a] * n + i];
    fk_frames<T, true>(d, qa, fr);
    for (int h = 0; h < 2; ++h)
      for (int c = 0; c < 12; ++c) frames[((int64_t)h * 12 + c) * n + i] = fr[h][c];
  }
  return 0;
}

template <typename T>
static int jac_impl(const gik_table_t* tab, int64_t n, const T* q, T* jac) {
  DevTable<T> d;
  int rc = build_dev_table<T>(*tab, d);
  if (rc) return rc;
  const int nq = d.nq;
  for (int64_t i = 0; i < n; ++i) {
    T qa[kActive], A[2][6][7];
    for (int a = 0; a < kActive; ++a) qa[a] = q[(int64_t)d.act_q[a] * n + i];
    frame_jacobians<T, true>(d, qa, A[0], A[1]);
    for (int h = 0; h < 2; ++h)
      for (int r = 0; r < 6; ++r) {
        for (int j = 0; j < nq; ++j) jac[(((int64_t)h * 6 + r) * nq + j) * n + i] = T(0);
        for (int k = 0; k < 7; ++k) {
          const int slot = k == 0 ? 0 : h * 6 + k;
          jac[(((int64_t)h * 6 + r) * nq + d.act_q[slot]) * n + i] = A[h][r][k];
        }
      }
  }
  return 0;
}

template <typename T>
static int solve_impl(const gik_table_t* tab, int64_t n, const T* q_init, const T* pose,
                      const gik_params_t* prm, T* q_out, uint8_t* conv, int32_t* iters, T* resid) {
  DevTable<T> d;
  int rc = build_dev_table<T>(*tab, d);
  if (rc) return rc;
  const T eps2 = (T)(prm->eps * prm->eps), dt = (T)prm->dt, lambda = (T)prm->damping;
  const bool generic = (prm->flags & 1) != 0;   // test hook: force the TZ = 0 instantiation
  const bool no_wrist = (prm->flags & 2) != 0;  // test hook: keep the Cholesky step where the spherical-wrist step would run
  const bool packed = (prm->flags & 4) != 0;    // fp32 only: the packed (left, right) iteration of the fp32 lane kernel
  PackedTable pt;
  if constexpr (sizeof(T) == 4) build_packed_table(d, pt);
  for (int64_t i = 0; i < n; ++i) {
    T q[kActive], cube[12], tgt[2][12], dq[kActive], rL = 0, rR = 0;
    for (int a = 0; a < kActive; ++a) q[a] = q_init[(int64_t)d.act_q[a] * n + i];
    for (int c = 0; c < 12; ++c) cube[c] = pose[(int64_t)c * n + i];
    hook_target(d.arm[0], cube, tgt[0]);
    hook_target(d.arm[1], cube, tgt[1]);
    int it = 0;
    bool ok = false;
    for (;;) {
      // same specialisation rule as choose_launch() in csrc/gik_kernels.cu
      const bool nx = (d.tzero & kNextageTZ) == kNextageTZ && !generic;
      bool done_packed = false;
      if constexpr (sizeof(T) == 4) {
        if (packed) {
          F2 q2[6], tgt2[12], dq2[6];
          float dq0;
          for (int k = 0; k < 6; ++k) q2[k] = F2(q[1 + k], q[7 + k]);
          for (int c = 0; c < 12; ++c) tgt2[c] = F2(tgt[0][c], tgt[1][c]);
          if (nx && lambda == T(0) && !no_wrist) ik_iteration_packed<kNextageTZ, true>(pt, q[0], q2, tgt2, lambda, dq0, dq2, rL, rR);
          else if (nx) ik_iteration_packed<kNextageTZ, false>(pt, q[0], q2, tgt2, lambda, dq0, dq2, rL, rR);
          else ik_iteration_packed<0, false>(pt, q[0], q2, tgt2, lambda, dq0, dq2, rL, rR);
          dq[0] = dq0;
          for (int k = 0; k < 6; ++k) { dq[1 + k] = dq2[k].x; dq[7 + k] = dq2[k].y; }
          done_packed = true;
        }
      }
      if (done_packed) {}
      else if (nx && lambda == T(0) && !no_wrist) ik_iteration<T, true, kNextageTZ, true>(d, q, tgt, lambda, dq, rL, rR);
      else if (nx) ik_iteration<T, true, kNextageTZ>(d, q, tgt, lambda, dq, rL, rR);
      else ik_iteration<T, true, 0>(d, q, tgt, lambda, dq, rL, rR);
      ok = (rL < eps2) && (rR < eps2) && (it < prm->max_iters);
      if (ok || it >= prm->max_iters) break;
      apply_step(d, q, dq, dt);
      ++it;
    }
    for (int a = 0; a < kActive; ++a) q_out[(int64_t)d.act_q[a] * n + i] = q[a];
    for (int p = 0; p < d.n_passive; ++p) {
      const int j = d.passive_q[p];
      T v = q_init[(int64_t)j * n + i];
      if (it > 0) v = min_(max_(d.qlo[j], v), d.qhi[j]);
      q_out[(int64_t)j * n + i] = v;
    }
    conv[i] = ok ? 1 : 0;
    if (iters) iters[i] = it;
    if (resid) { resid[i] = sqrt_(rL); resid[n + i] = sqrt_(rR); }
  }
  return 0;
}

// collision predicate over one pair list (PairList: 0 all pairs, 1 table/obstacle pairs, 2 the cube's own pairs),
// sequential over pairs (the kernel deals the same pairs to the lanes of a warp)
template <typename T>
static int collide_impl(const gik_table_t* tab, const gik_scene_t* scn, int64_t n, const T* q, const T* cube, int list,
                        double margin, uint8_t* out) {
  if (list < 0 || list >= kNumPairLists) return GIK_E_PARAM;
  int rc = validate_table(*tab);
  if (rc == 0) rc = validate_scene(*tab, *scn);
  if (rc) return rc;
  static DevScene<T> sc;
  static PairLists L;
  fill_dev_scene(*tab, *scn, sc);
  build_pair_lists(*tab, *scn, L);
  const uint8_t *pa = L.pairs[list][0], *pb = L.pairs[list][1];
  for (int64_t i = 0; i < n; ++i) {
    T oMi[GIK_MAX_NQ][12], oMg[GIK_MAX_GEOMS][12];
    if (q)
      for (int j = 0; j < sc.tree.nq; ++j)
        joint_placement(sc.tree, j, sc.tree.parent[j] < 0 ? (const T*)nullptr : oMi[sc.tree.parent[j]], q[(int64_t)j * n + i], oMi[j]);
    for (int g = 0; g < sc.n_geoms; ++g) place_geom(&sc, g, cube, n, i, q ? oMi : nullptr, oMg[g]);
    bool hit = false;
    for (int k = 0; k < L.n[list] && !hit; ++k) hit = pair_hits(sc.g[pa[k]], oMg[pa[k]], sc.g[pb[k]], oMg[pb[k]], (T)margin);
    out[i] = hit ? 1 : 0;
  }
  return 0;
}

// one pair of placed shapes: (type, R[9], p[3], size[3]) x 2 -> intersects?
template <typename T>
static int pair_impl(int ta, const double* Ra, const double* pa, const double* sa, int tb, const double* Rb, const double* pb,
                     const double* sb, double margin) {
  Shape<T> A, B;
  for (int k = 0; k < 9; ++k) { A.R[k] = (T)Ra[k]; B.R[k] = (T)Rb[k]; }
  A.p = {(T)pa[0], (T)pa[1], (T)pa[2]}; B.p = {(T)pb[0], (T)pb[1], (T)pb[2]};
  A.s0 = (T)sa[0]; A.s1 = (T)sa[1]; A.s2 = (T)sa[2]; A.type = ta;
  B.s0 = (T)sb[0]; B.s1 = (T)sb[1]; B.s2 = (T)sb[2]; B.type = tb;
  return gjk_intersect(A, B, (T)margin) ? 1 : 0;
}

extern "C" {
// structure mask the table builder derives (zero translations, spherical wrist, tip-aligned hand frames); < 0: error
long long hostsim_table_pattern(const gik_table_t* t) {
  DevTable<double> d;
  const int rc = build_dev_table<double>(*t, d);
  return rc ? (long long)rc : (long long)d.tzero;
}
// scalar functions of gik_core.cuh whose host and device forms share their code (polynomial atan2, log6)
void hostsim_atan2_pos_f64(int64_t n, const double* y, const double* x, double* out) {
  for (int64_t i = 0; i < n; ++i) out[i] = atan2_pos(y[i], x[i]);
}
void hostsim_atan2_pos_f32(int64_t n, const float* y, const float* x, float* out) {
  for (int64_t i = 0; i < n; ++i) out[i] = atan2_pos(y[i], x[i]);
}
// pair list `list` of the scene (gik_scene_attach's lists) -> a[n], b[n] with room for kPairListCap; returns n, < 0: error
int hostsim_pair_lists(const gik_table_t* t, const gik_scene_t* s, int list, uint8_t* a, uint8_t* b) {
  if (list < 0 || list >= kNumPairLists) return GIK_E_PARAM;
  int rc = validate_table(*t);
  if (rc == 0) rc = validate_scene(*t, *s);
  if (rc) return rc;
  static PairLists L;
  build_pair_lists(*t, *s, L);
  for (int k = 0; k < L.n[list]; ++k) { a[k] = L.pairs[list][0][k]; b[k] = L.pairs[list][1][k]; }
  return L.n[list];
}
int hostsim_collide_f32(const gik_table_t* t, const gik_scene_t* s, int64_t n, const float* q, const float* cube, int list, double m, uint8_t* o) { return collide_impl<float>(t, s, n, q, cube, list, m, o); }
int hostsim_collide_f64(const gik_table_t* t, const gik_scene_t* s, int64_t n, const double* q, const double* cube, int list, double m, uint8_t* o) { return collide_impl<double>(t, s, n, q, cube, list, m, o); }
int hostsim_pair_f32(int ta, const double* Ra, const double* pa, const double* sa, int tb, const double* Rb, const double* pb, const double* sb, double m) { return pair_impl<float>(ta, Ra, pa, sa, tb, Rb, pb, sb, m); }
int hostsim_pair_f64(int ta, const double* Ra, const double* pa, const double* sa, int tb, const double* Rb, const double* pb, const double* sb, double m) { return pair_impl<double>(ta, Ra, pa, sa, tb, Rb, pb, sb, m); }
int hostsim_fk_f32(const gik_table_t* t, int64_t n, const float* q, float* f) { return fk_impl<float>(t, n, q, f); }
int hostsim_fk_f64(const gik_table_t* t, int64_t n, const double* q, double* f) { return fk_impl<double>(t, n, q, f); }
int hostsim_jac_f32(const gik_table_t* t, int64_t n, const float* q, float* j) { return jac_impl<float>(t, n, q, j); }
int hostsim_jac_f64(const gik_table_t* t, int64_t n, const double* q, double* j) { return jac_impl<double>(t, n, q, j); }
int hostsim_solve_f32(const gik_table_t* t, int64_t n, const float* q0, const float* pose, const gik_params_t* p,
                      float* q, uint8_t* c, int32_t* it, float* r) {
  return solve_impl<float>(t, n, q0, pose, p, q, c, it, r);
}
int hostsim_solve_f64(const gik_table_t* t, int64_t n, const double* q0, const double* pose, const gik_params_t* p,
                      double* q, uint8_t* c, int32_t* it, double* r) {
  return solve_impl<double>(t, n, q0, pose, p, q, c, it, r);
}
}
