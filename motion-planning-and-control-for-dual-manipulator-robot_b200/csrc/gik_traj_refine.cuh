// gik_traj_refine.cuh -- refinement of fitted Bezier trajectories onto the grasp, many trajectories per call (included
// at the end of gik_kernels.cu, after gik_traj.cuh).  Semantics: include/gik.h, gik_traj_refine_*.
//
// The left hand leads, the right arm follows: only the right-arm columns (act_q[7..12]) of the free control points
// 3 .. n_ctrl-4 change, so with the chest, head and left-arm curves fixed the residual r_k = log6(C_L^-1 C_R) of sample
// k depends on six joints only and J_k = Ad(hook_R) J_R is square.  Levenberg-Marquardt on F = sum_k ||r_k||^2:
//   * one CTA per trajectory, persistent over the batch; control points, normal equations and factor in shared memory;
//   * threads take samples: q_k, FK and the LOCAL Jacobian of the IK kernels' hand chain (fk_frames / frame_jacobians),
//     r_k, and J^T J (21) / J^T r (6) in fp64 into a tile; then thread i owns item i of the normal equations (a 6x6
//     block of H for one pair of free control points, or 6 entries of g) and adds the tile's samples in ascending order;
//   * the damped system is factored (right-looking Cholesky, one row per thread) and solved (one row per thread and a
//     barrier per column), all in fp64.
// No floating-point atomics and no reduction whose order depends on timing: the outputs are identical between runs and
// do not depend on the batch.  The per-sample arithmetic, the assembly, the Cholesky solve and the box clamp are GIK_HD
// functions written for (tid, nth, sync): the kernel runs them with its 128 threads and __syncthreads, and
// tests/test_traj_refine_cpu.py with tid = 0, nth = 1 on the host.
#pragma once

namespace gik {

constexpr int kRefineThreads = 128;
constexpr int kRefineMinCtrl = 7, kRefineMaxCtrl = 26;   // 1 .. 20 free control points
// Levenberg-Marquardt constants: an accepted step divides lambda by kRefineDown, a rejected one multiplies it by
// kRefineUp; the loop ends once lambda exceeds kRefineLambdaMax (no step along the damped model lowers F any more).
constexpr double kRefineDown = 10.0, kRefineUp = 10.0, kRefineLambdaMax = 1e10;
// Cholesky pivot floor: max(d, kRefinePivotRel * (damped diagonal) + kRefinePivotAbs).  A free control point whose
// weights vanish at every sample (n_samples = 2) has a zero row in H and g; the floor gives it a zero step.
constexpr double kRefinePivotRel = 1e-12, kRefinePivotAbs = 1e-280;
constexpr int kRefineTileLd = 27;                        // tile row: J^T J (21), J^T r (6), then the nf free weights

struct RefineSync {                                      // the block barrier on the device, nothing on the host
  GIK_HD void operator()() const {
#if defined(__CUDA_ARCH__)
    __syncthreads();
#endif
  }
};

GIK_HD int refine_sym6(int c, int d) { return c >= d ? c * (c + 1) / 2 + d : d * (d + 1) / 2 + c; }
GIK_HD int refine_tri(int i) { return i * (i + 1) / 2; }   // start of row i of a packed lower triangle

// Cube placement hand frame H implies through hook (K, k): C = H * (K, k)^-1 = (R_H K^T, p_H - R_H K^T k).
template <typename T>
GIK_HD void refine_cube(const ArmConst<T>& ac, const T (&H)[12], T (&C)[12]) {
  const T* K = ac.hook_R;
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) C[3 * r + c] = H[3 * r] * K[3 * c] + H[3 * r + 1] * K[3 * c + 1] + H[3 * r + 2] * K[3 * c + 2];
    C[9 + r] = H[9 + r] - (C[3 * r] * ac.hook_p[0] + C[3 * r + 1] * ac.hook_p[1] + C[3 * r + 2] * ac.hook_p[2]);
  }
}

// Active joints of one sample: q_j = sum_i w[i] P_i[j], i ascending (as traj_point), with the right-arm columns of the
// free control points taken from X [nf][6].  P [n_ctrl][kActive]: the trajectory's control points in active-joint order.
template <typename T>
GIK_HD void refine_q(const T* w, const T* P, const T* X, int n_ctrl, T (&q)[kActive]) {
  for (int j = 0; j < kActive; ++j) {
    T acc = T(0);
    for (int i = 0; i < n_ctrl; ++i) {
      const bool x = j >= 7 && i >= 3 && i < n_ctrl - 3;
      acc += traj_ld(w + i) * (x ? X[(i - 3) * 6 + (j - 7)] : P[i * kActive + j]);
    }
    q[j] = acc;
  }
}

// Residual r = log6(C_L^-1 C_R) of the grasp at q and, with JAC, the model Jacobian J = Ad(hook_R) J_R: J_R = the six
// right-arm columns of RARM_EFF's LOCAL Jacobian (what gik_jac_* reports), since C_R(q + dq) = C_R exp(Ad(hook_R) J_R dq).
// fp64 uses the fast sincos (< 1 ulp); fp32 the accurate library one (the MUFU form is off by ~5e-7).
template <typename T, bool JAC>
GIK_HD void refine_sample(const DevTable<T>& tab, const T (&q)[kActive], T (&r)[6], T (&J)[6][6]) {
  constexpr bool kFast = sizeof(T) == 8;
  T fr[2][12], CL[12], CR[12];
  fk_frames<T, kFast>(tab, q, fr);
  refine_cube(tab.arm[0], fr[0], CL);
  refine_cube(tab.arm[1], fr[1], CR);
  se3_delta(CL, CR, r);
  if constexpr (JAC) {
    T AL[6][7], AR[6][7];
    frame_jacobians<T, kFast>(tab, q, AL, AR);
    const T* K = tab.arm[1].hook_R;
    const T* k = tab.arm[1].hook_p;
    for (int c = 0; c < 6; ++c) {          // Ad(K, k) [v; w] = [K v + k x (K w); K w]
      T Kv[3], Kw[3];
      for (int m = 0; m < 3; ++m) {
        Kv[m] = K[3 * m] * AR[0][1 + c] + K[3 * m + 1] * AR[1][1 + c] + K[3 * m + 2] * AR[2][1 + c];
        Kw[m] = K[3 * m] * AR[3][1 + c] + K[3 * m + 1] * AR[4][1 + c] + K[3 * m + 2] * AR[5][1 + c];
      }
      J[0][c] = Kv[0] + (k[1] * Kw[2] - k[2] * Kw[1]);
      J[1][c] = Kv[1] + (k[2] * Kw[0] - k[0] * Kw[2]);
      J[2][c] = Kv[2] + (k[0] * Kw[1] - k[1] * Kw[0]);
      J[3][c] = Kw[0]; J[4][c] = Kw[1]; J[5][c] = Kw[2];
    }
  }
}

// ||r||^2 in fp64
template <typename T>
GIK_HD double refine_r2(const T (&r)[6]) {
  double s = 0.0;
  for (int m = 0; m < 6; ++m) s += (double)r[m] * (double)r[m];
  return s;
}

// One tile row from a sample: G = J^T J (lower triangle, refine_sym6 order), b = J^T r, in fp64.
template <typename T>
GIK_HD void refine_normal(const T (&J)[6][6], const T (&r)[6], double* G, double* b) {
  for (int c = 0; c < 6; ++c) {
    for (int d = 0; d <= c; ++d) {
      double s = 0.0;
      for (int m = 0; m < 6; ++m) s += (double)J[m][c] * (double)J[m][d];
      G[refine_sym6(c, d)] = s;
    }
    double s = 0.0;
    for (int m = 0; m < 6; ++m) s += (double)J[m][c] * (double)r[m];
    b[c] = s;
  }
}

// Adds the cnt samples of a tile (rows of stride ld: G (21), b (6), the nf free weights) to item `item` of the normal
// equations, samples ascending.  H = sum_k (w_k w_k^T) (x) G_k, so each of its 6x6 blocks is symmetric: items
// 0 .. np-1 are the blocks M_ab = sum_k w_ka w_kb G_k of the pairs a >= b of free control points (21 entries each, at
// M + 21 * (a (a + 1) / 2 + b)); items np .. np + nf - 1 the gradient rows g_a = sum_k w_ka b_k (at g + 6 a).
GIK_HD void refine_accumulate(int item, int nf, int cnt, const double* tile, int ld, double* M, double* g) {
  const int np = nf * (nf + 1) / 2;
  if (item < np) {
    int a = 0;
    while (refine_tri(a + 1) <= item) ++a;
    const int b = item - refine_tri(a);
    double acc[21];
    for (int e = 0; e < 21; ++e) acc[e] = M[21 * item + e];
    for (int t = 0; t < cnt; ++t) {
      const double* row = tile + (int64_t)t * ld;
      const double wab = row[kRefineTileLd + a] * row[kRefineTileLd + b];
      for (int e = 0; e < 21; ++e) acc[e] += wab * row[e];
    }
    for (int e = 0; e < 21; ++e) M[21 * item + e] = acc[e];
  } else if (item < np + nf) {
    const int a = item - np;
    double acc[6];
    for (int c = 0; c < 6; ++c) acc[c] = g[6 * a + c];
    for (int t = 0; t < cnt; ++t) {
      const double* row = tile + (int64_t)t * ld;
      const double wa = row[kRefineTileLd + a];
      for (int c = 0; c < 6; ++c) acc[c] += wa * row[21 + c];
    }
    for (int c = 0; c < 6; ++c) g[6 * a + c] = acc[c];
  }
}

// The damped system: A = H + lambda diag(H) (packed lower triangle; unknown i = 6 a + c is joint c of free control
// point a), diag = its diagonal, z = -g.  Rows tid, tid + nth, ...
GIK_HD void refine_build(const double* M, const double* g, int nf, double lambda, double* A, double* diag, double* z,
                         int tid, int nth) {
  const int nu = 6 * nf;
  for (int i = tid; i < nu; i += nth) {
    const int a = i / 6, c = i % 6;
    double* row = A + refine_tri(i);
    for (int j = 0; j <= i; ++j) row[j] = M[21 * (refine_tri(a) + j / 6) + refine_sym6(c, j % 6)];
    row[i] += lambda * row[i];
    diag[i] = row[i];
    z[i] = -g[i];
  }
}

GIK_HD double refine_pivot(double d, double diag) {
  const double f = kRefinePivotRel * diag + kRefinePivotAbs;
  return sqrt(d > f ? d : f);
}

// In-place right-looking Cholesky A = L L^T of the packed lower triangle, with the pivot floor.  Column j: scale the
// rows below the pivot, then each row i > j subtracts L_ij L_kj from its entries k in (j, i] and, for i = j + 1, takes
// the next pivot.  Every entry sees its updates in column order whatever nth is.
template <class Sync>
GIK_HD void refine_cholesky(double* A, const double* diag, int nu, int tid, int nth, Sync sync) {
  if (tid == 0) A[0] = refine_pivot(A[0], diag[0]);
  for (int j = 0; j < nu; ++j) {
    sync();
    const double piv = A[refine_tri(j) + j];
    for (int i = j + 1 + tid; i < nu; i += nth) A[refine_tri(i) + j] /= piv;
    sync();
    for (int i = j + 1 + tid; i < nu; i += nth) {
      double* row = A + refine_tri(i);
      const double lij = row[j];
      for (int k = j + 1; k <= i; ++k) row[k] -= lij * A[refine_tri(k) + j];
      if (i == j + 1) row[i] = refine_pivot(row[i], diag[i]);
    }
  }
  sync();
}

// Solves L L^T x = z with the factor of refine_cholesky: forward substitution into y (held in y), then back substitution
// into z, which holds x on return.  One barrier per column.
template <class Sync>
GIK_HD void refine_solve(const double* L, double* z, double* y, int nu, int tid, int nth, Sync sync) {
  for (int j = 0; j < nu; ++j) {
    sync();
    const double yj = z[j] / L[refine_tri(j) + j];
    for (int i = j + 1 + tid; i < nu; i += nth) z[i] -= L[refine_tri(i) + j] * yj;
    if (tid == 0) y[j] = yj;
  }
  for (int j = nu - 1; j >= 0; --j) {
    sync();
    const double xj = y[j] / L[refine_tri(j) + j];
    for (int i = tid; i < j; i += nth) y[i] -= L[refine_tri(j) + i] * xj;
    if (tid == 0) z[j] = xj;
  }
  sync();
}

// New value of one unknown: x + d clamped to [min(lo, x0), max(hi, x0)], x0 = its input value.  A control point that
// starts inside the limits stays inside; one that starts outside never moves further out.  NaN passes through.
template <typename T>
GIK_HD T refine_clamp(T x, double d, T x0, T lo, T hi) {
  const T v = x + (T)d;
  const T lb = x0 < lo ? x0 : lo, hb = x0 > hi ? x0 : hi;
  return v < lb ? lb : (v > hb ? hb : v);
}

// Shared memory of one CTA for n_ctrl control points, in bytes: fp64 M, g, A, diag, z, y, the tile and the reduction
// buffer, then the storage-type control points P [n_ctrl][kActive], X, the trial X and the input X0 [nf][6].
GIK_HD size_t refine_smem_bytes(int n_ctrl, int elem) {
  const int nf = n_ctrl - 6, nu = 6 * nf;
  const size_t nd = (size_t)21 * refine_tri(nf) + 4 * (size_t)nu + refine_tri(nu) +
                    (size_t)kRefineThreads * (kRefineTileLd + nf) + 2 * kRefineThreads;
  return nd * sizeof(double) + (size_t)elem * ((size_t)n_ctrl * kActive + 3 * (size_t)nu);
}

#if defined(__CUDACC__)
template <typename T>
struct RefineArgs {
  int64_t n_traj;
  int32_t n_ctrl, n_samples, max_iters;
  double tol, lambda0;
  const T* weights;
  const T* ctrl;        // may equal ctrl_out: not __restrict__
  T* ctrl_out;
  double* obj_before;
  double* obj_after;
  T* grasp_err;
  int32_t* iters;
  int32_t* accepted;
};

// F = sum_k ||r_k||^2 and max_k ||r_k||^2 at the right-arm block X, for every thread: each thread sums its samples
// k = tid, tid + 128, ... in order, then a fixed tree over the threads.  (A NaN ||r_k||^2 makes F NaN.)
template <typename T>
__device__ void refine_eval(const DevTable<T>& tab, const RefineArgs<T>& a, const T* P, const T* X, double* red,
                            double& F, double& m2) {
  const int tid = threadIdx.x;
  double s = 0.0, mx = 0.0;
  for (int64_t k = tid; k < a.n_samples; k += kRefineThreads) {
    T q[kActive], r[6], J[6][6];
    refine_q(a.weights + k * a.n_ctrl, P, X, a.n_ctrl, q);
    refine_sample<T, false>(tab, q, r, J);
    const double r2 = refine_r2(r);
    s += r2;
    mx = r2 > mx ? r2 : mx;
  }
  red[tid] = s;
  red[kRefineThreads + tid] = mx;
  __syncthreads();
  for (int o = kRefineThreads / 2; o > 0; o >>= 1) {
    if (tid < o) {
      red[tid] += red[tid + o];
      const double b = red[kRefineThreads + tid + o];
      if (b > red[kRefineThreads + tid]) red[kRefineThreads + tid] = b;
    }
    __syncthreads();
  }
  F = red[0];
  m2 = red[kRefineThreads];
  __syncthreads();
}

template <typename T>
__global__ void __launch_bounds__(kRefineThreads)
gik_traj_refine_kernel(const __grid_constant__ DevTable<T> tab, const __grid_constant__ RefineArgs<T> a) {
  extern __shared__ double s_mem[];
  const int tid = threadIdx.x;
  const int n_ctrl = a.n_ctrl, nf = n_ctrl - 6, nu = 6 * nf, np = nf * (nf + 1) / 2, nq = tab.nq;
  const int ld = kRefineTileLd + nf;
  double* sM = s_mem;
  double* sg = sM + 21 * np;
  double* sA = sg + nu;
  double* sdiag = sA + refine_tri(nu);
  double* sz = sdiag + nu;
  double* sy = sz + nu;
  double* stile = sy + nu;
  double* sred = stile + kRefineThreads * ld;
  T* sP = reinterpret_cast<T*>(sred + 2 * kRefineThreads);
  T* sX = sP + n_ctrl * kActive;
  T* sXt = sX + nu;
  T* sX0 = sXt + nu;
  const RefineSync sync;

  for (int64_t n = blockIdx.x; n < a.n_traj; n += gridDim.x) {
    const T* C = a.ctrl + n * n_ctrl * nq;
    for (int e = tid; e < n_ctrl * kActive; e += kRefineThreads) sP[e] = C[(e / kActive) * nq + tab.act_q[e % kActive]];
    for (int e = tid; e < nu; e += kRefineThreads) sX[e] = sX0[e] = C[(3 + e / 6) * nq + tab.act_q[7 + e % 6]];
    __syncthreads();
    double F, m2;
    refine_eval(tab, a, sP, sX, sred, F, m2);
    const double F0 = F;
    int it = 0, acc = 0;
    if (isfinite(F)) {
      double lambda = a.lambda0;
      bool assembled = false;
      while (it < a.max_iters && !(sqrt(m2) <= a.tol)) {
        if (!assembled) {
          for (int e = tid; e < 21 * np + nu; e += kRefineThreads) sM[e] = 0.0;   // sg follows sM
          for (int64_t k0 = 0; k0 < a.n_samples; k0 += kRefineThreads) {
            const int cnt = (int)min((int64_t)kRefineThreads, a.n_samples - k0);
            __syncthreads();
            if (tid < cnt) {
              const int64_t k = k0 + tid;
              const T* w = a.weights + k * n_ctrl;
              T q[kActive], r[6], J[6][6];
              refine_q(w, sP, sX, n_ctrl, q);
              refine_sample<T, true>(tab, q, r, J);
              double* row = stile + tid * ld;
              refine_normal(J, r, row, row + 21);
              for (int f = 0; f < nf; ++f) row[kRefineTileLd + f] = (double)traj_ld(w + 3 + f);
            }
            __syncthreads();
            for (int item = tid; item < np + nf; item += kRefineThreads) refine_accumulate(item, nf, cnt, stile, ld, sM, sg);
          }
          assembled = true;
          __syncthreads();
        }
        refine_build(sM, sg, nf, lambda, sA, sdiag, sz, tid, kRefineThreads);
        refine_cholesky(sA, sdiag, nu, tid, kRefineThreads, sync);
        refine_solve(sA, sz, sy, nu, tid, kRefineThreads, sync);
        for (int e = tid; e < nu; e += kRefineThreads)
          sXt[e] = refine_clamp(sX[e], sz[e], sX0[e], tab.lo[7 + e % 6], tab.hi[7 + e % 6]);
        __syncthreads();
        double F1, m1;
        refine_eval(tab, a, sP, sXt, sred, F1, m1);
        ++it;
        if (F1 < F) {
          for (int e = tid; e < nu; e += kRefineThreads) sX[e] = sXt[e];
          F = F1; m2 = m1;
          lambda /= kRefineDown;
          ++acc;
          assembled = false;
          __syncthreads();
        } else {
          lambda *= kRefineUp;
          if (lambda > kRefineLambdaMax) break;
        }
      }
    }
    T* O = a.ctrl_out + n * n_ctrl * nq;
    if (O != C)
      for (int e = tid; e < n_ctrl * nq; e += kRefineThreads) O[e] = C[e];
    __syncthreads();
    for (int e = tid; e < nu; e += kRefineThreads) O[(3 + e / 6) * nq + tab.act_q[7 + e % 6]] = sX[e];
    if (tid == 0) {
      a.obj_before[n] = F0;
      a.obj_after[n] = F;
      a.grasp_err[n] = F == F ? (T)sqrt(m2) : T(INFINITY);
      a.iters[n] = it;
      a.accepted[n] = acc;
    }
    __syncthreads();
  }
}
#endif  // __CUDACC__

}  // namespace gik

#if defined(__CUDACC__)
namespace {

template <typename T>
int traj_refine_api(gik_handle_t h, int64_t n_traj, int32_t n_ctrl, int32_t n_samples, const T* weights, const T* ctrl,
                    int32_t max_iters, double tol, double damping, T* ctrl_out, double* obj_before, double* obj_after,
                    T* grasp_err, int32_t* iters, int32_t* accepted, void* stream) {
  if (n_traj < 0 || n_ctrl < gik::kRefineMinCtrl || n_ctrl > gik::kRefineMaxCtrl || n_samples < 2 ||
      n_samples > gik::kTrajMaxSamples)
    return GIK_E_SIZE;
  if (max_iters < 0 || !(tol >= 0.0) || !(damping > 0.0 && damping < INFINITY)) return GIK_E_PARAM;
  if (n_traj > 0 && (!weights || !ctrl || !ctrl_out || !obj_before || !obj_after || !grasp_err || !iters || !accepted))
    return GIK_E_NULL;
  if (bad_handle(h)) return GIK_E_HANDLE;
  if (n_traj == 0) return GIK_OK;
  DeviceGuard g(h->device);
  if (g.err != cudaSuccess) return (int)g.err;
  const size_t smem = gik::refine_smem_bytes(n_ctrl, (int)sizeof(T));
  auto kern = gik::gik_traj_refine_kernel<T>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  int occ = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, gik::kRefineThreads, smem);
  if (e != cudaSuccess) return (int)e;
  gik::RefineArgs<T> a{n_traj, n_ctrl, n_samples, max_iters, tol, damping, weights, ctrl, ctrl_out, obj_before,
                       obj_after, grasp_err, iters, accepted};
  return launch(h, kern, capped_grid(h, n_traj, 1, occ > 0 ? occ : 1), gik::kRefineThreads, smem, (cudaStream_t)stream,
                table_of<T>(h), a);
}

}  // namespace

extern "C" {
int gik_traj_refine_f32(gik_handle_t h, int64_t n_traj, int32_t n_ctrl, int32_t n_samples, const float* weights,
                        const float* ctrl, int32_t max_iters, double tol, double damping, float* ctrl_out,
                        double* obj_before, double* obj_after, float* grasp_err, int32_t* iters, int32_t* accepted,
                        void* s) {
  return traj_refine_api<float>(h, n_traj, n_ctrl, n_samples, weights, ctrl, max_iters, tol, damping, ctrl_out,
                                obj_before, obj_after, grasp_err, iters, accepted, s);
}
int gik_traj_refine_f64(gik_handle_t h, int64_t n_traj, int32_t n_ctrl, int32_t n_samples, const double* weights,
                        const double* ctrl, int32_t max_iters, double tol, double damping, double* ctrl_out,
                        double* obj_before, double* obj_after, double* grasp_err, int32_t* iters, int32_t* accepted,
                        void* s) {
  return traj_refine_api<double>(h, n_traj, n_ctrl, n_samples, weights, ctrl, max_iters, tol, damping, ctrl_out,
                                 obj_before, obj_after, grasp_err, iters, accepted, s);
}
}  // extern "C"
#endif  // __CUDACC__
