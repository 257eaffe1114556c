// gik_traj.cuh -- validity check of fitted Bezier trajectories at the controller's sample times, for many trajectories
// at once (included at the end of gik_kernels.cu: one translation unit, one library).  Semantics: include/gik.h,
// gik_traj_check_*.
//
// The reference learns whether a fitted trajectory can be executed only by running it in pybullet (control.py:416-463):
// the curve between the path vertices lies on no grasp manifold and its free control points are unconstrained.  Here
// every sample (n, k) of every trajectory is checked on the device: one warp per sample, trajectory-major, so the M
// warps of one trajectory share its control points through the read-only cache.  Lane j evaluates q_j, the warp walks
// the tree (warp_tree_fk), one lane derives both hand frames, the cube placement each hand implies and the grasp error,
// the lanes place the geometries with the left hand's cube (place_geom) and the pairs of list 3 go through the same
// broad phase with compaction and GJK on full warps of candidates as gik_collision_kernel.  Per trajectory only min /
// max reductions are kept (atomicMin of (sample << 3 | bits), atomicMax of the error's bits), so the outputs do not
// depend on the launch configuration or on the order in which warps finish.
//
// The per-sample arithmetic is GIK_HD: tests/test_traj_check_cpu.py compiles it with g++ against numpy.
#pragma once

namespace gik {

// Constants of the check that DevScene does not carry (from the handle's gik_table_t), passed as a __grid_constant__.
template <typename T>
struct TrajConst {
  int32_t hand_joint[2];
  T hand[2][12];                      // hand frame on its joint (LARM_EFF / RARM_EFF), R row-major then p
  T hook_inv[2][12];                  // inverse of the hook frame on the cube
  T lo[GIK_MAX_NQ], hi[GIK_MAX_NQ];   // joint limits widened by limit_tol
};

// (R, p)^-1 = (R^T, -R^T p), in fp64
inline void traj_inverse12(const double* R, const double* p, double* out) {
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) out[3 * r + c] = R[3 * c + r];
    out[9 + r] = -(R[r] * p[0] + R[3 + r] * p[1] + R[6 + r] * p[2]);
  }
}

template <typename T>
inline void fill_traj_const(const gik_table_t& t, double limit_tol, TrajConst<T>& c) {
  memset(&c, 0, sizeof(c));
  for (int h = 0; h < 2; ++h) {
    c.hand_joint[h] = t.hand_joint[h];
    double inv[12];
    traj_inverse12(t.hook_R[h], t.hook_p[h], inv);
    for (int k = 0; k < 9; ++k) c.hand[h][k] = (T)t.hand_R[h][k];
    for (int k = 0; k < 3; ++k) c.hand[h][9 + k] = (T)t.hand_p[h][k];
    for (int k = 0; k < 12; ++k) c.hook_inv[h][k] = (T)inv[k];
  }
  for (int j = 0; j < t.nq; ++j) {
    c.lo[j] = (T)(t.lower[j] - limit_tol);
    c.hi[j] = (T)(t.upper[j] + limit_tol);
  }
}

template <typename T>
GIK_HD T traj_ld(const T* p) {
#if defined(__CUDA_ARCH__)
  return __ldg(p);
#else
  return *p;
#endif
}

// One coordinate of a curve point: sum_i w[i] * c[i * ld], i ascending (w = the Bernstein weights of the sample).
template <typename T>
GIK_HD T traj_point(const T* w, const T* c, int n_ctrl, int ld) {
  T acc = T(0);
  for (int i = 0; i < n_ctrl; ++i) acc += traj_ld(w + i) * traj_ld(c + (int64_t)i * ld);
  return acc;
}

// Hand frame h in the world: H = oMi[hand_joint[h]] * hand offset.
template <typename T>
GIK_HD void traj_hand_frame(const TrajConst<T>& tc, const T (*oMi)[12], int h, T (&H)[12]) {
  se3_mul12(&oMi[tc.hand_joint[h]][0], tc.hand[h], H);
}

// Cube placement implied by hand h: C = H * hook_h^-1 (the cube whose hook h sits exactly on the hand).
template <typename T>
GIK_HD void traj_cube_from_hand(const TrajConst<T>& tc, const T (&H)[12], int h, T (&C)[12]) {
  se3_mul12(H, tc.hook_inv[h], C);
}

// Grasp error ||log6(C_L^-1 C_R)||_2: zero exactly when both hands sit on the hooks of one rigid cube.
template <typename T>
GIK_HD T traj_grasp_error(const T (&CL)[12], const T (&CR)[12]) {
  T xi[6];
  se3_delta(CL, CR, xi);
  return sqrt_(xi[0] * xi[0] + xi[1] * xi[1] + xi[2] * xi[2] + xi[3] * xi[3] + xi[4] * xi[4] + xi[5] * xi[5]);
}

// Per-trajectory key: (first bad sample << 3) | its bits; kTrajNone = no bad sample.
constexpr int32_t kTrajNone = 0x7fffffff;
constexpr int32_t kTrajMaxSamples = (1 << 28) - 1;

#if defined(__CUDACC__)
constexpr int kTrajWarps = 4;

__device__ __forceinline__ void atomic_max_nonneg(float* p, float v) { atomicMax((int*)p, __float_as_int(v)); }
__device__ __forceinline__ void atomic_max_nonneg(double* p, double v) {
  atomicMax((unsigned long long*)p, (unsigned long long)__double_as_longlong(v));
}

template <typename T>
__global__ void __launch_bounds__(256) gik_traj_init_kernel(int64_t n, int32_t* __restrict__ key, T* __restrict__ grasp_err) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    key[i] = kTrajNone;
    grasp_err[i] = T(0);
  }
}

__global__ void __launch_bounds__(256) gik_traj_finish_kernel(int64_t n, int32_t* __restrict__ first_bad,
                                                              uint8_t* __restrict__ valid, uint8_t* __restrict__ reason) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t key = first_bad[i];
    const bool none = key == kTrajNone;
    valid[i] = none ? 1 : 0;
    reason[i] = none ? 0 : (uint8_t)(key & 7);
    first_bad[i] = none ? -1 : key >> 3;
  }
}

template <typename T>
__global__ void __launch_bounds__(kTrajWarps * 32)
gik_traj_check_kernel(const __grid_constant__ TrajConst<T> tc, const DevScene<T>* __restrict__ sc,
                      const uint8_t* __restrict__ pa, const uint8_t* __restrict__ pb, int n_pairs, int64_t n_traj,
                      int n_ctrl, int n_samples, const T* __restrict__ weights, const T* __restrict__ ctrl, T grasp_tol,
                      int32_t* key, T* grasp_err, uint8_t* __restrict__ sample_flags) {
  __shared__ T s_oMi[kTrajWarps][GIK_MAX_NQ][12];
  __shared__ T s_oMg[kTrajWarps][GIK_MAX_GEOMS][12];
  __shared__ T s_cube[kTrajWarps][12];
  __shared__ uint16_t s_cand[kTrajWarps][kMaxCand];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int nq = sc->tree.nq, ng = sc->n_geoms;
  const int64_t total = n_traj * n_samples;
  const int64_t warps = (int64_t)gridDim.x * kTrajWarps;
  for (int64_t item = (int64_t)blockIdx.x * kTrajWarps + w; item < total; item += warps) {
    const int64_t n = item / n_samples;
    const int k = (int)(item - n * n_samples);
    // joint limits (NaN counts as outside)
    T qj = T(0);
    if (lane < nq) qj = traj_point(weights + (int64_t)k * n_ctrl, ctrl + n * n_ctrl * nq + lane, n_ctrl, nq);
    const bool outside = lane < nq && !(qj >= tc.lo[lane] && qj <= tc.hi[lane]);
    unsigned bits = __any_sync(0xffffffffu, outside) ? 1u : 0u;
    // grasp: both hands, the cube each implies, the error between the two cubes
    warp_tree_fk(sc, lane, [&](int) { return qj; }, s_oMi[w]);
    T ge = T(0);
    if (lane == 0) {
      T H[12], CL[12], CR[12];
      traj_hand_frame(tc, s_oMi[w], 0, H);
      traj_cube_from_hand(tc, H, 0, CL);
      traj_hand_frame(tc, s_oMi[w], 1, H);
      traj_cube_from_hand(tc, H, 1, CR);
      ge = traj_grasp_error(CL, CR);
#pragma unroll
      for (int c = 0; c < 12; ++c) s_cube[w][c] = CL[c];
    }
    ge = __shfl_sync(0xffffffffu, ge, 0);
    if (!(ge <= grasp_tol)) bits |= 2u;
    __syncwarp();
    // collisions of list 3 with the cube at C_L.  Without per-sample flags, a sample after the trajectory's first bad
    // one so far cannot change any output (the key is a minimum): its pair tests are skipped (a relaxed read).
    if (sample_flags || k <= (ld_relaxed(key + n) >> 3)) {
      for (int g = lane; g < ng; g += 32) place_geom(sc, g, &s_cube[w][0], s_oMi[w], &s_oMg[w][g][0]);
      __syncwarp();
      bool hit = false;
      int n_cand = 0;
      for (int k0 = 0; k0 < n_pairs && !hit; k0 += 32) {
        const int p = k0 + lane;
        bool pass = false;
        if (p < n_pairs) {
          const int a = pa[p], b = pb[p];
          const T* Ma = &s_oMg[w][a][0];
          const T* Mb = &s_oMg[w][b][0];
          const T dx = Ma[9] - Mb[9], dy = Ma[10] - Mb[10], dz = Ma[11] - Mb[11];
          const T reach = sc->g[a].bound + sc->g[b].bound;
          pass = dx * dx + dy * dy + dz * dz <= reach * reach;
        }
        const unsigned m = __ballot_sync(0xffffffffu, pass);
        if (n_cand + __popc(m) > kMaxCand) {
          // list full (never with the reference scene): test this round's survivors in place
          if (pass) hit = gjk_intersect(make_shape(sc->g[pa[p]], &s_oMg[w][pa[p]][0]), make_shape(sc->g[pb[p]], &s_oMg[w][pb[p]][0]), T(0));
          hit = __any_sync(0xffffffffu, hit);
        } else {
          if (pass) s_cand[w][n_cand + __popc(m & ((1u << lane) - 1u))] = (uint16_t)p;
          n_cand += __popc(m);
        }
      }
      __syncwarp();
      for (int c0 = 0; c0 < n_cand && !hit; c0 += 32) {
        if (c0 + lane < n_cand) {
          const int p = s_cand[w][c0 + lane];
          const int a = pa[p], b = pb[p];
          hit = gjk_intersect(make_shape(sc->g[a], &s_oMg[w][a][0]), make_shape(sc->g[b], &s_oMg[w][b][0]), T(0));
        }
        hit = __any_sync(0xffffffffu, hit);
      }
      if (hit) bits |= 4u;
    }
    if (lane == 0) {
      if (bits) atomicMin(key + n, (int32_t)(((unsigned)k << 3) | bits));
      atomic_max_nonneg(grasp_err + n, ge == ge ? ge : T(INFINITY));
      if (sample_flags) sample_flags[item] = (uint8_t)bits;
    }
    __syncwarp();
  }
}
#endif  // __CUDACC__

}  // namespace gik

#if defined(__CUDACC__)
namespace {

// Sizes, tolerances and pointers are checked before the handle and before any CUDA call.
template <typename T>
int traj_check_api(gik_handle_t h, int64_t n_traj, int32_t n_ctrl, int32_t n_samples, const T* weights, const T* ctrl,
                   double limit_tol, double grasp_tol, uint8_t* valid, int32_t* first_bad, uint8_t* reason, T* grasp_err,
                   uint8_t* sample_flags, void* stream) {
  if (n_traj < 0 || n_ctrl < 2 || n_samples < 2 || n_samples > gik::kTrajMaxSamples) return GIK_E_SIZE;
  if (n_traj > INT64_MAX / n_samples) return GIK_E_SIZE;
  if (!(limit_tol >= 0.0) || !(grasp_tol >= 0.0)) return GIK_E_PARAM;
  if (n_traj > 0 && (!weights || !ctrl || !valid || !first_bad || !reason || !grasp_err)) return GIK_E_NULL;
  if (bad_handle(h)) return GIK_E_HANDLE;
  if (!h->scene) return GIK_E_NOSCENE;
  if (n_traj == 0) return GIK_OK;
  DeviceGuard g(h->device);
  if (g.err != cudaSuccess) return (int)g.err;
  cudaStream_t st = (cudaStream_t)stream;
  gik::TrajConst<T> tc;
  gik::fill_traj_const(h->host, limit_tol, tc);
  gik_scene_dev* sd = h->scene;
  int64_t rb = (n_traj + 255) / 256;
  if (rb > (int64_t)h->sm_count * 8) rb = (int64_t)h->sm_count * 8;
  gik::gik_traj_init_kernel<T><<<(int)rb, 256, 0, st>>>(n_traj, first_bad, grasp_err);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;
  const int64_t total = n_traj * n_samples;
  int64_t blocks = (total + gik::kTrajWarps - 1) / gik::kTrajWarps;
  if (blocks > (int64_t)h->sm_count * 16) blocks = (int64_t)h->sm_count * 16;
  const uint8_t* pa = sd->pairs + (size_t)6 * GIK_MAX_PAIRS;
  gik::gik_traj_check_kernel<T><<<(int)blocks, gik::kTrajWarps * 32, 0, st>>>(
      tc, scene_of<T>(sd), pa, pa + gik::kTrajPairCap, sd->n_list[3], n_traj, n_ctrl, n_samples, weights, ctrl,
      (T)grasp_tol, first_bad, grasp_err, sample_flags);
  if ((e = cudaGetLastError()) != cudaSuccess) return (int)e;
  gik::gik_traj_finish_kernel<<<(int)rb, 256, 0, st>>>(n_traj, first_bad, valid, reason);
  return (int)cudaGetLastError();
}

}  // namespace

extern "C" {
int gik_traj_check_f32(gik_handle_t h, int64_t n_traj, int32_t n_ctrl, int32_t n_samples, const float* weights,
                       const float* ctrl, double limit_tol, double grasp_tol, uint8_t* valid, int32_t* first_bad,
                       uint8_t* reason, float* grasp_err, uint8_t* sample_flags, void* s) {
  return traj_check_api<float>(h, n_traj, n_ctrl, n_samples, weights, ctrl, limit_tol, grasp_tol, valid, first_bad, reason,
                               grasp_err, sample_flags, s);
}
int gik_traj_check_f64(gik_handle_t h, int64_t n_traj, int32_t n_ctrl, int32_t n_samples, const double* weights,
                       const double* ctrl, double limit_tol, double grasp_tol, uint8_t* valid, int32_t* first_bad,
                       uint8_t* reason, double* grasp_err, uint8_t* sample_flags, void* s) {
  return traj_check_api<double>(h, n_traj, n_ctrl, n_samples, weights, ctrl, limit_tol, grasp_tol, valid, first_bad, reason,
                                grasp_err, sample_flags, s);
}
}  // extern "C"
#endif  // __CUDACC__
