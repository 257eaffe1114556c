// gik_bezier.cuh -- the least-squares Bezier fit of `maketraj` (control.py:63-195) for many paths at once (included at the
// end of gik_kernels.cu: one translation unit, one library).
//
// The reference minimises sum_k |B(t_k) - q_k|^2 over the control points of a degree-n Bezier curve under position /
// velocity / acceleration constraints at both ends (SLSQP, control.py:110-158).  Those constraints pin three control points
// at each end (P0 = P1 = P2 = q0, Pn = Pn-1 = Pn-2 = q1; trajectory.py), and what is left is linear least squares in the
// free control points with the Bernstein matrix as design matrix -- the SAME matrix for every path with the same number
// of points, and for every joint.  So the host factors it once (pseudo-inverse in fp64, trajectory.py) and a fit is
//     rhs = path - w0 q0^T - w1 q1^T     [n_points][dim]
//     Pf  = pinv * rhs                   [n_free][dim]
//     cost = |basis * Pf - rhs|^2
// per path: one warp per path, operands in shared memory, rhs read once from HBM (the only traffic that scales:
// n_points * dim values in, (n_free + 6) * dim + 1 out).
#pragma once

namespace gik {

constexpr int kBezierWarps = 4;

template <typename T>
__global__ void __launch_bounds__(kBezierWarps * 32)
gik_bezier_fit_kernel(int64_t n_paths, int n_points, int dim, int n_ctrl, const T* __restrict__ pinv /* [n_free][n_points] */,
                      const T* __restrict__ basis /* [n_points][n_free] */, const T* __restrict__ w0, const T* __restrict__ w1,
                      const T* __restrict__ q0 /* [n_paths][dim] */, const T* __restrict__ q1,
                      const T* __restrict__ path /* [n_paths][n_points][dim] */, T* __restrict__ ctrl /* [n_paths][n_ctrl][dim] */,
                      T* __restrict__ cost) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* smem = reinterpret_cast<T*>(smem_raw);
  const int n_free = n_ctrl - 6;
  T* s_pinv = smem;                                  // [n_free][n_points]
  T* s_basis = s_pinv + n_free * n_points;           // [n_points][n_free]
  T* s_w0 = s_basis + n_points * n_free;             // [n_points]
  T* s_w1 = s_w0 + n_points;
  T* s_warp = s_w1 + n_points;                       // per warp: rhs [n_points][dim], Pf [n_free][dim]
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < n_free * n_points; i += blockDim.x) { s_pinv[i] = pinv[i]; s_basis[i] = basis[i]; }
  for (int i = threadIdx.x; i < n_points; i += blockDim.x) { s_w0[i] = w0[i]; s_w1[i] = w1[i]; }
  __syncthreads();
  T* rhs = s_warp + (size_t)w * (n_points + n_free) * dim;
  T* pf = rhs + n_points * dim;
  const int64_t warps = (int64_t)gridDim.x * kBezierWarps;
  for (int64_t p = (int64_t)blockIdx.x * kBezierWarps + w; p < n_paths; p += warps) {
    const T* pp = path + p * n_points * dim;
    for (int idx = lane; idx < n_points * dim; idx += 32) {
      const int k = idx / dim, d = idx - k * dim;
      rhs[idx] = pp[idx] - s_w0[k] * q0[p * dim + d] - s_w1[k] * q1[p * dim + d];
    }
    __syncwarp();
    for (int o = lane; o < n_free * dim; o += 32) {
      const int i = o / dim, d = o - i * dim;
      T acc = T(0);
      for (int k = 0; k < n_points; ++k) acc += s_pinv[i * n_points + k] * rhs[k * dim + d];
      pf[o] = acc;
    }
    __syncwarp();
    T c = T(0);
    for (int idx = lane; idx < n_points * dim; idx += 32) {
      const int k = idx / dim, d = idx - k * dim;
      T r = -rhs[idx];
      for (int i = 0; i < n_free; ++i) r += s_basis[k * n_free + i] * pf[i * dim + d];
      c += r * r;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if (lane == 0) cost[p] = c;
    T* cp = ctrl + p * n_ctrl * dim;
    for (int idx = lane; idx < n_ctrl * dim; idx += 32) {
      const int i = idx / dim, d = idx - i * dim;
      cp[idx] = i < 3 ? q0[p * dim + d] : (i >= n_ctrl - 3 ? q1[p * dim + d] : pf[(i - 3) * dim + d]);
    }
    __syncwarp();
  }
}

}  // namespace gik

namespace {

template <typename T>
int bezier_fit_api(gik_handle_t h, int64_t n_paths, int32_t n_points, int32_t dim, int32_t n_ctrl, const T* pinv, const T* basis,
                   const T* w0, const T* w1, const T* q0, const T* q1, const T* path, T* ctrl, T* cost, void* stream) {
  if (n_paths < 0 || n_points < 1 || dim < 1 || n_ctrl < 7) return GIK_E_SIZE;
  const int n_free = n_ctrl - 6;
  const size_t smem = sizeof(T) * ((size_t)2 * n_free * n_points + 2 * (size_t)n_points +
                                   (size_t)gik::kBezierWarps * (n_points + n_free) * dim);
  if (smem > 200 * 1024) return GIK_E_SIZE;
  if (n_paths > 0 && (!pinv || !basis || !w0 || !w1 || !q0 || !q1 || !path || !ctrl || !cost)) return GIK_E_NULL;
  if (bad_handle(h)) return GIK_E_HANDLE;
  if (n_paths == 0) return GIK_OK;
  DeviceGuard g(h->device);
  if (g.err != cudaSuccess) return (int)g.err;
  cudaError_t e = cudaFuncSetAttribute(gik::gik_bezier_fit_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  return launch(h, gik::gik_bezier_fit_kernel<T>, capped_grid(h, n_paths, gik::kBezierWarps, 4), gik::kBezierWarps * 32, smem,
                (cudaStream_t)stream, n_paths, n_points, dim, n_ctrl, pinv, basis, w0, w1, q0, q1, path, ctrl, cost);
}

}  // namespace

extern "C" {
int gik_bezier_fit_f32(gik_handle_t h, int64_t n_paths, int32_t n_points, int32_t dim, int32_t n_ctrl, const float* pinv,
                       const float* basis, const float* w0, const float* w1, const float* q0, const float* q1, const float* path,
                       float* ctrl, float* cost, void* s) {
  return bezier_fit_api<float>(h, n_paths, n_points, dim, n_ctrl, pinv, basis, w0, w1, q0, q1, path, ctrl, cost, s);
}
int gik_bezier_fit_f64(gik_handle_t h, int64_t n_paths, int32_t n_points, int32_t dim, int32_t n_ctrl, const double* pinv,
                       const double* basis, const double* w0, const double* w1, const double* q0, const double* q1,
                       const double* path, double* ctrl, double* cost, void* s) {
  return bezier_fit_api<double>(h, n_paths, n_points, dim, n_ctrl, pinv, basis, w0, w1, q0, q1, path, ctrl, cost, s);
}
}  // extern "C"
