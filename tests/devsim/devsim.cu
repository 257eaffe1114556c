// devsim.cu -- the device forms of the scalar functions of csrc/gik_core.cuh, run ON THE DEVICE, elementwise over
// device arrays (test-only; tests/test_gpu_device_functions.py loads it and compares with numpy longdouble).  The host
// build of the header (tests/hostsim) swaps these for the IEEE library forms, so only this build measures what the
// kernels compute: the MUFU .approx instructions, the fp64 seed + correction steps, __sincosf, the constant-bank
// Cody-Waite sincos and the packed F2 arithmetic.
#include <cuda_runtime.h>
#include "gik_core.cuh"

using namespace gik;

namespace {

// scalar ops: 0 rsqrt_(a), 1 rcp_(a), 2 sqrt_(a), 3 div_(a, b), 4 atan2_pos(a, b), 5 sincos_<true>(a), 6 sincos_<false>(a)
// out: [n] (ops 0-4) or [2][n] = (sin, cos) (ops 5, 6)
template <typename T>
__global__ void scalar_kernel(int op, int64_t n, const T* a, const T* b, T* out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const T x = a[i], y = b ? b[i] : T(0);
    T s, c;
    switch (op) {
      case 0: out[i] = rsqrt_(x); break;
      case 1: out[i] = rcp_(x); break;
      case 2: out[i] = sqrt_(x); break;
      case 3: out[i] = div_(x, y); break;
      case 4: out[i] = atan2_pos(x, y); break;
      case 5: sincos_<true>(x, s, c); out[i] = s; out[n + i] = c; break;
      case 6: sincos_<false>(x, s, c); out[i] = s; out[n + i] = c; break;
    }
  }
}

// The same on F2: element i of [n] arrays is half i % 2 of packed value i / 2 (n even).  Ops 0-2 and 4 as above,
// 3 = a * rcp_(b), the packed kernel's division.
__global__ void f2_kernel(int op, int64_t n, const float* a, const float* b, float* out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; 2 * i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const F2 x(a[2 * i], a[2 * i + 1]), y = b ? F2(b[2 * i], b[2 * i + 1]) : F2(0.0f);
    F2 r;
    switch (op) {
      case 0: r = rsqrt_(x); break;
      case 1: r = rcp_(x); break;
      case 2: r = sqrt_(x); break;
      case 3: r = x * rcp_(y); break;
      default: r = atan2_pos(x, y); break;
    }
    out[2 * i] = r.x; out[2 * i + 1] = r.y;
  }
}

// log6(R, p): R [9][n] row-major, p [3][n] -> e [6][n]
template <typename T>
__global__ void log6_kernel(int64_t n, const T* R, const T* p, T* e) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    T Ri[9], pi[3], ei[6];
    for (int k = 0; k < 9; ++k) Ri[k] = R[k * n + i];
    for (int k = 0; k < 3; ++k) pi[k] = p[k * n + i];
    log6(Ri, pi, ei);
    for (int k = 0; k < 6; ++k) e[k * n + i] = ei[k];
  }
}

// The packed form: problems 2j and 2j + 1 in the halves of one F2 (n even)
__global__ void log6_f2_kernel(int64_t n, const float* R, const float* p, float* e) {
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; 2 * j < n; j += (int64_t)gridDim.x * blockDim.x) {
    F2 Ri[9], pi[3], ei[6];
    for (int k = 0; k < 9; ++k) Ri[k] = F2(R[k * n + 2 * j], R[k * n + 2 * j + 1]);
    for (int k = 0; k < 3; ++k) pi[k] = F2(p[k * n + 2 * j], p[k * n + 2 * j + 1]);
    log6(Ri, pi, ei);
    for (int k = 0; k < 6; ++k) { e[k * n + 2 * j] = ei[k].x; e[k * n + 2 * j + 1] = ei[k].y; }
  }
}

int grid(int64_t n) { return (int)((n + 255) / 256 < 4096 ? (n + 255) / 256 : 4096); }

int finish() {
  const cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? (int)cudaDeviceSynchronize() : (int)e;
}

}  // namespace

extern "C" {
int devsim_scalar_f32(int op, int64_t n, const float* a, const float* b, float* out) {
  if (n > 0) scalar_kernel<float><<<grid(n), 256>>>(op, n, a, b, out);
  return finish();
}
int devsim_scalar_f64(int op, int64_t n, const double* a, const double* b, double* out) {
  if (n > 0) scalar_kernel<double><<<grid(n), 256>>>(op, n, a, b, out);
  return finish();
}
int devsim_scalar_f2(int op, int64_t n, const float* a, const float* b, float* out) {
  if (n % 2) return (int)cudaErrorInvalidValue;   // halves of packed values: an even count
  if (n > 0) f2_kernel<<<grid(n / 2), 256>>>(op, n, a, b, out);
  return finish();
}
int devsim_log6_f32(int64_t n, const float* R, const float* p, float* e) {
  if (n > 0) log6_kernel<float><<<grid(n), 256>>>(n, R, p, e);
  return finish();
}
int devsim_log6_f64(int64_t n, const double* R, const double* p, double* e) {
  if (n > 0) log6_kernel<double><<<grid(n), 256>>>(n, R, p, e);
  return finish();
}
int devsim_log6_f2(int64_t n, const float* R, const float* p, float* e) {
  if (n % 2) return (int)cudaErrorInvalidValue;
  if (n > 0) log6_f2_kernel<<<grid(n / 2), 256>>>(n, R, p, e);
  return finish();
}
}
