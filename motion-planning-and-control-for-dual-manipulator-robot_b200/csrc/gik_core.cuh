// gik_core.cuh -- per-problem arithmetic of the dual-arm grasp IK, one problem per thread, everything in
// registers.  Compiles for the device (nvcc, sm_100a) and -- for the CPU unit tests under tests/hostsim
// only -- as plain C++17.  Nothing here touches memory except through the DevTable reference, which on the
// device is a __constant__ object (constant-bank operands feed the FMAs directly).
//
// What one iteration computes (reference: inverse_geometry.py:56-89):
//   FK of both hands + both LOCAL frame Jacobians    (pin.framesForwardKinematics :58, computeFrameJacobian :75-76)
//   e_h = log6(hand_h^-1 * hook_h)                   (pin.log :66-67)
//   dq  = J^T (J J^T + lambda I)^-1 [e_L; e_R]       (np.linalg.pinv(J) @ error :83, lambda = 0)
// and the caller applies q <- clamp(q + dt dq)       (pin.integrate :86, projecttojointlimits :89).
//
// Structure that is exploited (DESIGN.md "Kernel math"):
//   * Each hand's chain is walked BACKWARDS from the hand frame, carrying the pose of the current joint
//     expressed in the hand frame.  That yields the LOCAL Jacobian columns directly (no world-frame FK, no
//     R_f^T rotations) and ends at hand^-1, which is exactly what the error needs.
//   * J = [c_L A_L 0; c_R 0 A_R] (chest column + two 6x6 arm blocks), so
//     J J^T + lambda I = blockdiag(A_L A_L^T + lambda I, A_R A_R^T + lambda I) + c c^T :
//     two 6x6 Cholesky factorisations and a Sherman-Morrison rank-1 correction replace the dense 12x12 solve.
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define GIK_HD __host__ __device__ __forceinline__
#else
#define GIK_HD inline __attribute__((always_inline))
#endif

#ifndef GIK_MAX_NQ
#define GIK_MAX_NQ 32
#endif

namespace gik {

constexpr int kActive = 13;  // chest + 6 + 6 joints that move the hands

// Axis of chain joint k (k = 0: chest, k = 1..6: arm joints root -> tip).  This pattern (z | z y y x y z) is
// the compiled-in structure of the fast path; gik_create() rejects tables that do not match it.
GIK_HD constexpr int chain_axis(int k) {
  return k == 0 ? 2 : k == 1 ? 2 : k == 2 ? 1 : k == 3 ? 1 : k == 4 ? 0 : k == 5 ? 1 : 2;
}

template <typename T>
struct ArmConst {
  T t[7][3];    // parent -> joint translation of chain joint k
  T finv_R[9];  // (hand frame offset on the tip joint)^-1, row-major
  T finv_p[3];
  T tip_lin[3]; // finv_p x finv_R[:, axis of the tip joint]: linear part of the (constant) LOCAL Jacobian column of the tip joint
  T g6[21];     // lower triangle (i >= j at i(i+1)/2 + j) of tip_col tip_col^T: the tip joint's constant share of G = A A^T
  T hook_R[9];  // hook frame on the cube
  T hook_p[3];
  T rw[3];      // wrist centre (common point of the axes of chain joints 4, 5, 6) in the hand frame; spherical-wrist tables only
  T tip_psi;    // tables with kTipZ: finv_R = Rot(z, tip_psi), so finv_R * Rot(z, -q6) = Rot(z, -(q6 - tip_psi))
};

template <typename T>
struct DevTable {
  ArmConst<T> arm[2];
  T lo[kActive], hi[kActive];          // limits of the active joints: 0 chest, 1-6 left, 7-12 right
  T qlo[GIK_MAX_NQ], qhi[GIK_MAX_NQ];  // limits in q order (passive joints)
  int32_t nq;
  int32_t act_q[kActive];              // q index of each active joint
  int32_t n_passive;
  int32_t passive_q[GIK_MAX_NQ];
  uint32_t tzero;                      // bit 3*K + c set <=> translation component c of chain joint K is 0 in BOTH arms
};

// Zero pattern of the Nextage joint translations (NextageaOpen.urdf:580-711): chest (0,0,z) | (x,y,z) | (0,0,z) |
// (0,y,z) | (x,0,z) | (x,0,0) | (0,0,z).  Kernels are instantiated for "no zeros known" (TZ = 0, any table of the
// compiled topology) and for this pattern; the launcher picks the specialisation when the table has at least these zeros.
constexpr uint32_t kNextageJointTZ = (3u << 0) | (3u << 6) | (1u << 9) | (1u << 13) | (6u << 15) | (3u << 18);
// Spherical wrist: joint 5's origin lies on joint 4's axis (t[5] = (x, 0, 0), joint 4 turns about x) and on joint 6's
// axis (t[6] = (0, 0, z), joint 6 turns about z), so the axes of chain joints 4, 5, 6 meet in one point.  Part of the
// Nextage pattern; the undamped step then decouples into two 3x3 solves per hand (hand_wrist_phase1).
constexpr uint32_t kWristTZ = (6u << 15) | (3u << 18);
// Tip-aligned hand frame: the rotation of the hand frame on the tip joint is a rotation about the tip joint's own axis
// (LARM_EFF / RARM_EFF: rpy = (0, 0, 1.5708), NextageaOpen.urdf), so in the HAND frame the tip axis is the constant
// (0, 0, 1), the first step of the backward walk is one rotation by q6 - psi with no arithmetic, and the next one acts
// on a matrix with four zeros: 44 of the wrist step's ~340 packed operations disappear (hand_wrist_phase1).
constexpr uint32_t kTipZ = 1u << 24;
constexpr uint32_t kNextageTZ = kNextageJointTZ | kTipZ;
static_assert((kNextageTZ & kWristTZ) == kWristTZ, "the Nextage pattern includes the spherical wrist");

// ------------------------------------------------------------------------------------------------------
// scalar helpers
// ------------------------------------------------------------------------------------------------------
template <typename T> struct Num;
template <> struct Num<float> {
  static constexpr float kPivotFloor = 1e-30f;  // Cholesky pivot guard (singular arm Jacobian)
  static constexpr float kSeriesT2 = 0.25f;     // theta^2 below which log6's alpha/beta use their series
  static constexpr float kTinyS = 1e-18f;
  static constexpr float kRcpCap = 1e12f;       // |1 / det| cap of the 3x3 solves (singular arm / wrist)
};
template <> struct Num<double> {
  static constexpr double kPivotFloor = 1e-280;
  static constexpr double kSeriesT2 = 1e-4;
  static constexpr double kTinyS = 1e-150;
  static constexpr double kRcpCap = 1e100;
};

// fp32 device versions are single MUFU instructions (rsqrt/sqrt/rcp .approx.ftz, <= 2 ulp): the IEEE library
// forms carry denormal pre-scaling, Newton steps and slow-path calls that cost issue slots and branch bubbles in
// the descent loop.  Inputs here are never denormal where it matters (pivots are floored, norms are >= 0).
GIK_HD float rsqrt_(float x) {
#ifdef __CUDA_ARCH__
  float r;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
#else
  return 1.0f / sqrtf(x);
#endif
}
// fp64 device versions: MUFU seed (rsqrt/rcp.approx.ftz.f64, ~2^-22 relative) + ONE third-order correction step
// (5 / 3 FP64-pipe instructions; two Newton steps, 7 / 4, measured no more accurate).  Accuracy on the B200 from the
// floors to 1e12 (tests/test_gpu_device_functions.py): 1.1e-16 / 1.4e-16 relative; no special-case paths: operands are floored.
GIK_HD double rsqrt_(double x) {
#ifdef __CUDA_ARCH__
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  // one third-order step: y (1 + e/2 + 3 e^2 / 8), e = 1 - x y^2; seed error 2^-22 -> ~1e-20 before rounding
  const double e = fma(-(x * y), y, 1.0);
  return fma(y * e, fma(e, 0.375, 0.5), y);
#else
  return 1.0 / sqrt(x);
#endif
}
GIK_HD float rcp_(float b) {
#ifdef __CUDA_ARCH__
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(b));
  return r;
#else
  return 1.0f / b;
#endif
}
GIK_HD double rcp_(double b) {
#ifdef __CUDA_ARCH__
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(b));
  // one third-order step: y (1 + e + e^2), e = 1 - b y
  const double e = fma(-b, y, 1.0);
  return fma(fma(y, e, y), e, y);
#else
  return 1.0 / b;
#endif
}
#ifdef __CUDA_ARCH__
GIK_HD float div_(float a, float b) { return a * rcp_(b); }
GIK_HD double div_(double a, double b) { return a * rcp_(b); }
#else
GIK_HD float div_(float a, float b) { return a / b; }
GIK_HD double div_(double a, double b) { return a / b; }
#endif
GIK_HD float sqrt_(float x) {
#ifdef __CUDA_ARCH__
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
#else
  return sqrtf(x);
#endif
}
GIK_HD double sqrt_(double x) { return sqrt(x); }
GIK_HD float max_(float a, float b) { return fmaxf(a, b); }
GIK_HD double max_(double a, double b) { return fmax(a, b); }
GIK_HD float min_(float a, float b) { return fminf(a, b); }
GIK_HD double min_(double a, double b) { return fmin(a, b); }
// atan2(y, x) for y >= 0 (the only case log6 needs: y = |vee(R - R^T)| / 2), result in [0, pi].
// fp32: branch-free, one reciprocal + degree-7 polynomial in t = (min/max)^2 fitted on [0, 1] (abs error
// 1.1e-7, relative 1.5e-7 measured against atan in fp64; on the device, with the MUFU reciprocal and the rounding of
// results up to pi, 3.0e-7 absolute); the library atan2f is ~2x the instructions plus branches.
GIK_HD float atan2_pos(float y, float x) {
  const float ax = fabsf(x);
  const float mn = min_(y, ax), mx = max_(max_(y, ax), 1e-30f);
  const float a = div_(mn, mx), t = a * a;
  float p = 3.8667389163e-03f;
  p = p * t + -2.0026747651e-02f;
  p = p * t + 4.8914321553e-02f;
  p = p * t + -8.0096817182e-02f;
  p = p * t + 1.0865759085e-01f;
  p = p * t + -1.4257044926e-01f;
  p = p * t + 1.9998681172e-01f;
  p = p * t + -3.3333323101e-01f;     // (Estrin's scheme, half the dependent depth: config 4 25.2 -> 25.4 ms, not kept)
  float r = (a * t) * p + a;
  r = y > ax ? 1.57079632679489662f - r : r;
  return x < 0.0f ? 3.14159265358979324f - r : r;
}
// fp64: one division + a degree-10 polynomial in u^2 after reducing the ratio to |u| <= tan(pi/8)
// (mn/mx > tan(pi/8): atan(mn/mx) = pi/4 + atan((mn - mx)/(mn + mx))).  Coefficients: interpolation of
// (atan(u) - u)/u^3 at the Chebyshev nodes of u^2 in [0, tan^2(pi/8)], computed in 50-digit arithmetic; max abs error
// of the double evaluation 5.6e-17 on a 2001-point grid (= rounding).  Branch-free, constants are constant-bank
// loads on the device (the library atan2 spends ~40 UMOV on its 64-bit immediates plus a division slow path).
#define GIK_ATAN64_COEFFS                                                                                      \
  -0.3333333333333333, 0.1999999999999552, -0.14285714284666542, 0.11111111015256361, -0.09090904578123903,  \
      0.07692183190826087, -0.06664511447381948, 0.0585814891280221, -0.0508544973794026, 0.03923165829558719, \
      -0.01917688711906226
#if defined(__CUDACC__)
static __constant__ double kAtan64[11] = {GIK_ATAN64_COEFFS};
#endif
GIK_HD double atan2_pos(double y, double x) {
#ifdef __CUDA_ARCH__
  const double* K = kAtan64;
#else
  static const double K[11] = {GIK_ATAN64_COEFFS};
#endif
  const double ax = fabs(x);
  const double mn = min_(y, ax), mx = max_(max_(y, ax), 1e-300);
  const bool big = mn > 0.41421356237309503 * mx;
  const double num = big ? mn - mx : mn, den = big ? mn + mx : mx;
  const double u = div_(num, den), z = u * u;
  double p = fma(K[10], z, K[9]);
  p = fma(p, z, K[8]); p = fma(p, z, K[7]); p = fma(p, z, K[6]); p = fma(p, z, K[5]);
  p = fma(p, z, K[4]); p = fma(p, z, K[3]); p = fma(p, z, K[2]); p = fma(p, z, K[1]); p = fma(p, z, K[0]);
  double r = fma(u * z, p, u);
  r = big ? r + 0.78539816339744831 : r;
  r = y > ax ? 1.57079632679489662 - r : r;
  return x < 0.0 ? 3.14159265358979324 - r : r;
}

// ------------------------------------------------------------------------------------------------------
// F2: two fp32 values in one 64-bit register pair, operated on by Blackwell's packed FFMA2 / FMUL2 / FADD2
// (PTX fma/mul/add/sub.rn.f32x2, sm_100+).  One packed instruction does the work of two scalar ones in ONE issue slot
// (measured on B200, tools/probes/ffma2.cu: 68.4 TFLOP/s with three register operands, where scalar FFMA with three
// register operands stops at 45 TFLOP/s on register-file bandwidth).  The two hands of one problem run the same
// operation sequence on different data, so the fp32 lane kernel carries (left, right) in the halves of an F2.
// ptxas contracts mul.f32x2 + add/sub.f32x2 into FFMA2 and folds negations into operand modifiers, so the templates
// below are instantiated with T = F2 unchanged.  On the host (unit tests) the halves are plain floats.
// ------------------------------------------------------------------------------------------------------
struct F2 {
  float x, y;
  GIK_HD F2() {}
  GIK_HD F2(float a) : x(a), y(a) {}
  GIK_HD F2(double a) : x((float)a), y((float)a) {}
  GIK_HD F2(int a) : x((float)a), y((float)a) {}
  GIK_HD F2(float a, float b) : x(a), y(b) {}
};
#ifdef __CUDA_ARCH__
GIK_HD unsigned long long f2_pack(F2 a) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a.x), "f"(a.y));
  return r;
}
GIK_HD F2 f2_unpack(unsigned long long r) {
  F2 a;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a.x), "=f"(a.y) : "l"(r));
  return a;
}
GIK_HD F2 operator*(F2 a, F2 b) {
  unsigned long long d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(f2_pack(a)), "l"(f2_pack(b)));
  return f2_unpack(d);
}
GIK_HD F2 operator+(F2 a, F2 b) {
  unsigned long long d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(f2_pack(a)), "l"(f2_pack(b)));
  return f2_unpack(d);
}
GIK_HD F2 operator-(F2 a, F2 b) {
  unsigned long long d;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(f2_pack(a)), "l"(f2_pack(b)));
  return f2_unpack(d);
}
#else
GIK_HD F2 operator*(F2 a, F2 b) { return F2(a.x * b.x, a.y * b.y); }
GIK_HD F2 operator+(F2 a, F2 b) { return F2(a.x + b.x, a.y + b.y); }
GIK_HD F2 operator-(F2 a, F2 b) { return F2(a.x - b.x, a.y - b.y); }
#endif
GIK_HD F2 operator-(F2 a) { return F2(-a.x, -a.y); }
GIK_HD F2& operator+=(F2& a, F2 b) { a = a + b; return a; }
GIK_HD F2& operator-=(F2& a, F2 b) { a = a - b; return a; }
GIK_HD F2 max_(F2 a, F2 b) { return F2(max_(a.x, b.x), max_(a.y, b.y)); }
GIK_HD F2 min_(F2 a, F2 b) { return F2(min_(a.x, b.x), min_(a.y, b.y)); }
GIK_HD F2 rsqrt_(F2 a) { return F2(rsqrt_(a.x), rsqrt_(a.y)); }
GIK_HD F2 rcp_(F2 a) { return F2(rcp_(a.x), rcp_(a.y)); }
GIK_HD F2 sqrt_(F2 a) { return F2(sqrt_(a.x), sqrt_(a.y)); }
GIK_HD F2 abs_(F2 a) { return F2(fabsf(a.x), fabsf(a.y)); }
// per-half predicates and selects (FSETP / FSEL on the ALU pipe, which the FMA-bound loop has to spare)
struct B2 { bool x, y; };
GIK_HD B2 gt_(F2 a, F2 b) { return {a.x > b.x, a.y > b.y}; }
GIK_HD B2 ge_(F2 a, F2 b) { return {a.x >= b.x, a.y >= b.y}; }
GIK_HD B2 lt_(F2 a, F2 b) { return {a.x < b.x, a.y < b.y}; }
GIK_HD F2 sel_(B2 c, F2 a, F2 b) { return F2(c.x ? a.x : b.x, c.y ? a.y : b.y); }
// atan2_pos on both halves: the same degree-7 polynomial as the scalar fp32 form, evaluated with packed FMAs
GIK_HD F2 atan2_pos(F2 y, F2 x) {
  const F2 ax = abs_(x);
  const F2 mn = min_(y, ax), mx = max_(max_(y, ax), F2(1e-30f));
  const F2 a = mn * rcp_(mx), t = a * a;
  F2 p = F2(3.8667389163e-03f);
  p = p * t + F2(-2.0026747651e-02f);
  p = p * t + F2(4.8914321553e-02f);
  p = p * t + F2(-8.0096817182e-02f);
  p = p * t + F2(1.0865759085e-01f);
  p = p * t + F2(-1.4257044926e-01f);
  p = p * t + F2(1.9998681172e-01f);
  p = p * t + F2(-3.3333323101e-01f);
  F2 r = (a * t) * p + a;
  r = sel_(gt_(y, ax), F2(1.57079632679489662f) - r, r);
  return sel_(lt_(x, F2(0.0f)), F2(3.14159265358979324f) - r, r);
}
template <> struct Num<F2> { static constexpr float kPivotFloor = 1e-30f; static constexpr float kRcpCap = 1e12f; };

// FAST = MUFU-based sin/cos (abs error measured 4.0e-7 on [-pi, pi] -- above the 3.6e-7 CUDA documents for __sinf /
// __cosf -- and 7.1e-7 over the joint arguments, [-5.15, 4.71] on Nextage); accurate otherwise.
template <bool FAST>
GIK_HD void sincos_(float x, float& s, float& c) {
#ifdef __CUDA_ARCH__
  if (FAST) __sincosf(x, &s, &c); else sincosf(x, &s, &c);
#else
  s = sinf(x); c = cosf(x);
#endif
}
// fp64, FAST: Cody-Waite reduction by multiples of pi/2 (two-term pi/2, exact-product FMAs) + the classic degree-13 /
// degree-14 minimax kernels on |r| <= pi/4 (coefficients of the fdlibm __kernel_sin / __kernel_cos polynomials;
// < 1 ulp each; 1.7e-16 absolute measured on the B200 for |x| <= 1e6, the library 1.3e-16).  Same arithmetic class as the library sincos, but every constant is a constant-bank OPERAND of its
// DFMA: the library form materialises its 64-bit immediates with UMOV pairs inside the descent loop (~30 per call,
// 15 % of the loop's issue slots in the round-1 fp64 capture) and carries a slow-path branch for huge arguments.
// Valid for |x| < 2^50 (far beyond any joint range); NaN/inf propagate.
#if defined(__CUDACC__)
static __constant__ double kSinCos64[18] = {
    6.36619772367581382433e-01,   // 0: 2/pi
    6755399441055744.0,           // 1: 1.5 * 2^52 (round-to-nearest-integer magic)
    -1.57079632679489655800e+00,  // 2: -(pi/2 high)
    -6.12323399573676603587e-17,  // 3: -(pi/2 low)
    -1.66666666666666324348e-01,  // 4: S1
    8.33333333332248946124e-03,   // 5: S2
    -1.98412698298579493134e-04,  // 6: S3
    2.75573137070700676789e-06,   // 7: S4
    -2.50507602534068634195e-08,  // 8: S5
    1.58969099521155010221e-10,   // 9: S6
    4.16666666666666019037e-02,   // 10: C1
    -1.38888888888741095749e-03,  // 11: C2
    2.48015872894767294178e-05,   // 12: C3
    -2.75573143513906633035e-07,  // 13: C4
    2.08757232129817482790e-09,   // 14: C5
    -1.13596475577881948265e-11,  // 15: C6
    -0.5, 1.0};
#endif
template <bool FAST>
GIK_HD void sincos_(double x, double& s, double& c) {
#ifdef __CUDA_ARCH__
  if (FAST) {
    const double* K = kSinCos64;
    const double t = fma(x, K[0], K[1]);
    const int k = __double2loint(t);
    const double kd = t - K[1];
    double r = fma(kd, K[2], x);
    r = fma(kd, K[3], r);
    const double z = r * r;
    double ps = fma(K[9], z, K[8]);
    ps = fma(ps, z, K[7]); ps = fma(ps, z, K[6]); ps = fma(ps, z, K[5]); ps = fma(ps, z, K[4]);
    double pc = fma(K[15], z, K[14]);
    pc = fma(pc, z, K[13]); pc = fma(pc, z, K[12]); pc = fma(pc, z, K[11]); pc = fma(pc, z, K[10]);
    const double sr = fma(r * z, ps, r);
    const double cr = fma(z * z, pc, fma(z, K[16], K[17]));
    const bool odd = k & 1;
    double so = odd ? cr : sr, co = odd ? sr : cr;
    // sign flips on the high word: sin negative in quadrants 2, 3; cos negative in quadrants 1, 2
    so = __hiloint2double(__double2hiint(so) ^ ((k & 2) << 30), __double2loint(so));
    co = __hiloint2double(__double2hiint(co) ^ (((k + 1) & 2) << 30), __double2loint(co));
    s = so; c = co;
  } else {
    sincos(x, &s, &c);
  }
#else
  s = sin(x); c = cos(x);
#endif
}

// ------------------------------------------------------------------------------------------------------
// log6: SE3 (R row-major, p) -> [v; w].  Same function as pinocchio's log6/log3 (pin.log at
// inverse_geometry.py:66-67); theta is taken as atan2(|vee(R - R^T)|/2, (tr R - 1)/2), which equals
// acos((tr R - 1)/2) for a rotation matrix but stays accurate in fp32 near theta = 0.
// ------------------------------------------------------------------------------------------------------
// In two functions: log6_pre is straight-line code (theta, the common-case w = theta/(2 sin theta) vee(R - R^T), alpha,
// beta -- a chain of dependent MUFU results), log6_post holds the one data-dependent branch (pinocchio's form near
// theta = pi, rare) and the assembly of [v; w].  (Written this way to try orderings that put independent work between
// the halves; none of them paid -- DESIGN.md "Tried and dropped" -- but the split itself measured 5 % faster on the
// edge projection and is kept.)
template <typename T>
struct Log6Mid { T vx, vy, vz, d0, d1, d2, c, theta, wx, wy, wz, alpha, beta; };

// log6_pre_v: the same from vee(R - R^T) and tr R alone (all the common case needs of R); the diagonal m.d0..d2, read
// only by the near-pi form, is then the caller's to fill when log6_near_pi(m) says so (hand_error_post).
template <typename T>
GIK_HD void log6_pre_v(T vx, T vy, T vz, T tr, Log6Mid<T>& m);
template <typename T>
GIK_HD void log6_pre(const T (&R)[9], Log6Mid<T>& m) {
  log6_pre_v(R[7] - R[5], R[2] - R[6], R[3] - R[1], R[0] + R[4] + R[8], m);
  m.d0 = R[0]; m.d1 = R[4]; m.d2 = R[8];
}
template <typename T>
GIK_HD bool log6_near_pi(const Log6Mid<T>& m) { return m.theta >= T(3.14159265358979323846 - 1e-2); }
template <typename T>
GIK_HD void log6_pre_v(T vx, T vy, T vz, T tr, Log6Mid<T>& m) {
  const T c = min_(max_((tr - T(1)) * T(0.5), T(-1)), T(1));
  const T s = T(0.5) * sqrt_(vx * vx + vy * vy + vz * vz);
  const T theta = atan2_pos(s, c);
  const T fac = s > Num<T>::kTinyS ? T(0.5) * div_(theta, s) : T(0.5);  // theta / (2 sin theta)
  m.wx = fac * vx; m.wy = fac * vy; m.wz = fac * vz;
  const T t2 = theta * theta;
  // alpha = (theta/2) cot(theta/2), beta = (1 - alpha) / theta^2; cot(theta/2) = (1+c)/s = s/(1-c)
  const bool front = c >= T(0);
  const T num = front ? T(1) + c : s;
  const T den = front ? s : T(1) - c;
  T alpha = T(0.5) * theta * div_(num, max_(den, Num<T>::kTinyS));
  T beta = div_(T(1) - alpha, max_(t2, Num<T>::kTinyS));
  // (The series also SHORTENS the dependent chain of the latency-bound scalar kernels -- its inputs are ready long before
  // the reciprocals of the general form: dropping it cost config 4 1.7 %.  The packed form below drops it.)
  if (t2 < Num<T>::kSeriesT2) {
    alpha = T(1) - t2 * (T(1.0 / 12) + t2 * (T(1.0 / 720) + t2 * T(1.0 / 30240)));
    beta = T(1.0 / 12) + t2 * (T(1.0 / 720) + t2 * (T(1.0 / 30240) + t2 * T(1.0 / 1209600)));
  }
  m.vx = vx; m.vy = vy; m.vz = vz;
  m.c = c; m.theta = theta; m.alpha = alpha; m.beta = beta;
}

template <typename T>
GIK_HD void log6_post(const Log6Mid<T>& m, const T (&p)[3], T (&e)[6]) {
  T wx = m.wx, wy = m.wy, wz = m.wz;
  if (log6_near_pi(m)) {
    // pinocchio's explicit branch near pi: |w_i| from the diagonal, sign from the antisymmetric part
    const T cphi = -m.c;
    const T beta = div_(m.theta * m.theta, T(1) + cphi);
    const T t0 = (m.d0 + cphi) * beta, t1 = (m.d1 + cphi) * beta, t2 = (m.d2 + cphi) * beta;
    wx = (m.vx > T(0) ? T(1) : T(-1)) * (t0 > T(0) ? sqrt_(t0) : T(0));
    wy = (m.vy > T(0) ? T(1) : T(-1)) * (t1 > T(0) ? sqrt_(t1) : T(0));
    wz = (m.vz > T(0) ? T(1) : T(-1)) * (t2 > T(0) ? sqrt_(t2) : T(0));
  }
  const T wp = m.beta * (wx * p[0] + wy * p[1] + wz * p[2]);
  e[0] = m.alpha * p[0] - T(0.5) * (wy * p[2] - wz * p[1]) + wp * wx;
  e[1] = m.alpha * p[1] - T(0.5) * (wz * p[0] - wx * p[2]) + wp * wy;
  e[2] = m.alpha * p[2] - T(0.5) * (wx * p[1] - wy * p[0]) + wp * wz;
  e[3] = wx; e[4] = wy; e[5] = wz;
}

// Both hands at once (packed fp32 lane kernel): the two log6 evaluations are the same straight-line sequence on
// different data, so they run on the halves of F2 values -- packed FMAs, per-half MUFU results and selects.  The series
// forms of alpha / beta are evaluated unconditionally and selected (7 packed FMAs instead of a divergent branch); the
// near-pi form (rare) falls back to the scalar code on each half.
GIK_HD bool log6_near_pi(const Log6Mid<F2>& m) {
  const float lim = 3.14159265358979323846f - 1e-2f;
  return m.theta.x >= lim || m.theta.y >= lim;
}
GIK_HD void log6_pre_v(F2 vx, F2 vy, F2 vz, F2 tr, Log6Mid<F2>& m) {
  const F2 c = min_(max_((tr - F2(1.0f)) * F2(0.5f), F2(-1.0f)), F2(1.0f));
  const F2 s = F2(0.5f) * sqrt_(vx * vx + vy * vy + vz * vz);
  const F2 theta = atan2_pos(s, c);
  const F2 tiny = F2(Num<float>::kTinyS);
  const F2 fac = sel_(gt_(s, tiny), F2(0.5f) * (theta * rcp_(s)), F2(0.5f));
  m.wx = fac * vx; m.wy = fac * vy; m.wz = fac * vz;
  const F2 t2 = theta * theta;
  const B2 front = ge_(c, F2(0.0f));
  const F2 num = sel_(front, F2(1.0f) + c, s);
  const F2 den = sel_(front, s, F2(1.0f) - c);
  const F2 alpha_g = F2(0.5f) * theta * (num * rcp_(max_(den, tiny)));
  const F2 beta_g = (F2(1.0f) - alpha_g) * rcp_(max_(t2, tiny));
  // The packed kernel is bound by FMA-pipe slots, and fp32 needs no series near theta = 0: alpha = (theta / s) (1 + c) / 2
  // is a product of factors that each keep their relative accuracy (theta is computed FROM s, so the ratio is clean),
  // and beta = (1 - alpha) / theta^2 -- whose cancellation costs it ~1e-7 / theta^2 absolute -- enters e only as
  // beta (w.p) w with |w| = theta: an error of ~1e-7 |p|, the same as alpha's own rounding.  Seven packed FMAs and two
  // selects less per iteration: config 2 45.8 -> 47.1 M solves/s.
  m.alpha = sel_(gt_(s, tiny), alpha_g, F2(1.0f));     // (exactly zero rotation error: theta = 0 would zero the product)
  m.beta = beta_g;
  m.vx = vx; m.vy = vy; m.vz = vz;
  m.c = c; m.theta = theta;
}
GIK_HD void log6_pre(const F2 (&R)[9], Log6Mid<F2>& m) {
  log6_pre_v(R[7] - R[5], R[2] - R[6], R[3] - R[1], R[0] + R[4] + R[8], m);
  m.d0 = R[0]; m.d1 = R[4]; m.d2 = R[8];
}

GIK_HD void log6_post(const Log6Mid<F2>& m, const F2 (&p)[3], F2 (&e)[6]) {
  if (log6_near_pi(m)) {                           // pinocchio's near-pi form on either hand: scalar code per half
    Log6Mid<float> ml, mr;
    ml.vx = m.vx.x; ml.vy = m.vy.x; ml.vz = m.vz.x; ml.d0 = m.d0.x; ml.d1 = m.d1.x; ml.d2 = m.d2.x; ml.c = m.c.x;
    ml.theta = m.theta.x; ml.wx = m.wx.x; ml.wy = m.wy.x; ml.wz = m.wz.x; ml.alpha = m.alpha.x; ml.beta = m.beta.x;
    mr.vx = m.vx.y; mr.vy = m.vy.y; mr.vz = m.vz.y; mr.d0 = m.d0.y; mr.d1 = m.d1.y; mr.d2 = m.d2.y; mr.c = m.c.y;
    mr.theta = m.theta.y; mr.wx = m.wx.y; mr.wy = m.wy.y; mr.wz = m.wz.y; mr.alpha = m.alpha.y; mr.beta = m.beta.y;
    const float pl[3] = {p[0].x, p[1].x, p[2].x}, pr[3] = {p[0].y, p[1].y, p[2].y};
    float el[6], er[6];
    log6_post(ml, pl, el);
    log6_post(mr, pr, er);
#pragma unroll
    for (int i = 0; i < 6; ++i) e[i] = F2(el[i], er[i]);
    return;
  }
  const F2 wx = m.wx, wy = m.wy, wz = m.wz;
  const F2 wp = m.beta * (wx * p[0] + wy * p[1] + wz * p[2]);
  e[0] = m.alpha * p[0] - F2(0.5f) * (wy * p[2] - wz * p[1]) + wp * wx;
  e[1] = m.alpha * p[1] - F2(0.5f) * (wz * p[0] - wx * p[2]) + wp * wy;
  e[2] = m.alpha * p[2] - F2(0.5f) * (wx * p[1] - wy * p[0]) + wp * wz;
  e[3] = wx; e[4] = wy; e[5] = wz;
}

template <typename T>
GIK_HD void log6(const T (&R)[9], const T (&p)[3], T (&e)[6]) {
  Log6Mid<T> m;
  log6_pre(R, m);
  log6_post(m, p, e);
}

// ------------------------------------------------------------------------------------------------------
// Backward walk of one hand's chain.  (B, b) is the pose of the current joint frame expressed in the hand
// frame; A[:, K] receives the LOCAL Jacobian column of chain joint K ([linear; angular]).  On return (B, b)
// is hand^-1 in the world.  OFF maps chain joint K >= 1 to its slot in the active-joint arrays.
// ------------------------------------------------------------------------------------------------------
template <typename T, int K, int OFF, uint32_t TZ>
GIK_HD void chain_step(const ArmConst<T>& ac, const T (&cs)[kActive], const T (&sn)[kActive], T (&B)[9],
                       T (&b)[3], T (&A)[6][7]) {
  constexpr int AX = chain_axis(K), I = (AX + 1) % 3, J = (AX + 2) % 3;
  constexpr int SLOT = K == 0 ? 0 : OFF + K;
  const T ax = B[AX], ay = B[3 + AX], az = B[6 + AX];
  if constexpr (K == 6) {  // (B, b) is still the constant frame offset: the column is a table constant
    A[0][K] = ac.tip_lin[0]; A[1][K] = ac.tip_lin[1]; A[2][K] = ac.tip_lin[2];
  } else {
    A[0][K] = b[1] * az - b[2] * ay;
    A[1][K] = b[2] * ax - b[0] * az;
    A[2][K] = b[0] * ay - b[1] * ax;
  }
  A[3][K] = ax; A[4][K] = ay; A[5][K] = az;
  const T c = cs[SLOT], s = sn[SLOT];
#pragma unroll
  for (int r = 0; r < 3; ++r) {  // B <- B * Rot(axis, -q)
    const T bi = B[3 * r + I], bj = B[3 * r + J];
    B[3 * r + I] = c * bi - s * bj;
    B[3 * r + J] = s * bi + c * bj;
  }
#pragma unroll
  for (int r = 0; r < 3; ++r) {  // b <- b - B * t, one FMA per non-zero translation component
    if constexpr (!((TZ >> (3 * K + 0)) & 1u)) b[r] -= B[3 * r] * ac.t[K][0];
    if constexpr (!((TZ >> (3 * K + 1)) & 1u)) b[r] -= B[3 * r + 1] * ac.t[K][1];
    if constexpr (!((TZ >> (3 * K + 2)) & 1u)) b[r] -= B[3 * r + 2] * ac.t[K][2];
  }
  if constexpr (K > 0) chain_step<T, K - 1, OFF, TZ>(ac, cs, sn, B, b, A);
}

template <typename T, int OFF, uint32_t TZ>
GIK_HD void hand_chain(const ArmConst<T>& ac, const T (&cs)[kActive], const T (&sn)[kActive], T (&B)[9],
                       T (&b)[3], T (&A)[6][7]) {
#pragma unroll
  for (int i = 0; i < 9; ++i) B[i] = ac.finv_R[i];
#pragma unroll
  for (int i = 0; i < 3; ++i) b[i] = ac.finv_p[i];
  chain_step<T, 6, OFF, TZ>(ac, cs, sn, B, b, A);
}

// hook target of one hand: cube * hook offset (tools.getcubeplacement, tools.py:54-59)
template <typename T>
GIK_HD void hook_target(const ArmConst<T>& ac, const T (&cube)[12], T (&tgt)[12]) {
#pragma unroll
  for (int r = 0; r < 3; ++r) {
#pragma unroll
    for (int c = 0; c < 3; ++c)
      tgt[3 * r + c] = cube[3 * r] * ac.hook_R[c] + cube[3 * r + 1] * ac.hook_R[3 + c] +
                       cube[3 * r + 2] * ac.hook_R[6 + c];
    tgt[9 + r] = cube[9 + r] + cube[3 * r] * ac.hook_p[0] + cube[3 * r + 1] * ac.hook_p[1] +
                 cube[3 * r + 2] * ac.hook_p[2];
  }
}

// e = log6(hand^-1 * target), hand^-1 = (B, b); in two halves (see log6_pre / log6_post)
template <typename T>
struct ErrMid { Log6Mid<T> m; T p[3]; };
template <typename T>
GIK_HD void hand_error_pre(const T (&B)[9], const T (&b)[3], const T (&tgt)[12], ErrMid<T>& em) {
  T R[9];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
#pragma unroll
    for (int c = 0; c < 3; ++c)
      R[3 * r + c] = B[3 * r] * tgt[c] + B[3 * r + 1] * tgt[3 + c] + B[3 * r + 2] * tgt[6 + c];
    em.p[r] = b[r] + B[3 * r] * tgt[9] + B[3 * r + 1] * tgt[10] + B[3 * r + 2] * tgt[11];
  }
  log6_pre(R, em.m);
}
// (Measured and dropped: trace and antisymmetric part of R accumulated directly -- the same 27 products, five additions
// fewer, the diagonal only near theta = pi: config 2 fp32 45.8 -> 44.6 M solves/s, config 4 24.8 -> 25.0 ms.  Three
// six-term accumulation chains are longer than nine three-term ones, and ptxas spilled more.)
template <typename T>
GIK_HD void hand_error_post(const ErrMid<T>& em, T (&e)[6]) { log6_post(em.m, em.p, e); }

// One hand's share of the damped least-squares step, in two phases around the only coupling between the hands (the
// chest joint).  With G = A A^T + lambda I = L L^T (A = 6x6 arm block, c = chest column):
//   phase 1: yf = L^-1 e, zf = L^-1 c, Sy = zf.yf = c.G^-1 e, Sz = zf.zf = c.G^-1 c
//   [both hands: kappa = dq_chest = (SyL + SyR) / (1 + SzL + SzR), Sherman-Morrison]
//   phase 2: dq_arm = A^T L^-T (yf - kappa zf)        (= A^T G^-1 (e - kappa c))
// so the two right-hand sides share the forward substitution and need ONE backward substitution and ONE A^T product.
template <typename T>
struct HandState {
  T A[6][6];     // arm block of the LOCAL Jacobian (columns of the six arm joints)
  T L[6][6];     // Cholesky factor, strictly lower part (scaled), inv[j] = 1 / L[j][j]
  T inv[6];
  T yf[6], zf[6];
};

// G = A A^T + lambda I (arm block, lower triangle) and its Cholesky factor into hs.L / hs.inv.
// Two structural facts of the compiled chain save 30 of the 126 Gram products: the tip joint's column is constant, so
// its outer product comes from the table (ac.g6; G6 = false keeps the products -- fp64, where the lane and pair
// kernels stay bit-identical, and callers whose constants are lane-indexed constant loads: config 4 measured 45.1 ms
// with the table against 40.3 before the pair kernel kept its constants in registers); and chain joints 2 and 3 turn
// about the same axis with a rotation-free placement between them, so their angular parts A[3..5][2] and A[3..5][3]
// are the same values -- the angular-angular block takes 2 a a^T once and the angular-linear block a (l_2 + l_3)^T.
template <typename T, bool G6>
GIK_HD void gram_cholesky(const ArmConst<T>& ac, const T (&A)[6][7], T lambda, HandState<T>& hs) {
  static_assert(chain_axis(2) == chain_axis(3), "parallel consecutive axes assumed by the Gram shortcut");
  T (&L)[6][6] = hs.L;
  T l23[3], a2[3];
#pragma unroll
  for (int j = 0; j < 3; ++j) { l23[j] = A[j][2] + A[j][3]; a2[j] = A[3 + j][2] + A[3 + j][2]; }
#pragma unroll
  for (int i = 0; i < 6; ++i)
#pragma unroll
    for (int j = 0; j <= i; ++j) {
      T g;
      if constexpr (G6) {
        const T g0 = (i == j) ? ac.g6[i * (i + 1) / 2 + j] + lambda : ac.g6[i * (i + 1) / 2 + j];
        g = A[i][1] * A[j][1] + g0;
      } else {
        g = (i == j) ? A[i][1] * A[j][1] + lambda : A[i][1] * A[j][1];
        g += A[i][6] * A[j][6];
      }
      if (i >= 3 && j >= 3) g += a2[i - 3] * A[j][2];
      else if (i >= 3) g += A[i][2] * l23[j];
      else { g += A[i][2] * A[j][2]; g += A[i][3] * A[j][3]; }
      g += A[i][4] * A[j][4];
      g += A[i][5] * A[j][5];
      L[i][j] = g;
    }
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    T d = L[j][j];
#pragma unroll
    for (int k = 0; k < j; ++k) d -= L[j][k] * L[j][k];
    hs.inv[j] = rsqrt_(max_(d, Num<T>::kPivotFloor));
#pragma unroll
    for (int i = j + 1; i < 6; ++i) {
      T v = L[i][j];
#pragma unroll
      for (int k = 0; k < j; ++k) v -= L[i][k] * L[j][k];
      L[i][j] = v * hs.inv[j];
    }
  }
}

template <typename T, int OFF, uint32_t TZ, bool G6 = true>
GIK_HD void hand_phase1(const ArmConst<T>& ac, const T (&cs)[kActive], const T (&sn)[kActive], const T (&tgt)[12],
                        T lambda, HandState<T>& hs, T& Sy, T& Sz, T& resid2) {
  T B[9], b[3], A[6][7], e[6];
  hand_chain<T, OFF, TZ>(ac, cs, sn, B, b, A);
  ErrMid<T> em;
  hand_error_pre(B, b, tgt, em);
  hand_error_post(em, e);
  resid2 = e[0] * e[0] + e[1] * e[1] + e[2] * e[2] + e[3] * e[3] + e[4] * e[4] + e[5] * e[5];   // ||e||^2
  gram_cholesky<T, G6>(ac, A, lambda, hs);
  // forward substitution of both right-hand sides: e and the chest column c = A[:,0]
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    T a = e[j], cc = A[j][0];
#pragma unroll
    for (int k = 0; k < j; ++k) { a -= hs.L[j][k] * hs.yf[k]; cc -= hs.L[j][k] * hs.zf[k]; }
    hs.yf[j] = a * hs.inv[j]; hs.zf[j] = cc * hs.inv[j];
  }
  Sy = hs.zf[0] * hs.yf[0]; Sz = hs.zf[0] * hs.zf[0];
#pragma unroll
  for (int i = 1; i < 6; ++i) { Sy += hs.zf[i] * hs.yf[i]; Sz += hs.zf[i] * hs.zf[i]; }
#pragma unroll
  for (int i = 0; i < 6; ++i)
#pragma unroll
    for (int k = 0; k < 6; ++k) hs.A[i][k] = A[i][k + 1];
}

template <typename T>
GIK_HD void hand_phase2(const HandState<T>& hs, T kappa, T (&dq)[6]) {
  T t[6];
#pragma unroll
  for (int j = 0; j < 6; ++j) t[j] = hs.yf[j] - kappa * hs.zf[j];
#pragma unroll
  for (int j = 5; j >= 0; --j) {      // backward substitution L^T x = t
    T a = t[j];
#pragma unroll
    for (int k = j + 1; k < 6; ++k) a -= hs.L[k][j] * t[k];
    t[j] = a * hs.inv[j];
  }
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    T a = hs.A[0][k] * t[0];
#pragma unroll
    for (int i = 1; i < 6; ++i) a += hs.A[i][k] * t[i];
    dq[k] = a;
  }
}

// ------------------------------------------------------------------------------------------------------
// Spherical-wrist form of the UNDAMPED step (lambda = 0; tables with kWristTZ).
//
// With J = [c_L A_L 0; c_R 0 A_R] of full row rank, pinv(J) e = J^T (J J^T)^-1 e, and because the arm blocks A are
// SQUARE, A^T (A A^T)^-1 = A^-1: with u = A^-1 e, w = A^-1 c (per hand)
//     dq_chest = kappa = (u_L.w_L + u_R.w_R) / (1 + |w_L|^2 + |w_R|^2),      dq_arm = u - kappa w
// (Sherman-Morrison on blockdiag(A A^T) + c c^T, the same identity as the Cholesky path, with G^-1 = A^-T A^-1).  No Gram
// matrix, no factorisation of A A^T, no A^T product, and the conditioning is cond(A) instead of cond(A)^2.
// The min-norm solution is unchanged when both sides are multiplied by an invertible X (J -> X J, e -> X e), so every
// hand's rows may be expressed at ANOTHER REFERENCE POINT: v' = v + w x r moves the point where the linear velocity
// is taken from the hand origin to r.  At the WRIST CENTRE (the common point of the axes of chain joints 4, 5, 6) the
// linear parts of those three columns vanish, A' = [M 0; Wa Wb] is block triangular, and A'^-1 is two 3x3 solves:
//     M x_123 = rhs_v                      M = [m1 m2 m3], m_K = (b_K - r) x a_K           (Cramer, one reciprocal)
//     Wb x_456 = rhs_w - Wa x_123          Wb = [a4 a5 a6] with a5 _|_ a4, a5 _|_ a6, |a_K| = 1 (consecutive
//                                          perpendicular axes):  x5 = a5.rho, x4 = (n.rho)/(n.a4) with n = a5 x a6,
//                                          x6 = a6.rho - (a6.a4) x4                                  (one reciprocal)
// The chain is walked as before (backwards from the hand frame) with the translation taken relative to the wrist
// centre: it is exactly 0 at joint 5, so only joints 0..3 need their linear parts.  Reciprocals are capped
// (Num<T>::kRcpCap) where the arm or the wrist is singular, as the Cholesky path floors its pivots.
// ------------------------------------------------------------------------------------------------------
template <typename T>
struct WristState { T u[6], w[6]; };

template <typename T, int K, int OFF>
GIK_HD void chain_rotate(const T (&cs)[kActive], const T (&sn)[kActive], T (&B)[9]) {   // B <- B * Rot(axis_K, -q_K)
  constexpr int AX = chain_axis(K), I = (AX + 1) % 3, J = (AX + 2) % 3;
  constexpr int SLOT = K == 0 ? 0 : OFF + K;
  const T c = cs[SLOT], s = sn[SLOT];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const T bi = B[3 * r + I], bj = B[3 * r + J];
    B[3 * r + I] = c * bi - s * bj;
    B[3 * r + J] = s * bi + c * bj;
  }
}
template <typename T, int K, uint32_t TZ>
GIK_HD void chain_translate(const ArmConst<T>& ac, const T (&B)[9], T (&b)[3]) {       // b <- b - B * t_K
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    if constexpr (!((TZ >> (3 * K + 0)) & 1u)) b[r] -= B[3 * r] * ac.t[K][0];
    if constexpr (!((TZ >> (3 * K + 1)) & 1u)) b[r] -= B[3 * r + 1] * ac.t[K][1];
    if constexpr (!((TZ >> (3 * K + 2)) & 1u)) b[r] -= B[3 * r + 2] * ac.t[K][2];
  }
}
template <typename T>
GIK_HD void cross3(const T (&a)[3], const T (&b)[3], T (&o)[3]) {
  o[0] = a[1] * b[2] - a[2] * b[1];
  o[1] = a[2] * b[0] - a[0] * b[2];
  o[2] = a[0] * b[1] - a[1] * b[0];
}
template <typename T>
GIK_HD T dot3(const T (&a)[3], const T (&b)[3]) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
template <typename T>
GIK_HD T rcp_capped(T d) { return min_(max_(rcp_(d), T(-Num<T>::kRcpCap)), T(Num<T>::kRcpCap)); }

template <typename T, int OFF, uint32_t TZ>
GIK_HD void hand_wrist_phase1(const ArmConst<T>& ac, const T (&cs)[kActive], const T (&sn)[kActive], const T (&tgt)[12],
                              WristState<T>& ws, T& Sy, T& Sz, T& resid2) {
  static_assert((TZ & kWristTZ) == kWristTZ, "spherical-wrist path instantiated for a table pattern without one");
  static_assert(chain_axis(4) == 0 && chain_axis(5) == 1 && chain_axis(6) == 2 && chain_axis(2) == 1 && chain_axis(3) == 1 &&
                chain_axis(1) == 2 && chain_axis(0) == 2, "axis pattern assumed below");
  constexpr bool TIPZ = (TZ & kTipZ) != 0;
  T B[9], b[3], a4[3], a5[3], a6[3];
  if constexpr (TIPZ) {
    // finv_R * Rot(z, -q6) = Rot(z, -theta), theta = q6 - tip_psi (cs / sn of the tip slot are those of theta):
    // B = [ct st 0; -st ct 0; 0 0 1], a6 = (0, 0, 1), a5 = (st, ct, 0).  Joint 5 (y) then acts on those zeros, and row 2
    // of joint 4's rotation (x) starts from (s5, 0, c5).
    const T ct = cs[OFF + 6], st = sn[OFF + 6], c5 = cs[OFF + 5], s5 = sn[OFF + 5], c4 = cs[OFF + 4], s4 = sn[OFF + 4];
    a5[0] = st; a5[1] = ct;
    B[0] = c5 * ct; B[3] = -(c5 * st); B[6] = s5;
    const T b02 = -(s5 * ct), b12 = s5 * st;
#pragma unroll
    for (int r = 0; r < 3; ++r) { a4[r] = B[3 * r]; b[r] = -(B[3 * r] * ac.t[5][0]); }
    // joint 4 (x): columns 1, 2 <- (c4 b1 - s4 b2, s4 b1 + c4 b2)
    B[1] = c4 * st - s4 * b02; B[2] = s4 * st + c4 * b02;
    B[4] = c4 * ct - s4 * b12; B[5] = s4 * ct + c4 * b12;
    B[7] = -(s4 * c5);         B[8] = c4 * c5;
  } else {
#pragma unroll
    for (int i = 0; i < 9; ++i) B[i] = ac.finv_R[i];
    // joint 6 (z): its axis is constant in the hand frame; after its step the translation relative to the wrist centre is 0
    a6[0] = B[2]; a6[1] = B[5]; a6[2] = B[8];
    chain_rotate<T, 6, OFF>(cs, sn, B);
    // joint 5 (y)
    a5[0] = B[1]; a5[1] = B[4]; a5[2] = B[7];
    chain_rotate<T, 5, OFF>(cs, sn, B);
#pragma unroll
    for (int r = 0; r < 3; ++r) b[r] = -(B[3 * r] * ac.t[5][0]);
    // joint 4 (x): still on the wrist centre's axes -- no linear part
#pragma unroll
    for (int r = 0; r < 3; ++r) a4[r] = B[3 * r];
    chain_rotate<T, 4, OFF>(cs, sn, B);
  }
  chain_translate<T, 4, TZ>(ac, B, b);
  // joints 3, 2 (y, y: parallel axes, the rotation about y leaves column 1 alone), 1 (z), chest (z: the same axis as joint 1)
  const T ay[3] = {B[1], B[4], B[7]};
  T m3[3], m2[3], m1[3], m0[3];
  cross3(b, ay, m3);
  chain_rotate<T, 3, OFF>(cs, sn, B);
  chain_translate<T, 3, TZ>(ac, B, b);
  cross3(b, ay, m2);
  chain_rotate<T, 2, OFF>(cs, sn, B);
  chain_translate<T, 2, TZ>(ac, B, b);
  const T az[3] = {B[2], B[5], B[8]};
  cross3(b, az, m1);
  chain_rotate<T, 1, OFF>(cs, sn, B);
  chain_translate<T, 1, TZ>(ac, B, b);
  cross3(b, az, m0);
  chain_rotate<T, 0, OFF>(cs, sn, B);
  chain_translate<T, 0, TZ>(ac, B, b);
  // (B, b + rw) = hand^-1: the error in the hand frame, then moved to the wrist centre
  T bf[3], e[6];
#pragma unroll
  for (int r = 0; r < 3; ++r) bf[r] = b[r] + ac.rw[r];
  ErrMid<T> em;
  hand_error_pre(B, bf, tgt, em);
  hand_error_post(em, e);
  resid2 = e[0] * e[0] + e[1] * e[1] + e[2] * e[2] + e[3] * e[3] + e[4] * e[4] + e[5] * e[5];
  const T ew[3] = {e[3], e[4], e[5]};
  T ev[3];
  cross3(ew, ac.rw, ev);
#pragma unroll
  for (int r = 0; r < 3; ++r) ev[r] += e[r];
  // M x_123 = rhs_v for rhs = e' and the chest column c' = [m0; az]
  T c1[3], c2[3], c3[3];
  cross3(m2, m3, c1);
  cross3(m3, m1, c2);
  cross3(m1, m2, c3);
  const T rdet = rcp_capped(dot3(m1, c1));
  T (&u)[6] = ws.u;
  T (&w)[6] = ws.w;
  u[0] = dot3(c1, ev) * rdet; u[1] = dot3(c2, ev) * rdet; u[2] = dot3(c3, ev) * rdet;
  w[0] = dot3(c1, m0) * rdet; w[1] = dot3(c2, m0) * rdet; w[2] = dot3(c3, m0) * rdet;
  // rho = rhs_w - a1 x1 - ay (x2 + x3)
  T ru[3], rc[3];
  const T su = u[1] + u[2], sw = w[1] + w[2], w0m = T(1) - w[0];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    ru[r] = ew[r] - az[r] * u[0] - ay[r] * su;
    rc[r] = az[r] * w0m - ay[r] * sw;
  }
  // wrist: [a4 a5 a6] x_456 = rho
  if constexpr (TIPZ) {
    // a6 = (0, 0, 1), a5 = (st, ct, 0), n = a5 x a6 = (ct, -st, 0), n.a4 = c5, a6.a4 = s5
    const T ct = a5[1], st = a5[0], s5 = a4[2];
    const T rd = rcp_capped(cs[OFF + 5]);
    u[3] = (ct * ru[0] - st * ru[1]) * rd; u[4] = st * ru[0] + ct * ru[1]; u[5] = ru[2] - s5 * u[3];
    w[3] = (ct * rc[0] - st * rc[1]) * rd; w[4] = st * rc[0] + ct * rc[1]; w[5] = rc[2] - s5 * w[3];
  } else {
    T n[3];
    cross3(a5, a6, n);
    const T rd = rcp_capped(dot3(n, a4)), g = dot3(a6, a4);
    u[3] = dot3(n, ru) * rd; u[4] = dot3(a5, ru); u[5] = dot3(a6, ru) - g * u[3];
    w[3] = dot3(n, rc) * rd; w[4] = dot3(a5, rc); w[5] = dot3(a6, rc) - g * w[3];
  }
  Sy = u[0] * w[0]; Sz = w[0] * w[0];
#pragma unroll
  for (int i = 1; i < 6; ++i) { Sy += u[i] * w[i]; Sz += w[i] * w[i]; }
}

template <typename T>
GIK_HD void hand_wrist_phase2(const WristState<T>& ws, T kappa, T (&dq)[6]) {
#pragma unroll
  for (int k = 0; k < 6; ++k) dq[k] = ws.u[k] - kappa * ws.w[k];
}

// Sherman-Morrison coupling of the two arm blocks through the shared chest joint: dq_chest = c.D^-1 e / (1 + c.D^-1 c)
template <typename T>
GIK_HD T chest_rate(T SyL, T SzL, T SyR, T SzR) { return div_(SyL + SyR, T(1) + (SzL + SzR)); }

// One full iteration at q: SQUARED residual norms of both hands and the step direction dq = J^+ e.  (The predicate
// ||e|| < eps of inverse_geometry.py:70 is evaluated as ||e||^2 < eps^2; the norm itself is only taken when a result is stored.)
template <typename T, bool FAST, uint32_t TZ = 0, bool WRIST = false>
GIK_HD void ik_iteration(const DevTable<T>& tab, const T (&q)[kActive], const T (&tgt)[2][12], T lambda,
                         T (&dq)[kActive], T& resid2L, T& resid2R) {
  T cs[kActive], sn[kActive];
#pragma unroll
  for (int i = 0; i < kActive; ++i) {
    // tip-aligned wrist step: the tip joints' slots carry the angle q6 - tip_psi (hand_wrist_phase1)
    const T ang = (WRIST && (TZ & kTipZ) && (i == 6 || i == 12)) ? q[i] - tab.arm[i / 12].tip_psi : q[i];
    sincos_<FAST>(ang, sn[i], cs[i]);
  }
  T SyL, SzL, SyR, SzR;
  if constexpr (WRIST) {          // lambda = 0 on a spherical-wrist table: two 3x3 solves per hand
    WristState<T> wL, wR;
    hand_wrist_phase1<T, 0, TZ>(tab.arm[0], cs, sn, tgt[0], wL, SyL, SzL, resid2L);
    hand_wrist_phase1<T, 6, TZ>(tab.arm[1], cs, sn, tgt[1], wR, SyR, SzR, resid2R);
    const T kappa = chest_rate(SyL, SzL, SyR, SzR);
    dq[0] = kappa;
    T dL[6], dR[6];
    hand_wrist_phase2(wL, kappa, dL);
    hand_wrist_phase2(wR, kappa, dR);
#pragma unroll
    for (int k = 0; k < 6; ++k) { dq[1 + k] = dL[k]; dq[7 + k] = dR[k]; }
    return;
  }
  HandState<T> hL, hR;
  // the fp64 lane kernel keeps the tip products so that it stays bit-identical to the fp64 pair kernel (the default)
  constexpr bool G6 = sizeof(T) == 4;
  hand_phase1<T, 0, TZ, G6>(tab.arm[0], cs, sn, tgt[0], lambda, hL, SyL, SzL, resid2L);
  hand_phase1<T, 6, TZ, G6>(tab.arm[1], cs, sn, tgt[1], lambda, hR, SyR, SzR, resid2R);
  const T kappa = chest_rate(SyL, SzL, SyR, SzR);
  dq[0] = kappa;
  T dL[6], dR[6];
  hand_phase2(hL, kappa, dL);
  hand_phase2(hR, kappa, dR);
#pragma unroll
  for (int k = 0; k < 6; ++k) { dq[1 + k] = dL[k]; dq[7 + k] = dR[k]; }
}

// fp32 lane kernel: the same iteration with (left, right) packed.  State: chest angle q0, arm angles q2[k] =
// (q_L[k], q_R[k]), targets tgt2 = (left hook target, right hook target).  Returns the squared residuals and applies
// nothing: the caller updates q0 with dq0 and q2 with dq2.
struct PackedTable {
  ArmConst<F2> arm;        // (left, right) constants of the two chains
  F2 lo[6], hi[6];         // arm joint limits
  float lo0, hi0;          // chest limits
};

template <uint32_t TZ, bool WRIST = false>
GIK_HD void ik_iteration_packed(const PackedTable& pt, float q0, const F2 (&q2)[6], const F2 (&tgt2)[12], float lambda,
                                float& dq0, F2 (&dq2)[6], float& resid2L, float& resid2R) {
  F2 cs[kActive], sn[kActive];      // only chain slots 0..6 are used
  {
    float s, c;
    sincos_<true>(q0, s, c);
    cs[0] = F2(c); sn[0] = F2(s);
  }
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    float sl, cl, sr, cr;
    // tip-aligned wrist step: the tip joint's slot carries the angle q6 - tip_psi (hand_wrist_phase1)
    const bool tip = WRIST && (TZ & kTipZ) && k == 5;
    sincos_<true>(tip ? q2[k].x - pt.arm.tip_psi.x : q2[k].x, sl, cl);
    sincos_<true>(tip ? q2[k].y - pt.arm.tip_psi.y : q2[k].y, sr, cr);
    cs[1 + k] = F2(cl, cr); sn[1 + k] = F2(sl, sr);
  }
  F2 Sy, Sz, r2;
  if constexpr (WRIST) {
    WristState<F2> ws;
    hand_wrist_phase1<F2, 0, TZ>(pt.arm, cs, sn, tgt2, ws, Sy, Sz, r2);
    const float kappa = chest_rate(Sy.x, Sz.x, Sy.y, Sz.y);
    dq0 = kappa;
    hand_wrist_phase2(ws, F2(kappa), dq2);
  } else {
    HandState<F2> hs;
    hand_phase1<F2, 0, TZ, true>(pt.arm, cs, sn, tgt2, F2(lambda), hs, Sy, Sz, r2);
    const float kappa = chest_rate(Sy.x, Sz.x, Sy.y, Sz.y);
    dq0 = kappa;
    hand_phase2(hs, F2(kappa), dq2);
  }
  resid2L = r2.x; resid2R = r2.y;
}

// q <- clamp(q + dt dq)  (pin.integrate on an all-revolute model :86, projecttojointlimits :89)
template <typename T>
GIK_HD void apply_step(const DevTable<T>& tab, T (&q)[kActive], const T (&dq)[kActive], T dt) {
#pragma unroll
  for (int i = 0; i < kActive; ++i) q[i] = min_(max_(tab.lo[i], q[i] + dt * dq[i]), tab.hi[i]);
}

// Residual norms only (no Jacobian use) -- used for the final evaluation of an exhausted problem.
template <typename T, bool FAST>
GIK_HD void fk_frames(const DevTable<T>& tab, const T (&q)[kActive], T (&frames)[2][12]) {
  T cs[kActive], sn[kActive];
#pragma unroll
  for (int i = 0; i < kActive; ++i) sincos_<FAST>(q[i], sn[i], cs[i]);
  T B[9], b[3], A[6][7];
  hand_chain<T, 0, 0>(tab.arm[0], cs, sn, B, b, A);
#pragma unroll
  for (int r = 0; r < 3; ++r) {  // invert: R = B^T, p = -B^T b
#pragma unroll
    for (int c = 0; c < 3; ++c) frames[0][3 * r + c] = B[3 * c + r];
    frames[0][9 + r] = -(B[r] * b[0] + B[3 + r] * b[1] + B[6 + r] * b[2]);
  }
  hand_chain<T, 6, 0>(tab.arm[1], cs, sn, B, b, A);
#pragma unroll
  for (int r = 0; r < 3; ++r) {
#pragma unroll
    for (int c = 0; c < 3; ++c) frames[1][3 * r + c] = B[3 * c + r];
    frames[1][9 + r] = -(B[r] * b[0] + B[3 + r] * b[1] + B[6 + r] * b[2]);
  }
}

template <typename T, bool FAST>
GIK_HD void frame_jacobians(const DevTable<T>& tab, const T (&q)[kActive], T (&AL)[6][7], T (&AR)[6][7]) {
  T cs[kActive], sn[kActive];
#pragma unroll
  for (int i = 0; i < kActive; ++i) sincos_<FAST>(q[i], sn[i], cs[i]);
  T B[9], b[3];
  hand_chain<T, 0, 0>(tab.arm[0], cs, sn, B, b, AL);
  hand_chain<T, 6, 0>(tab.arm[1], cs, sn, B, b, AR);
}

}  // namespace gik

// ------------------------------------------------------------------------------------------------------
// SE3 interpolation for the edge march: pin.SE3.Interpolate(A, B, alpha) = A * exp6(alpha * log6(A^-1 B))
// (path.py:141).  Poses are 12-vectors: rotation row-major (9) + translation (3).
// ------------------------------------------------------------------------------------------------------
namespace gik {

// xi = log6(A^-1 B)
template <typename T>
GIK_HD void se3_delta(const T (&A)[12], const T (&Bp)[12], T (&xi)[6]) {
  T R[9], p[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
#pragma unroll
    for (int c = 0; c < 3; ++c) R[3 * r + c] = A[r] * Bp[c] + A[3 + r] * Bp[3 + c] + A[6 + r] * Bp[6 + c];
    p[r] = A[r] * (Bp[9] - A[9]) + A[3 + r] * (Bp[10] - A[10]) + A[6 + r] * (Bp[11] - A[11]);
  }
  log6(R, p, xi);
}

// out = A * exp6(alpha * xi)
template <typename T>
GIK_HD void se3_advance(const T (&A)[12], const T (&xi)[6], T alpha, T (&out)[12]) {
  const T vx = alpha * xi[0], vy = alpha * xi[1], vz = alpha * xi[2];
  const T wx = alpha * xi[3], wy = alpha * xi[4], wz = alpha * xi[5];
  const T t2 = wx * wx + wy * wy + wz * wz;
  T a, b, c;  // sin(t)/t, (1-cos t)/t^2, (t - sin t)/t^3
  if (t2 < Num<T>::kSeriesT2) {
    a = T(1) - t2 * (T(1.0 / 6) - t2 * (T(1.0 / 120) - t2 * (T(1.0 / 5040) - t2 * T(1.0 / 362880))));
    b = T(0.5) - t2 * (T(1.0 / 24) - t2 * (T(1.0 / 720) - t2 * (T(1.0 / 40320) - t2 * T(1.0 / 3628800))));
    c = T(1.0 / 6) - t2 * (T(1.0 / 120) - t2 * (T(1.0 / 5040) - t2 * (T(1.0 / 362880) - t2 * T(1.0 / 39916800))));
  } else {
    const T t = sqrt_(t2);
    T st, ct;
    sincos_<false>(t, st, ct);
    a = st / t; b = (T(1) - ct) / t2; c = (t - st) / (t2 * t);
  }
  // E = I + a W + b W^2 ; V = I + b W + c W^2 ; W^2 = w w^T - t2 I
  T E[9], d[3];
  E[0] = T(1) + b * (wx * wx - t2); E[1] = -a * wz + b * wx * wy;       E[2] = a * wy + b * wx * wz;
  E[3] = a * wz + b * wx * wy;      E[4] = T(1) + b * (wy * wy - t2);   E[5] = -a * wx + b * wy * wz;
  E[6] = -a * wy + b * wx * wz;     E[7] = a * wx + b * wy * wz;        E[8] = T(1) + b * (wz * wz - t2);
  const T wv = wx * vx + wy * vy + wz * vz;
  d[0] = vx + b * (wy * vz - wz * vy) + c * (wx * wv - t2 * vx);
  d[1] = vy + b * (wz * vx - wx * vz) + c * (wy * wv - t2 * vy);
  d[2] = vz + b * (wx * vy - wy * vx) + c * (wz * wv - t2 * vz);
#pragma unroll
  for (int r = 0; r < 3; ++r) {
#pragma unroll
    for (int cc = 0; cc < 3; ++cc)
      out[3 * r + cc] = A[3 * r] * E[cc] + A[3 * r + 1] * E[3 + cc] + A[3 * r + 2] * E[6 + cc];
    out[9 + r] = A[9 + r] + A[3 * r] * d[0] + A[3 * r + 1] * d[1] + A[3 * r + 2] * d[2];
  }
}

// Placement of step s of an edge marched in nsteps steps, xi = se3_delta(A, B): A * exp6((s / nsteps) xi).  The edge
// kernels solve each step for it and the tree kernels store it with the step's configuration.
template <typename T>
GIK_HD void edge_placement(const T (&A)[12], const T (&xi)[6], int s, int nsteps, T (&out)[12]) {
  se3_advance(A, xi, T(s) / T(nsteps), out);
}

}  // namespace gik
