"""log6 and the SE3 interpolation over the full rotation range, on the CPU: the GIK_HD code of csrc/gik_core.cuh
(scalar fp64 / fp32, and the packed fp32 form with one half near pi and the other not) compiled with g++ against an
extended-precision reference built from a known axis and angle, and against pinocchio's semantics (oracle); the host
copy path.se3_interpolate against the C oracle; and the kernel arithmetic of the IK descent on cubes whose hands start
up to pi away from their targets.  The angle grid puts points on both sides of every branch: the fp64 series threshold
(theta = 0.01), the fp32 series threshold (theta = 0.5), and pinocchio's near-pi form (theta >= pi - 1e-2)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from conftest import ROOT, make_poses, rot_rpy

CSRC = os.path.join(ROOT, "motion-planning-and-control-for-dual-manipulator-robot_b200", "csrc")
PI = np.pi
NEAR_PI = PI - 1e-2                                 # pinocchio's log3 switches to its near-pi form at this angle
THETAS = [0.0, 1e-9, 1e-4, 0.0099, 0.0101, 0.4999, 0.5001, 1.0, 2.0, PI / 2,
          PI - 0.0101, PI - 0.0099, PI - 1e-3, PI - 1e-5, PI - 1e-7, PI]
COORD_AXES = [np.array(a, float) for a in ((1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1))]

HARNESS = r"""
#include <stdint.h>
#include "gik_core.cuh"
using namespace gik;

// M: poses [n][12] (rotation row-major, translation) -> e [n][6] = log6(M) = [v; w]
template <typename T>
static void log6_rows(int64_t n, const double* M, double* e) {
  for (int64_t i = 0; i < n; ++i) {
    T R[9], p[3], o[6];
    for (int k = 0; k < 9; ++k) R[k] = (T)M[i * 12 + k];
    for (int k = 0; k < 3; ++k) p[k] = (T)M[i * 12 + 9 + k];
    log6(R, p, o);
    for (int k = 0; k < 6; ++k) e[i * 6 + k] = o[k];
  }
}
// SE3 interpolation of the edge and tree kernels: A exp6(alpha log6(A^-1 B))
template <typename T>
static void interp_rows(int64_t n, const double* A, const double* B, const double* al, double* out) {
  for (int64_t i = 0; i < n; ++i) {
    T a[12], b[12], xi[6], o[12];
    for (int k = 0; k < 12; ++k) { a[k] = (T)A[i * 12 + k]; b[k] = (T)B[i * 12 + k]; }
    se3_delta(a, b, xi);
    se3_advance(a, xi, (T)al[i], o);
    for (int k = 0; k < 12; ++k) out[i * 12 + k] = o[k];
  }
}

extern "C" {
void h_log6_f64(int64_t n, const double* M, double* e) { log6_rows<double>(n, M, e); }
void h_log6_f32(int64_t n, const double* M, double* e) { log6_rows<float>(n, M, e); }
// packed fp32 (both hands of the lane kernel): problem i of Mx in the .x half, problem i of My in the .y half
void h_log6_f2(int64_t n, const double* Mx, const double* My, double* ex, double* ey) {
  for (int64_t i = 0; i < n; ++i) {
    F2 R[9], p[3], o[6];
    for (int k = 0; k < 9; ++k) R[k] = F2((float)Mx[i * 12 + k], (float)My[i * 12 + k]);
    for (int k = 0; k < 3; ++k) p[k] = F2((float)Mx[i * 12 + 9 + k], (float)My[i * 12 + 9 + k]);
    log6(R, p, o);
    for (int k = 0; k < 6; ++k) { ex[i * 6 + k] = o[k].x; ey[i * 6 + k] = o[k].y; }
  }
}
void h_interp_f64(int64_t n, const double* A, const double* B, const double* al, double* out) { interp_rows<double>(n, A, B, al, out); }
void h_interp_f32(int64_t n, const double* A, const double* B, const double* al, double* out) { interp_rows<float>(n, A, B, al, out); }
}
"""


@pytest.fixture(scope="module")
def rot_lib(tmp_path_factory):
    d = tmp_path_factory.mktemp("rotation_harness")
    src = d / "harness.cpp"
    src.write_text(HARNESS)
    out = d / "librot.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-I", CSRC,
                    "-I", os.path.join(ROOT, "include"), "-o", str(out), str(src)], check=True)
    return ctypes.CDLL(str(out))


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _rows(x):
    return np.ascontiguousarray(x, np.float64)


def dev_log6(lib, M, prec):
    M = _rows(M)
    e = np.zeros((len(M), 6))
    getattr(lib, f"h_log6_{prec}")(ctypes.c_int64(len(M)), _p(M), _p(e))
    return e


def dev_log6_packed(lib, Mx, My):
    Mx, My = _rows(Mx), _rows(My)
    ex, ey = np.zeros((len(Mx), 6)), np.zeros((len(Mx), 6))
    lib.h_log6_f2(ctypes.c_int64(len(Mx)), _p(Mx), _p(My), _p(ex), _p(ey))
    return ex, ey


def dev_interp(lib, A, B, alpha, prec):
    A, B, al = _rows(A), _rows(B), _rows(alpha)
    out = np.zeros((len(A), 12))
    getattr(lib, f"h_interp_{prec}")(ctypes.c_int64(len(A)), _p(A), _p(B), _p(al), _p(out))
    return out


# ------------------------------------------------------------------------------------- extended-precision reference
LD = np.longdouble
PI_LD = np.arccos(LD(-1))


def _hat(w):
    return np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]], dtype=LD)


def exp6_ld(xi):
    """pinocchio exp6 of [v; w] in long double -> (R, p)."""
    v, w = np.asarray(xi[:3], LD), np.asarray(xi[3:], LD)
    t2 = (w * w).sum()
    t = np.sqrt(t2)
    if t < LD(1e-2):
        a = 1 - t2 / 6 + t2 * t2 / 120 - t2 ** 3 / 5040
        b = LD(0.5) - t2 / 24 + t2 * t2 / 720 - t2 ** 3 / 40320
        c = LD(1) / 6 - t2 / 120 + t2 * t2 / 5040 - t2 ** 3 / 362880
    else:
        a, b, c = np.sin(t) / t, (1 - np.cos(t)) / t2, (t - np.sin(t)) / (t2 * t)
    W = _hat(w)
    W2 = W @ W
    eye = np.eye(3, dtype=LD)
    return eye + a * W + b * W2, (eye + b * W + c * W2) @ v


def log6_exact_ld(u, theta, p):
    """The exact log6 of (R(u, theta), p) for theta < pi: w = theta u, v = alpha p - w x p / 2 + beta (w.p) w."""
    th = PI_LD if theta == PI else LD(theta)
    w = np.asarray(u, LD) * th
    p = np.asarray(p, LD)
    t2 = th * th
    if th < LD(1e-3):
        alpha, beta = 1 - t2 / 12 - t2 * t2 / 720, LD(1) / 12 + t2 / 720
    else:
        alpha = th / 2 / np.tan(th / 2)
        beta = (1 - alpha) / t2
    v = alpha * p - np.cross(w, p) / 2 + beta * (w @ p) * w
    return np.concatenate([v, w])


def pose_ld(u, theta, p):
    """(R(u, theta), p) as a 12-row in long double; theta == pi is taken as the long-double pi."""
    th = PI_LD if theta == PI else LD(theta)
    R, _ = exp6_ld(np.concatenate([np.zeros(3, LD), np.asarray(u, LD) * th]))
    return np.concatenate([R.reshape(9), np.asarray(p, LD)])


def mul_ld(A, B):
    Ra, Rb = A[:9].reshape(3, 3), B[:9].reshape(3, 3)
    return np.concatenate([(Ra @ Rb).reshape(9), A[9:] + Ra @ B[9:]])


def _axes(rng, n_random):
    ax = [(a, True) for a in COORD_AXES] + [(np.array([1.0, 1.0, 0.0]) / np.sqrt(2), False)]
    for _ in range(n_random):
        u = rng.standard_normal(3)
        ax.append((u / np.linalg.norm(u), False))
    return ax


def grid_cases(seed, n_random=4):
    """Every (theta, axis) of the grid with a random translation: list of dicts (theta, u, coord, zero, p); `coord`: a
    coordinate axis, `zero`: an axis with a zero component (all coordinate axes, and (1, 1, 0) / sqrt 2)."""
    rng = np.random.default_rng(seed)
    cases = []
    for th in THETAS:
        for u, coord in _axes(rng, n_random):
            cases.append(dict(theta=th, u=u, coord=coord, zero=bool((u == 0).any()), p=rng.uniform(-0.5, 0.5, 3)))
    return cases


def band_tol(prec, theta, zero):
    """Bound on |kernel - exact| for a log6 / interpolation at relative angle theta about an axis with (`zero`) or
    without a zero component."""
    if prec == "f64":
        return 1e-10 if theta < NEAR_PI else 1e-7
    if theta <= 2.0:
        return 1e-6
    if theta < NEAR_PI:
        return 2e-5
    # pinocchio's near-pi form takes sqrt of the diagonal: a component of w that should be 0 is the square root of fp32
    # rounding noise (~3e-4)
    return 1e-3 if zero else 1e-4


def fp32_resolvable(theta, coord, exact_zeros=True):
    """fp32 can tell theta u from -theta u: the antisymmetric part 2 sin(theta) u is above the rounding of R.  A
    rotation about a coordinate axis given directly keeps its exact zeros (`exact_zeros`); as A^-1 B of two rotated
    placements it carries rounding noise in every entry."""
    if theta >= PI:
        return False
    if coord:
        return exact_zeros or PI - theta >= 1e-5
    return PI - theta >= 1e-4


# ----------------------------------------------------------------------------------------------------------- log6
def _log6_inputs(cases, dtype):
    M = np.array([pose_ld(c["u"], c["theta"], c["p"]) for c in cases]).astype(dtype)
    return M.astype(np.float64)


def _check_log6(e, cases, prec, M):
    """e [n,6] kernel logs of the rows M [n,12] (already rounded to the kernel's precision)."""
    from oracle import grasp_ik_np as o
    worst = {}
    for i, c in enumerate(cases):
        th, u, coord = c["theta"], c["u"], c["coord"]
        R = M[i, :9].reshape(3, 3)
        if th < PI and (prec == "f64" or fp32_resolvable(th, coord)):
            ref = log6_exact_ld(u, th, c["p"]).astype(np.float64)
            err = np.abs(e[i] - ref).max()
            tol = band_tol(prec, th, c["zero"])
            assert err < tol, (prec, th, u, err, e[i], ref)
            band = "near_pi" if th >= NEAR_PI else "far"
            worst[band] = max(worst.get(band, 0.0), err)
        else:
            # exactly pi (or below fp32 resolution): the direction of the turn is rounding noise.  |w| = theta, |w_i| =
            # theta |u_i|; on a coordinate axis w is a valid logarithm (exp(w) = R) whichever sign it took
            tol = 1e-7 if prec == "f64" else 1e-3
            w = e[i, 3:]
            assert abs(np.linalg.norm(w) - th) < tol, (prec, th, u, w)
            assert np.abs(np.abs(w) - th * np.abs(u)).max() < tol, (prec, th, u, w)
            if coord:
                Rw, _ = exp6_ld(np.concatenate([np.zeros(3), w]))
                assert np.abs(Rw.astype(np.float64) - R).max() < tol, (prec, th, u, w)
        if prec == "f64":
            # pinocchio's semantics on the very same matrix: the signs of the near-pi form are decided by the same
            # comparisons, so kernel and oracle agree even where the exact log is not defined
            ref_o = o.log6(R, M[i, 9:])
            assert np.abs(e[i] - ref_o).max() < band_tol("f64", th, c["zero"]), (th, u, e[i], ref_o)
    return worst


@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_log6_over_the_rotation_range(rot_lib, prec):
    cases = grid_cases(1)
    M = _log6_inputs(cases, np.float64 if prec == "f64" else np.float32)
    e = dev_log6(rot_lib, M, prec)
    worst = _check_log6(e, cases, prec, M)
    print(f"log6 {prec}: worst |err| per band {worst}")
    assert {"far", "near_pi"} <= set(worst)


def test_packed_log6_with_one_half_near_pi(rot_lib):
    # the packed fp32 form evaluates both hands at once and falls back to the scalar near-pi form for BOTH halves when
    # either is near pi: every pair here has one half in the near-pi band and the other outside it
    cases = grid_cases(2)
    near = [i for i, c in enumerate(cases) if c["theta"] >= NEAR_PI]
    far = [i for i, c in enumerate(cases) if c["theta"] < NEAR_PI]
    ix = near + far
    iy = [far[k % len(far)] for k in range(len(near))] + [near[k % len(near)] for k in range(len(far))]
    M = _log6_inputs(cases, np.float32)
    ex, ey = dev_log6_packed(rot_lib, M[ix], M[iy])
    assert all((cases[a]["theta"] >= NEAR_PI) != (cases[b]["theta"] >= NEAR_PI) for a, b in zip(ix, iy))
    _check_log6(ex, [cases[i] for i in ix], "f32", M[ix])
    _check_log6(ey, [cases[i] for i in iy], "f32", M[iy])
    # both halves far from pi: the packed straight-line form (no series) against the exact log
    iy2 = far[1:] + far[:1]
    ex, ey = dev_log6_packed(rot_lib, M[far], M[iy2])
    _check_log6(ex, [cases[i] for i in far], "f32", M[far])
    _check_log6(ey, [cases[i] for i in iy2], "f32", M[iy2])


# ---------------------------------------------------------------------------------------------------- interpolation
def _interp_cases(seed):
    """Edges A -> B = A (R(u, theta), p) over the grid, A a random placement; alpha in {0, random, 1} for each."""
    rng = np.random.default_rng(seed + 100)
    cases, A, B, al = [], [], [], []
    for c in grid_cases(seed):
        u0 = rng.standard_normal(3)
        a = pose_ld(u0 / np.linalg.norm(u0), rng.uniform(0, PI), rng.uniform(-0.5, 0.5, 3))
        b = mul_ld(a, pose_ld(c["u"], c["theta"], c["p"]))
        for alpha in (0.0, rng.uniform(0.05, 0.95), 1.0):
            cases.append(dict(c, alpha=alpha, a_ld=a))
            A.append(a); B.append(b); al.append(alpha)
    return cases, np.array(A), np.array(B), np.array(al)


def _interp_exact(c, sign=1.0):
    """A exp6(alpha log6(M)), M = (R(u, theta), p); sign = -1 takes the other logarithm of a half turn, about -u."""
    R, p = exp6_ld(c["alpha"] * log6_exact_ld(sign * c["u"], c["theta"], c["p"]))
    return mul_ld(c["a_ld"], np.concatenate([R.reshape(9), p])).astype(np.float64)


def _check_interp(out, cases, prec, B):
    worst = {}
    for i, c in enumerate(cases):
        th, coord, alpha = c["theta"], c["coord"], c["alpha"]
        tol = band_tol(prec, th, c["zero"])
        if th < PI and (prec == "f64" or fp32_resolvable(th, coord, False)):
            err = np.abs(out[i] - _interp_exact(c)).max()
            band = "near_pi" if th >= NEAR_PI else "far"
            worst[band] = max(worst.get(band, 0.0), err)
            assert err < tol, (prec, th, c["u"], alpha, err)
        elif coord:
            # exactly pi: alpha = 1 lands on B; in between, a turn about u either way round
            if alpha == 1.0:
                assert np.abs(out[i] - B[i]).max() < tol, (prec, th, c["u"])
            else:
                err = min(np.abs(out[i] - _interp_exact(c, s)).max() for s in (1.0, -1.0))
                assert err < tol, (prec, th, c["u"], alpha, err)
    return worst


@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_edge_interpolation_over_the_rotation_range(rot_lib, c_oracle, prec):
    cases, A, B, al = _interp_cases(3)
    dt = np.float64 if prec == "f64" else np.float32
    A, B = A.astype(dt).astype(np.float64), B.astype(dt).astype(np.float64)
    out = dev_interp(rot_lib, A, B, al, prec)
    worst = _check_interp(out, cases, prec, B)
    print(f"se3_delta + se3_advance {prec}: worst |err| per band {worst}")
    # pinocchio's semantics (C oracle) on the same inputs, wherever the turn's direction is not rounding noise.  (The
    # oracle takes theta = acos((tr R - 1) / 2) and then divides by sin(theta): on the slightly non-orthonormal
    # fp32-rounded inputs that is ill-conditioned near pi (1e-3 at pi - 0.0101), so for fp32 it is a reference up to
    # theta = 2 and the exact log above bounds the rest.)
    ref = c_oracle.interpolate(A, B, al)
    for i, c in enumerate(cases):
        if c["theta"] < PI and (prec == "f64" or c["theta"] <= 2.0):
            assert np.abs(out[i] - ref[i]).max() < band_tol(prec, c["theta"], c["zero"]), (c["theta"], c["u"])


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_host_se3_interpolate_over_the_rotation_range(c_oracle, dtype):
    # path.se3_interpolate places the cube for the scene tests and the returned cube paths: it must be pinocchio's
    # interpolation at every angle, for fp32 inputs too (it takes log6 in fp64 and rounds the twist to fp32)
    from gik_b200.path import se3_interpolate
    cases, A, B, al = _interp_cases(4)
    ndt = np.float64 if dtype == torch.float64 else np.float32
    A, B = A.astype(ndt), B.astype(ndt)
    out = se3_interpolate(torch.from_numpy(A), torch.from_numpy(B), torch.from_numpy(al.astype(ndt)))
    assert out.dtype == dtype
    out = out.double().numpy()
    alq = al.astype(ndt).astype(np.float64)
    ref = c_oracle.interpolate(A.astype(np.float64), B.astype(np.float64), alq)
    rnd = 0.0 if dtype == torch.float64 else 1e-6            # the rounding of the result to fp32
    for i, c in enumerate(cases):
        if c["theta"] < PI and (dtype == torch.float64 or c["theta"] <= 2.0):     # (see the kernel test above)
            assert np.abs(out[i] - ref[i]).max() < band_tol("f64", c["theta"], c["zero"]) + rnd, (c["theta"], c["u"], c["alpha"])
    # exactly pi about a coordinate axis: alpha = 1 lands on B, in between a half turn either way round
    _check_interp(out, [dict(c, alpha=a) for c, a in zip(cases, alq)], "f64" if dtype == torch.float64 else "f32",
                  B.astype(np.float64))
    # a cube yawed by exactly pi from the identity, the way a caller writes it
    a = np.zeros((3, 12)); a[:, [0, 4, 8]] = 1; a[:, 9:] = [0.3, -0.1, 1.0]
    b = a.copy(); b[:, :9] = rot_rpy(0, 0, np.pi).reshape(9); b[:, 9:] += [0.05, 0.02, 0.0]
    o2 = se3_interpolate(torch.from_numpy(a).to(dtype), torch.from_numpy(b).to(dtype),
                         torch.tensor([0.5, 1.0, 0.25], dtype=dtype)).double().numpy()
    tol = 1e-12 if dtype == torch.float64 else 1e-6
    assert np.abs(o2[1] - b[1]).max() < tol
    assert np.abs(o2[0, :9] - rot_rpy(0, 0, np.pi / 2).reshape(9)).max() < tol
    assert np.abs(o2 - c_oracle.interpolate(a, b, np.array([0.5, 1.0, 0.25]))).max() < tol


def test_host_se3_interpolate_reproduces_the_kernel_on_translations(rot_lib):
    # an edge without rotation (every edge the planner samples): the host placements are the kernel's bit for bit, in
    # both precisions, so the scene tests and the returned cube paths use exactly the placements the kernel solved for
    from gik_b200.path import se3_interpolate
    rng = np.random.default_rng(6)
    n = 2000
    A = np.zeros((n, 12)); A[:, [0, 4, 8]] = 1; A[:, 9:] = rng.uniform(-1, 1.5, (n, 3))
    B = A.copy(); B[:, 9:] = rng.uniform(-1, 1.5, (n, 3))
    ns = rng.integers(1, 40, n)
    k = rng.integers(1, ns + 1)
    for dtype, ndt, prec in ((torch.float32, np.float32, "f32"), (torch.float64, np.float64, "f64")):
        alpha = torch.from_numpy(k).to(dtype) / torch.from_numpy(ns).to(dtype)            # the kernel's T(k) / T(ns)
        host = se3_interpolate(torch.from_numpy(A).to(dtype), torch.from_numpy(B).to(dtype), alpha).numpy()
        dev = dev_interp(rot_lib, A.astype(ndt), B.astype(ndt), alpha.double().numpy(), prec).astype(ndt)
        assert np.array_equal(host, dev), prec


# ------------------------------------------------------------------------------------------- IK under large rotations
def large_rotation_batch(c_oracle, table_c, n, seed):
    """Solve problems whose hands start up to half a turn from their hooks -> (q_init [n,15], cube [n,12]).  Cubes in
    the reference sampler box, a fifth of them of each of three kinds, from q_init = 0:
      * yawed by exactly +-pi/2: one hand then starts half a turn (within 1e-2) from its hook;
      * uniform yaw;
      * uniform yaw with roll and pitch up to 0.3;
    and two fifths warm-started half a turn away: the oracle's solution for a cube of the kind above, with the second
    wrist joint (a y axis, joint 7 or 13) turned by pi - delta, delta in [1e-3, 9e-3] (a turn whose direction fp32 still
    resolves).  The +-pi/2 cubes do not converge within the reference's 1000 iterations (measured: none of them); the
    warm starts converge about half of the time."""
    from oracle import grasp_ik_np as o
    rng = np.random.default_rng(seed)
    P = make_poses(n, seed, "sampler")
    Q0 = np.zeros((n, 15))
    kind = rng.permutation(np.arange(n) % 5)
    yaw = rng.uniform(-np.pi, np.pi, n)
    rp = rng.uniform(-0.3, 0.3, (n, 2)) * (kind == 2)[:, None]
    yaw[kind == 0] = np.where(rng.random((kind == 0).sum()) < 0.5, np.pi / 2, -np.pi / 2)
    for i in range(n):
        P[i, :9] = rot_rpy(rp[i, 0], rp[i, 1], yaw[i]).reshape(9)
    warm = np.flatnonzero(kind >= 3)
    pool = make_poses(8 * len(warm), seed + 1, "sampler")
    for i, (r, p, y) in enumerate(zip(*rng.uniform([-0.3, -0.3, -np.pi], [0.3, 0.3, np.pi], (len(pool), 3)).T)):
        pool[i, :9] = rot_rpy(r, p, y).reshape(9)
    qp, okp, _, _ = c_oracle.solve(table_c, np.zeros((len(pool), 15)), pool)
    k = 0
    for i in warm:
        while True:
            j, k = k, k + 1
            assert k <= len(pool), "not enough converged warm starts"
            if not okp[j]:
                continue
            q = qp[j].copy()
            delta = rng.uniform(1e-3, 9e-3)
            for jt in rng.permutation([7, 13]):
                t = q[jt] - (np.pi - delta) if q[jt] > o.LOWER[jt] + np.pi else q[jt] + (np.pi - delta)
                if o.LOWER[jt] <= t <= o.UPPER[jt]:
                    q[jt] = t
                    break
            else:
                continue
            Q0[i], P[i] = q, pool[j]
            break
    return Q0, P


def start_angles(Q0, P):
    """Rotation error angle of each hand at q_init: [n,2]."""
    from oracle import grasp_ik_np as o
    th = np.zeros((len(P), 2))
    for i, row in enumerate(P):
        tg = o.hook_targets(row[:9].reshape(3, 3), row[9:])
        fk = o.forward_kinematics(Q0[i])
        for h in (0, 1):
            th[i, h] = np.linalg.norm(o.hand_error(Q0[i], h, tg[h], fk)[3:])
    return th


def test_large_rotation_batch_reaches_the_near_pi_branch(table_c, c_oracle):
    from oracle import grasp_ik_np as o
    Q0, P = large_rotation_batch(c_oracle, table_c, 300, 5)
    near = start_angles(Q0, P).max(axis=1) >= NEAR_PI
    print(f"large-rotation batch: {near.mean():.2f} of the problems start with a hand in the near-pi band")
    assert near.mean() >= 1 / 3
    assert (Q0 >= o.LOWER).all() and (Q0 <= o.UPPER).all()


@pytest.mark.parametrize("dtype,flags", [(np.float64, 0), (np.float64, 2), (np.float64, 1), (np.float32, 0), (np.float32, 4)])
def test_host_ik_arithmetic_under_large_rotations(table_c, hostsim, c_oracle, dtype, flags):
    # the descent of every solve path (scalar fp64 wrist / Cholesky / generic, scalar and packed fp32) on problems whose
    # hands start up to half a turn from their hooks, against the C oracle
    n = 300
    Q0, P = large_rotation_batch(c_oracle, table_c, n, 5)
    qo, oko, ito, _ = c_oracle.solve(table_c, Q0, P)
    q, ok, it, r = hostsim.solve(table_c, Q0, P, dtype, flags=flags)
    both = ok & oko
    d = np.abs(q[both] - qo[both]).max(axis=1)
    print(f"hostsim {np.dtype(dtype).name} flags {flags}: {both.mean():.2f} converged in both, flags differ on "
          f"{(ok != oko).sum()}, worst |dq| {d.max():.1e}")
    assert both.mean() >= 0.3
    assert (r[ok] < 1e-3).all()
    if dtype == np.float64:
        assert (ok != oko).sum() <= 1
        assert np.quantile(d, 0.99) < 1e-9 and (it[both] == ito[both]).mean() >= 0.99
    else:
        assert (ok != oko).sum() <= 3
        assert np.quantile(d, 0.99) < 1e-3 and np.quantile(np.abs(it[both] - ito[both]), 0.99) <= 2
