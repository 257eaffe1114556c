"""The trajectory refinement's arithmetic (csrc/gik_traj_refine.cuh) on the CPU: the GIK_HD residual, model Jacobian,
normal-equation assembly, Cholesky solve and box clamp compiled with g++ (tid = 0, nth = 1: the kernel's loops run
serially) against numpy, the C oracle and tests/traj_oracle.py; the argument checks of the C entries (no GPU needed)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from traj_oracle import cubes_from_hands, grasp_error

CSRC = os.path.join(ROOT, "motion-planning-and-control-for-dual-manipulator-robot_b200", "csrc")

HARNESS = r"""
#include <stdint.h>
#include <new>
#include "gik_table.h"
#include "gik_traj.cuh"
#include "gik_traj_refine.cuh"
using namespace gik;

template <typename T>
static int resid(const gik_table_t* t, const T* q15, T* r, T* J) {
  DevTable<T>* d = new DevTable<T>();
  const int rc = build_dev_table(*t, *d);
  T q[kActive], rr[6], JJ[6][6];
  for (int k = 0; k < kActive; ++k) q[k] = q15[d->act_q[k]];
  refine_sample<T, true>(*d, q, rr, JJ);
  for (int m = 0; m < 6; ++m) {
    r[m] = rr[m];
    for (int c = 0; c < 6; ++c) J[6 * m + c] = JJ[m][c];
  }
  delete d;
  return rc;
}

// The kernel's assembly for S samples, serially: tiles of kRefineThreads samples, tile rows from refine_normal and the
// free weights, every item accumulated tile by tile.
static void assemble(int nf, int S, const double* J, const double* r, const double* w, double* M, double* g) {
  const int np = nf * (nf + 1) / 2, ld = kRefineTileLd + nf;
  for (int e = 0; e < 21 * np; ++e) M[e] = 0.0;
  for (int e = 0; e < 6 * nf; ++e) g[e] = 0.0;
  double* tile = new double[kRefineThreads * ld];
  for (int k0 = 0; k0 < S; k0 += kRefineThreads) {
    const int cnt = S - k0 < kRefineThreads ? S - k0 : kRefineThreads;
    for (int t = 0; t < cnt; ++t) {
      const int k = k0 + t;
      double JJ[6][6], rr[6];
      for (int m = 0; m < 6; ++m) {
        rr[m] = r[6 * k + m];
        for (int c = 0; c < 6; ++c) JJ[m][c] = J[36 * k + 6 * m + c];
      }
      double* row = tile + t * ld;
      refine_normal(JJ, rr, row, row + 21);
      for (int f = 0; f < nf; ++f) row[kRefineTileLd + f] = w[k * nf + f];
    }
    for (int item = 0; item < np + nf; ++item) refine_accumulate(item, nf, cnt, tile, ld, M, g);
  }
  delete[] tile;
}

extern "C" {
int h_resid_f64(const gik_table_t* t, const double* q, double* r, double* J) { return resid(t, q, r, J); }
int h_resid_f32(const gik_table_t* t, const float* q, float* r, float* J) { return resid(t, q, r, J); }
void h_assemble(int nf, int S, const double* J, const double* r, const double* w, double* M, double* g) {
  assemble(nf, S, J, r, w, M, g);
}
void h_build(const double* M, const double* g, int nf, double lambda, double* A, double* diag, double* z) {
  refine_build(M, g, nf, lambda, A, diag, z, 0, 1);
}
void h_chol_solve(double* A, const double* diag, double* z, double* y, int nu) {
  refine_cholesky(A, diag, nu, 0, 1, RefineSync());
  refine_solve(A, z, y, nu, 0, 1, RefineSync());
}
double h_clamp_f64(double x, double d, double x0, double lo, double hi) { return refine_clamp(x, d, x0, lo, hi); }
float h_clamp_f32(float x, double d, float x0, float lo, float hi) { return refine_clamp(x, d, x0, lo, hi); }
}
"""

DT = {"f64": np.float64, "f32": np.float32}


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    d = tmp_path_factory.mktemp("refine_harness")
    src = d / "harness.cpp"
    src.write_text(HARNESS)
    out = d / "librefine.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-I", CSRC,
                    "-I", os.path.join(ROOT, "include"), "-o", str(out), str(src)], check=True)
    L = ctypes.CDLL(str(out))
    L.h_build.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_double] + [ctypes.c_void_p] * 3
    L.h_clamp_f64.restype = ctypes.c_double
    L.h_clamp_f64.argtypes = [ctypes.c_double] * 5
    L.h_clamp_f32.restype = ctypes.c_float
    L.h_clamp_f32.argtypes = [ctypes.c_float, ctypes.c_double, ctypes.c_float, ctypes.c_float, ctypes.c_float]
    return L


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _resid(lib, table_c, q, sfx):
    r = np.zeros(6, DT[sfx]); J = np.zeros(36, DT[sfx])
    assert getattr(lib, f"h_resid_{sfx}")(ctypes.byref(table_c), _p(np.ascontiguousarray(q, DT[sfx])), _p(r), _p(J)) == 0
    return r.astype(float), J.reshape(6, 6).astype(float)


def _right_arm(table):
    """q indices of the right arm's six joints, root to tip (act_q[7..12])."""
    chain, k = [], int(table.hand_joint[1])
    while k >= 0:
        chain.append(k); k = int(table.parent[k])
    return chain[::-1][1:]


@pytest.mark.parametrize("sfx,tol", [("f64", 1e-11), ("f32", 2e-5)])
def test_residual_matches_numpy_log6_and_the_check_oracle(lib, table, table_c, c_oracle, sfx, tol):
    from oracle import grasp_ik_np
    rng = np.random.default_rng(21)
    Q = rng.uniform(table.lower, table.upper, (48, 15))
    HR, Hp = c_oracle.fk(table_c, Q)
    for i in range(len(Q)):
        r, _ = _resid(lib, table_c, Q[i].astype(DT[sfx]).astype(float), sfx)
        CL, CR = cubes_from_hands(table, HR[i], Hp[i])
        if sfx == "f32":            # the same configuration as the fp32 call sees it
            HR32, Hp32 = c_oracle.fk(table_c, Q[i:i + 1].astype(np.float32).astype(float))
            CL, CR = cubes_from_hands(table, HR32[0], Hp32[0])
        ref = grasp_ik_np.log6(CL[0].T @ CR[0], CL[0].T @ (CR[1] - CL[1]))
        assert np.abs(r - ref).max() < tol * max(1.0, np.abs(ref).max()), (i, r, ref)
        assert abs(np.linalg.norm(r) - grasp_error(CL, CR)) < tol * max(1.0, np.linalg.norm(ref))


def _on_one_cube(lib, table, table_c, c_oracle, n):
    """Configurations where both hands sit exactly on one cube: converged IK solutions (residuals up to 1e-3), then the
    right arm alone driven to r = 0 by Newton steps with the model Jacobian (exact at r = 0)."""
    rng = np.random.default_rng(22)
    P = np.zeros((4 * n, 12)); P[:, [0, 4, 8]] = 1
    P[:, 9:] = rng.uniform([0.25, -0.3, 0.95], [0.5, 0.3, 1.2], (4 * n, 3))
    q, ok, _, _ = c_oracle.solve(table_c, np.zeros((4 * n, 15)), P)
    arm = _right_arm(table)
    out = []
    for qi in q[ok.astype(bool)][:n]:
        qi = qi.copy()
        for _ in range(30):
            r, J = _resid(lib, table_c, qi, "f64")
            if np.linalg.norm(r) < 1e-14:
                break
            qi[arm] -= np.linalg.solve(J, r)
        assert np.linalg.norm(_resid(lib, table_c, qi, "f64")[0]) < 1e-13
        out.append(qi)
    assert len(out) >= n // 2
    return out


def test_model_jacobian_matches_central_differences_on_the_grasp(lib, table, table_c, c_oracle):
    arm = _right_arm(table)
    h = 1e-6
    for q in _on_one_cube(lib, table, table_c, c_oracle, 8):
        _, J = _resid(lib, table_c, q, "f64")
        num = np.zeros((6, 6))
        for c, j in enumerate(arm):
            qp, qm = q.copy(), q.copy()
            qp[j] += h; qm[j] -= h
            num[:, c] = (_resid(lib, table_c, qp, "f64")[0] - _resid(lib, table_c, qm, "f64")[0]) / (2 * h)
        assert np.abs(J - num).max() < 1e-6, np.abs(J - num).max()


def test_model_jacobian_is_the_adjoint_of_the_local_jacobian(lib, table, table_c, c_oracle):
    """J = Ad(hook_R) J_R with J_R the right-arm columns of the C oracle's LOCAL Jacobian of RARM_EFF."""
    rng = np.random.default_rng(23)
    Q = rng.uniform(table.lower, table.upper, (16, 15))
    Jo = c_oracle.jac(table_c, Q)                       # [n, 2, 6, nq]
    K = np.asarray(table.hook_R[1]).reshape(3, 3); k = np.asarray(table.hook_p[1])
    kx = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    Ad = np.block([[K, kx @ K], [np.zeros((3, 3)), K]])
    for i in range(len(Q)):
        _, J = _resid(lib, table_c, Q[i], "f64")
        assert np.abs(J - Ad @ np.asarray(Jo[i])[1][:, _right_arm(table)]).max() < 1e-12


def _dense(A, nu):
    D = np.zeros((nu, nu))
    for i in range(nu):
        D[i, :i + 1] = A[i * (i + 1) // 2:i * (i + 1) // 2 + i + 1]
    return D


@pytest.mark.parametrize("nf,S", [(15, 301), (1, 2), (20, 128), (4, 1000)])
def test_assembly_matches_einsum_and_the_solve_matches_numpy(lib, nf, S):
    rng = np.random.default_rng(nf * 1000 + S)
    J = rng.normal(size=(S, 6, 6)); r = rng.normal(size=(S, 6)) * 1e-2
    w = rng.uniform(0, 1, (S, nf))
    np_ = nf * (nf + 1) // 2; nu = 6 * nf
    M = np.zeros(21 * np_); g = np.zeros(nu)
    lib.h_assemble(nf, S, _p(J), _p(r), _p(w), _p(M), _p(g))
    H_ref = np.einsum("ka,kb,kmc,kmd->acbd", w, w, J, J).reshape(nu, nu)
    g_ref = np.einsum("ka,kmc,km->ac", w, J, r).reshape(nu)
    lam = 1e-3
    A = np.zeros(nu * (nu + 1) // 2); diag = np.zeros(nu); z = np.zeros(nu); y = np.zeros(nu)
    lib.h_build(_p(M), _p(g), nf, lam, _p(A), _p(diag), _p(z))
    Ad = _dense(A, nu)
    Hd = H_ref + lam * np.diag(np.diag(H_ref))
    assert np.abs(Ad - np.tril(Hd)).max() < 1e-12 * np.abs(Hd).max()
    assert np.array_equal(diag, np.diag(Ad)) and np.abs(z + g_ref).max() < 1e-12 * max(1.0, np.abs(g_ref).max())
    lib.h_chol_solve(_p(A), _p(diag), _p(z), _p(y), nu)
    L = _dense(A, nu)
    assert np.abs(L @ L.T - Hd).max() < 1e-10 * np.abs(Hd).max()
    ref = np.linalg.solve(Hd, -g_ref)
    assert np.abs(z - ref).max() < 1e-8 * max(1.0, np.abs(ref).max()), np.abs(z - ref).max()


def test_zero_rows_get_a_zero_step(lib):
    """n_samples = 2 puts every sample at u = 0 or 1, where the free control points weigh nothing: H = 0, g = 0, and the
    pivot floor turns that into delta = 0 (not NaN)."""
    nf, nu = 3, 18
    M = np.zeros(21 * 6); g = np.zeros(nu)
    A = np.zeros(nu * (nu + 1) // 2); diag = np.zeros(nu); z = np.zeros(nu); y = np.zeros(nu)
    lib.h_build(_p(M), _p(g), nf, 1e-3, _p(A), _p(diag), _p(z))
    lib.h_chol_solve(_p(A), _p(diag), _p(z), _p(y), nu)
    assert np.array_equal(z, np.zeros(nu))


@pytest.mark.parametrize("sfx", ["f64", "f32"])
def test_box_clamp(lib, sfx):
    f = getattr(lib, f"h_clamp_{sfx}")
    rng = np.random.default_rng(24)
    lo, hi = -1.0, 2.0
    for _ in range(2000):
        x0 = float(DT[sfx](rng.choice([rng.uniform(lo, hi), rng.uniform(-3, lo), rng.uniform(hi, 4), lo, hi])))
        x = float(DT[sfx](rng.uniform(min(lo, x0), max(hi, x0))))     # any value the box allows
        d = float(rng.normal(0, 2))
        v = f(x, d, x0, lo, hi)
        if lo <= x0 <= hi:
            assert lo <= v <= hi                              # inside stays inside
        else:
            assert min(lo, x0) <= v <= max(hi, x0)            # outside never moves further out
            assert abs(v - (lo + hi) / 2) <= abs(x0 - (lo + hi) / 2) + 1e-6
        if min(lo, x0) <= x + d <= max(hi, x0):
            assert v == DT[sfx](DT[sfx](x) + DT[sfx](d))      # an unclamped step is the plain sum
    assert np.isnan(f(0.5, float("nan"), 0.5, lo, hi))        # NaN passes through (the trial is then rejected)


def test_traj_refine_entries_reject_bad_arguments_without_gpu():
    from gik_b200 import _cabi
    lib = _cabi.lib()
    x = ctypes.c_void_p(8)          # never dereferenced: every call below is refused before any memory access
    for sfx in ("f32", "f64"):
        f = getattr(lib, f"gik_traj_refine_{sfx}")
        ok = [x] * 8                # weights, ctrl, then ctrl_out, obj_before, obj_after, grasp_err, iters, accepted
        args = lambda n=4, nc=21, m=1501, it=8, tol=1e-3, lam=1e-3, p=ok: (None, n, nc, m, p[0], p[1], it, tol, lam,
                                                                            *p[2:], None)
        assert f(*args()) == -6                                   # GIK_E_HANDLE
        assert f(*args(n=-1)) == -2                               # GIK_E_SIZE
        assert f(*args(nc=6)) == -2 and f(*args(nc=27)) == -2 and f(*args(nc=-3)) == -2
        assert f(*args(nc=7)) == -6 and f(*args(nc=26)) == -6
        assert f(*args(m=1)) == -2 and f(*args(m=-5)) == -2 and f(*args(m=1 << 28)) == -2
        assert f(*args(it=-1)) == -5 and f(*args(tol=-1e-9)) == -5 and f(*args(tol=float("nan"))) == -5   # GIK_E_PARAM
        for lam in (0.0, -1.0, float("nan"), float("inf")):
            assert f(*args(lam=lam)) == -5
        assert f(*args(it=0, tol=0.0)) == -6
        for i in range(8):
            bad = list(ok); bad[i] = None
            assert f(*args(p=bad)) == -1                          # GIK_E_NULL
        assert f(*args(n=0, p=[None] * 8)) == -6                  # no pointers needed for n = 0, still a handle
