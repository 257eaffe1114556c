"""The trajectory check's per-sample arithmetic (csrc/gik_traj.cuh) on the CPU: the GIK_HD Bernstein sum, hand frames,
cube-from-hand and grasp error compiled with g++ in fp64 and fp32 against numpy and the C oracle; maketraj_paths on CPU
tensors against maketraj; list 3 of the packaged scene; the argument checks of the C entries (no GPU needed)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from conftest import ROOT, rot_rpy
from traj_oracle import cubes_from_hands, grasp_error, list3_pairs

CSRC = os.path.join(ROOT, "motion-planning-and-control-for-dual-manipulator-robot_b200", "csrc")

HARNESS = r"""
#include <stdint.h>
#include <new>
#include "gik_table.h"
#include "gik_traj.cuh"
using namespace gik;

// world placements of every joint, parents first (what warp_tree_fk computes level by level)
template <typename T>
static void tree_fk(const gik_table_t* t, const T* q, T (*oMi)[12]) {
  gik_scene_t* s = new gik_scene_t();
  DevScene<T>* d = new DevScene<T>();
  fill_dev_scene(*t, *s, *d);
  for (int j = 0; j < t->nq; ++j)
    joint_placement(d->tree, j, t->parent[j] < 0 ? (const T*)nullptr : oMi[t->parent[j]], q[j], oMi[j]);
  delete d; delete s;
}

template <typename T>
static T sample(const gik_table_t* t, const T* q, T* H, T* C) {
  TrajConst<T> tc;
  fill_traj_const(*t, 0.0, tc);
  T oMi[GIK_MAX_NQ][12];
  tree_fk(t, q, oMi);
  T h[12], c[2][12];
  for (int k = 0; k < 2; ++k) {
    traj_hand_frame(tc, oMi, k, h);
    traj_cube_from_hand(tc, h, k, c[k]);
    for (int i = 0; i < 12; ++i) { H[12 * k + i] = h[i]; C[12 * k + i] = c[k][i]; }
  }
  return traj_grasp_error(c[0], c[1]);
}

template <typename T>
static void cube_from_hand(const gik_table_t* t, int k, const T* H, T* C) {
  TrajConst<T> tc;
  fill_traj_const(*t, 0.0, tc);
  T h[12], c[12];
  for (int i = 0; i < 12; ++i) h[i] = H[i];
  traj_cube_from_hand(tc, h, k, c);
  for (int i = 0; i < 12; ++i) C[i] = c[i];
}

template <typename T>
static T gerr(const T* A, const T* B) {
  T a[12], b[12];
  for (int i = 0; i < 12; ++i) { a[i] = A[i]; b[i] = B[i]; }
  return traj_grasp_error(a, b);
}

extern "C" {
double h_point_f64(const double* w, const double* c, int n, int ld) { return traj_point(w, c, n, ld); }
float h_point_f32(const float* w, const float* c, int n, int ld) { return traj_point(w, c, n, ld); }
double h_sample_f64(const gik_table_t* t, const double* q, double* H, double* C) { return sample(t, q, H, C); }
float h_sample_f32(const gik_table_t* t, const float* q, float* H, float* C) { return sample(t, q, H, C); }
void h_cube_f64(const gik_table_t* t, int k, const double* H, double* C) { cube_from_hand(t, k, H, C); }
void h_cube_f32(const gik_table_t* t, int k, const float* H, float* C) { cube_from_hand(t, k, H, C); }
double h_gerr_f64(const double* A, const double* B) { return gerr(A, B); }
float h_gerr_f32(const float* A, const float* B) { return gerr(A, B); }
void h_limits_f64(const gik_table_t* t, double tol, double* lo, double* hi) {
  TrajConst<double> tc;
  fill_traj_const(*t, tol, tc);
  for (int j = 0; j < t->nq; ++j) { lo[j] = tc.lo[j]; hi[j] = tc.hi[j]; }
}
}
"""

DT = {"f64": np.float64, "f32": np.float32}


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    d = tmp_path_factory.mktemp("traj_harness")
    src = d / "harness.cpp"
    src.write_text(HARNESS)
    out = d / "libtraj.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-I", CSRC,
                    "-I", os.path.join(ROOT, "include"), "-o", str(out), str(src)], check=True)
    L = ctypes.CDLL(str(out))
    for s in ("f64", "f32"):
        ct = ctypes.c_double if s == "f64" else ctypes.c_float
        getattr(L, f"h_point_{s}").restype = ct
        getattr(L, f"h_sample_{s}").restype = ct
        getattr(L, f"h_gerr_{s}").restype = ct
    return L


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _m12(R, p):
    return np.concatenate([np.asarray(R).reshape(9), p])


def _rot(axis, angle):
    a = np.asarray(axis, float); a /= np.linalg.norm(a)
    K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return np.eye(3) + np.sin(angle) * K + (1 - np.cos(angle)) * K @ K


@pytest.mark.parametrize("sfx,tol", [("f64", 1e-13), ("f32", 2e-6)])
def test_bernstein_sum_matches_de_casteljau(lib, sfx, tol):
    from gik_b200.trajectory import Bezier, sample_weights
    rng = np.random.default_rng(0)
    f = getattr(lib, f"h_point_{sfx}")
    for n_ctrl in (2, 3, 7, 21):
        P = rng.uniform(-2, 2, (n_ctrl, 15))
        curve = Bezier(list(P), t_min=0.0, t_max=15.0)
        M = 101
        W = sample_weights(n_ctrl, M).astype(DT[sfx])
        Pc = np.ascontiguousarray(P.astype(DT[sfx]))
        for k in range(M):
            ref = curve(15.0 * k / (M - 1))
            for j in (0, 7, 14):
                got = f(_p(np.ascontiguousarray(W[k])), _p(Pc[:, j:]), n_ctrl, 15)
                assert abs(got - ref[j]) <= tol * max(1.0, abs(ref[j])), (n_ctrl, k, j)


def test_limits_are_widened_in_fp64(lib, table, table_c):
    lo, hi = np.empty(15), np.empty(15)
    lib.h_limits_f64(ctypes.byref(table_c), ctypes.c_double(1e-6), _p(lo), _p(hi))
    assert np.array_equal(lo, np.asarray(table.lower) - 1e-6) and np.array_equal(hi, np.asarray(table.upper) + 1e-6)


@pytest.mark.parametrize("sfx,tol", [("f64", 1e-12), ("f32", 1e-5)])
def test_hand_frames_and_cubes_match_the_oracle(lib, table, table_c, c_oracle, sfx, tol):
    rng = np.random.default_rng(1)
    Q = rng.uniform(table.lower, table.upper, (64, 15))
    HR, Hp = c_oracle.fk(table_c, Q)
    f = getattr(lib, f"h_sample_{sfx}")
    for i in range(len(Q)):
        H = np.zeros(24, DT[sfx]); C = np.zeros(24, DT[sfx])
        g = f(ctypes.byref(table_c), _p(np.ascontiguousarray(Q[i].astype(DT[sfx]))), _p(H), _p(C))
        for h in range(2):
            assert np.abs(H[12 * h:12 * h + 12] - _m12(HR[i, h], Hp[i, h])).max() < tol
        cubes = cubes_from_hands(table, HR[i], Hp[i])
        for h in range(2):
            assert np.abs(C[12 * h:12 * h + 12] - _m12(*cubes[h])).max() < tol
        assert abs(g - grasp_error(*cubes)) < 10 * tol


@pytest.mark.parametrize("sfx", ["f64", "f32"])
def test_cube_from_hand_inverts_the_hook(lib, table, table_c, sfx):
    rng = np.random.default_rng(2)
    f = getattr(lib, f"h_cube_{sfx}")
    for h in range(2):
        for _ in range(10):
            R = rot_rpy(*rng.uniform(-3, 3, 3)); p = rng.uniform(-1, 1, 3)
            C = np.zeros(12, DT[sfx])
            f(ctypes.byref(table_c), h, _p(_m12(R, p).astype(DT[sfx])), _p(C))
            # the hook of that cube is the hand: C * hook_h = H
            CR, Cp = C[:9].astype(float).reshape(3, 3), C[9:].astype(float)
            hR, hp = np.asarray(table.hook_R[h]), np.asarray(table.hook_p[h])
            tol = 1e-12 if sfx == "f64" else 2e-6
            assert np.abs(CR @ hR - R).max() < tol and np.abs(Cp + CR @ hp - p).max() < tol


# angles on both sides of the near-pi threshold (pi - 1e-2), exactly pi, and ordinary ones
ANGLES = [0.0, 1e-7, 1e-3, 0.3, 1.5, 3.0, np.pi - 2e-2, np.pi - 1e-2 + 1e-4, np.pi - 1e-4, np.pi - 1e-7, np.pi]
AXES = [(0, 0, 1), (1, 0, 0), (0, 1, 1), (1, 2, 3), (-1, 0.5, 0.2)]


def _exact_g(axis, angle, d):
    """||log6((Rot(axis, angle), d))|| from the known axis and angle (no log of a rounded matrix)."""
    a = np.asarray(axis, float) / np.linalg.norm(axis)
    w, t = angle * a, angle
    if t < 1e-6:
        alpha, beta = 1.0 - t * t / 12, 1.0 / 12
    else:
        alpha = t * np.sin(t) / (2 * (1 - np.cos(t)))
        beta = 1 / t ** 2 - np.sin(t) / (2 * t * (1 - np.cos(t)))
    v = alpha * d - 0.5 * np.cross(w, d) + beta * np.dot(w, d) * w
    return float(np.linalg.norm(np.concatenate([v, w])))


@pytest.mark.parametrize("sfx", ["f64", "f32"])
def test_grasp_error_matches_numpy_log6_through_a_half_turn(lib, sfx):
    from oracle import grasp_ik_np
    rng = np.random.default_rng(3)
    f = getattr(lib, f"h_gerr_{sfx}")
    tol = 1e-10 if sfx == "f64" else 2e-6
    for ang in ANGLES:
        for ax in AXES:
            RL = rot_rpy(*rng.uniform(-3, 3, 3)); pL = rng.uniform(-0.5, 0.5, 3)
            D = _rot(ax, ang); d = rng.uniform(-0.1, 0.1, 3)
            RR, pR = RL @ D, pL + RL @ d
            got = f(_p(_m12(RL, pL).astype(DT[sfx])), _p(_m12(RR, pR).astype(DT[sfx])))
            if ang == np.pi:
                # exactly a half turn: the direction of the turn is rounding noise, only |w| = pi is determined
                assert got >= np.pi - tol, (ax, got)
                continue
            assert abs(got - _exact_g(ax, ang, d)) < tol, (ang, ax, got)
            if ang <= np.pi - 1e-4:       # numpy's arccos loses 1e-16 / sin(theta) closer to pi
                ref = np.linalg.norm(grasp_ik_np.log6(RL.T @ RR, RL.T @ (pR - pL)))
                assert abs(got - ref) < tol, (ang, ax, got, ref)
    # a pure half turn about a coordinate axis, no translation: g = pi
    I12 = _m12(np.eye(3), np.zeros(3)).astype(DT[sfx])
    assert abs(f(_p(I12), _p(_m12(_rot((0, 0, 1), np.pi), np.zeros(3)).astype(DT[sfx]))) - np.pi) < (1e-12 if sfx == "f64" else 1e-6)


def test_converged_ik_solution_places_the_cube_within_its_residual(lib, table, table_c, c_oracle, golden):
    rng = np.random.default_rng(4)
    n = 16
    P = np.zeros((n, 12)); P[:, [0, 4, 8]] = 1
    P[:, 9:] = rng.uniform([0.25, -0.3, 0.95], [0.5, 0.3, 1.2], (n, 3))
    P[3, :9] = rot_rpy(0, 0, 0.4).reshape(9)
    P[0, 9:] = golden["cases"][0]["cube_p"]
    q, ok, _, res = c_oracle.solve(table_c, np.zeros((n, 15)), P)
    assert ok.sum() >= n // 2
    from oracle import grasp_ik_np
    for i in np.nonzero(ok)[0]:
        H = np.zeros(24); C = np.zeros(24)
        g = lib.h_sample_f64(ctypes.byref(table_c), _p(q[i]), _p(H), _p(C))
        cube = P[i]
        # C_L^-1 * cube: the IK residual of the left hand, conjugated by the hook (same angle, lever arm |hook_p|)
        CL_R, CL_p = C[:9].reshape(3, 3), C[9:12]
        e = grasp_ik_np.log6(CL_R.T @ cube[:9].reshape(3, 3), CL_R.T @ (cube[9:] - CL_p))
        lever = 1.0 + np.linalg.norm(table.hook_p[0])
        assert np.linalg.norm(e) <= lever * res[i, 0] + 1e-12
        assert g <= lever * (res[i, 0] + res[i, 1]) + 1e-12


def test_maketraj_paths_equals_maketraj_per_path():
    from gik_b200.trajectory import maketraj, maketraj_batch, maketraj_paths
    rng = np.random.default_rng(5)
    lens = [5, 0, 12, 5, 30, 1, 12, 2, 64]
    # planner-like paths: short steps from a random start
    q = np.concatenate([rng.uniform(-1, 1, (1, 15)) + np.cumsum(rng.normal(0, 0.02, (n, 15)), axis=0) for n in lens])
    off = np.concatenate([[0], np.cumsum(lens)])
    q0 = np.stack([q[o] if n else np.zeros(15) for o, n in zip(off[:-1], lens)])
    q1 = np.stack([q[o + n - 1] if n else np.zeros(15) for o, n in zip(off[:-1], lens)])
    ctrl, cost = maketraj_paths(torch.from_numpy(q0), torch.from_numpy(q1), torch.from_numpy(q), torch.from_numpy(off))
    assert ctrl.shape == (len(lens), 21, 15) and cost.shape == (len(lens),)
    for i, n in enumerate(lens):
        if n == 0:
            assert torch.isnan(ctrl[i]).all() and cost[i] == float("inf")
            continue
        path = q[off[i]:off[i + 1]]
        # the path fitted alone
        c1, k1 = maketraj_batch(torch.from_numpy(q0[i:i + 1]), torch.from_numpy(q1[i:i + 1]), torch.from_numpy(path[None]))
        assert np.abs(ctrl[i].numpy() - c1[0].numpy()).max() < 1e-12 and abs(float(cost[i] - k1[0])) < 1e-12
        # the reference's maketraj (numpy lstsq): the same least-squares solution up to the fit's conditioning (the
        # Bernstein design matrix has a condition number of about 2e5; paths of fewer than 15 points have min-norm fits)
        (curve, _, _), _ = maketraj(q0[i], q1[i], path, 15.0)
        ref = np.array(curve.control_points_)
        assert np.abs(ctrl[i].numpy() - ref).max() < 1e-9 * max(1.0, np.abs(ref).max()), (i, n)


def test_list3_of_the_packaged_scene(table):
    import gik_b200
    sc = gik_b200.nextage_scene()
    hands = tuple(int(j) for j in table.hand_joint)
    L3 = list3_pairs(sc, hands)
    on_hand = [g for g, geom in enumerate(sc.geoms) if geom.joint in hands]
    cube_hand = [(a, b) for a, b in sc.pairs if (a == sc.cube and b in on_hand) or (b == sc.cube and a in on_hand)]
    assert len(on_hand) == 4 and len(cube_hand) == 4
    assert len(L3) == len(sc.pairs) - 4 + 1 == 742                # + the cube-table pair; the obstacle-cube pair is listed
    as_sets = [frozenset(p) for p in L3.tolist()]
    assert len(set(as_sets)) == len(as_sets)
    assert not any(sc.cube in p and (set(p) - {sc.cube}) & set(on_hand) for p in as_sets)
    assert as_sets.count(frozenset((sc.obstacle, sc.cube))) == 1 and as_sets.count(frozenset((sc.table, sc.cube))) == 1
    # every other pair of the scene is kept
    assert set(as_sets) >= {frozenset(p) for p in sc.pairs.tolist()} - {frozenset(p) for p in cube_hand}


def test_traj_check_entries_reject_bad_arguments_without_gpu():
    from gik_b200 import _cabi
    lib = _cabi.lib()
    x = ctypes.c_void_p(8)          # never dereferenced: every call below is refused before any memory access
    for sfx in ("f32", "f64"):
        f = getattr(lib, f"gik_traj_check_{sfx}")
        ok = [x] * 6                # weights, ctrl, then valid, first_bad, reason, grasp_err
        args = lambda n=4, nc=21, m=1501, lt=1e-6, gt=1e-2, p=ok, flags=None: (None, n, nc, m, p[0], p[1], lt, gt, *p[2:], flags, None)
        assert f(*args()) == -6                                   # GIK_E_HANDLE
        assert f(*args(n=-1)) == -2                               # GIK_E_SIZE
        assert f(*args(nc=1)) == -2 and f(*args(nc=-3)) == -2
        assert f(*args(m=1)) == -2 and f(*args(m=-5)) == -2 and f(*args(m=1 << 28)) == -2
        assert f(*args(lt=-1e-9)) == -5 and f(*args(gt=-1.0)) == -5 and f(*args(gt=float("nan"))) == -5   # GIK_E_PARAM
        for i in range(6):
            bad = list(ok); bad[i] = None
            assert f(*args(p=bad)) == -1                          # GIK_E_NULL
        assert f(*args(n=0, p=[None] * 6)) == -6                  # no pointers needed for n = 0, still a handle
