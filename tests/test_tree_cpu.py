"""The device-side RRT-connect trees (csrc/gik_tree.cuh) on the CPU: the GIK_HD nearest-vertex scan, tree append and
path walk compiled with g++ against Python restatements of path.computepath's nearest(), grow() and _get_path(), plus
the argument checks of the C entries (no GPU needed)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from conftest import ROOT

CSRC = os.path.join(ROOT, "motion-planning-and-control-for-dual-manipulator-robot_b200", "csrc")

HARNESS = r"""
#include <stdint.h>
#include "gik_core.cuh"
#include "gik_tree.cuh"
using namespace gik;

// the nearest-vertex kernel's work for one target: 32 lanes scan residue classes, then the xor-butterfly merge
template <typename T>
static void nearest(int nq, int64_t cap, const T* tree, int nv, int64_t n, const T* targets, int32_t* out) {
  for (int64_t t = 0; t < n; ++t) {
    double bd[32]; int bi[32];
    for (int l = 0; l < 32; ++l) { bd[l] = 1.0 / 0.0; bi[l] = -1; tree_scan_nearest(tree, cap, nv, targets + t * nq, nq, l, 32, bd[l], bi[l]); }
    for (int o = 16; o > 0; o >>= 1) {
      double nd[32]; int ni[32];
      for (int l = 0; l < 32; ++l) {
        nd[l] = bd[l]; ni[l] = bi[l];
        const double od = bd[l ^ o]; const int oi = bi[l ^ o];
        if (oi >= 0 && (bi[l] < 0 || tree_better(od, oi, bd[l], bi[l]))) { nd[l] = od; ni[l] = oi; }
      }
      for (int l = 0; l < 32; ++l) { bd[l] = nd[l]; bi[l] = ni[l]; }
    }
    out[t] = bi[0];
  }
}

extern "C" {
void h_nearest_f64(int nq, int64_t cap, const double* tree, int nv, int64_t n, const double* tg, int32_t* out) { nearest(nq, cap, tree, nv, n, tg, out); }
void h_nearest_f32(int nq, int64_t cap, const float* tree, int nv, int64_t n, const float* tg, int32_t* out) { nearest(nq, cap, tree, nv, n, tg, out); }
int h_append_f64(int nq, int64_t cap, int max_steps, int64_t E, int64_t e0, int64_t e1, double* verts, double* cubes,
                 int32_t* parent, int32_t* n_verts, const int32_t* near, const double* q_start, const double* pose_a,
                 const double* pose_b, const int32_t* num_steps, const int32_t* n_valid, const double* q_path, int32_t* seg_end) {
  return tree_append(nq, cap, max_steps, E, e0, e1, verts, cubes, parent, n_verts, near, q_start, pose_a, pose_b,
                     num_steps, n_valid, q_path, seg_end);
}
int64_t h_path_f64(int nq, int64_t cap, const double* vs, const double* cs, const int32_t* ps, int nvs, int s,
                   const double* vg, const double* cg, const int32_t* pg, int nvg, int g, double* q, double* cube) {
  return tree_write_path(nq, cap, vs, cs, ps, nvs, s, vg, cg, pg, nvg, g, q, cube);
}
}
"""


@pytest.fixture(scope="module")
def tree_lib(tmp_path_factory):
    d = tmp_path_factory.mktemp("tree_harness")
    src = d / "harness.cpp"
    src.write_text(HARNESS)
    out = d / "libtree.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-I", CSRC,
                    "-I", os.path.join(ROOT, "include"), "-o", str(out), str(src)], check=True)
    return ctypes.CDLL(str(out))


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _nearest(lib, P, T, dtype=np.float64, cap=None):
    """P [nv,nq] tree vertices, T [n,nq] targets -> harness indices (tree stored [nq][cap])."""
    nv, nq = P.shape
    cap = cap or nv + 3
    tree = np.zeros((nq, cap), dtype); tree[:, :nv] = P.T
    tg = np.ascontiguousarray(T, dtype)
    out = np.full(len(T), -7, np.int32)
    f = lib.h_nearest_f64 if dtype == np.float64 else lib.h_nearest_f32
    f(ctypes.c_int(nq), ctypes.c_int64(cap), _p(tree), ctypes.c_int(nv), ctypes.c_int64(len(T)), _p(tg), _p(out))
    return out


def _numpy_nearest(P, T):          # nearest() of path.computepath
    return ((P[None, :, :] - T[:, None, :]) ** 2).sum(axis=2).argmin(axis=1)


@pytest.mark.parametrize("nv", [1, 2, 31, 32, 33, 200, 1000])
def test_scan_matches_numpy_argmin_on_random_trees(tree_lib, nv):
    rng = np.random.default_rng(nv)
    P = rng.uniform(-2, 2, (nv, 15)); T = rng.uniform(-2, 2, (64, 15))
    assert (_nearest(tree_lib, P, T) == _numpy_nearest(P, T)).all()
    # fp32 storage: distances still in fp64 of the stored values
    P32, T32 = P.astype(np.float32), T.astype(np.float32)
    assert (_nearest(tree_lib, P32, T32, np.float32) == _numpy_nearest(P32.astype(float), T32.astype(float))).all()


def test_scan_ties_go_to_the_lowest_index(tree_lib):
    # grow() re-adds the nearest vertex as every segment's first vertex: exact duplicates in the tree
    rng = np.random.default_rng(1)
    base = rng.uniform(-1, 1, (40, 15))
    P = base[rng.integers(0, 40, 300)]                                   # every vertex duplicated several times
    T = np.vstack([base[:20] + rng.normal(0, 1e-3, (20, 15)), base[20:]])
    got = _nearest(tree_lib, P, T)
    assert (got == _numpy_nearest(P, T)).all()
    for t, i in enumerate(got):                                          # and the first of its duplicates
        assert i == np.flatnonzero((P == P[i]).all(axis=1))[0]
    # a target at the same distance from two distinct vertices
    P = np.zeros((64, 15)); P[5, 0] = 1.0; P[40, 0] = -1.0; P[:5] = 9; P[6:40] = 9; P[41:] = 9
    assert _nearest(tree_lib, P, np.zeros((1, 15)))[0] == 5 == _numpy_nearest(P, np.zeros((1, 15)))[0]


def test_scan_single_vertex_and_one_ulp_apart(tree_lib):
    rng = np.random.default_rng(2)
    P = rng.uniform(-1, 1, (1, 15)); T = rng.uniform(-1, 1, (8, 15))
    assert (_nearest(tree_lib, P, T) == 0).all()
    # distances that differ by one ulp: vertex k moved by the smallest step that changes its squared distance
    x = rng.uniform(0.1, 1, (1, 15))
    P = np.repeat(x, 40, axis=0)
    for k in range(40):
        P[k, k % 15] = np.nextafter(P[k, k % 15], 2.0 if k % 2 else -2.0)
    d = ((P[None] - np.zeros((1, 1, 15))) ** 2).sum(axis=2)[0]
    assert len(np.unique(d)) > 1 and np.diff(np.unique(d)).min() <= 4 * np.spacing(d.max())
    assert _nearest(tree_lib, P, np.zeros((1, 15)))[0] == _numpy_nearest(P, np.zeros((1, 15)))[0]


def test_scan_sum_order_matters_and_other_nq_sum_left_to_right(tree_lib):
    rng = np.random.default_rng(3)
    P = rng.standard_normal((300, 15)); T = rng.standard_normal((200, 15))
    assert (_nearest(tree_lib, P, T) == _numpy_nearest(P, T)).all()
    P7, T7 = P[:, :7].copy(), T[:, :7].copy()                             # nq != 15
    sq = (P7[None] - T7[:, None]) ** 2
    ltr = np.zeros(sq.shape[:2])
    for c in range(7):
        ltr = ltr + sq[:, :, c]
    assert (_nearest(tree_lib, P7, T7) == ltr.argmin(axis=1)).all()


# ---------------------------------------------------------------------------------------------------------- append
def _se3_rows(A, B, alpha):
    from gik_b200.path import se3_interpolate
    return se3_interpolate(torch.from_numpy(A), torch.from_numpy(B), torch.as_tensor(alpha, dtype=torch.float64)).numpy()


def _grow_ref(G, C, near, segs):    # grow() of path.computepath (path.py:284-291 here)
    ends = []
    for k, (sq, sc) in enumerate(segs):
        for j in range(len(sq)):
            G.append((len(G) - 1 if j > 0 else int(near[k]), sq[j]))
            C.append(sc[j])
        ends.append(len(G) - 1)
    return ends


def _random_edges(rng, n_edges, nq, S, rotate):
    A = np.zeros((n_edges, 12)); A[:, [0, 4, 8]] = 1; A[:, 9:] = rng.uniform(0.2, 0.5, (n_edges, 3))
    B = A.copy(); B[:, 9:] += rng.uniform(-0.1, 0.1, (n_edges, 3))
    if rotate:
        from conftest import rot_rpy
        for e in range(n_edges):
            B[e, :9] = rot_rpy(*rng.uniform(-0.5, 0.5, 3)).reshape(9)
    ns = rng.integers(1, S + 1, n_edges).astype(np.int32)
    nv = np.minimum(rng.integers(0, S + 1, n_edges), ns).astype(np.int32)
    nv[0] = 0
    qs = rng.uniform(-1, 1, (n_edges, nq))
    path = rng.uniform(-1, 1, (S, nq, n_edges))
    return A, B, ns, nv, qs, path


@pytest.mark.parametrize("rotate", [False, True])
def test_append_reproduces_grow(tree_lib, rotate):
    rng = np.random.default_rng(4 + rotate)
    nq, S, cap, E = 15, 6, 80, 7
    n0 = 5
    G = [(None if i == 0 else i - 1, rng.uniform(-1, 1, nq)) for i in range(n0)]
    C = [rng.uniform(-1, 1, 12) for _ in range(n0)]
    verts = np.zeros((nq, cap)); cubes = np.zeros((12, cap)); parent = np.full(cap, -9, np.int32)
    for i, ((par, q), c) in enumerate(zip(G, C)):
        verts[:, i] = q; cubes[:, i] = c; parent[i] = -1 if par is None else par
    n_verts = np.array([n0], np.int32)
    A, B, ns, nv, qs, path = _random_edges(rng, E, nq, S, rotate)
    near = rng.integers(0, n0, E).astype(np.int32)
    nv[3] = -1                                                             # an idle slot: no segment
    qsT, AT, BT = [np.ascontiguousarray(x.T) for x in (qs, A, B)]
    seg_end = np.zeros(E, np.int32)
    ok = tree_lib.h_append_f64(nq, ctypes.c_int64(cap), S, ctypes.c_int64(E), ctypes.c_int64(0), ctypes.c_int64(E),
                               _p(verts), _p(cubes), _p(parent), _p(n_verts), _p(near), _p(qsT), _p(AT), _p(BT), _p(ns),
                               _p(nv), _p(np.ascontiguousarray(path)), _p(seg_end))
    assert ok == 1
    keep = [k for k in range(E) if nv[k] >= 0]
    segs = []
    for k in keep:
        sq = np.vstack([qs[k][None], path[:nv[k], :, k]])
        sc = np.vstack([A[k][None]] + ([_se3_rows(np.tile(A[k], (nv[k], 1)), np.tile(B[k], (nv[k], 1)),
                                                  np.arange(1, nv[k] + 1) / ns[k])] if nv[k] else []))
        segs.append((sq, sc))
    ends = _grow_ref(G, C, near[keep], segs)
    assert n_verts[0] == len(G)
    assert list(seg_end[keep]) == ends and seg_end[3] == -1
    for i, (par, q) in enumerate(G):
        assert parent[i] == (-1 if par is None else par)
        assert np.array_equal(verts[:, i], q)
        assert np.abs(cubes[:, i] - C[i]).max() <= (1e-12 if rotate else 0.0)
    assert (parent[len(G):] == -9).all()


def test_append_overflow_leaves_the_tree_unchanged(tree_lib):
    rng = np.random.default_rng(6)
    nq, S, E = 15, 5, 4
    A, B, ns, nv, qs, path = _random_edges(rng, E, nq, S, False)
    need = int((nv + 1).sum())
    for cap, fits in ((1 + need, True), (need, False)):
        verts = np.zeros((nq, cap)); cubes = np.zeros((12, cap)); parent = np.full(cap, -9, np.int32); parent[0] = -1
        n_verts = np.array([1], np.int32)
        before = (verts.copy(), cubes.copy(), parent.copy())
        seg_end = np.zeros(E, np.int32)
        ok = tree_lib.h_append_f64(nq, ctypes.c_int64(cap), S, ctypes.c_int64(E), ctypes.c_int64(0), ctypes.c_int64(E),
                                   _p(verts), _p(cubes), _p(parent), _p(n_verts), _p(np.zeros(E, np.int32)),
                                   _p(np.ascontiguousarray(qs.T)), _p(np.ascontiguousarray(A.T)), _p(np.ascontiguousarray(B.T)),
                                   _p(ns), _p(nv), _p(np.ascontiguousarray(path)), _p(seg_end))
        assert ok == int(fits)
        if fits:
            assert n_verts[0] == cap and seg_end[-1] == cap - 1
        else:
            assert n_verts[0] == 1 and (seg_end == -1).all()
            assert all(np.array_equal(x, y) for x, y in zip(before, (verts, cubes, parent)))


# ---------------------------------------------------------------------------------------------------------- paths
def _get_path_ref(G, node):         # path._get_path
    from gik_b200.path import _get_path
    return _get_path(G, node)


def _random_tree(rng, n, nq):
    G = [(None, rng.uniform(-1, 1, nq))]
    for i in range(1, n):
        G.append((int(rng.integers(0, i)), rng.uniform(-1, 1, nq)))
    return G


def test_path_assembly_equals_get_path(tree_lib):
    rng = np.random.default_rng(7)
    nq, cap = 15, 64
    for trial in range(20):
        Gs, Gg = _random_tree(rng, int(rng.integers(1, 40)), nq), _random_tree(rng, int(rng.integers(1, 40)), nq)
        arrs = []
        for G in (Gs, Gg):
            v = np.zeros((nq, cap)); c = np.zeros((12, cap)); p = np.full(cap, -1, np.int32)
            for i, (par, q) in enumerate(G):
                v[:, i] = q; c[:, i] = np.arange(12) + 100 * i; p[i] = -1 if par is None else par
            arrs.append((v, c, p))
        s, g = int(rng.integers(0, len(Gs))), int(rng.integers(0, len(Gg)))
        ref = _get_path_ref(Gs, s) + _get_path_ref(Gg, g)[::-1]
        q = np.zeros((2 * cap, nq)); cube = np.zeros((2 * cap, 12))
        (vs, cs, ps), (vg, cg, pg) = arrs
        n = tree_lib.h_path_f64(nq, ctypes.c_int64(cap), _p(vs), _p(cs), _p(ps), len(Gs), s, _p(vg), _p(cg), _p(pg),
                                len(Gg), g, _p(q), _p(cube))
        assert n == len(ref)
        assert all(np.array_equal(q[r], ref[r]) for r in range(n))
        # the cube rows follow their vertices
        idx_s = [int(x) for x in cube[:n, 0] // 100]
        assert all(np.array_equal(vs[:, i] if r < len(_get_path_ref(Gs, s)) else vg[:, i], q[r]) for r, i in enumerate(idx_s))
    # an end that is not a vertex: no path
    n = tree_lib.h_path_f64(nq, ctypes.c_int64(cap), _p(vs), _p(cs), _p(ps), len(Gs), -1, _p(vg), _p(cg), _p(pg),
                            len(Gg), 0, _p(q), _p(cube))
    assert n == 0


# ---------------------------------------------------------------------------------------------------------- C ABI
def test_tree_entries_reject_bad_arguments_without_gpu():
    from gik_b200 import _cabi
    lib = _cabi.lib()
    x = ctypes.c_void_p(8)          # never dereferenced: every call below is refused before any memory access
    for sfx in ("f32", "f64"):
        near = getattr(lib, f"gik_tree_nearest_{sfx}")
        assert near(None, 2, 8, x, x, 4, x, x, x, None) == -6                       # GIK_E_HANDLE
        assert near(None, -1, 8, x, x, 4, x, x, x, None) == -2                      # GIK_E_SIZE
        assert near(None, 2, 0, x, x, 4, x, x, x, None) == -2
        assert near(None, 2, 8, x, x, -4, x, x, x, None) == -2
        assert near(None, 2, 8, None, x, 4, x, x, x, None) == -1                    # GIK_E_NULL
        assert near(None, 2, 8, x, x, 4, x, x, None, None) == -1
        grow = getattr(lib, f"gik_tree_grow_{sfx}")
        ok = [x] * 9                # edge_tree, near, q_start, pose_a, pose_b, num_steps, n_valid, q_path, seg_end
        assert grow(None, 2, 8, x, x, x, x, x, 4, 3, *ok, None) == -6
        assert grow(None, 2, 8, x, x, x, x, x, -4, 3, *ok, None) == -2
        assert grow(None, 2, 8, x, x, x, x, x, 4, -3, *ok, None) == -2
        for i in range(9):
            bad = list(ok); bad[i] = None
            assert grow(None, 2, 8, x, x, x, x, x, 4, 3, *bad, None) == -1
        assert grow(None, 2, 8, x, None, x, x, x, 4, 3, *ok, None) == -1
        assert grow(None, 2, 8, x, x, x, x, None, 4, 3, *ok, None) == -1           # overflow flags
        paths = getattr(lib, f"gik_tree_paths_{sfx}")
        assert paths(None, 3, 8, x, x, x, x, x, x, x, None, None, None) == -6      # size query
        assert paths(None, 3, 8, x, x, x, x, x, x, x, x, x, None) == -6
        assert paths(None, -3, 8, x, x, x, x, x, x, x, None, None, None) == -2
        assert paths(None, 3, 8, x, x, x, x, x, x, None, None, None, None) == -1   # offsets
        assert paths(None, 3, 8, x, x, x, x, x, x, x, x, None, None) == -1         # q without cube
