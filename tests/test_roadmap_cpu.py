"""Grasp roadmap (csrc/gik_roadmap.cuh) on the CPU: the GIK_HD kNN slot rule, edge judgement, relaxation, predecessor and
goal rules compiled with g++ and run the way the kernels run them, against a stable numpy argsort, a numpy restatement
of the edge rules (bit for bit) and scipy's Dijkstra; plus the argument checks of the C entries (no GPU needed)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from test_shortcut_cpu import _norm

CSRC = os.path.join(ROOT, "motion-planning-and-control-for-dual-manipulator-robot_b200", "csrc")

HARNESS = r"""
#include <stdint.h>
#include <string.h>
#include <math.h>
#include "gik_core.cuh"
#include "gik_tree.cuh"
#include "gik_shortcut.cuh"
#include "gik_roadmap.cuh"
using namespace gik;

// the kNN kernel's work for one warp per point: slot l = lane l; per chunk of 32 vertices the lanes whose candidate
// beats slot k - 1 are inserted in lane order, every slot updated from its own and the previous slot's entry
template <typename T>
static void knn_all(int N, int k, const T* cube, int64_t P, const T* points, int32_t* nbr) {
  for (int64_t p = 0; p < P; ++p) {
    const T* pt = points ? points + p * 12 : cube + p * 12;
    const int self = points ? -1 : (int)p;
    double d[32]; int id[32];
    for (int l = 0; l < 32; ++l) { d[l] = INFINITY; id[l] = kRmNone; }
    for (int v0 = 0; v0 < N; v0 += 32) {
      double cd[32]; bool in[32];
      const double td = d[k - 1]; const int ti = id[k - 1];
      for (int l = 0; l < 32; ++l) {
        const int v = v0 + l;
        cd[l] = v < N && v != self ? rm_dist(cube + (int64_t)v * 12, pt) : INFINITY;
        in[l] = v < N && v != self && tree_better(cd[l], v, td, ti);
      }
      for (int src = 0; src < 32; ++src) {
        if (!in[src]) continue;
        double nd[32]; int ni[32];
        for (int l = 0; l < 32; ++l)
          rm_knn_slot(l == 0, d[l], id[l], l ? d[l - 1] : d[0], l ? id[l - 1] : id[0], cd[src], v0 + src, nd[l], ni[l]);
        for (int l = 0; l < 32; ++l) { d[l] = nd[l]; id[l] = ni[l]; }
      }
    }
    for (int l = 0; l < k; ++l) nbr[p * k + l] = id[l];
  }
}

// the SSSP kernel's work for one query, its threads run one after the other
static void sssp_one(int N, int ka, int64_t E, const int64_t* row_ptr, const int32_t* dst, const double* w,
                     const int32_t* av, const double* aw, uint64_t* dist, int32_t* mark, int32_t* gp, double* len) {
  for (int v = 0; v < N; ++v) { dist[v] = rm_bits(INFINITY); mark[v] = -1; }
  for (int s = 0; s < ka; ++s) {
    const int a = av[s];
    if (a >= 0 && a < N && aw[s] < INFINITY && rm_lower(dist + a, aw[s])) mark[a] = 0;
  }
  for (int round = 1;; ++round) {
    bool ch = false;
    for (int u = 0; u < N; ++u)
      if (rm_load(mark + u) == round - 1) ch |= rm_relax(N, E, row_ptr, dst, w, dist, mark, u, round);
    if (!ch) break;
  }
  int32_t* pred = mark;
  for (int v = 0; v < N; ++v) pred[v] = kRmNone;
  for (int s = 0; s < ka; ++s) {
    const int a = av[s];
    if (a >= 0 && a < N && aw[s] < INFINITY && rm_bits(aw[s]) == dist[a]) rm_min(pred + a, -1);
  }
  for (int u = 0; u < N; ++u) rm_pred(N, E, row_ptr, dst, w, dist, pred, u);
  for (int v = 0; v < N; ++v) if (pred[v] == kRmNone) pred[v] = -2;
  *gp = rm_goal(N, ka, av, aw, dist, *len);
}

extern "C" {
void h_knn_f64(int N, int k, const double* c, int64_t P, const double* p, int32_t* nbr) { knn_all(N, k, c, P, p, nbr); }
void h_knn_f32(int N, int k, const float* c, int64_t P, const float* p, int32_t* nbr) { knn_all(N, k, c, P, p, nbr); }
void h_weight_f64(int nq, int64_t E, int S, const double* qf, const double* qt, const int32_t* ns, const int32_t* nv,
                  const double* qp, double tol, double* w) {
  for (int64_t e = 0; e < E; ++e) w[e] = rm_edge_weight(nq, qf + e * nq, qt + e * nq, ns[e], nv[e], S, qp, E, e, tol);
}
void h_weight_f32(int nq, int64_t E, int S, const float* qf, const float* qt, const int32_t* ns, const int32_t* nv,
                  const float* qp, double tol, double* w) {
  for (int64_t e = 0; e < E; ++e) w[e] = rm_edge_weight(nq, qf + e * nq, qt + e * nq, ns[e], nv[e], S, qp, E, e, tol);
}
void h_sssp(int N, int ka, int64_t E, const int64_t* row_ptr, const int32_t* dst, const double* w, const int32_t* av,
            const double* aw, double* dist, int32_t* pred, int32_t* gp, double* len) {
  sssp_one(N, ka, E, row_ptr, dst, w, av, aw, (uint64_t*)dist, pred, gp, len);
}
}
"""


@pytest.fixture(scope="module")
def rm_lib(tmp_path_factory):
    d = tmp_path_factory.mktemp("roadmap_harness")
    src = d / "harness.cpp"
    src.write_text(HARNESS)
    out = d / "libroadmap.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-I", CSRC,
                    "-I", os.path.join(ROOT, "include"), "-o", str(out), str(src)], check=True)
    return ctypes.CDLL(str(out))


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


# ------------------------------------------------------------------------------------------------ kNN
def knn_reference(cube, k, points=None):
    """Stable argsort of the fp64 translation distances sqrt((dx^2 + dy^2) + dz^2); a vertex excludes itself."""
    V = cube[:, 9:].astype(np.float64)
    P = V if points is None else points[:, 9:].astype(np.float64)
    d = P[:, None, :] - V[None, :, :]
    sq = d * d
    dist = np.sqrt((sq[..., 0] + sq[..., 1]) + sq[..., 2])
    if points is None:
        np.fill_diagonal(dist, np.inf)
    return np.argsort(dist, axis=1, kind="stable")[:, :k].astype(np.int32)


def _knn(lib, cube, k, points=None):
    sfx = "f64" if cube.dtype == np.float64 else "f32"
    P = cube.shape[0] if points is None else points.shape[0]
    nbr = np.zeros((P, k), np.int32)
    getattr(lib, f"h_knn_{sfx}")(cube.shape[0], k, _p(cube), ctypes.c_int64(P), None if points is None else _p(points),
                                 _p(nbr))
    return nbr


def _grid_cubes(rng, n, dtype, step=0.25):
    """Translations on a coarse grid: many exactly equal distances (ties), exact in fp32 and fp64."""
    c = np.zeros((n, 12)); c[:, [0, 4, 8]] = 1
    c[:, 9:] = rng.integers(-4, 5, (n, 3)) * step
    return np.ascontiguousarray(c.astype(dtype))


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("N,k", [(2, 1), (33, 32), (100, 16), (257, 8), (70, 5)])
def test_knn_matches_a_stable_argsort(rm_lib, dtype, N, k):
    rng = np.random.default_rng(N * 100 + k)
    for cube in (_grid_cubes(rng, N, dtype),
                 np.ascontiguousarray(np.hstack([np.tile(np.eye(3).reshape(9), (N, 1)), rng.uniform(-1, 1, (N, 3))]).astype(dtype))):
        assert np.array_equal(_knn(rm_lib, cube, k), knn_reference(cube, k))
        pts = _grid_cubes(rng, 40, dtype)
        kp = min(k, N - 1)
        assert np.array_equal(_knn(rm_lib, cube, kp, pts), knn_reference(cube, kp, pts))


def test_knn_ties_go_to_the_lower_index(rm_lib):
    cube = np.zeros((40, 12)); cube[:, [0, 4, 8]] = 1
    cube[:, 9] = np.where(np.arange(40) % 2 == 0, 1.0, -1.0)          # every vertex at distance 1 from the origin
    pts = np.zeros((1, 12)); pts[0, [0, 4, 8]] = 1
    assert list(_knn(rm_lib, cube, 7, pts)[0]) == list(range(7))
    assert list(_knn(rm_lib, cube, 3)[0]) == [2, 4, 6]                 # vertex 0: its distance-0 twins, itself excluded


# ------------------------------------------------------------------------------------------------ edge judgement
def weight_reference(q_from, q_to, ns, nv, q_path, tol, S):
    E = q_from.shape[0]
    w = np.full(E, np.inf)
    for e in range(E):
        m = int(ns[e])
        if not (1 <= m <= S and nv[e] == m):
            continue
        s = [q_path[t, :, e] for t in range(m)]
        if not (_norm(s[m - 1], q_to[e]) < tol):
            continue
        rows = [q_from[e]] + s[:m - 1] + [q_to[e]]
        L = 0.0
        for r in range(1, len(rows)):
            L = L + _norm(rows[r], rows[r - 1])
        w[e] = L
    return w


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("tol", [0.5, 0.05, 0.25])
def test_edge_acceptance_and_weight_match_the_restatement(rm_lib, dtype, tol):
    rng = np.random.default_rng(int(tol * 100) + (dtype == np.float32))
    nq, E, S = 15, 300, 6
    q_from = rng.uniform(-1, 1, (E, nq)).astype(dtype)
    q_to = (q_from + rng.normal(0, 0.3, (E, nq))).astype(dtype)
    ns = rng.integers(1, S + 2, E).astype(np.int32)                   # some above S: rejected
    nv = ns.copy(); nv[rng.uniform(size=E) < 0.15] -= 1
    q_path = np.zeros((S, nq, E), dtype)
    for e in range(E):
        m = min(ns[e], S)
        for t in range(m):
            a = (t + 1) / ns[e]
            q_path[t, :, e] = (1 - a) * q_from[e] + a * q_to[e] + rng.normal(0, 0.1 if t < m - 1 else 0.01, nq)
    q_path[0, :, 0] = q_to[0]; ns[0] = nv[0] = 1                     # lands exactly: weight ||q_to - q_from||
    q_path[0, :, 1] = q_to[1]; q_path[0, 0, 1] += np.float32(0.25); ns[1] = nv[1] = 1   # misses by exactly 0.25
    w = np.zeros(E)
    sfx = "f64" if dtype == np.float64 else "f32"
    getattr(rm_lib, f"h_weight_{sfx}")(nq, ctypes.c_int64(E), S, _p(q_from), _p(q_to), _p(ns), _p(nv), _p(q_path),
                                       ctypes.c_double(tol), _p(w))
    ref = weight_reference(q_from, q_to, ns, nv, q_path, tol, S)
    assert np.array_equal(w, ref)                                     # bit for bit, +inf where rejected
    assert w[0] == _norm(q_to[0], q_from[0])
    assert np.isfinite(w[1]) == (tol > 0.25)
    assert np.isfinite(w).sum() > 10 and (~np.isfinite(w)).sum() > 10


# ------------------------------------------------------------------------------------------------ shortest paths
def _sssp(lib, N, row_ptr, dst, w, av, aw):
    ka = (len(av) - 1) // 2
    dist, pred = np.zeros(N), np.zeros(N, np.int32)
    gp, ln = np.zeros(1, np.int32), np.zeros(1)
    args = [np.ascontiguousarray(x, t) for x, t in ((row_ptr, np.int64), (dst, np.int32), (w, np.float64),
                                                    (av, np.int32), (aw, np.float64))]
    lib.h_sssp(N, ka, ctypes.c_int64(len(dst)), *[_p(x) for x in args], _p(dist), _p(pred), _p(gp), _p(ln))
    return dist, pred, int(gp[0]), float(ln[0])


def scipy_reference(N, row_ptr, dst, w, av, aw, preds=True):
    """Dijkstra from a virtual start (node N) over the roadmap plus the attachments, to a virtual goal (node N + 1); then
    the predecessor (unless not `preds`) and goal rules restated from the final distances."""
    from scipy.sparse import csr_matrix
    from scipy.sparse.csgraph import dijkstra
    ka = (len(av) - 1) // 2
    src = np.repeat(np.arange(N), np.diff(row_ptr))
    rows, cols, vals = list(src), list(dst), list(w)
    for s in range(2 * ka + 1):
        if np.isfinite(aw[s]):
            rows.append(N if s < ka or s == 2 * ka else av[s])
            cols.append(N + 1 if s >= ka else av[s])
            vals.append(aw[s])
    G = csr_matrix((vals, (rows, cols)), shape=(N + 2, N + 2))
    d = dijkstra(G, directed=True, indices=N)
    dist = d[:N]
    pred = np.full(N, -2, np.int32)
    for v in range(N if preds else 0):
        if not np.isfinite(dist[v]):
            continue
        if any(av[s] == v and aw[s] == dist[v] for s in range(ka)):
            pred[v] = -1
            continue
        cand = [u for u, x, ww in zip(src, dst, w) if x == v and np.isfinite(dist[u]) and dist[u] + ww == dist[v]]
        pred[v] = min(cand)
    best, gp = aw[2 * ka], (-1 if np.isfinite(aw[2 * ka]) else -2)
    for s in range(ka, 2 * ka):
        b = av[s]
        if np.isfinite(aw[s]) and np.isfinite(dist[b]):
            c = dist[b] + aw[s]
            if c < best or (c == best and gp >= 0 and b < gp):
                best, gp = c, b
    return dist, pred, gp, (d[N + 1] if gp != -2 else np.inf)


def _random_graph(rng, N, k, ka, quantised):
    nbr = np.stack([rng.choice(np.delete(np.arange(N), i), k, replace=False) for i in range(N)])
    keep = rng.uniform(size=(N, k)) < 0.7
    row_ptr = np.concatenate([[0], np.cumsum(keep.sum(1))]).astype(np.int64)
    dst = nbr[keep].astype(np.int32)
    w = rng.integers(1, 5, len(dst)) * 0.125 if quantised else rng.uniform(0.01, 1.0, len(dst))
    av = np.concatenate([rng.choice(N, ka, replace=False), rng.choice(N, ka, replace=False), [-1]]).astype(np.int32)
    aw = rng.integers(1, 5, 2 * ka + 1) * 0.125 if quantised else rng.uniform(0.01, 1.0, 2 * ka + 1)
    aw[rng.uniform(size=2 * ka + 1) < 0.3] = np.inf
    return row_ptr, dst, w, av, aw


@pytest.mark.parametrize("seed", range(12))
def test_relaxation_and_predecessors_match_dijkstra(rm_lib, seed):
    rng = np.random.default_rng(seed)
    N, k, ka = int(rng.integers(5, 120)), int(rng.integers(1, 6)), int(rng.integers(1, 5))
    k = min(k, N - 1)
    g = _random_graph(rng, N, k, ka, quantised=seed % 2 == 1)       # quantised weights: many equal-length paths
    dist, pred, gp, ln = _sssp(rm_lib, N, *g)
    rdist, rpred, rgp, rln = scipy_reference(N, *g)
    assert np.array_equal(dist, rdist)                                # exactly
    assert np.array_equal(pred, rpred) and gp == rgp
    assert ln == rln or (np.isinf(ln) and np.isinf(rln))


@pytest.mark.parametrize("direct,expect_gp", [(4.0, -1), (np.inf, 3), (5.0, 3)])
def test_scripted_graph_with_equal_weight_ties(rm_lib, direct, expect_gp):
    # start -> 0 (1), start -> 1 (1), start -> 4 (2); 0 -> 2, 1 -> 2, 2 -> 3 (1 each), 0 -> 3 (2), 0 -> 4 (1), 5 isolated
    # goal: 3 -> goal (1), 4 -> goal (2), 5 -> goal rejected: 3 and 4 reach the goal at 4, as the direct edge does at 4
    N = 6
    edges = {0: [(2, 1.0), (3, 2.0), (4, 1.0)], 1: [(2, 1.0)], 2: [(3, 1.0)], 3: [], 4: [], 5: []}
    row_ptr = np.concatenate([[0], np.cumsum([len(edges[u]) for u in range(N)])])
    dst = [v for u in range(N) for v, _ in edges[u]]
    w = [x for u in range(N) for _, x in edges[u]]
    av = [0, 1, 4, 4, 3, 5, -1]
    aw = [1.0, 1.0, 2.0, 2.0, 1.0, np.inf, direct]
    dist, pred, gp, ln = _sssp(rm_lib, N, row_ptr, dst, w, av, aw)
    assert list(dist) == [1, 1, 2, 3, 2, np.inf]
    assert list(pred) == [-1, -1, 0, 0, -1, -2]                       # ties: the virtual start, then the smallest u
    assert gp == expect_gp and ln == 4.0
    rdist, rpred, rgp, rln = scipy_reference(N, np.array(row_ptr), np.array(dst), np.array(w), np.array(av), np.array(aw))
    assert np.array_equal(dist, rdist) and np.array_equal(pred, rpred) and gp == rgp and ln == rln


def test_unconnected_query(rm_lib):
    row_ptr, dst, w = np.array([0, 1, 1]), np.array([1]), np.array([0.5])
    dist, pred, gp, ln = _sssp(rm_lib, 2, row_ptr, dst, w, np.array([0, 0, -1]), np.array([np.inf, 1.0, np.inf]))
    assert gp == -2 and np.isinf(ln) and list(pred) == [-2, -2] and np.isinf(dist).all()


# ------------------------------------------------------------------------------------------------ C ABI
def test_roadmap_entries_reject_bad_arguments_without_gpu():
    from gik_b200 import _cabi
    lib = _cabi.lib()
    x = ctypes.c_void_p(8)          # never dereferenced: every call below is refused before any memory access
    for sfx in ("f32", "f64"):
        knn = getattr(lib, f"gik_knn_{sfx}")
        assert knn(None, 10, 4, x, 5, x, x, None) == -6                  # GIK_E_HANDLE
        assert knn(None, 10, 4, x, 10, None, x, None) == -6              # the vertices themselves
        for N, k, P, pts in ((10, 0, 5, x), (10, 33, 5, x), (10, 10, 5, x), (10, 4, -1, x), (10, 4, 5, None)):
            assert knn(None, N, k, x, P, pts, x, None) == -2, (N, k, P)   # GIK_E_SIZE
        assert knn(None, 33, 32, x, 5, x, x, None) == -6
        assert knn(None, 10, 4, None, 5, x, x, None) == -1 and knn(None, 10, 4, x, 5, x, None, None) == -1
        assert knn(None, 10, 4, None, 0, x, None, None) == -6

        ed = getattr(lib, f"gik_roadmap_edges_{sfx}")
        p5 = [x] * 5
        assert ed(None, 4, 3, *p5, ctypes.c_double(0.5), x, None) == -6
        assert ed(None, -1, 3, *p5, ctypes.c_double(0.5), x, None) == -2 and ed(None, 4, -1, *p5, ctypes.c_double(0.5), x, None) == -2
        assert ed(None, 4, 3, *p5, ctypes.c_double(-1.0), x, None) == -5
        assert ed(None, 4, 3, *p5, ctypes.c_double(float("nan")), x, None) == -5
        for i in range(5):
            bad = list(p5); bad[i] = None
            assert ed(None, 4, 3, *bad, ctypes.c_double(0.5), x, None) == -1, i
        bad = list(p5); bad[4] = None
        assert ed(None, 4, 0, *bad, ctypes.c_double(0.5), x, None) == -6   # q_path only when max_steps > 0
        assert ed(None, 4, 3, *p5, ctypes.c_double(0.5), None, None) == -1

        pa = getattr(lib, f"gik_roadmap_paths_{sfx}")
        p19 = [x] * 19
        assert pa(None, 3, 10, 4, 5, 20, *p19, None, None, None) == -6
        assert pa(None, 3, 10, 4, 5, 20, *p19, x, x, None) == -6
        assert pa(None, 3, 10, 4, 5, 20, *p19, x, None, None) == -1
        for args in ((-1, 10, 4, 5, 20), (3, 0, 4, 5, 20), (3, 10, 33, 5, 20), (3, 10, -1, 5, 20), (3, 10, 4, -1, 20),
                     (3, 10, 4, 5, -1)):
            assert pa(None, *args, *p19, None, None, None) == -2, args
        for i in range(19):
            bad = list(p19); bad[i] = None
            want = -6 if i == 6 else -1                                   # steps may be NULL
            assert pa(None, 3, 10, 4, 5, 20, *bad, None, None, None) == want, i
        bad = list(p19); bad[3] = bad[4] = None
        assert pa(None, 3, 10, 4, 5, 0, *bad, None, None, None) == -6      # no edges: dst, ns not needed
        bad = list(p19); bad[14] = None
        assert pa(None, 3, 10, 4, 0, 20, *bad, None, None, None) == -6     # att_path only when max_steps > 0

    ss = lib.gik_roadmap_sssp
    p11 = [x] * 11
    assert ss(None, 3, 10, 4, 20, *p11, None) == -6
    for args in ((-1, 10, 4, 20), (3, 0, 4, 20), (3, 10, 33, 20), (3, 10, -1, 20), (3, 10, 4, -1)):
        assert ss(None, *args, *p11, None) == -2, args
    for i in range(11):
        bad = list(p11); bad[i] = None
        assert ss(None, 3, 10, 4, 20, *bad, None) == -1, i
    bad = list(p11); bad[1] = bad[2] = None
    assert ss(None, 3, 10, 4, 0, *bad, None) == -6                          # no edges: dst, weight not needed
    assert ss(None, 0, 10, 4, 20, *([None] * 11), None) == -6
