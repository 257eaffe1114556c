"""Path shortcutting (csrc/gik_shortcut.cuh) on the CPU: the GIK_HD candidate judgement, choice, length and row writer
compiled with g++ and run the way the two kernels run them, against a numpy restatement of the rules in
include/gik.h, bit for bit; plus the argument checks of the C entries and the range of planner._draw_pairs (no GPU
needed)."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest
import torch

from conftest import ROOT

CSRC = os.path.join(ROOT, "motion-planning-and-control-for-dual-manipulator-robot_b200", "csrc")

HARNESS = r"""
#include <stdint.h>
#include <math.h>
#include "gik_core.cuh"
#include "gik_tree.cuh"
#include "gik_shortcut.cuh"
using namespace gik;

// the select kernel's work: per path, lanes 0..31 judge candidate k = lane (k < K), xor-butterfly merge, lane 0
// writes; then the inclusive scan of the row counts
template <typename T>
static void select_all(int nq, int64_t Q, int K, int max_steps, const int64_t* off, const T* q, const int32_t* pi,
                       const int32_t* pj, const int32_t* ns, const int32_t* nv, const T* q_path, double tol,
                       int32_t* chosen, double* length, int64_t* off_out) {
  const int64_t E = Q * K;
  off_out[0] = 0;
  for (int64_t p = 0; p < Q; ++p) {
    const int64_t o = off[p], n = off[p + 1] - o;
    double bg[32]; int bk[32];
    for (int l = 0; l < 32; ++l) {
      bg[l] = 0.0; bk[l] = -1;
      if (l < K) {
        const int64_t e = p * K + l;
        double g;
        if (sc_candidate(nq, n, q + o * nq, pi[e], pj[e], ns[e], nv[e], max_steps, q_path, E, e, tol, g)) { bg[l] = g; bk[l] = l; }
      }
    }
    for (int s = 16; s > 0; s >>= 1) {
      double ng[32]; int nk[32];
      for (int l = 0; l < 32; ++l) {
        ng[l] = bg[l]; nk[l] = bk[l];
        if (sc_better(bg[l ^ s], bk[l ^ s], bg[l], bk[l])) { ng[l] = bg[l ^ s]; nk[l] = bk[l ^ s]; }
      }
      for (int l = 0; l < 32; ++l) { bg[l] = ng[l]; bk[l] = nk[l]; }
    }
    const int k = bk[0];
    const int64_t e = p * K + (k < 0 ? 0 : k);
    int i = 0, j = 0, m = 0;
    int64_t n_out = n;
    if (k >= 0) { i = pi[e]; j = pj[e]; m = ns[e]; n_out = n - (j - i) + m; }
    chosen[p] = k;
    length[p] = sc_length(nq, n_out, k >= 0, q + o * nq, i, j, m, q_path, E, e);
    off_out[p + 1] = off_out[p] + n_out;
  }
}

// the write kernel's work: per path, every output row
template <typename T>
static void write_all(int nq, int64_t Q, int K, const int64_t* off, const T* q, const T* cube, const int32_t* pi,
                      const int32_t* pj, const int32_t* ns, const T* q_path, const int32_t* chosen, const int64_t* off_out,
                      T* q_out, T* cube_out) {
  const int64_t E = Q * K;
  for (int64_t p = 0; p < Q; ++p) {
    const int64_t o = off[p], oo = off_out[p], n_out = off_out[p + 1] - oo;
    const int k = chosen[p];
    const bool ch = k >= 0;
    const int64_t e = ch ? p * K + k : 0;
    const int i = ch ? pi[e] : 0, j = ch ? pj[e] : 0, m = ch ? ns[e] : 0;
    T ci[12], xi[6] = {};
    for (int c = 0; c < 12; ++c) ci[c] = ch ? cube[(o + i) * 12 + c] : T(0);
    if (ch && m > 1) {
      T cj[12];
      for (int c = 0; c < 12; ++c) cj[c] = cube[(o + j) * 12 + c];
      se3_delta(ci, cj, xi);
    }
    for (int64_t r = 0; r < n_out; ++r)
      sc_write_row(r, ch, nq, q + o * nq, cube + o * 12, i, j, m, q_path, E, e, ci, xi, q_out + oo * nq, cube_out + oo * 12);
  }
}

#define ENTRIES(T, SFX)                                                                                                \
  void h_select_##SFX(int nq, int64_t Q, int K, int S, const int64_t* off, const T* q, const int32_t* pi,               \
                      const int32_t* pj, const int32_t* ns, const int32_t* nv, const T* qp, double tol, int32_t* ch,   \
                      double* len, int64_t* oo) { select_all(nq, Q, K, S, off, q, pi, pj, ns, nv, qp, tol, ch, len, oo); } \
  void h_write_##SFX(int nq, int64_t Q, int K, const int64_t* off, const T* q, const T* cube, const int32_t* pi,        \
                     const int32_t* pj, const int32_t* ns, const T* qp, const int32_t* ch, const int64_t* oo, T* qo,   \
                     T* co) { write_all(nq, Q, K, off, q, cube, pi, pj, ns, qp, ch, oo, qo, co); }
extern "C" {
ENTRIES(double, f64)
ENTRIES(float, f32)
}
"""


@pytest.fixture(scope="module")
def sc_lib(tmp_path_factory):
    d = tmp_path_factory.mktemp("shortcut_harness")
    src = d / "harness.cpp"
    src.write_text(HARNESS)
    out = d / "libshortcut.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-I", CSRC,
                    "-I", os.path.join(ROOT, "include"), "-o", str(out), str(src)], check=True)
    return ctypes.CDLL(str(out))


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


# ------------------------------------------------------------------------------------------------ numpy restatement
def _norm(a, b):
    """||a - b|| in fp64: differences and squares of the stored values, summed left to right."""
    s = 0.0
    for x, y in zip(a.tolist(), b.tolist()):
        d = float(x) - float(y)
        s = s + d * d
    return math.sqrt(s)


def _path_length(rows):
    L = 0.0
    for r in range(1, len(rows)):
        L = L + _norm(rows[r], rows[r - 1])
    return L


def _placements(ci, cj, ns, dtype):
    from gik_b200.path import se3_interpolate
    m = np.arange(1, ns)
    if len(m) == 0:
        return np.zeros((0, 12), dtype)
    A = torch.from_numpy(np.tile(ci, (len(m), 1)))
    B = torch.from_numpy(np.tile(cj, (len(m), 1)))
    return se3_interpolate(A, B, torch.from_numpy(m.astype(dtype)) / torch.tensor(ns, dtype=A.dtype)).numpy()


def _reference(paths, pi, pj, ns, nv, q_path, tol, S):
    """-> chosen [Q], length [Q], list of (q, cube) output paths."""
    Q, K = pi.shape
    chosen, length, out = np.full(Q, -1, np.int32), np.zeros(Q), []
    for p, (q, cube) in enumerate(paths):
        n = len(q)
        best, bg = -1, None
        for k in range(K):
            e = p * K + k
            i, j, m = int(pi[p, k]), int(pj[p, k]), int(ns[p, k])
            if not (i >= 0 and j >= i + 2 and j <= n - 1 and 1 <= m <= S and nv[p, k] == m):
                continue
            s = [q_path[t, :, e] for t in range(m)]                 # s[t] = step t + 1
            if not (_norm(s[m - 1], q[j]) < tol):
                continue
            l_old = 0.0
            for t in range(i, j):
                l_old = l_old + _norm(q[t + 1], q[t])
            if m == 1:
                l_new = _norm(q[j], q[i])
            else:
                l_new = _norm(s[0], q[i])
                for t in range(1, m - 1):
                    l_new = l_new + _norm(s[t], s[t - 1])
                l_new = l_new + _norm(q[j], s[m - 2])
            g = l_old - l_new
            if g > 0 and (best < 0 or g > bg):
                best, bg = k, g
        chosen[p] = best
        if best < 0:
            out.append((q.copy(), cube.copy()))
        else:
            e = p * K + best
            i, j, m = int(pi[p, best]), int(pj[p, best]), int(ns[p, best])
            steps = np.stack([q_path[t, :, e] for t in range(m - 1)]) if m > 1 else np.zeros((0, q.shape[1]), q.dtype)
            out.append((np.vstack([q[:i + 1], steps, q[j:]]),
                        np.vstack([cube[:i + 1], _placements(cube[i], cube[j], m, q.dtype), cube[j:]])))
        length[p] = _path_length(out[-1][0])
    return chosen, length, out


def _run(lib, sfx, paths, pi, pj, ns, nv, q_path, tol, S, nq):
    Q, K = pi.shape
    dt = q_path.dtype
    off = np.zeros(Q + 1, np.int64)
    off[1:] = np.cumsum([len(q) for q, _ in paths])
    q = np.ascontiguousarray(np.vstack([x for x, _ in paths] + [np.zeros((0, nq), dt)]), dt)
    cube = np.ascontiguousarray(np.vstack([c for _, c in paths] + [np.zeros((0, 12), dt)]), dt)
    ch, ln, oo = np.zeros(Q, np.int32), np.zeros(Q), np.zeros(Q + 1, np.int64)
    a = [np.ascontiguousarray(x, np.int32) for x in (pi, pj, ns, nv)]
    qp = np.ascontiguousarray(q_path)
    getattr(lib, f"h_select_{sfx}")(nq, ctypes.c_int64(Q), K, S, _p(off), _p(q), *[_p(x) for x in a], _p(qp),
                                    ctypes.c_double(tol), _p(ch), _p(ln), _p(oo))
    qo, co = np.zeros((oo[-1], nq), dt), np.zeros((oo[-1], 12), dt)
    getattr(lib, f"h_write_{sfx}")(nq, ctypes.c_int64(Q), K, _p(off), _p(q), _p(cube), *[_p(x) for x in a[:3]], _p(qp),
                                   _p(ch), _p(oo), _p(qo), _p(co))
    return ch, ln, [(qo[oo[p]:oo[p + 1]], co[oo[p]:oo[p + 1]]) for p in range(Q)]


# ------------------------------------------------------------------------------------------------ fabricated rounds
def _fabricate(rng, dtype, rotate):
    """Paths of 0 .. 30 rows with cube translations along a line, K = 7 candidates each, and edge outputs: steps near
    the straight line from q_i to q_j (so some candidates shorten the path), ns in 1 .. S (some above S, some
    idle), n_valid mostly ns, and the special cases below."""
    nq, K, S = 15, 7, 6
    lens = [5, 0, 2, 3, 12, 30, 1, 8, 6, 9, 4, 3]
    paths = []
    for n in lens:
        q = rng.uniform(-1, 1, (n, nq))
        if n > 4:
            q[2] = q[1]                                              # grow() stores each segment's start twice
        cube = np.zeros((n, 12)); cube[:, [0, 4, 8]] = 1
        cube[:, 9:] = np.array([0.3, -0.2, 0.95]) + np.cumsum(rng.uniform(-0.02, 0.02, (n, 3)), axis=0)
        if rotate and n:
            from conftest import rot_rpy
            for r in range(n):
                cube[r, :9] = rot_rpy(*rng.uniform(-0.4, 0.4, 3)).reshape(9)
        paths.append((q.astype(dtype), cube.astype(dtype)))
    Q = len(paths)
    from gik_b200.planner import _draw_pairs
    n_t = torch.tensor(lens, dtype=torch.int64)
    pi, pj = [x.numpy().copy() for x in _draw_pairs(n_t, K, torch.Generator().manual_seed(int(rng.integers(1 << 30))))]
    ns = rng.integers(1, S + 1, (Q, K)).astype(np.int32)
    ns[rng.uniform(size=(Q, K)) < 0.1] = S + 1                      # more steps than the launch had: rejected
    ns[pi < 0] = 0
    nv = ns.copy()
    nv[rng.uniform(size=(Q, K)) < 0.15] -= 1                        # a step failed or collided
    E = Q * K
    q_path = np.zeros((S, nq, E), dtype)
    for p, (q, _) in enumerate(paths):
        for k in range(K):
            e, i, j, m = p * K + k, pi[p, k], pj[p, k], min(ns[p, k], S)
            if i < 0:
                continue
            for t in range(m):
                a = (t + 1) / ns[p, k]
                q_path[t, :, e] = ((1 - a) * q[i].astype(float) + a * q[j].astype(float)
                                   + rng.normal(0, 0.05 if t < m - 1 else 0.02, nq)).astype(dtype)
            q_path[m:, :, e] = 0
    # path 0 (5 rows): scripted candidates
    q0 = paths[0][0]
    q0[:, 0] = 0.5
    q0[1] = q0[0]                                                    # rows 0, 1 equal: (0, 2) with ns = 1 gains nothing
    q0[2] = q0[0]
    q0[2, 1] = q0[0, 1] + 0.5                                        # ... unless row 2 moves; see candidate 2 below
    cand = [(0, 2, 1), (1, 4, 2), (1, 4, 2), (0, 3, 3), (1, 4, 2), (1, 3, 1), (0, 4, 1)]
    for k, (i, j, m) in enumerate(cand):
        pi[0, k], pj[0, k], ns[0, k], nv[0, k] = i, j, m, m
    q_path[:, :, :K] = 0
    # k = 0: ns = 1, s_1 = q_2 exactly; L_old = |q1 - q0| + |q2 - q1| = 0 + |q2 - q0| = L_new: zero gain, rejected
    q_path[0, :, 0] = q0[2]
    # k = 1, 2, 4: the same edge with the same gain (a tie): k = 1 must win; its last step misses q_4 by exactly 0.25
    # in component 0 (0.5 -> 0.75): accepted only while join_tol > 0.25
    for k in (1, 2, 4):
        q_path[0, :, k] = (0.5 * (q0[1].astype(float) + q0[4].astype(float))).astype(dtype)
        q_path[1, :, k] = q0[4]
        q_path[1, 0, k] = 0.75
    # k = 3: n_valid < ns
    nv[0, 3] = 2
    q_path[:3, :, 3] = q0[3]
    # k = 5: ns = 1, s_1 at q_3: accepted whenever it shortens the path; k = 6: a gap of 2 at the join, rejected
    q_path[0, :, 5] = q0[3]
    q_path[0, :, 6] = q0[4]
    q_path[0, 0, 6] = 2.5
    return paths, pi, pj, ns, nv, q_path, S, nq


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("rotate", [False, True])
@pytest.mark.parametrize("tol", [0.5, 0.25, 0.2500001, 0.05])
def test_select_and_splice_match_the_restatement(sc_lib, dtype, rotate, tol):
    rng = np.random.default_rng(int(tol * 1e7) % 1000 + 10 * rotate + (dtype == np.float32))
    paths, pi, pj, ns, nv, q_path, S, nq = _fabricate(rng, dtype, rotate)
    sfx = "f64" if dtype == np.float64 else "f32"
    ch, ln, out = _run(sc_lib, sfx, paths, pi, pj, ns, nv, q_path, tol, S, nq)
    rch, rln, rout = _reference(paths, pi, pj, ns, nv, q_path, tol, S)
    assert np.array_equal(ch, rch)
    assert np.array_equal(ln, rln)                                    # bit for bit
    pl_tol = 0.0 if not rotate else (1e-12 if dtype == np.float64 else 2e-6)
    for (q, c), (rq, rc), (q_in, c_in) in zip(out, rout, paths):
        assert q.shape == rq.shape and np.array_equal(q, rq)
        assert c.shape == rc.shape and np.abs(c.astype(float) - rc.astype(float)).max(initial=0.0) <= pl_tol
        if len(q_in):                                                 # the ends are kept bit for bit
            assert np.array_equal(q[0], q_in[0]) and np.array_equal(q[-1], q_in[-1])
            assert np.array_equal(c[0], c_in[0]) and np.array_equal(c[-1], c_in[-1])
        assert _path_length(q) <= _path_length(q_in)
    # the scripted path 0: the tie goes to candidate 1 when the join gap of 0.25 is inside join_tol, else to 5
    assert ch[0] == (1 if tol > 0.25 else 5)
    # what the fabricated round covers
    assert (ch[[1, 2, 6]] == -1).all()                                # empty, 2-vertex and 1-vertex paths
    if tol >= 0.25:                                                   # (at 0.05 the fabricated joins mostly miss)
        assert (ch >= 0).sum() >= 4


def test_no_candidates_computes_lengths_only(sc_lib):
    rng = np.random.default_rng(3)
    paths, pi, pj, ns, nv, q_path, S, nq = _fabricate(rng, np.float64, False)
    e = np.zeros((len(paths), 0), np.int32)
    ch, ln, out = _run(sc_lib, "f64", paths, e, e, e, e, np.zeros((S, nq, 0)), 0.5, S, nq)
    assert (ch == -1).all()
    assert np.array_equal(ln, [_path_length(q) for q, _ in paths])
    assert all(np.array_equal(q, q0) and np.array_equal(c, c0) for (q, c), (q0, c0) in zip(out, paths))


# ------------------------------------------------------------------------------------------------ pair draw
def test_draw_pairs_range_and_coverage():
    from gik_b200.planner import _draw_pairs
    n = torch.tensor([0, 1, 2, 3, 4, 7, 50, 3, 200], dtype=torch.int64)
    K = 32
    g = torch.Generator().manual_seed(0)
    seen = {}
    for _ in range(200):
        i, j = _draw_pairs(n, K, g)
        assert i.dtype == torch.int32 and j.dtype == torch.int32 and i.shape == (len(n), K)
        for p, m in enumerate(n.tolist()):
            if m < 3:
                assert (i[p] == -1).all() and (j[p] == -1).all()
                continue
            assert (i[p] >= 0).all() and (j[p] >= i[p] + 2).all() and (j[p] <= m - 1).all()
            seen.setdefault(p, set()).update(zip(i[p].tolist(), j[p].tolist()))
    for p, m in enumerate(n.tolist()):                               # every pair of the short paths is drawn
        if 3 <= m <= 7:
            assert len(seen[p]) == (m - 1) * (m - 2) // 2
    # the same generator state gives the same pairs
    a = _draw_pairs(n, 5, torch.Generator().manual_seed(9))
    b = _draw_pairs(n, 5, torch.Generator().manual_seed(9))
    assert all(torch.equal(x, y) for x, y in zip(a, b))


# ------------------------------------------------------------------------------------------------ C ABI
def test_shortcut_entries_reject_bad_arguments_without_gpu():
    from gik_b200 import _cabi
    lib = _cabi.lib()
    x = ctypes.c_void_p(8)          # never dereferenced: every call below is refused before any memory access
    for sfx in ("f32", "f64"):
        f = getattr(lib, f"gik_path_shortcut_{sfx}")

        def call(Q=3, K=4, S=5, tol=0.5, p=None, out=(None, None)):
            p = [x] * 9 if p is None else p      # offsets, q, cube, pair_i, pair_j, num_steps, n_valid, q_path, + 3 outs
            return f(None, Q, K, S, *p[:8], ctypes.c_double(tol), *p[8:], x, x, *out, None)

        p9 = [x] * 9
        assert call() == -6                                          # GIK_E_HANDLE (size query)
        assert call(out=(x, x)) == -6
        assert call(Q=-1) == -2 and call(K=-1) == -2 and call(K=33) == -2 and call(S=-1) == -2   # GIK_E_SIZE
        assert call(K=32) == -6
        assert call(tol=-1e-9) == -5 and call(tol=float("nan")) == -5 # GIK_E_PARAM
        assert call(Q=-1, tol=-1.0) == -2                             # sizes are checked first
        for i in range(8):
            bad = list(p9); bad[i] = None
            assert call(p=bad) == -1, i                               # GIK_E_NULL
        bad = list(p9); bad[8] = None
        assert call(p=bad) == -1                                      # chosen
        assert f(None, 3, 4, 5, *p9[:8], ctypes.c_double(0.5), x, None, x, None, None, None) == -1   # length
        assert f(None, 3, 4, 5, *p9[:8], ctypes.c_double(0.5), x, x, None, None, None, None) == -1   # offsets_out
        assert call(out=(x, None)) == -1 and call(out=(None, x)) == -1  # q_out without cube_out
        none4 = [x, x, x, None, None, None, None, None, x]
        assert call(K=0, p=none4) == -6                               # K = 0: no candidate arrays needed
        nopath = list(p9); nopath[7] = None
        assert call(S=0, p=nopath) == -6 and call(S=1, p=nopath) == -1  # q_path only when max_steps > 0
        assert call(Q=0, p=[None] * 9) == -6
