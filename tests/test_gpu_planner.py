"""Batched RRT-connect (planner.computepath_batch) and its tree kernels (csrc/gik_tree.cuh) on the GPU: kernel parity
with Python restatements of computepath's nearest() / grow() / _get_path(), replay parity with computepath on
scripted targets, no cross-talk between queries, and the validity of unscripted plans checked with the oracle."""
import json
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN

pytestmark = pytest.mark.gpu

A_REF = np.array([0.33, -0.3, 0.93]); B_REF = np.array([0.4, 0.11, 0.93])     # config.py:36-37


@pytest.fixture(scope="module")
def solver(table):
    import gik_b200
    s = gik_b200.GraspIK(table, "cuda:0").attach_scene()
    yield s
    s.close()


def _pose(p):
    P = np.zeros(12); P[[0, 4, 8]] = 1; P[9:] = p
    return P


# ------------------------------------------------------------------------------------------------ 1. kernel parity
def _random_trees(rng, n_trees, cap, nq, dtype):
    n_verts = rng.integers(1, cap + 1, n_trees).astype(np.int32)
    n_verts[0] = 1
    verts = rng.uniform(-1, 1, (n_trees, nq, cap))
    dup = rng.integers(0, cap, (n_trees, cap // 3))                       # duplicated vertices (ties)
    for t in range(n_trees):
        verts[t][:, dup[t]] = verts[t][:, :1]
    verts = verts.astype(np.float32 if dtype == torch.float32 else np.float64)
    parent = np.full((n_trees, cap), -1, np.int32)
    for t in range(n_trees):
        for i in range(1, cap):
            parent[t, i] = rng.integers(0, i)
    cubes = rng.uniform(-1, 1, (n_trees, 12, cap)).astype(verts.dtype)
    return verts, cubes, parent, n_verts


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_tree_kernels_match_the_restatements(solver, dtype):
    from gik_b200.path import _get_path, se3_interpolate
    rng = np.random.default_rng(11)
    nq, cap, n_trees = 15, 97, 12
    verts, cubes, parent, n_verts = _random_trees(rng, n_trees, cap, nq, dtype)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()     # noqa: E731
    # nearest: ragged trees, targets near duplicated vertices
    tt = rng.integers(0, n_trees, 300).astype(np.int32)
    T = rng.uniform(-1, 1, (300, nq)).astype(verts.dtype)
    T[::3] = verts[tt[::3], :, 0]
    got = solver.tree_nearest(d(verts), d(n_verts), d(T), d(tt)).cpu().numpy()
    for i in range(300):
        P = verts[tt[i], :, :n_verts[tt[i]]].T.astype(np.float64)
        assert got[i] == ((P[None] - T[i].astype(np.float64)[None, None]) ** 2).sum(axis=2).argmin(axis=1)[0]
    # grow: real edges from the edge kernel, appended to trees 2, 5, 5, 5, 7, 8, 8
    tree = np.array([2, 5, 5, 5, 7, 8, 8], np.int32)
    E = len(tree)
    nv0 = np.minimum(n_verts, 40).astype(np.int32); nv0[tree] = np.minimum(nv0[tree], 20)
    near = np.array([rng.integers(0, nv0[t]) for t in tree], np.int32)
    gold_q = np.array(json.load(open(os.path.join(GOLDEN, "ik_golden.json")))["cases"][0]["q"])
    qs = np.tile(gold_q, (E, 1))
    A = np.tile(_pose(A_REF), (E, 1))
    B = A.copy(); B[:, 9:] = rng.uniform([0.3, -0.3, 1.0], [0.45, 0.1, 1.2], (E, 3))
    ns = (np.floor(np.linalg.norm(A[:, 9:] - B[:, 9:], axis=1) / 0.025) + 1).astype(np.int32)
    S = int(ns.max())
    q_soa, pa, pb = d(qs.T).to(dtype), d(A.T).to(dtype), d(B.T).to(dtype)
    path, nv, _ = solver.project_edges_soa(q_soa, pa, pb, d(ns), S)
    nv = nv.cpu().numpy().copy(); nv[4] = -1                             # an idle slot
    tv, tc, tp, tn = d(verts), d(cubes), d(parent), d(nv0)
    ovf = torch.zeros(n_trees, dtype=torch.uint8, device="cuda:0")
    seg_end = solver.tree_grow(tv, tc, tp, tn, ovf, d(tree), d(near), q_soa, pa, pb, d(ns), d(nv), path).cpu().numpy()
    qp = path.cpu().numpy()
    for t in np.unique(tree):
        G = [(None if parent[t, i] < 0 else int(parent[t, i]), verts[t, :, i]) for i in range(nv0[t])]
        C = [cubes[t, :, i] for i in range(nv0[t])]
        ends = []
        for e in np.flatnonzero(tree == t):
            if nv[e] < 0:
                assert seg_end[e] == -1
                continue
            m = int(nv[e])
            poses = se3_interpolate(torch.from_numpy(A[e:e + 1]).to(dtype).expand(m, 12),
                                    torch.from_numpy(B[e:e + 1]).to(dtype).expand(m, 12),
                                    torch.arange(1, m + 1, dtype=dtype) / int(ns[e])).numpy() if m else np.zeros((0, 12))
            seg = [(qs[e].astype(verts.dtype), A[e].astype(verts.dtype))] + [(qp[j, :, e], poses[j]) for j in range(m)]
            for j, (q, c) in enumerate(seg):
                G.append((len(G) - 1 if j else int(near[e]), q)); C.append(c)
            ends.append(len(G) - 1)
            assert seg_end[e] == ends[-1]
        assert tn[t].item() == len(G)
        V, Cu, Pa = tv[t].cpu().numpy(), tc[t].cpu().numpy(), tp[t].cpu().numpy()
        for i in range(len(G)):
            assert Pa[i] == (-1 if G[i][0] is None else G[i][0])
            assert np.array_equal(V[:, i], G[i][1])
            # identity rotations: the placement each step was solved for, exactly
            assert np.array_equal(Cu[:, i], C[i])
    assert not ovf.any()
    # overflow: a tree that cannot take its edges stays unchanged and is flagged
    tn2 = torch.full((n_trees,), cap - 1, dtype=torch.int32, device="cuda:0")
    before = tv.clone()
    se2 = solver.tree_grow(tv, tc, tp, tn2, ovf, d(tree), d(near), q_soa, pa, pb, d(ns), d(nv), path)
    assert (se2 == -1).all() and (tn2 == cap - 1).all() and torch.equal(tv, before)
    full = np.unique(tree[nv >= 0])                                       # (tree 7 only has the idle slot)
    assert ovf.cpu().numpy()[full].all() and ovf.sum().item() == len(full)
    # paths: Q = n_trees / 2 queries
    Q = n_trees // 2
    tnp = tn.cpu().numpy()
    se = np.array([rng.integers(0, tnp[i]) for i in range(Q)], np.int32); se[1] = -1
    ge = np.array([rng.integers(0, tnp[Q + i]) for i in range(Q)], np.int32)
    q, cube, off = solver.tree_paths(tv, tc, tp, tn, d(se), d(ge))
    q, cube, off = q.cpu().numpy(), cube.cpu().numpy(), off.cpu().numpy()
    V, Cu, Pa = tv.cpu().numpy(), tc.cpu().numpy(), tp.cpu().numpy()
    for i in range(Q):
        if se[i] < 0:
            assert off[i + 1] == off[i]
            continue
        Gs = [(None if Pa[i, k] < 0 else int(Pa[i, k]), (V[i, :, k], Cu[i, :, k])) for k in range(tnp[i])]
        Gg = [(None if Pa[Q + i, k] < 0 else int(Pa[Q + i, k]), (V[Q + i, :, k], Cu[Q + i, :, k])) for k in range(tnp[Q + i])]
        ref = _get_path(Gs, int(se[i])) + _get_path(Gg, int(ge[i]))[::-1]
        assert off[i + 1] - off[i] == len(ref)
        for r, (qv, cv) in enumerate(ref):
            assert np.array_equal(q[off[i] + r], qv) and np.array_equal(cube[off[i] + r], cv)


# ------------------------------------------------------------------------------------------------ scripted targets
class Script:
    """Targets as a deterministic function of (query id, call index n = (retry * per_retry + iteration) * K + k)."""

    def __init__(self, pools):
        self.pools = pools                   # script id -> list of valid (q, placement [3]) samples

    @staticmethod
    def _h(s, n, salt):
        return ((int(s) * 1000003 + int(n) * 7919 + salt * 104729) * 2654435761) % (1 << 32)

    def coin(self, s, n):
        return self._h(s, n, 1) / float(1 << 32)

    def sample(self, s, n):
        pool = self.pools[s % len(self.pools)]
        return pool[self._h(s, n, 2) % len(pool)]


class FakeRng:
    def __init__(self, script, s):
        self.script, self.s, self.n = script, s, 0

    def random(self):
        self.cur = self.n
        self.n += 1
        return self.script.coin(self.s, self.cur)


def _pools(solver, n_pools=9):
    import gik_b200
    g = torch.Generator(device="cuda:0").manual_seed(5)
    pools = []
    for i in range(n_pools):
        q, pl, ok = gik_b200.sample_grasp_poses_batch(solver, 512, _pose(A_REF), _pose(B_REF), dtype=torch.float64, generator=g)
        idx = torch.nonzero(ok).flatten()[:64 + i].cpu()
        pools.append(list(zip(q[idx].cpu().numpy(), pl[idx].cpu().numpy())))
    return pools


def _queries(solver, golden):
    from gik_b200 import experiments
    q0 = np.array(golden["cases"][0]["q"]); qe = np.array(golden["cases"][1]["q"])
    c0 = np.array(golden["cases"][0]["cube_p"]); c1 = np.array(golden["cases"][1]["cube_p"])
    g = torch.Generator(device="cuda:0").manual_seed(6)
    q, pl = experiments.random_endpoints(solver, (np.eye(3), A_REF), (np.eye(3), B_REF), (0.1, 0.1, 0.1), 16, generator=g)
    q, pl = q.cpu().numpy(), pl.cpu().numpy()
    QI = np.vstack([q0, q[:8]]); QG = np.vstack([qe, q[8:]])
    CI = np.vstack([_pose(c0)] + [_pose(p) for p in pl[:8]]); CG = np.vstack([_pose(c1)] + [_pose(p) for p in pl[8:]])
    return QI, QG, CI, CG


def _sequential(monkeypatch, solver, script, s, qi, qg, ci, cg, K):
    import gik_b200
    from gik_b200 import path as path_mod
    rng = FakeRng(script, s)
    monkeypatch.setattr(path_mod._SamplePool, "next", lambda self: script.sample(s, rng.cur))
    P, st = gik_b200.computepath(qi, qg, ci, cg, robot=solver, rng=rng, dtype=torch.float64, expand=K, return_stats=True)
    monkeypatch.undo()
    return P, st


def _batch(monkeypatch, solver, script, ids, QI, QG, CI, CG, K):
    import gik_b200
    from gik_b200 import planner
    per_retry = -(-250 // K)
    ids = np.asarray(ids)

    def draw(solver_, query, retry, iteration, K_, q_goal, cube_start, cube_goal, dtype, generator):
        qh, rh, ih = query.cpu().numpy(), retry.cpu().numpy(), iteration.cpu().numpy()
        A = len(qh)
        q = np.zeros((A, K_, solver_.nq)); c = np.zeros((A, K_, 12))
        gq, gc = q_goal.cpu().numpy(), cube_goal.cpu().numpy()
        for a in range(A):
            for k in range(K_):
                n = (rh[a] * per_retry + ih[a]) * K_ + k
                s = int(ids[qh[a]])
                if script.coin(s, n) < 0.1:
                    q[a, k], c[a, k] = gq[a], gc[a]
                else:
                    qq, p = script.sample(s, n)
                    q[a, k], c[a, k] = qq, _pose(p)
        dev = q_goal.device
        return (torch.from_numpy(q).to(dev, dtype), torch.from_numpy(c).to(dev, dtype),
                torch.ones((A, K_), dtype=torch.bool, device=dev))

    monkeypatch.setattr(planner, "_draw_targets", draw)
    out = gik_b200.computepath_batch(QI, QG, CI, CG, robot=solver, dtype=torch.float64, expand=K)
    monkeypatch.undo()
    q, cube, off, st = out
    off = off.cpu().numpy()
    return ([q[off[i]:off[i + 1]].cpu().numpy() for i in range(len(off) - 1)],
            [cube[off[i]:off[i + 1]].cpu().numpy() for i in range(len(off) - 1)],
            {k: v.cpu().numpy() for k, v in st.items()})


# ------------------------------------------------------------------------------------------------ 2. replay parity
@pytest.mark.parametrize("K", [1, 8])
def test_replay_parity_with_computepath(solver, golden, monkeypatch, K):
    script = Script(_pools(solver))
    QI, QG, CI, CG = _queries(solver, golden)
    for s in range(len(QI)):
        P, st = _sequential(monkeypatch, solver, script, s, QI[s], QG[s], CI[s], CG[s], K)
        qb, cb, sb = _batch(monkeypatch, solver, script, [s], QI[s:s + 1], QG[s:s + 1], CI[s:s + 1], CG[s:s + 1], K)
        print(f"K={K} query {s}: {len(P)} vertices, {st}; batch {len(qb[0])} vertices, iterations {sb['iterations'][0]}")
        assert len(qb[0]) == len(P)
        assert sb["iterations"][0] == st["iterations"] and sb["retries"][0] == st["retries"] and sb["edges"][0] == st["edges"]
        if P:
            assert np.abs(qb[0] - np.array(P)).max() <= 1e-12
            assert sb["vertices"][0] == st["vertices"]
            # the stored placements: start / goal placements at the ends, steps of at most one step_size in between
            assert np.array_equal(cb[0][0], CI[s]) and np.array_equal(cb[0][-1], CG[s])


# ------------------------------------------------------------------------------------------------ 3. no cross-talk
def test_no_cross_talk_between_queries(solver, golden, monkeypatch):
    K = 8
    script = Script(_pools(solver))
    QI, QG, CI, CG = _queries(solver, golden)
    singles = [_batch(monkeypatch, solver, script, [s], QI[s:s + 1], QG[s:s + 1], CI[s:s + 1], CG[s:s + 1], K)
               for s in range(9)]
    nine = _batch(monkeypatch, solver, script, list(range(9)), QI, QG, CI, CG, K)
    pad = 256
    order = np.random.default_rng(3).permutation(pad)                   # the 9 queries at scattered rows
    ids = np.arange(pad) + 100
    rows = order[:9]
    ids[rows] = np.arange(9)
    src = np.where(ids < 100, ids, ids % 9)
    big = _batch(monkeypatch, solver, script, ids, QI[src], QG[src], CI[src], CG[src], K)
    for s in range(9):
        for res, i in ((nine, s), (big, rows[s])):
            assert np.array_equal(res[0][i], singles[s][0][0]) and np.array_equal(res[1][i], singles[s][1][0])
            for k in ("iterations", "retries", "edges", "vertices", "overflows"):
                assert res[2][k][i] == singles[s][2][k][0]


# ------------------------------------------------------------------------------------------------ 4. unscripted plans
@pytest.mark.parametrize("sd", [0.1, 0.2])
def test_unscripted_plans_are_valid(solver, table, table_c, scene_c, c_oracle, sd):
    import gik_b200
    from gik_b200 import experiments
    Q, K, tol, step = 256, 8, 0.5, 0.025
    g = torch.Generator(device="cuda:0").manual_seed(int(sd * 100))
    q, pl = experiments.random_endpoints(solver, (np.eye(3), A_REF), (np.eye(3), B_REF), (sd, sd, sd), 2 * Q, generator=g)
    qi, qg, ci, cg = q[:Q], q[Q:], pl[:Q], pl[Q:]
    qp, cp, off, st = gik_b200.computepath_batch(qi, qg, ci, cg, robot=solver, generator=g, expand=K)
    qp, cp, off = qp.cpu().numpy(), cp.cpu().numpy(), off.cpu().numpy()
    qi, qg = qi.cpu().numpy(), qg.cpu().numpy()
    st = {k: v.cpu().numpy() for k, v in st.items()}
    ok = off[1:] > off[:-1]
    print(f"sigma {sd}: success {ok.mean():.3f}, iterations mean {st['iterations'].mean():.2f} max {st['iterations'].max()}")
    if sd == 0.1:
        assert ok.mean() >= 0.95
    assert (st["iterations"] <= (st["retries"] + 1) * -(-250 // K)).all() and (st["overflows"] == 0).all()
    assert (st["retries"][~ok] == 10).all()
    # every path, checked all at once with the oracle
    assert (np.abs(cp[:, [0, 4, 8]] - 1).max() == 0) and np.abs(cp[:, [1, 2, 3, 5, 6, 7]]).max() == 0
    assert (qp >= table.lower - 1e-9).all() and (qp <= table.upper + 1e-9).all()
    R, p = c_oracle.fk(table_c, qp)
    assert np.abs(np.linalg.norm(p[:, 0] - p[:, 1], axis=1) - 0.1).max() < 3e-3
    assert (c_oracle.scene_distance(table_c, scene_c, qp, None, mode=1, cull=0.3) > 0).all()
    _, conv, it, _ = c_oracle.solve(table_c, qp, cp, max_iters=1)
    assert conv.all() and (it == 0).all()                                # converged for its own stored placement
    assert (c_oracle.scene_distance(table_c, scene_c, None, cp, mode=2) > 0).all()
    for i in np.flatnonzero(ok):
        Qp, Cp = qp[off[i]:off[i + 1]], cp[off[i]:off[i + 1]]
        assert np.array_equal(Qp[0], qi[i]) and np.array_equal(Qp[-1], qg[i])
        assert np.array_equal(Cp[0, 9:], ci[i].cpu().numpy()) and np.array_equal(Cp[-1, 9:], cg[i].cpu().numpy())
        move = np.linalg.norm(np.diff(Cp[:, 9:], axis=0), axis=1)
        big = np.flatnonzero(move > step + 1e-9)
        assert len(big) <= 1
        gaps = np.linalg.norm(np.diff(Qp, axis=0), axis=1)
        assert (gaps[big] < tol).all() and gaps.min() < tol


# ------------------------------------------------------------------------------------------------ 5. experiment
def test_trials_experiment_batch(solver):
    from gik_b200 import experiments
    a, b = (np.eye(3), A_REF), (np.eye(3), B_REF)
    seq = experiments.rrt_connect_trials(solver, a, b, std_devs=[(0.1, 0.1, 0.1)], trials=6,
                                         generator=torch.Generator(device="cuda:0").manual_seed(4), rng=np.random.default_rng(4))
    bat = experiments.rrt_connect_trials_batch(solver, a, b, std_devs=[(0.1, 0.1, 0.1)], trials=32,
                                               generator=torch.Generator(device="cuda:0").manual_seed(4))
    assert set(bat[0]) == set(seq[0]) and bat[0]["std_dev"] == (0.1, 0.1, 0.1)
    assert bat[0]["success_rate"] >= min(seq[0]["success_rate"], 95.0) and bat[0]["min_iterations"] >= 1
