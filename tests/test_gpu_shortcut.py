"""Path shortcutting (planner.shortcut_paths_batch, csrc/gik_shortcut.cuh) on the GPU: kernel parity with the numpy
restatement of tests/test_shortcut_cpu.py on real edge-launch outputs, the invariants of shortcut unscripted plans
checked with the oracle, no cross-talk between paths, determinism and the rounds = 0 pass-through."""
import numpy as np
import pytest
import torch

from test_shortcut_cpu import _path_length, _reference

pytestmark = pytest.mark.gpu

A_REF = np.array([0.33, -0.3, 0.93]); B_REF = np.array([0.4, 0.11, 0.93])     # config.py:36-37
DTYPES = [torch.float32, torch.float64]


@pytest.fixture(scope="module")
def solver(table):
    import gik_b200
    s = gik_b200.GraspIK(table, "cuda:0").attach_scene()
    yield s
    s.close()


_PLANS = {}


def _plans(solver, sd, Q=256):
    """computepath_batch's paths for Q random endpoint pairs at spread sd (fp64, planned once per module)."""
    if (sd, Q) not in _PLANS:
        import gik_b200
        from gik_b200 import experiments
        g = torch.Generator(device="cuda:0").manual_seed(int(sd * 100) + 7)
        q, pl = experiments.random_endpoints(solver, (np.eye(3), A_REF), (np.eye(3), B_REF), (sd, sd, sd), 2 * Q, generator=g)
        qp, cp, off, _ = gik_b200.computepath_batch(q[:Q], q[Q:], pl[:Q], pl[Q:], robot=solver, generator=g)
        _PLANS[(sd, Q)] = (qp, cp, off)
    return _PLANS[(sd, Q)]


def _split(q, cube, off):
    q, cube, off = q.cpu().numpy(), cube.cpu().numpy(), off.cpu().numpy()
    return [(q[off[p]:off[p + 1]], cube[off[p]:off[p + 1]]) for p in range(len(off) - 1)]


# ------------------------------------------------------------------------------------------------ 1. kernel parity
@pytest.mark.parametrize("dtype", DTYPES)
def test_kernel_matches_the_restatement_on_real_edges(solver, dtype, monkeypatch):
    import gik_b200
    qp, cp, off = _plans(solver, 0.1)
    calls = []
    real = solver.path_shortcut

    def spy(q, cube, offsets, pi, pj, ns, nv, q_path, *, join_tol):
        out = real(q, cube, offsets, pi, pj, ns, nv, q_path, join_tol=join_tol)
        calls.append(([t.cpu().numpy() for t in (q, cube, offsets, pi, pj, ns, nv, q_path)], join_tol,
                      [t.cpu().numpy() for t in out]))
        return out

    monkeypatch.setattr(solver, "path_shortcut", spy)
    for tol in (0.5, 0.05):
        g = torch.Generator(device="cuda:0").manual_seed(1)
        gik_b200.shortcut_paths_batch(qp.to(dtype), cp.to(dtype), off, robot=solver, rounds=3, generator=g, join_tol=tol)
    monkeypatch.undo()
    assert len(calls) == 6
    accepted = 0
    for (q, cube, o, pi, pj, ns, nv, q_path), tol, (q2, c2, o2, ch, ln) in calls:
        paths = [(q[o[p]:o[p + 1]], cube[o[p]:o[p + 1]]) for p in range(len(o) - 1)]
        rch, rln, rout = _reference(paths, pi, pj, ns, nv, q_path, tol, q_path.shape[0])
        assert np.array_equal(ch, rch) and np.array_equal(ln, rln)
        for p, (rq, rc) in enumerate(rout):
            # identity rotations: the host interpolation equals the kernel's placements bit for bit
            assert np.array_equal(q2[o2[p]:o2[p + 1]], rq) and np.array_equal(c2[o2[p]:o2[p + 1]], rc)
        accepted += (ch >= 0).sum()
        # the real edges cover the cases: cut or failed edges, joins outside the tolerance, accepted ones
        assert (nv < ns).any() and (ns >= 1).any()
    assert accepted > 0


# ------------------------------------------------------------------------------------------------ 2. unscripted plans
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("sd", [0.1, 0.2])
def test_unscripted_shortcuts_keep_the_invariants(solver, table, table_c, scene_c, c_oracle, sd, dtype):
    import gik_b200
    step = 0.025
    qp, cp, off = _plans(solver, sd)
    qp, cp = qp.to(dtype), cp.to(dtype)
    g = torch.Generator(device="cuda:0").manual_seed(3)
    qs, cs, offs, st = gik_b200.shortcut_paths_batch(qp, cp, off, robot=solver, generator=g)
    _, _, _, st0 = gik_b200.shortcut_paths_batch(qp, cp, off, robot=solver, rounds=0)
    before, after = _split(qp, cp, off), _split(qs, cs, offs)
    sc, ln, ln0 = st["shortcuts"].cpu().numpy(), st["length"].cpu().numpy(), st0["length"].cpu().numpy()
    n0 = np.array([len(q) for q, _ in before]); n1 = np.array([len(q) for q, _ in after])
    print(f"sigma {sd} {dtype}: shortcuts mean {sc.mean():.2f}, vertices {n0.sum()} -> {n1.sum()}, "
          f"length {ln0.sum():.2f} -> {ln.sum():.2f}")
    # every splice has gain > 0 on its own partial sums; the total, summed again left to right over the new rows, can
    # come out a few ulps above the old total when a gain is within rounding of zero
    print(f"largest relative length change {((ln - ln0) / np.maximum(ln0, 1e-300)).max():.3e}")
    assert sc.sum() > 0 and (ln <= ln0 * (1 + 1e-12)).all() and ln.sum() < ln0.sum()
    assert ((n0 == 0) == (n1 == 0)).all() and (n1[n0 < 3] == n0[n0 < 3]).all() and (sc[n0 < 3] == 0).all()
    for (q, c), (q1, c1), L in zip(before, after, ln):
        if not len(q):
            continue
        assert np.array_equal(q1[0], q[0]) and np.array_equal(q1[-1], q[-1])
        assert np.array_equal(c1[0], c[0]) and np.array_equal(c1[-1], c[-1])
        assert L == _path_length(q1)
        big0 = np.linalg.norm(np.diff(c[:, 9:].astype(float), axis=0), axis=1) > step + 1e-6
        big1 = np.linalg.norm(np.diff(c1[:, 9:].astype(float), axis=0), axis=1) > step + 1e-6
        assert big1.sum() <= big0.sum()
    # every row, checked all at once with the oracle (in fp64, as test_gpu_planner checks the planner's rows)
    Q64, C64 = qs.double().cpu().numpy(), cs.double().cpu().numpy()
    assert (np.abs(C64[:, [0, 4, 8]] - 1).max() == 0) and np.abs(C64[:, [1, 2, 3, 5, 6, 7]]).max() == 0
    assert (Q64 >= table.lower - 1e-6).all() and (Q64 <= table.upper + 1e-6).all()
    assert (c_oracle.scene_distance(table_c, scene_c, Q64, None, mode=1, cull=0.3) > 0).all()
    # a grasp for its own stored placement; fp32 rows passed the fp32 kernel's residual test, which the fp64 oracle
    # can see up to fp32 rounding above eps
    eps = 1e-3 if dtype == torch.float64 else 1.01e-3
    _, conv, it, _ = c_oracle.solve(table_c, Q64, C64, max_iters=1)
    print(f"rows at the oracle's eps: {conv.mean():.5f} converged")
    _, conv, it, _ = c_oracle.solve(table_c, Q64, C64, eps=eps, max_iters=1)
    assert conv.all() and (it == 0).all()
    assert (c_oracle.scene_distance(table_c, scene_c, None, C64, mode=2) > 0).all()


# ------------------------------------------------------------------------------------------------ 3. no cross-talk
def _script(monkeypatch):
    """_draw_pairs as a function of (path length, round, k) only: a path's draws do not depend on its neighbours."""
    from gik_b200 import planner
    state = {"round": 0}

    def draw(n, K, generator):
        r = state["round"]
        state["round"] += 1
        h = (n[:, None] * 2654435761 + r * 40503 + torch.arange(K, device=n.device)[None, :] * 97) % 1000003
        m = (n - 1).clamp_min(2)[:, None]
        x = h % m
        y = (h // 7) % (m - 1)
        y = y + (y >= x).long()
        i, j = torch.minimum(x, y), torch.maximum(x, y) + 1
        ok = (n >= 3)[:, None]
        return torch.where(ok, i, -1).to(torch.int32), torch.where(ok, j, -1).to(torch.int32)

    monkeypatch.setattr(planner, "_draw_pairs", draw)
    return state


@pytest.mark.parametrize("dtype", DTYPES)
def test_no_cross_talk_between_paths(solver, dtype, monkeypatch):
    import gik_b200
    qp, cp, off = _plans(solver, 0.1)
    paths = [(q, c) for q, c in _split(qp, cp, off) if len(q) >= 3][:9]
    assert len(paths) == 9

    def run(sel):
        rows = [paths[s] if s >= 0 else (np.zeros((0, 15)), np.zeros((0, 12))) for s in sel]
        o = np.zeros(len(rows) + 1, np.int64); o[1:] = np.cumsum([len(q) for q, _ in rows])
        q = torch.from_numpy(np.vstack([r[0] for r in rows])).to("cuda:0", dtype)
        c = torch.from_numpy(np.vstack([r[1] for r in rows])).to("cuda:0", dtype)
        state = _script(monkeypatch)
        out = gik_b200.shortcut_paths_batch(q, c, torch.from_numpy(o), robot=solver, rounds=4)
        monkeypatch.undo()
        assert state["round"] == 4
        return _split(*out[:3]), {k: v.cpu().numpy() for k, v in out[3].items()}

    singles = [run([s]) for s in range(9)]
    nine = run(list(range(9)))
    order = np.random.default_rng(3).permutation(256)
    sel = np.arange(256) % 9
    sel[order[:40]] = -1                                                 # empty paths among them
    rows = order[40:49]
    sel[rows] = np.arange(9)
    big = run(sel)
    assert sum(singles[s][1]["shortcuts"][0] for s in range(9)) > 0
    for s in range(9):
        for res, i in ((nine, s), (big, rows[s])):
            assert np.array_equal(res[0][i][0], singles[s][0][0][0]) and np.array_equal(res[0][i][1], singles[s][0][0][1])
            for k in ("shortcuts", "length"):
                assert res[1][k][i] == singles[s][1][k][0]
    assert all(len(big[0][i][0]) == 0 for i in order[:40])


# ------------------------------------------------------------------------------------------------ 4. determinism, rounds = 0
@pytest.mark.parametrize("dtype", DTYPES)
def test_same_seed_same_output_and_rounds_zero_passes_through(solver, dtype):
    import gik_b200
    qp, cp, off = _plans(solver, 0.2)
    qp, cp = qp.to(dtype), cp.to(dtype)
    outs = []
    for _ in range(2):
        g = torch.Generator(device="cuda:0").manual_seed(11)
        outs.append(gik_b200.shortcut_paths_batch(qp, cp, off, robot=solver, rounds=4, generator=g))
    (a, b) = outs
    assert all(torch.equal(x, y) for x, y in zip(a[:3], b[:3]))
    assert all(torch.equal(a[3][k], b[3][k]) for k in a[3])
    q0, c0, o0, st0 = gik_b200.shortcut_paths_batch(qp, cp, off, robot=solver, rounds=0)
    assert torch.equal(q0, qp) and torch.equal(c0, cp) and torch.equal(o0.cpu(), off.cpu())
    assert (st0["shortcuts"] == 0).all()
    assert np.array_equal(st0["length"].cpu().numpy(), [_path_length(q) for q, _ in _split(qp, cp, off)])
