"""Grasp roadmap (roadmap.build_roadmap / query_roadmap_batch, csrc/gik_roadmap.cuh) on the GPU, fp32 and fp64: vertices
and edge steps checked with the C oracle, kNN against numpy, edge weights against the numpy restatement bit for bit,
query lengths against scipy's Dijkstra exactly, path invariants, determinism and batch independence, edge cases and
the downstream fit and check."""
import io

import numpy as np
import pytest
import torch

from test_roadmap_cpu import knn_reference, scipy_reference, weight_reference
from test_shortcut_cpu import _path_length

pytestmark = pytest.mark.gpu

A_REF = np.array([0.33, -0.3, 0.93]); B_REF = np.array([0.4, 0.11, 0.93])     # config.py:36-37
A, B = (np.eye(3), A_REF), (np.eye(3), B_REF)
DTYPES = [torch.float32, torch.float64]
N, K, STEP = 1024, 8, 0.025


@pytest.fixture(scope="module")
def solver(table):
    import gik_b200
    s = gik_b200.GraspIK(table, "cuda:0").attach_scene()
    yield s
    s.close()


_RM = {}


def _roadmap(solver, dtype):
    """A roadmap per dtype, built once per module with the calls to roadmap_edges recorded."""
    if dtype not in _RM:
        import gik_b200
        calls = []
        real = solver.roadmap_edges

        def spy(q_from, q_to, ns, nv, q_path, *, join_tol):
            w = real(q_from, q_to, ns, nv, q_path, join_tol=join_tol)
            calls.append([t.cpu().numpy() for t in (q_from, q_to, ns, nv, q_path, w)] + [join_tol])
            return w

        solver.roadmap_edges = spy
        try:
            rm = gik_b200.build_roadmap(A, B, N, k=K, dtype=dtype, robot=solver,
                                        generator=torch.Generator(device="cuda:0").manual_seed(5))
        finally:
            del solver.roadmap_edges
        _RM[dtype] = (rm, calls[0])
    return _RM[dtype]


def _endpoints(solver, dtype, Q=64, sd=0.1, seed=3):
    from gik_b200 import experiments
    g = torch.Generator(device="cuda:0").manual_seed(seed)
    q, pl = experiments.random_endpoints(solver, A, B, (sd, sd, sd), 2 * Q, generator=g)
    return q[:Q].to(dtype), q[Q:].to(dtype), pl[:Q].to(dtype), pl[Q:].to(dtype)


def _oracle_rows(table, table_c, scene_c, c_oracle, Qr, Cr, dtype, clearance=False):
    Qr, Cr = np.asarray(Qr, np.float64), np.asarray(Cr, np.float64)
    assert (Qr >= table.lower - 1e-9).all() and (Qr <= table.upper + 1e-9).all()
    assert (c_oracle.scene_distance(table_c, scene_c, Qr, None, mode=1, cull=0.3) > 0).all()
    assert (c_oracle.scene_distance(table_c, scene_c, None, Cr, mode=2) > 0).all()
    # a grasp for its own placement; fp32 rows passed the fp32 kernel's residual test, which the fp64 oracle can see up
    # to fp32 rounding above eps
    eps = 1e-3 if dtype == torch.float64 else 1.01e-3
    _, conv, it, _ = c_oracle.solve(table_c, Qr, Cr, eps=eps, max_iters=1)
    assert conv.all() and (it == 0).all()
    if clearance:
        d = c_oracle.scene_distance(table_c, scene_c, Qr, Cr, mode=1)
        assert (d >= 0.04 - (1e-9 if dtype == torch.float64 else 1e-5)).all()


# ------------------------------------------------------------------------------------------------ 1-3. the build
@pytest.mark.parametrize("dtype", DTYPES)
def test_vertices_knn_and_edges(solver, table, table_c, scene_c, c_oracle, dtype):
    from gik_b200.path import se3_interpolate
    rm, (qf, qt, ns_all, nv_all, q_path, w_all, tol) = _roadmap(solver, dtype)
    q, cube = rm.q.cpu().numpy(), rm.cube.cpu().numpy()
    assert q.shape == (N, 15) and cube.shape == (N, 12) and rm.drawn >= N
    print(f"{dtype}: {rm.drawn} drawn for {N} vertices, {rm.dst.numel()} of {N * K} edges accepted, "
          f"{rm.steps.shape[0]} step rows")
    # 1. vertices
    lo, hi = np.array(rm.box[0]), np.array(rm.box[1])
    assert (cube[:, 9:] >= lo - 1e-6).all() and (cube[:, 9:] <= hi + 1e-6).all()
    assert np.array_equal(cube[:, :9], np.tile(np.eye(3).reshape(9), (N, 1)).astype(cube.dtype))
    _oracle_rows(table, table_c, scene_c, c_oracle, q, cube, dtype, clearance=True)
    # 2. kNN
    nbr = solver.knn(rm.cube, K).cpu().numpy()
    assert np.array_equal(nbr, knn_reference(cube, K))
    # 3. edges: the recorded judgement equals the restatement, the roadmap keeps exactly the accepted edges
    ref = weight_reference(qf, qt, ns_all, nv_all, q_path, tol, q_path.shape[0])
    assert np.array_equal(w_all, ref)
    keep = np.isfinite(ref)
    row_ptr, dst, ns = rm.row_ptr.cpu().numpy(), rm.dst.cpu().numpy(), rm.ns.cpu().numpy()
    src = np.repeat(np.arange(N), np.diff(row_ptr))
    assert np.array_equal(dst, nbr.reshape(-1)[keep]) and np.array_equal(src, np.repeat(np.arange(N), K)[keep])
    assert np.array_equal(rm.weight.cpu().numpy(), ref[keep]) and np.array_equal(ns, ns_all[keep])
    assert 0 < keep.sum() < N * K
    steps, sp = rm.steps.cpu().numpy(), rm.step_ptr.cpu().numpy()
    assert np.array_equal(np.diff(sp), ns - 1)
    rows_c = []
    for e in range(len(dst)):
        i, j, m = src[e], dst[e], ns[e]
        rows = [q[i]] + list(steps[sp[e]:sp[e + 1]]) + [q[j]]
        assert _path_length(rows) == rm.weight[e].item()                 # the weight of the stored rows
        if m > 1:
            a = torch.from_numpy(np.tile(cube[i], (m - 1, 1))); b = torch.from_numpy(np.tile(cube[j], (m - 1, 1)))
            rows_c.append(se3_interpolate(a, b, torch.arange(1, m, dtype=a.dtype) / m).numpy())
    if rows_c:
        _oracle_rows(table, table_c, scene_c, c_oracle, steps, np.vstack(rows_c), dtype)


# ------------------------------------------------------------------------------------------------ 4-5. queries
def _query(solver, rm, *args, **kw):
    """query_roadmap_batch with the sssp inputs recorded."""
    import gik_b200
    rec = {}
    real = solver.roadmap_sssp

    def spy(row_ptr, dst, weight, att_vertex, att_weight):
        out = real(row_ptr, dst, weight, att_vertex, att_weight)
        rec["att"] = (att_vertex.cpu().numpy(), att_weight.cpu().numpy())
        return out

    solver.roadmap_sssp = spy
    try:
        out = gik_b200.query_roadmap_batch(rm, *args, robot=solver, **kw)
    finally:
        del solver.roadmap_sssp
    return out, rec


def _split(q, cube, off):
    q, cube, off = q.cpu().numpy(), cube.cpu().numpy(), off.cpu().numpy()
    return [(q[off[p]:off[p + 1]], cube[off[p]:off[p + 1]]) for p in range(len(off) - 1)]


@pytest.mark.parametrize("dtype", DTYPES)
def test_query_lengths_and_paths(solver, table, table_c, scene_c, c_oracle, dtype):
    rm, _ = _roadmap(solver, dtype)
    qi, qg, ci, cg = _endpoints(solver, dtype)
    (q, cube, off, st), rec = _query(solver, rm, qi, qg, ci, cg)
    st = {k: v.cpu().numpy() for k, v in st.items()}
    av, aw = rec["att"]
    row_ptr, dst, w = rm.row_ptr.cpu().numpy(), rm.dst.cpu().numpy(), rm.weight.cpu().numpy()
    paths = _split(q, cube, off)
    ok = st["connected"].astype(bool)
    print(f"{dtype}: {ok.sum()} of {len(ok)} connected, vertices mean {st['vertices'][ok].mean():.1f}, "
          f"attachments {st['attach_start'].mean():.1f} / {st['attach_goal'].mean():.1f}")
    assert ok.mean() >= 0.5
    for p in range(len(ok)):
        _, _, rgp, rln = scipy_reference(N, row_ptr, dst, w, av[p], aw[p], preds=False)
        assert st["length"][p] == rln or (np.isinf(rln) and np.isinf(st["length"][p]))   # exactly
        assert st["attach_start"][p] == np.isfinite(aw[p][:K]).sum() and st["attach_goal"][p] == np.isfinite(aw[p][K:2 * K]).sum()
        Qp, Cp = paths[p]
        assert (len(Qp) > 0) == ok[p]
        if not ok[p]:
            continue
        # the path's own length, summed left to right over its rows: the same up to the association of the sums
        assert abs(_path_length(Qp) - st["length"][p]) <= 1e-12 * st["length"][p]
        assert np.array_equal(Qp[0], qi[p].cpu().numpy()) and np.array_equal(Qp[-1], qg[p].cpu().numpy())
        assert np.array_equal(Cp[0], np.concatenate([np.eye(3).reshape(9), ci[p].cpu().numpy()]).astype(Cp.dtype))
        assert np.array_equal(Cp[-1], np.concatenate([np.eye(3).reshape(9), cg[p].cpu().numpy()]).astype(Cp.dtype))
        move = np.linalg.norm(np.diff(Cp[:, 9:].astype(np.float64), axis=0), axis=1)
        assert (move <= STEP + 1e-9).all()                               # no connection jump
    allq, allc = q.cpu().numpy(), cube.cpu().numpy()
    _oracle_rows(table, table_c, scene_c, c_oracle, allq, allc, dtype)


# ------------------------------------------------------------------------------------------------ 6. determinism
@pytest.mark.parametrize("dtype", DTYPES)
def test_same_seed_alone_or_in_a_batch_and_between_runs(solver, dtype):
    import gik_b200
    rm, _ = _roadmap(solver, dtype)
    again = gik_b200.build_roadmap(A, B, N, k=K, dtype=dtype, robot=solver,
                                   generator=torch.Generator(device="cuda:0").manual_seed(5))
    for f in vars(rm):
        a, b = getattr(rm, f), getattr(again, f)
        assert torch.equal(a, b) if torch.is_tensor(a) else a == b, f
    qi, qg, ci, cg = _endpoints(solver, dtype, seed=9)
    batch = gik_b200.query_roadmap_batch(rm, qi, qg, ci, cg, robot=solver)
    twice = gik_b200.query_roadmap_batch(rm, qi, qg, ci, cg, robot=solver)
    assert all(torch.equal(x, y) for x, y in zip(batch[:3], twice[:3]))
    assert all(torch.equal(batch[3][k], twice[3][k]) for k in batch[3])
    paths = _split(*batch[:3])
    for p in (0, 17, 63):
        one = gik_b200.query_roadmap_batch(rm, qi[p:p + 1], qg[p:p + 1], ci[p:p + 1], cg[p:p + 1], robot=solver)
        (q1, c1), = _split(*one[:3])
        assert np.array_equal(q1, paths[p][0]) and np.array_equal(c1, paths[p][1])
        for k in one[3]:
            assert one[3][k][0].item() == batch[3][k][p].item(), k


# ------------------------------------------------------------------------------------------------ 7. edge cases
@pytest.mark.parametrize("dtype", DTYPES)
def test_edge_cases(solver, dtype):
    import gik_b200
    rm, _ = _roadmap(solver, dtype)
    qi, qg, ci, cg = _endpoints(solver, dtype, Q=4, seed=11)
    q, cube, off, st = gik_b200.query_roadmap_batch(rm, qi[:0], qg[:0], ci[:0], cg[:0], robot=solver)
    assert q.shape == (0, 15) and cube.shape == (0, 12) and off.tolist() == [0] and st["length"].numel() == 0
    for k in (0, 33, -1):
        with pytest.raises(ValueError):
            gik_b200.query_roadmap_batch(rm, qi, qg, ci, cg, k_attach=k, robot=solver)
        with pytest.raises(ValueError):
            gik_b200.build_roadmap(A, B, 64, k=k, dtype=dtype, robot=solver)
    with pytest.raises(ValueError):
        gik_b200.build_roadmap(A, B, 8, k=8, dtype=dtype, robot=solver)        # k > N - 1
    # start == goal: the direct edge of length 0, two rows
    q, cube, off, st = gik_b200.query_roadmap_batch(rm, qi[:1], qi[:1], ci[:1], ci[:1], robot=solver)
    assert off.tolist() == [0, 2] and st["length"][0].item() == 0.0 and st["vertices"][0].item() == 0
    assert torch.equal(q[0], qi[0]) and torch.equal(q[1], qi[0])
    # a goal nobody can reach: an empty path
    far = cg[:1].clone(); far[0, 2] = 2.5
    q, cube, off, st = gik_b200.query_roadmap_batch(rm, qi[:2], qg[:2], ci[:2], torch.cat([far, cg[1:2]]), robot=solver)
    assert st["connected"][0].item() == 0 and off[1].item() == 0 and np.isinf(st["length"][0].item())
    assert st["attach_goal"][0].item() == 0
    # torch.save of the fields round-trips the roadmap
    buf = io.BytesIO()
    torch.save(vars(rm), buf)
    buf.seek(0)
    back = gik_b200.Roadmap(**torch.load(buf, weights_only=False))
    a = gik_b200.query_roadmap_batch(rm, qi, qg, ci, cg, robot=solver)
    b = gik_b200.query_roadmap_batch(back, qi, qg, ci, cg, robot=solver)
    assert all(torch.equal(x, y) for x, y in zip(a[:3], b[:3]))


# ------------------------------------------------------------------------------------------------ 8. downstream
def test_downstream_fit_and_check_accept_the_output(solver):
    import gik_b200
    rm, _ = _roadmap(solver, torch.float64)
    qi, qg, ci, cg = _endpoints(solver, torch.float64, Q=32, seed=13)
    q, cube, off, st = gik_b200.query_roadmap_batch(rm, qi, qg, ci, cg, robot=solver)
    ctrl, cost = gik_b200.maketraj_paths(qi, qg, q, off, solver=solver)
    ok = st["connected"].bool()
    assert torch.isfinite(cost[ok]).all() and torch.isinf(cost[~ok]).all()
    chk = gik_b200.check_trajectories_batch(ctrl[ok], solver=solver)
    print(f"roadmap paths: {int(chk['valid'].sum())} of {int(ok.sum())} fitted trajectories valid")
    assert chk["valid"].shape == (int(ok.sum()),)
    sc = gik_b200.shortcut_paths_batch(q, cube, off, robot=solver, rounds=2)
    assert sc[2].shape == off.shape
