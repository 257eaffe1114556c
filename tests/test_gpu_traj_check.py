"""The trajectory check (gik_traj_check_*, csrc/gik_traj.cuh) on the GPU against an oracle built here for every sample:
numpy Bernstein evaluation in fp64, the C oracle's FK, the numpy log6 and the C oracle's pair distances on the scene
without the cube-hand pairs (mode 0) plus the cube's own pairs (mode 2), with the cube at the left hand's placement."""
import ctypes

import numpy as np
import pytest
import torch

from traj_oracle import oracle_flags, oracle_samples, reduce_flags

pytestmark = pytest.mark.gpu

A = (np.eye(3), np.array([0.33, -0.3, 0.93]))                     # config.py:36-37
B = (np.eye(3), np.array([0.4, 0.11, 0.93]))
GRASP_TOL, LIMIT_TOL = 1e-2, 1e-6
M = 201                 # samples per trajectory in the oracle comparisons (the oracle is the slow side)


@pytest.fixture(scope="module")
def solver(table):
    import gik_b200
    s = gik_b200.GraspIK(table, "cuda:0").attach_scene()
    yield s
    s.close()


@pytest.fixture(scope="module")
def batch(solver, table):
    """ctrl [N, 21, 15] fp64 numpy: constant trajectories at converged grasp poses, planner paths fitted by
    maketraj_paths, control points perturbed around grasp poses, a sweep into the robot's zero configuration (which
    collides), and one control point pushed past a joint limit."""
    import gik_b200
    from gik_b200 import experiments
    rng = np.random.default_rng(11)
    g = torch.Generator(device="cuda:0").manual_seed(11)
    P = np.zeros((32, 12)); P[:, [0, 4, 8]] = 1
    P[:, 9:] = rng.uniform([0.25, -0.3, 0.95], [0.5, 0.3, 1.2], (32, 3))
    q, ok = solver.solve(torch.zeros(15), torch.from_numpy(P), dtype=torch.float64)
    grasp = q.cpu().numpy()[ok.cpu().numpy().astype(bool)][:10]
    assert len(grasp) >= 6
    rows = [np.repeat(qg[None], 21, axis=0) for qg in grasp]                               # constant
    qe, pl = experiments.random_endpoints(solver, A, B, (0.1, 0.1, 0.1), 12, generator=g)
    qp, _, off, _ = gik_b200.computepath_batch(qe[:6], qe[6:], pl[:6], pl[6:], robot=solver, generator=g)
    ctrl, _ = gik_b200.maketraj_paths(qe[:6], qe[6:], qp, off, solver=solver)
    fitted = ctrl.cpu().numpy()[(off[1:] > off[:-1]).cpu().numpy()]
    assert len(fitted) >= 3
    rows += list(fitted)
    for k in range(8):                                                                      # perturbed
        c = np.repeat(grasp[k % len(grasp)][None], 21, axis=0)
        c[3:-3] += rng.normal(0, 0.02 * (1 + k), (15, 15))
        rows.append(c)
    rows.append(np.linspace(grasp[0], np.zeros(15), 21))                                    # into q = 0
    # past a limit: every free control point of one joint 0.5 rad above its upper limit, so that the middle of the curve
    # (where the pinned end points weigh 4e-4 in all) is outside by about 0.5 rad whatever the grasp pose
    c = np.repeat(grasp[1][None], 21, axis=0); c[3:-3, 5] = table.upper[5] + 0.5; rows.append(c)
    return np.stack(rows)


def _run(solver, ctrl, dtype, per_sample=True, n_samples=M):
    from gik_b200 import check_trajectories_batch
    r = check_trajectories_batch(torch.as_tensor(ctrl, dtype=dtype, device="cuda:0"), n_samples=n_samples,
                                 grasp_tol=GRASP_TOL, limit_tol=LIMIT_TOL, per_sample=per_sample, solver=solver)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in r.items()}


@pytest.mark.parametrize("dtype,band_d,band_g,band_q,tol_g", [(torch.float64, 1e-6, 1e-9, 1e-12, 1e-9),
                                                              (torch.float32, 1e-4, 1e-4, 1e-5, 1e-4)])
def test_per_sample_flags_match_the_oracle(solver, table, c_oracle, batch, dtype, band_d, band_g, band_q, tol_g):
    import gik_b200
    ctrl = batch.astype(np.float32).astype(np.float64) if dtype == torch.float32 else batch
    o = oracle_samples(c_oracle, table, gik_b200.nextage_scene(), ctrl, M, LIMIT_TOL)
    ref = oracle_flags(o, GRASP_TOL)
    r = _run(solver, ctrl, dtype)
    got = r["sample_flags"]
    sure_c = (o["dist"] == 0) | (o["dist"] > band_d)
    sure_g = np.abs(o["g"] - GRASP_TOL) > band_g
    sure_q = np.abs(o["margin"]) > band_q
    for bit, sure in ((1, sure_q), (2, sure_g), (4, sure_c)):
        assert sure.mean() > 0.7
        assert ((got & bit) == (ref & bit))[sure].all(), (bit, np.argwhere(((got & bit) != (ref & bit)) & sure)[:5])
        assert (ref & bit).any() and (got & bit).any(), bit                  # every reason occurs in the batch
    assert np.abs(r["grasp_err"] - o["g"].max(axis=1)).max() < tol_g
    # constant trajectories at converged grasp poses: valid unless the oracle finds a collision there.  (In fp32 the
    # Bernstein sum of a joint that sits on its limit is off by ~1e-6 relative, about limit_tol: only the grasp bit.)
    for i in range(6):
        assert ((got[i] & 2) == 0).all()
        if dtype == torch.float64 and sure_c[i].all():
            assert ((got[i] & 1) == 0).all() and r["valid"][i] == (not (ref[i] & 4).any())
    # the reductions are those of the per-sample flags
    v, fb, rs = reduce_flags(got)
    assert (r["valid"] == v).all() and (r["first_bad"] == fb).all() and (r["reason"] == rs).all()


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_outputs_do_not_depend_on_the_batch_or_the_run(solver, batch, dtype):
    keys = ("valid", "first_bad", "reason", "grasp_err")
    full = _run(solver, batch, dtype, n_samples=1501)
    v, fb, rs = reduce_flags(full["sample_flags"])
    assert (full["valid"] == v).all() and (full["first_bad"] == fb).all() and (full["reason"] == rs).all()
    lean = _run(solver, batch, dtype, per_sample=False, n_samples=1501)
    again = _run(solver, batch, dtype, per_sample=False, n_samples=1501)
    for k in keys:
        assert np.array_equal(full[k], lean[k]) and np.array_equal(lean[k], again[k]), k
    N = len(batch)
    big = batch[np.arange(1024) % N]
    r_big = _run(solver, big, dtype, per_sample=False, n_samples=1501)
    for i in range(N):
        alone = _run(solver, batch[i:i + 1], dtype, per_sample=False, n_samples=1501)
        nine = _run(solver, np.concatenate([batch[(i + 1 + np.arange(4)) % N], batch[i:i + 1],
                                            batch[(i + 5 + np.arange(4)) % N]]), dtype, per_sample=False, n_samples=1501)
        for k in keys:
            assert alone[k][0] == full[k][i] == nine[k][4] == r_big[k][i] == r_big[k][i + N], (i, k)


def test_check_trajectory_equals_the_batch_row(solver, batch):
    from gik_b200 import check_trajectory
    from gik_b200.trajectory import maketraj
    rng = np.random.default_rng(12)
    path = batch[0, 0] + np.cumsum(rng.normal(0, 0.01, (40, 15)), axis=0)
    (curve, _, _), _ = maketraj(path[0], path[-1], path, 15.0)
    one = check_trajectory(curve, per_sample=True, solver=solver)
    ctrl = np.concatenate([batch[:3], np.array(curve.control_points_)[None], batch[3:5]])
    r = _run(solver, ctrl, torch.float64, n_samples=1501)
    assert one["valid"] == bool(r["valid"][3]) and one["first_bad"] == r["first_bad"][3]
    assert one["reason"] == r["reason"][3] and one["grasp_err"] == r["grasp_err"][3]
    assert np.array_equal(one["sample_flags"].cpu().numpy(), r["sample_flags"][3])


def test_error_codes_and_guard_columns(solver, table, batch):
    import gik_b200
    from gik_b200 import _cabi
    from gik_b200.trajectory import sample_weights
    lib = _cabi.lib()
    dev = "cuda:0"
    N, Ms = 5, 33
    for dtype, sfx in ((torch.float64, "f64"), (torch.float32, "f32")):
        f = getattr(lib, f"gik_traj_check_{sfx}")
        W = torch.as_tensor(sample_weights(21, Ms), dtype=dtype, device=dev)
        C = torch.as_tensor(batch[-N:], dtype=dtype, device=dev).contiguous()
        valid = torch.full((N + 2,), 0xAB, dtype=torch.uint8, device=dev)
        first = torch.full((N + 2,), 12345, dtype=torch.int32, device=dev)
        reason = torch.full((N + 2,), 0xCD, dtype=torch.uint8, device=dev)
        gerr = torch.full((N + 2,), 7.5, dtype=dtype, device=dev)
        flags = torch.full(((N + 2) * Ms,), 0xEE, dtype=torch.uint8, device=dev)
        outs = (valid, first, reason, gerr)
        keep = [t.clone() for t in outs] + [flags.clone()]
        ptr = lambda t, off=1: ctypes.c_void_p(t.data_ptr() + off * t.element_size())

        def call(h=solver._h, n=N, nc=21, m=Ms, lt=LIMIT_TOL, gt=GRASP_TOL, w=ptr(W, 0), c=ptr(C, 0), fl=None):
            rc = f(h, n, nc, m, w, c, lt, gt, *[ptr(t) for t in outs], fl if fl is not None else ptr(flags, Ms), None)
            torch.cuda.synchronize()
            return rc

        assert call(n=-1) == -2 and call(nc=1) == -2 and call(m=1) == -2 and call(m=-4) == -2
        assert call(lt=-1e-3) == -5 and call(gt=-1e-3) == -5
        assert call(w=None) == -1 and call(c=None) == -1
        assert call(h=None) == -6
        assert call(n=0) == 0
        bare = gik_b200.GraspIK(table, dev)                   # no scene attached
        assert call(h=bare._h) == -7
        bare.close()
        for t, k in zip(outs + (flags,), keep):
            assert torch.equal(t, k)                          # refused calls write nothing
        assert call() == 0
        for t, k in zip(outs, keep):
            assert torch.equal(t[0], k[0]) and torch.equal(t[-1], k[-1]) and not torch.equal(t[1:-1], k[1:-1])
        assert (flags[:Ms] == 0xEE).all() and (flags[(N + 1) * Ms:] == 0xEE).all()
        ref = solver.check_trajectories(C, W, limit_tol=LIMIT_TOL, grasp_tol=GRASP_TOL, per_sample=True)
        for t, x in zip(outs, ref[:4]):
            assert torch.equal(t[1:-1], x)
        assert torch.equal(flags[Ms:(N + 1) * Ms].reshape(N, Ms), ref[4])
