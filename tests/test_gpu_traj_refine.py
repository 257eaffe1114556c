"""Trajectory refinement (gik_traj_refine_*, csrc/gik_traj_refine.cuh) on the GPU: recovery of perturbed trajectories
on the grasp, the invariants of include/gik.h on planner-fitted and perturbed trajectories, pass-through cases,
independence from the batch and the run, one Levenberg-Marquardt step against a numpy restatement built on the C
oracle's FK and Jacobian, and the C entry's error codes."""
import ctypes

import numpy as np
import pytest
import torch

from traj_oracle import cubes_from_hands, sample_weights

pytestmark = pytest.mark.gpu

A = (np.eye(3), np.array([0.33, -0.3, 0.93]))                     # config.py:36-37
B = (np.eye(3), np.array([0.4, 0.11, 0.93]))
DAMPING = 1e-3


@pytest.fixture(scope="module")
def solver(table):
    import gik_b200
    s = gik_b200.GraspIK(table, "cuda:0").attach_scene()
    yield s
    s.close()


def _right_arm(table):
    chain, k = [], int(table.hand_joint[1])
    while k >= 0:
        chain.append(k); k = int(table.parent[k])
    return chain[::-1][1:]


def _residual(c_oracle, table, Q):
    """r = log6(C_L^-1 C_R) [n, 6] and the model Jacobian Ad(hook_R) J_R [n, 6, 6] from the C oracle."""
    from oracle import grasp_ik_np
    tc = table.to_c()
    HR, Hp = c_oracle.fk(tc, Q)
    Jo = c_oracle.jac(tc, Q)
    K = np.asarray(table.hook_R[1]).reshape(3, 3); k = np.asarray(table.hook_p[1])
    kx = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    Ad = np.block([[K, kx @ K], [np.zeros((3, 3)), K]])
    arm = _right_arm(table)
    r = np.empty((len(Q), 6)); J = np.empty((len(Q), 6, 6))
    for s in range(len(Q)):
        CL, CR = cubes_from_hands(table, HR[s], Hp[s])
        r[s] = grasp_ik_np.log6(CL[0].T @ CR[0], CL[0].T @ (CR[1] - CL[1]))
        J[s] = Ad @ Jo[s, 1][:, arm]
    return r, J


@pytest.fixture(scope="module")
def grasp(solver, table, c_oracle):
    """Grasp poses with r = 0: converged IK solutions, the right arm then driven onto the left hand's cube by Newton
    steps (inside the joint limits)."""
    rng = np.random.default_rng(31)
    P = np.zeros((32, 12)); P[:, [0, 4, 8]] = 1
    P[:, 9:] = rng.uniform([0.25, -0.3, 0.95], [0.5, 0.3, 1.2], (32, 3))
    q, ok = solver.solve(torch.zeros(15), torch.from_numpy(P), dtype=torch.float64)
    arm = _right_arm(table)
    out = []
    for qi in q.cpu().numpy()[ok.cpu().numpy().astype(bool)]:
        for _ in range(20):
            r, J = _residual(c_oracle, table, qi[None])
            qi[arm] -= np.linalg.solve(J[0], r[0])
        inside = (qi >= table.lower).all() and (qi <= table.upper).all()
        if np.linalg.norm(_residual(c_oracle, table, qi[None])[0]) < 1e-13 and inside:
            out.append(qi)
    assert len(out) >= 6
    return np.stack(out[:8])


@pytest.fixture(scope="module")
def batch(solver, table, grasp):
    """ctrl [N, 21, 15] fp64: planner paths fitted by maketraj_paths, control points perturbed around grasp poses, a
    sweep into the robot's zero configuration, and one control point pushed past a joint limit (as in
    test_gpu_traj_check.py), plus right-arm control points pushed past the right arm's limits."""
    import gik_b200
    from gik_b200 import experiments
    rng = np.random.default_rng(32)
    g = torch.Generator(device="cuda:0").manual_seed(32)
    qe, pl = experiments.random_endpoints(solver, A, B, (0.1, 0.1, 0.1), 16, generator=g)
    qp, _, off, _ = gik_b200.computepath_batch(qe[:8], qe[8:], pl[:8], pl[8:], robot=solver, generator=g)
    ctrl, _ = gik_b200.maketraj_paths(qe[:8], qe[8:], qp, off, solver=solver)
    rows = list(ctrl.cpu().numpy()[(off[1:] > off[:-1]).cpu().numpy()])
    assert len(rows) >= 4
    for k in range(6):
        c = np.repeat(grasp[k % len(grasp)][None], 21, axis=0)
        c[3:-3] += rng.normal(0, 0.02 * (1 + k), (15, 15))
        rows.append(c)
    rows.append(np.linspace(grasp[0], np.zeros(15), 21))
    c = np.repeat(grasp[1][None], 21, axis=0); c[3:-3, 5] = table.upper[5] + 0.5; rows.append(c)
    arm = _right_arm(table)
    c = np.repeat(grasp[2][None], 21, axis=0); c[5:9, arm[1]] = table.upper[arm[1]] + 0.3
    c[10:12, arm[3]] = table.lower[arm[3]] - 0.2; rows.append(c)
    return np.stack(rows)


def _refine(solver, ctrl, dtype, n_samples=1501, max_iters=8, tol=0.0):
    from gik_b200 import refine_trajectories_batch
    r = refine_trajectories_batch(torch.as_tensor(ctrl, dtype=dtype, device="cuda:0"), n_samples=n_samples,
                                  max_iters=max_iters, tol=tol, solver=solver)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in r.items()}


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint64 if a.dtype == np.float64 else np.uint32)


@pytest.mark.parametrize("dtype,bound", [(torch.float64, 1e-8), (torch.float32, 1e-4)])
@pytest.mark.parametrize("sigma", [0.01, 0.05])
def test_recovers_perturbed_right_arm(solver, table, grasp, dtype, bound, sigma):
    """Constant trajectories on an exact grasp with the right arm's free control points perturbed: the unperturbed
    control points are a zero of F inside the box, and the refinement finds it.  fp32: r is then the rounding of the
    fp32 forward kinematics (single-precision rotations over a chain about a metre long: a few 1e-7 per sample, up to a
    few 1e-6 in the worst samples), not the perturbation; 1e-4 leaves a margin of more than 10 over that floor."""
    rng = np.random.default_rng(int(sigma * 1000))
    arm = _right_arm(table)
    ctrl = np.repeat(grasp[:, None], 21, axis=1)
    for c in ctrl:
        c[3:-3, arm] += rng.normal(0, sigma, (15, 6))
    r = _refine(solver, ctrl, dtype, max_iters=40)
    assert (r["grasp_err"] < bound).all(), r["grasp_err"]
    assert (r["accepted"] >= 1).all() and (r["obj_after"] < r["obj_before"]).all()


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_invariants(solver, table, batch, dtype):
    from gik_b200 import check_trajectories_batch
    arm = _right_arm(table)
    src = batch.astype(np.float32) if dtype == torch.float32 else batch
    r = _refine(solver, src, dtype)
    out = r["ctrl"]
    keep = np.ones(out.shape, bool); keep[:, 3:-3, arm] = False
    assert np.array_equal(_bits(out)[keep], _bits(src)[keep])         # pinned rows and every other column, bit for bit
    assert (r["obj_after"] <= r["obj_before"]).all()
    assert (r["accepted"] >= 1).sum() >= len(batch) - 2
    lo, hi = np.asarray(table.lower)[arm], np.asarray(table.upper)[arm]
    x0, x1 = src[:, 3:-3][:, :, arm].astype(float), out[:, 3:-3][:, :, arm].astype(float)
    inside = (x0 >= lo) & (x0 <= hi)
    assert ((x1 >= lo) & (x1 <= hi))[inside].all()                     # inside stays inside
    assert (np.abs(x1 - (lo + hi) / 2) <= np.maximum(np.abs(x0 - (lo + hi) / 2), (hi - lo) / 2))[~inside].all()
    assert (~inside).any()
    chk = check_trajectories_batch(torch.as_tensor(out, device="cuda:0"), n_samples=1501, solver=solver)
    tol = 1e-9 if dtype == torch.float64 else 1e-5
    assert np.abs(chk["grasp_err"].cpu().numpy() - r["grasp_err"]).max() < tol


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_zero_iterations_and_nan_pass_through(solver, batch, dtype):
    src = batch.astype(np.float32) if dtype == torch.float32 else batch
    r0 = _refine(solver, src, dtype, max_iters=0)
    assert np.array_equal(_bits(r0["ctrl"]), _bits(src)) and (r0["iters"] == 0).all() and (r0["accepted"] == 0).all()
    assert np.array_equal(r0["obj_before"], r0["obj_after"])
    bad = src[0].copy(); bad[10] = np.nan                             # F is NaN
    mixed = np.concatenate([src[:3], bad[None], src[3:]])
    r = _refine(solver, mixed, dtype)
    ref = _refine(solver, src, dtype)
    assert np.array_equal(_bits(r["ctrl"][3]), _bits(bad)) and r["iters"][3] == 0 and r["accepted"][3] == 0
    assert np.isnan(r["obj_before"][3]) and np.isnan(r["obj_after"][3]) and r["grasp_err"][3] == np.inf
    others = np.r_[0:3, 4:len(mixed)]
    for k in ("ctrl", "obj_before", "obj_after", "grasp_err", "iters", "accepted"):
        assert np.array_equal(r[k][others], ref[k]), k


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_outputs_do_not_depend_on_the_batch_or_the_run(solver, batch, dtype):
    keys = ("ctrl", "obj_before", "obj_after", "grasp_err", "iters", "accepted")
    full = _refine(solver, batch, dtype)
    again = _refine(solver, batch, dtype)
    N = len(batch)
    big = _refine(solver, batch[np.arange(1024) % N], dtype)
    for k in keys:
        assert np.array_equal(full[k], again[k]), k
    for i in range(N):
        alone = _refine(solver, batch[i:i + 1], dtype)
        nine = _refine(solver, np.concatenate([batch[(i + 1 + np.arange(4)) % N], batch[i:i + 1],
                                               batch[(i + 5 + np.arange(4)) % N]]), dtype)
        for k in keys:
            assert np.array_equal(alone[k][0], full[k][i]) and np.array_equal(nine[k][4], full[k][i]), (i, k)
            assert np.array_equal(big[k][i], full[k][i]) and np.array_equal(big[k][i + N], full[k][i]), (i, k)


def test_one_step_matches_a_numpy_restatement(solver, table, c_oracle, batch):
    """max_iters = 1: H and g from the C oracle's FK and LOCAL Jacobian, (H + lambda diag H) delta = -g, the box clamp,
    and the step kept only if F drops."""
    M = 201
    W = sample_weights(21, M)
    arm = _right_arm(table)
    r = _refine(solver, batch, torch.float64, n_samples=M, max_iters=1)
    lo, hi = np.asarray(table.lower)[arm], np.asarray(table.upper)[arm]
    stepped = 0
    for n, c in enumerate(batch):
        rr, J = _residual(c_oracle, table, W @ c)
        F = (rr ** 2).sum()
        w = W[:, 3:-3]
        H = np.einsum("ka,kb,kmc,kmd->acbd", w, w, J, J).reshape(90, 90)
        g = np.einsum("ka,kmc,km->ac", w, J, rr).reshape(90)
        d = np.linalg.solve(H + DAMPING * np.diag(np.diag(H)), -g).reshape(15, 6)
        x0 = c[3:-3][:, arm]
        x1 = np.clip(x0 + d, np.minimum(lo, x0), np.maximum(hi, x0))
        c1 = c.copy()
        for a_ in range(15):
            c1[3 + a_, arm] = x1[a_]
        F1 = (_residual(c_oracle, table, W @ c1)[0] ** 2).sum()
        assert abs(r["obj_before"][n] - F) <= 1e-10 * max(F, 1e-12)
        if F1 < F * (1 - 1e-9):
            stepped += 1
            assert r["accepted"][n] == 1 and np.abs(r["ctrl"][n] - c1).max() < 1e-8, (n, np.abs(r["ctrl"][n] - c1).max())
            assert abs(r["obj_after"][n] - F1) <= 1e-8 * F1 + 1e-18
        elif F1 > F * (1 + 1e-9):
            assert r["accepted"][n] == 0 and np.array_equal(r["ctrl"][n], c)
    assert stepped >= len(batch) // 2


def test_error_codes_and_guard_columns(solver, table, batch):
    import gik_b200
    from gik_b200 import _cabi
    from gik_b200.trajectory import sample_weights as weights
    lib = _cabi.lib()
    dev = "cuda:0"
    N, Ms = 5, 33
    for dtype, sfx in ((torch.float64, "f64"), (torch.float32, "f32")):
        f = getattr(lib, f"gik_traj_refine_{sfx}")
        W = torch.as_tensor(weights(21, Ms), dtype=dtype, device=dev)
        C = torch.as_tensor(batch[-N:], dtype=dtype, device=dev).contiguous()
        out = torch.full((N + 2, 21, 15), 3.25, dtype=dtype, device=dev)
        before = torch.full((N + 2,), 7.5, dtype=torch.float64, device=dev)
        after = torch.full((N + 2,), 8.5, dtype=torch.float64, device=dev)
        gerr = torch.full((N + 2,), 9.5, dtype=dtype, device=dev)
        iters = torch.full((N + 2,), 12345, dtype=torch.int32, device=dev)
        acc = torch.full((N + 2,), 54321, dtype=torch.int32, device=dev)
        outs = (out, before, after, gerr, iters, acc)
        keep = [t.clone() for t in outs]
        ptr = lambda t, off=1: ctypes.c_void_p(t.data_ptr() + off * t[0].numel() * t.element_size())   # noqa: E731

        def call(h=solver._h, n=N, nc=21, m=Ms, it=4, tol=0.0, lam=DAMPING, w=ptr(W, 0), c=ptr(C, 0)):
            rc = f(h, n, nc, m, w, c, it, tol, lam, *[ptr(t) for t in outs], None)
            torch.cuda.synchronize()
            return rc

        assert call(n=-1) == -2 and call(nc=6) == -2 and call(nc=27) == -2 and call(m=1) == -2
        assert call(it=-1) == -5 and call(tol=-1e-3) == -5 and call(lam=0.0) == -5 and call(lam=float("nan")) == -5
        assert call(w=None) == -1 and call(c=None) == -1
        assert call(h=None) == -6
        assert call(n=0) == 0
        for t, k in zip(outs, keep):
            assert torch.equal(t, k)                          # refused calls write nothing
        bare = gik_b200.GraspIK(table, dev)                   # no scene needed
        assert call(h=bare._h) == 0
        bare.close()
        for t, k in zip(outs, keep):
            assert torch.equal(t[0], k[0]) and torch.equal(t[-1], k[-1]) and not torch.equal(t[1:-1], k[1:-1])
        ref = solver.refine_trajectories(C, W, max_iters=4, tol=0.0, damping=DAMPING)
        for t, x in zip(outs, ref):
            assert torch.equal(t[1:-1], x)
        # in place: ctrl_out = ctrl
        Cp = C.clone()
        assert f(solver._h, N, 21, Ms, ptr(W, 0), ptr(Cp, 0), 4, 0.0, DAMPING, ptr(Cp, 0),
                 *[ptr(t) for t in outs[1:]], None) == 0
        torch.cuda.synchronize()
        assert torch.equal(Cp, ref[0])
