"""The kernels over the full rotation range on the GPU: solves whose hands start up to half a turn from their hooks
(pinocchio's near-pi form of log6 in every solve mapping, the success predicate's descent and replay), edges that turn
the cube by up to pi (the edge kernel's and gik_tree_grow's SE3 interpolation), and the host bookkeeping of
project_path / project_edges_batch on such edges -- against the C oracle on the same seeded inputs."""
import json
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, make_poses, rot_rpy
from test_gpu_parity import _assert_q_close
from test_rotation_range_cpu import (NEAR_PI, PI, THETAS, band_tol, fp32_resolvable, large_rotation_batch, pose_ld,
                                     start_angles)

pytestmark = pytest.mark.gpu
EPS = 1e-3


@pytest.fixture(scope="module")
def solver(table):
    import gik_b200
    s = gik_b200.GraspIK(table, "cuda:0").attach_scene()
    yield s
    s.close()


@pytest.fixture(scope="module")
def batch(table_c, c_oracle):
    """1,500 large-rotation problems (test_rotation_range_cpu.large_rotation_batch) and the oracle's solve of them."""
    Q0, P = large_rotation_batch(c_oracle, table_c, 1500, 31)
    near = start_angles(Q0, P).max(axis=1) >= NEAR_PI
    ref = c_oracle.solve(table_c, Q0, P)
    print(f"large-rotation batch: {near.mean():.2f} start with a hand in the near-pi band, "
          f"{ref[1].mean():.2f} converge in the oracle")
    return Q0, P, near, ref


def _soa(a, dtype):
    return torch.as_tensor(np.ascontiguousarray(np.asarray(a).T), dtype=dtype, device="cuda:0")


def _t(a, dtype=torch.float64):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device="cuda:0")


# ------------------------------------------------------------------------------------------------------------ solve
# Bounds per mapping: (flag agreement, q quantile bound, problems allowed beyond the outlier bound).  The half-turned
# warm starts make this batch more sensitive than the workspace batches of test_gpu_parity: on a few of them every pair
# of implementations of the same iteration agrees to 1e-13 for ~100 iterations, then diverges exponentially to O(1)
# differences in q within ~70 more (measured with the kernel arithmetic built for the host against the oracle, so not a
# device effect) and lands on a different flag or another point of the self-motion manifold.  Measured on an NVIDIA
# B200 (1000 W), 1,500 problems: flags differ on 2 (fp64), 3 (fp32 wrist forms), 12 (fp32 Cholesky form) problems; the
# host build of the same arithmetic: 2-4, 3-4 and 4-8.  The fp32 Cholesky form squares the condition number
# (test_gpu_parity.test_wrist_form_equals_cholesky_form): its 99.5 % quantile of |q - q_oracle| is 1.5e-3 - 3.2e-3 in
# the host build, against 4.2e-4 for the wrist forms.
SOLVE_BOUNDS = {"f64": (0.997, 1e-9, 4), "f32": (0.995, 1e-3, 4), "f32+chol": (0.985, 5e-3, 8)}


@pytest.mark.parametrize("dtype,kernel", [(torch.float64, None), (torch.float64, "lane"), (torch.float64, "pair+chol"),
                                          (torch.float32, "lane"), (torch.float32, "lane1"), (torch.float32, "pair"),
                                          (torch.float32, "lane+chol")])
def test_solve_under_large_rotations_matches_oracle(solver, batch, dtype, kernel):
    Q0, P, near, (qo, oko, ito, _) = batch
    assert near.mean() >= 1 / 3
    q, ok, it, res = solver.solve_soa(_soa(Q0, dtype), _soa(P, dtype), kernel=kernel)
    q = q.t().double().cpu().numpy(); ok = ok.bool().cpu().numpy(); it = it.cpu().numpy()
    res = res.t().double().cpu().numpy()
    both = ok & oko
    d = np.abs(q[both] - qo[both]).max(axis=1)
    print(f"{dtype} {kernel}: {both.mean():.2f} converged in both ({(both & near).sum()} of them from near pi), "
          f"flags differ on {(ok != oko).sum()}, |dq| 99.5 % {np.quantile(d, 0.995):.1e}, "
          f"{(d >= 5e-3).sum()} beyond 5e-3, worst {d.max():.1e}")
    key = "f64" if dtype == torch.float64 else ("f32+chol" if "chol" in kernel else "f32")
    agree, tol, n_far = SOLVE_BOUNDS[key]
    assert (ok == oko).mean() >= agree
    assert both.mean() >= 0.3 and (both & near).sum() >= 100
    assert (res[ok] < EPS).all()
    if dtype == torch.float64:
        _assert_q_close(q[both], qo[both], tol, n_far=n_far)
        assert (it[both] == ito[both]).mean() >= 0.995
        assert (it[~ok] == 1000).all()
    else:
        _assert_q_close(q[both], qo[both], tol, tol_outlier=5e-2, n_far=n_far)
        assert np.quantile(np.abs(it[both] - ito[both]), 0.995) <= 2


def test_fp64_large_batch_instantiation_under_large_rotations(solver, batch):
    # more than 16 * 8 * SMs problems: the pair kernel's large-batch instantiation, bit for bit the lane kernel
    Q0, P, _, _ = batch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = 16 * 8 * sms + 517
    assert solver.kernel_name(n, torch.float64).startswith("gik_solve_pair_kernel<double")
    idx = np.arange(n) % len(P)
    q0, pose = _soa(Q0[idx], torch.float64), _soa(P[idx], torch.float64)
    a = solver.solve_soa(q0, pose)
    b = solver.solve_soa(q0, pose, kernel="lane")
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    assert a[1].float().mean().item() >= 0.3


def test_success_predicate_under_large_rotations(solver, batch, table_c, scene_c, c_oracle):
    # gik_solve_success_f64: the descent, the collision test, the continuation of converged-but-colliding problems and
    # their replay, on problems that start near pi
    Q0, P, near, _ = batch
    n = 200
    Q0, P, near = Q0[:n], P[:n], near[:n]
    qo, oko, ito, evo = c_oracle.solve_success(table_c, scene_c, Q0, P, return_ever=True)
    q, succ, conv, it, _ = solver.solve_success_soa(_soa(Q0, torch.float64), _soa(P, torch.float64))
    succ = succ.bool().cpu().numpy(); it = it.cpu().numpy(); q = q.t().cpu().numpy()
    print(f"success predicate: {succ.mean():.2f} succeed, {(evo & ~oko).sum()} converged but colliding, "
          f"{near.sum()} start near pi")
    assert (succ == oko).all()
    assert (it == ito).mean() >= 0.98
    assert oko.sum() >= 10 and (oko & near).sum() >= 5
    d = np.abs(q - qo).max(axis=1)
    assert np.quantile(d[oko], 0.95) < 1e-9
    # one collision test at the configuration the descent stopped at: a success there is a success of the reference
    # loop too, with the same q and iteration count
    q2, s2, _, it2, _ = solver.solve_success_soa(_soa(Q0, torch.float64), _soa(P, torch.float64),
                                                 descend_while_colliding=False)
    s2 = s2.bool().cpu().numpy()
    assert (s2 & ~oko).sum() == 0 and s2.sum() >= 5
    assert np.abs(q2.t().cpu().numpy()[s2] - qo[s2]).max() < 1e-8 and (it2.cpu().numpy()[s2] == ito[s2]).all()


# ------------------------------------------------------------------------------------------------------------ edges
def _rotation_edges(seed):
    """Relative rotations of the edges: the angle grid about z (exactly pi written the way a caller would,
    rot_rpy(0, 0, pi)) and about random axes (exactly pi excluded: its direction is rounding noise there).
    -> (R [m,9], theta [m], axis has a zero component [m])."""
    rng = np.random.default_rng(seed)
    rows = []
    for th in THETAS:
        axes = [np.array([0.0, 0.0, 1.0])] + [u / np.linalg.norm(u) for u in rng.standard_normal((2, 3))]
        for k, u in enumerate(axes):
            if th == PI and k:
                continue
            R = rot_rpy(0, 0, np.pi) if th == PI else pose_ld(u, th, np.zeros(3))[:9].astype(float).reshape(3, 3)
            rows.append((R.reshape(9), th, k == 0))
    return np.array([r[0] for r in rows]), np.array([r[1] for r in rows]), np.array([r[2] for r in rows])


@pytest.fixture(scope="module")
def edges(table_c, c_oracle):
    """Edges A -> B, A a cube placement with identity rotation at which the oracle converges from q = 0 (three per
    relative rotation), B = (R, A's translation + up to 5 cm).  -> (A, B, theta, zero, q at A)."""
    R, th, zero = [np.concatenate([x] * 3) for x in _rotation_edges(41)]
    pool = make_poses(6 * len(R), 43, "sampler")
    qp, okp, _, _ = c_oracle.solve(table_c, np.zeros((len(pool), 15)), pool)
    take = np.flatnonzero(okp)[:len(R)]
    assert len(take) == len(R)
    A = pool[take]
    B = A.copy()
    B[:, :9] = R
    B[:, 9:] += np.random.default_rng(42).uniform(-0.05, 0.05, (len(A), 3))
    return A, B, th, zero, qp[take]


def test_project_edges_under_large_rotations_matches_oracle(solver, edges, table_c, c_oracle):
    import gik_b200
    A, B, th, zero, q0 = edges
    E, S = len(A), 6
    assert E >= 40 and (th == PI).any() and (th >= NEAR_PI).sum() >= 10
    ns = np.random.default_rng(44).integers(1, S + 1, size=E).astype(np.int32)
    path_o, nv_o, it_o = c_oracle.project_edges(table_c, q0, A, B, ns, S)
    path, nv, itt = gik_b200.project_edges_batch(solver, _t(q0), _t(A), _t(B), num_steps=ns, max_steps=S,
                                                 dtype=torch.float64, return_info=True)
    nv = nv.cpu().numpy()
    print(f"rotation edges: {E}, complete in the oracle {(nv_o == ns).sum()}, of them near pi {((nv_o == ns) & (th >= NEAR_PI)).sum()}")
    assert np.array_equal(nv, nv_o) and np.array_equal(itt.cpu().numpy(), it_o)
    assert ((nv_o >= 1) & (th >= NEAR_PI)).sum() >= 3
    path = path.cpu().numpy()
    for e in range(E):
        assert np.abs(path[e, :nv_o[e]] - path_o[e, :nv_o[e]]).max(initial=0) < 1e-8
    path32, nv32 = gik_b200.project_edges_batch(solver, _t(q0), _t(A), _t(B), num_steps=ns, max_steps=S,
                                                dtype=torch.float32)
    same = nv32.cpu().numpy() == nv_o
    print(f"fp32: {(~same).sum()} of {E} edges stop at a different step")
    assert (~same).sum() <= max(1, E // 50)
    for e in np.nonzero(same)[0]:
        assert np.abs(path32[e, :nv_o[e]].double().cpu().numpy() - path_o[e, :nv_o[e]]).max(initial=0) < 2e-3


def _grow_cubes(solver, A, B, ns, dtype):
    """gik_tree_grow_* with every step valid, one tree per edge: -> the placements it stored [E, S, 12]."""
    E, S = len(A), int(ns.max())
    nq = solver.nq
    verts = torch.zeros((E, nq, S + 2), dtype=dtype, device="cuda:0")
    cubes = torch.zeros((E, 12, S + 2), dtype=dtype, device="cuda:0")
    parent = torch.full((E, S + 2), -1, dtype=torch.int32, device="cuda:0")
    n_verts = torch.ones(E, dtype=torch.int32, device="cuda:0")
    ovf = torch.zeros(E, dtype=torch.uint8, device="cuda:0")
    i32 = lambda a: torch.as_tensor(np.ascontiguousarray(a, np.int32), device="cuda:0")    # noqa: E731
    seg = solver.tree_grow(verts, cubes, parent, n_verts, ovf, i32(np.arange(E)), i32(np.zeros(E)),
                           torch.zeros((nq, E), dtype=dtype, device="cuda:0"), _soa(A, dtype), _soa(B, dtype), i32(ns),
                           i32(ns), torch.zeros((S, nq, E), dtype=dtype, device="cuda:0"))
    assert not ovf.any() and (seg.cpu().numpy() == 1 + ns).all()
    return cubes[:, :, 2:].permute(0, 2, 1).double().cpu().numpy()


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_tree_grow_placements_over_the_rotation_range(solver, edges, c_oracle, dtype):
    A, B, th, zero, _ = edges
    E = len(A)
    ns = np.random.default_rng(45).integers(1, 9, size=E).astype(np.int32)
    prec = "f64" if dtype == torch.float64 else "f32"
    cubes = _grow_cubes(solver, A, B, ns, dtype)
    worst = {}
    for e in range(E):
        # the oracle on the fp64 edge (for fp32 the bound includes the rounding of the inputs, as in the CPU tests:
        # the oracle's own acos form is ill-conditioned near pi on fp32-rounded matrices).  A has an identity rotation,
        # so A^-1 B is B's rotation exactly; at exactly pi about z the sin(pi) = 1.2e-16 of rot_rpy fixes the
        # direction of the turn in both precisions
        if prec == "f32" and th[e] < PI and not fp32_resolvable(th[e], zero[e]):
            continue
        al = np.arange(1, ns[e] + 1) / ns[e]
        ref = c_oracle.interpolate(np.tile(A[e], (ns[e], 1)), np.tile(B[e], (ns[e], 1)), al)
        err = np.abs(cubes[e, :ns[e]] - ref).max()
        band = "near_pi" if th[e] >= NEAR_PI else "far"
        worst[band] = max(worst.get(band, 0.0), err)
        assert err < band_tol(prec, th[e], zero[e]), (th[e], e, err)
        assert np.abs(cubes[e, ns[e] - 1] - B[e]).max() < band_tol(prec, th[e], zero[e])
    print(f"tree_grow {prec}: worst |err| per band {worst}")


# ------------------------------------------------------------------------------------------------------- end to end
def test_project_path_lands_on_a_half_turned_cube(solver, c_oracle, table_c):
    # one step that yaws the cube by exactly pi (the reference's second golden grasp converges there): the returned
    # cube path ends on B, and it is the oracle's march
    import gik_b200
    g = json.load(open(os.path.join(GOLDEN, "ik_golden.json")))["cases"][1]
    q0 = np.array(g["q"])
    a = (np.eye(3), np.array(g["cube_p"]))
    b = (rot_rpy(0, 0, np.pi), np.array(g["cube_p"]) + [0.01, 0.0, 0.0])
    A = np.concatenate([a[0].reshape(9), a[1]]); B = np.concatenate([b[0].reshape(9), b[1]])
    _, nv_o, _ = c_oracle.project_edges(table_c, q0[None], A[None], B[None], np.array([1], np.int32), 1)
    assert nv_o[0] == 1
    rp, cp = gik_b200.project_path(solver, None, q0, a, b)
    assert len(rp) == len(cp) == 2
    assert np.abs(np.asarray(cp[-1]) - B).max() < 1e-12
    # and half way along a two-step edge: a quarter turn, the way the kernel turned
    from gik_b200.path import se3_interpolate
    mid = se3_interpolate(torch.from_numpy(A[None]), torch.from_numpy(B[None]), 0.5).numpy()[0]
    assert np.abs(mid - c_oracle.interpolate(A[None], B[None], np.array([0.5]))[0]).max() < 1e-12


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_scene_tests_use_the_placements_the_kernel_solved_for(solver, edges, table_c, scene_c, c_oracle, dtype):
    # project_edges_batch(scene_tests=True) tests each step's cube and robot at the placement the host interpolates;
    # it must be the placement the edge kernel solved for (the one gik_tree_grow stores, the same device code)
    import gik_b200
    from gik_b200.path import se3_interpolate
    A, B, th, zero, q0 = edges
    E, S = len(A), 6
    ns = np.random.default_rng(46).integers(1, S + 1, size=E).astype(np.int32)
    prec = "f64" if dtype == torch.float64 else "f32"
    a12, b12 = _t(A, dtype), _t(B, dtype)
    cubes = _grow_cubes(solver, A, B, ns, dtype)
    for e in range(E):
        if prec == "f32" and th[e] < PI and not fp32_resolvable(th[e], zero[e]):
            continue
        al = torch.arange(1, ns[e] + 1, dtype=dtype, device="cuda:0") / int(ns[e])     # as _cut_at_first_collision
        m = int(ns[e])
        host = se3_interpolate(a12[e:e + 1].expand(m, 12), b12[e:e + 1].expand(m, 12), al).double().cpu().numpy()
        assert np.abs(host - cubes[e, :ns[e]]).max() < band_tol(prec, th[e], zero[e]), (th[e], e)
    # the cut itself (fp64): the first step whose cube or robot the oracle finds in collision, at the oracle's placement
    if dtype == torch.float64:
        path, nv = gik_b200.project_edges_batch(solver, _t(q0), a12, b12, num_steps=ns, max_steps=S, dtype=dtype)
        path_c, nv_c = gik_b200.project_edges_batch(solver, _t(q0), a12, b12, num_steps=ns, max_steps=S, dtype=dtype,
                                                    scene_tests=True)
        nv, nv_c, path = nv.cpu().numpy(), nv_c.cpu().numpy(), path.cpu().numpy()
        checked = 0
        for e in range(E):
            if nv[e] == 0:
                continue
            al = np.arange(1, nv[e] + 1) / ns[e]
            pl = c_oracle.interpolate(np.tile(A[e], (nv[e], 1)), np.tile(B[e], (nv[e], 1)), al)
            d_cube = c_oracle.scene_distance(table_c, scene_c, None, pl, mode=2)
            d_rob = c_oracle.scene_distance(table_c, scene_c, path[e, :nv[e]], pl, mode=0, cull=0.05)
            d = np.minimum(d_cube, d_rob)
            if ((d > 0) & (d < 1e-6)).any():
                continue                                                    # a step at the collision boundary
            bad = np.flatnonzero(d == 0)
            assert nv_c[e] == (bad[0] if len(bad) else nv[e]), (e, th[e], nv_c[e], nv[e], d)
            checked += 1
        print(f"scene tests: {checked} edges checked, {(nv_c < nv).sum()} cut by a collision")
        assert checked >= E // 2
