"""GPU collision kernels (through the C ABI) against the CPU oracle (alternating projections, oracle/collision_oracle.inc)
on the same seeded inputs, plus the reference's known answers."""
import numpy as np
import pytest
import torch

from conftest import rot_rpy

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def solver(table):
    import gik_b200
    s = gik_b200.GraspIK(table, "cuda:0").attach_scene()
    yield s
    s.close()


def _t(a, dtype):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device="cuda:0")


def _inputs(table, n, seed):
    rng = np.random.default_rng(seed)
    Q = rng.uniform(table.lower, table.upper, size=(n, 15)) * 0.7
    Q[0] = 0.0
    P = np.zeros((n, 12)); P[:, [0, 4, 8]] = 1
    P[:, 9:] = rng.uniform([0.2, -0.4, 0.93], [0.6, 0.4, 1.4], size=(n, 3))
    P[1::5, :9] = rot_rpy(0, 0, 0.5).reshape(9)
    return Q, P


@pytest.mark.parametrize("dtype,band", [(torch.float64, 1e-6), (torch.float32, 1e-4)])
def test_collision_and_clearance_match_oracle(solver, table, table_c, scene_c, c_oracle, dtype, band):
    n = 1203                                                       # not a multiple of the warps per block
    Q, P = _inputs(table, n, 3)
    d_all = c_oracle.scene_distance(table_c, scene_c, Q, P, mode=0, cull=0.05)
    d_obs = c_oracle.scene_distance(table_c, scene_c, Q, P, mode=1, cull=0.2)
    qs, ps = _t(Q, dtype).t().contiguous(), _t(P, dtype).t().contiguous()
    col = solver.collision_soa(qs, ps).bool().cpu().numpy()
    sure = (d_all == 0) | (d_all > band)
    assert sure.mean() > 0.95 and (col[sure] == (d_all[sure] == 0)).all()
    assert col[0]                                                  # collision(robot, q0) is True (lab_instructions.ipynb:252)
    assert 0.05 < col.mean() < 0.98
    clear = solver.clearance_soa(qs, ps, 0.04).bool().cpu().numpy()
    sure = np.abs(d_obs - 0.04) > 10 * band
    assert (clear[sure] == (d_obs[sure] >= 0.04)).all()
    # row-major convenience + default cube placement of the scene
    c2 = solver.collision(_t(Q[:64], dtype), _t(P[:64], dtype)).cpu().numpy()
    assert (c2 == col[:64]).all()
    d_def = c_oracle.scene_distance(table_c, scene_c, Q[:64], None, mode=0, cull=0.05)
    c3 = solver.collision(_t(Q[:64], dtype)).cpu().numpy()
    sure = (d_def == 0) | (d_def > band)
    assert (c3[sure] == (d_def[sure] == 0)).all()


@pytest.mark.parametrize("dtype,tol,typical", [(torch.float64, 5e-5, 1e-6), (torch.float32, 2e-4, 5e-5)])
def test_obstacle_distance_matches_oracle(solver, table, table_c, scene_c, c_oracle, dtype, tol, typical):
    # distanceToObstacle as a value (tools.py:38-51): gik_obstacle_distance_* (GJK bisection in the kernel, one launch)
    # against the oracle's alternating-projection distances, incl. the cap and the 0 on intersection
    n = 1203
    Q, P = _inputs(table, n, 11)
    d_ref = c_oracle.scene_distance(table_c, scene_c, Q, P, mode=1)            # exact for every pair (no cull)
    qs, ps = _t(Q, dtype).t().contiguous(), _t(P, dtype).t().contiguous()
    d = solver.obstacle_distance_soa(qs, ps, 2.0).double().cpu().numpy()
    assert d.shape == (n,) and (d >= 0).all() and (d <= 2.0).all()
    assert ((d == 0) == (d_ref == 0))[(d_ref == 0) | (d_ref > 10 * tol)].all()
    assert 0.1 < (d_ref > 0).mean() < 0.95
    # two different algorithms (GJK bisection here, alternating projections in the oracle, which converges linearly on
    # nearly parallel faces): round-off level agreement on almost every configuration, 1e-5 m on the worst
    err = np.abs(d - np.minimum(d_ref, 2.0))
    assert err.max() < tol and np.quantile(err, 0.95) < typical
    # cap below the true distance: the value is the cap; consistent with the boolean clearance kernel
    d_cap = solver.obstacle_distance_soa(qs, ps, 0.04).double().cpu().numpy()
    assert np.abs(d_cap - np.minimum(d_ref, 0.04)).max() < tol
    clear = solver.clearance_soa(qs, ps, 0.04).bool().cpu().numpy()
    sure = np.abs(d_ref - 0.04) > 10 * tol
    assert (clear[sure] == (d_cap[sure] >= 0.04 - tol)).all()
    # default cube placement of the scene, and an empty batch
    d_def = solver.obstacle_distance_soa(qs[:, :64].contiguous(), None, 2.0).double().cpu().numpy()
    assert np.abs(d_def - np.minimum(c_oracle.scene_distance(table_c, scene_c, Q[:64], None, mode=1), 2.0)).max() < tol
    assert solver.obstacle_distance_soa(qs[:, :0].contiguous(), None).shape == (0,)


def test_cube_collision_matches_oracle(solver, table_c, scene_c, c_oracle):
    rng = np.random.default_rng(5)
    n = 999
    P = np.zeros((n, 12)); P[:, [0, 4, 8]] = 1
    P[:, 9:] = rng.uniform([0.2, -0.3, 0.85], [0.65, 0.15, 1.1], size=(n, 3))
    P[::3, :9] = rot_rpy(0.1, -0.2, 0.6).reshape(9)
    dc = c_oracle.scene_distance(table_c, scene_c, None, P, mode=2)
    for dtype, band in ((torch.float64, 1e-6), (torch.float32, 1e-4)):
        got = solver.cube_collision_soa(_t(P, dtype).t().contiguous()).bool().cpu().numpy()
        sure = (dc == 0) | (dc > band)
        assert (got[sure] == (dc[sure] == 0)).all() and 0.1 < got.mean() < 0.9


def test_golden_grasp_poses_are_collision_free(solver, golden):
    Q = np.array([c["q"] for c in golden["cases"]])
    P = np.array([c["cube_R"] + c["cube_p"] for c in golden["cases"]], float)
    for dtype in (torch.float64, torch.float32):
        assert not solver.collision(_t(Q, dtype), _t(P, dtype)).any()      # the reference returned success=True for both
    assert solver.collision(_t(Q, torch.float64)).any() is not None


def test_collision_error_codes_in_check_order(table):
    import ctypes
    import gik_b200
    from gik_b200 import _cabi
    s = gik_b200.GraspIK(table, "cuda:0")
    z = ctypes.c_void_p(0)
    x = ctypes.c_void_p(8)                                                     # never dereferenced
    assert _cabi.lib().gik_collision_f32(s._h, 4, x, z, x, z) == -7           # GIK_E_NOSCENE
    assert _cabi.lib().gik_collision_f32(s._h, 4, z, z, z, z) == -1           # pointers are checked before the scene
    s.attach_scene()
    assert _cabi.lib().gik_collision_f32(s._h, 4, z, z, z, z) == -1           # GIK_E_NULL
    assert _cabi.lib().gik_collision_f32(s._h, 0, z, z, z, z) == 0
    bad = gik_b200.nextage_scene()
    bad.geoms[3].joint = 99
    with pytest.raises(_cabi.GikError):
        s.attach_scene(bad)
    s.close()


def test_full_success_predicate_matches_oracle(solver, table_c, scene_c, c_oracle):
    # computeqgrasppose WITH the collision term (inverse_geometry.py:70, 97-98), including the reference's
    # keep-descending-while-colliding tail: same success flags, same iteration counts, same q
    from conftest import make_poses
    import gik_b200
    n = 96
    P = make_poses(n, 77)
    qo, oko, ito = c_oracle.solve_success(table_c, scene_c, np.zeros((n, 15)), P)
    q, ok, info = gik_b200.computeqgrasppose_batch(solver, torch.zeros(15), _t(P, torch.float64), dtype=torch.float64,
                                                   collision=True, return_info=True)
    ok = ok.cpu().numpy(); q = q.cpu().numpy(); it = info.iters.cpu().numpy()
    assert (ok == oko).all()
    assert (it == ito).mean() >= 0.98
    d = np.abs(q - qo).max(axis=1)
    assert np.quantile(d[ok], 0.95) < 1e-9 and np.quantile(d, 0.9) < 1e-6
    _, conv = solver.solve(torch.zeros(15), _t(P, torch.float64), dtype=torch.float64)
    conv = conv.cpu().numpy()
    assert (conv & ~ok).sum() >= 5                     # the batch does contain converged-but-colliding problems
    assert (it[conv & ~ok] == 1000).all()              # ... which kept descending to the iteration cap, like the reference
    # skipping the extra descent gives the same decisions on this batch
    q2, s2, c2, it2, _ = solver.solve_success_soa(torch.zeros((15, n), dtype=torch.float64, device="cuda:0"),
                                                  _t(P, torch.float64).t().contiguous(), descend_while_colliding=False)
    assert (s2.bool().cpu().numpy() == oko).all()
    # single-call drop-in: full reference semantics without pinocchio (GPU collision on the packaged scene)
    i_bad = int(np.nonzero(conv & ~ok)[0][0]); i_good = int(np.nonzero(ok)[0][0])
    for i in (i_bad, i_good):
        qs, ss = gik_b200.computeqgrasppose(None, np.zeros(15), None, (np.eye(3), P[i, 9:]))
        assert ss == bool(oko[i]) and np.abs(qs - qo[i]).max() < 1e-6


def test_batched_sampler_applies_every_reference_filter(solver, table_c, scene_c, c_oracle):
    import gik_b200
    g = torch.Generator(device="cuda:0").manual_seed(9)
    a = (np.eye(3), np.array([0.33, -0.3, 0.93])); b = (np.eye(3), np.array([0.4, 0.11, 0.93]))   # config.py:36-37
    q, pl, ok = gik_b200.sample_grasp_poses_batch(solver, 2048, a, b, dtype=torch.float64, generator=g)
    pl_np = pl.cpu().numpy(); okn = ok.cpu().numpy(); qn = q.cpu().numpy()
    assert 0.02 < okn.mean() < 0.6
    assert (pl_np[:, 0] >= 0.33).all() and (pl_np[:, 0] <= 0.4).all() and (pl_np[:, 2] >= 1.05).all() and (pl_np[:, 2] <= 1.4).all()
    P = np.zeros((len(pl_np), 12)); P[:, [0, 4, 8]] = 1; P[:, 9:] = pl_np
    idx = np.nonzero(okn)[0][:40]
    # accepted samples satisfy every predicate of path.sample_cube_placement according to the oracle
    assert (c_oracle.scene_distance(table_c, scene_c, None, P[idx], mode=2) > 0).all()             # path.py:51-54
    assert (c_oracle.scene_distance(table_c, scene_c, qn[idx], P[idx], mode=0, cull=0.05) > 0).all()  # :57-59
    assert (c_oracle.scene_distance(table_c, scene_c, qn[idx], P[idx], mode=1, cull=0.2) >= 0.04 - 1e-6).all()   # :61-62


def test_rrt_connect_driver_end_to_end(solver, table, table_c, scene_c, c_oracle, golden):
    # path.computepath (path.py:194-278) on the reference's own query: carry the cube from CUBE_PLACEMENT to
    # CUBE_PLACEMENT_TARGET over the obstacle, starting and ending at the recorded grasp poses
    import time
    import gik_b200
    q0 = np.array(golden["cases"][0]["q"]); qe = np.array(golden["cases"][1]["q"])
    a = (np.eye(3), np.array(golden["cases"][0]["cube_p"])); b = (np.eye(3), np.array(golden["cases"][1]["cube_p"]))
    t0 = time.perf_counter()
    path, stats = gik_b200.computepath(q0, qe, a, b, robot=solver, rng=np.random.default_rng(0),
                                       generator=torch.Generator(device="cuda:0").manual_seed(0), return_stats=True)
    dt = time.perf_counter() - t0
    print(f"computepath: {len(path)} configurations, {stats}, {dt:.2f} s")
    assert len(path) >= 3 and np.array_equal(path[0], q0) and np.array_equal(path[-1], qe)
    Q = np.array(path)
    assert (Q >= table.lower - 1e-9).all() and (Q <= table.upper + 1e-9).all()
    # every vertex still holds the cube: the two hand frames are one cube width apart (hooks at +-0.05, cube_small.urdf:34-48)
    R, p = c_oracle.fk(table_c, Q)
    assert np.abs(np.linalg.norm(p[:, 0] - p[:, 1], axis=1) - 0.1).max() < 3e-3
    # ... and stays clear of the table and the obstacle (robot geometries; oracle distances)
    assert (c_oracle.scene_distance(table_c, scene_c, Q, None, mode=1, cull=0.3) > 0).all()
    # consecutive vertices inside a segment move the cube by at most one step (0.025 m): hands move accordingly
    mid = 0.5 * (p[:, 0] + p[:, 1])
    jumps = np.linalg.norm(np.diff(mid, axis=0), axis=1)
    assert np.quantile(jumps, 0.9) < 0.03


def test_rrt_connect_batched_expansion(solver, table, table_c, scene_c, c_oracle, golden):
    # expand = K tree extensions per iteration through one launch of the edge kernel (path.py:194-278 rules unchanged):
    # expand=1 is the reference loop; both must return a valid path within the reference's extension budget per retry
    import time
    import gik_b200
    q0 = np.array(golden["cases"][0]["q"]); qe = np.array(golden["cases"][1]["q"])
    a = (np.eye(3), np.array(golden["cases"][0]["cube_p"])); b = (np.eye(3), np.array(golden["cases"][1]["cube_p"]))
    its = {}
    for K in (1, 8):
        tot = 0
        for seed in (1, 2, 3):
            t0 = time.perf_counter()
            path, stats = gik_b200.computepath(q0, qe, a, b, robot=solver, rng=np.random.default_rng(seed), expand=K,
                                               generator=torch.Generator(device="cuda:0").manual_seed(seed), return_stats=True)
            print(f"expand={K} seed={seed}: {len(path)} configurations, {stats}, {time.perf_counter() - t0:.2f} s")
            assert len(path) >= 3 and np.array_equal(path[0], q0) and np.array_equal(path[-1], qe) and stats["expand"] == K
            Q = np.array(path)
            assert (Q >= table.lower - 1e-9).all() and (Q <= table.upper + 1e-9).all()
            R, p = c_oracle.fk(table_c, Q)
            assert np.abs(np.linalg.norm(p[:, 0] - p[:, 1], axis=1) - 0.1).max() < 3e-3
            assert (c_oracle.scene_distance(table_c, scene_c, Q, None, mode=1, cull=0.3) > 0).all()
            mid = 0.5 * (p[:, 0] + p[:, 1])
            assert np.quantile(np.linalg.norm(np.diff(mid, axis=0), axis=1), 0.9) < 0.03
            assert stats["iterations"] <= (stats["retries"] + 1) * -(-250 // K) and stats["edges"] == 2 * K * stats["iterations"]
            tot += stats["iterations"]
        its[K] = tot
    print("iterations over the three seeds:", its)     # (speed claim: tools/probes/rrt_probe.py, DESIGN.md section 4)


def test_success_rate_experiment_matches_oracle(solver, table_c, scene_c, c_oracle):
    # inverse_geometry_TESTS.py:474-561 in batch form: the same placements through the oracle give the same tally
    from gik_b200 import experiments
    a = (np.eye(3), np.array([0.33, -0.3, 0.93])); b = (np.eye(3), np.array([0.4, 0.11, 0.93]))
    g = torch.Generator(device="cuda:0").manual_seed(3)
    res = experiments.grasp_success_rate(solver, a, b, std_devs=[(0.1, 0.1, 0.1), (0.4, 0.4, 0.4)], trials=48, generator=g)
    assert [r[2] for r in res] == [48, 48] and all(0.0 <= r[1] <= 100.0 for r in res)
    # replay the first spread's placements through the CPU oracle
    g = torch.Generator(device="cuda:0").manual_seed(3)
    pl = experiments.sample_gaussian_placements(48 * 4, a, b, (0.1, 0.1, 0.1), device="cuda:0", generator=g).cpu().numpy()
    lo = np.minimum(a[1], b[1]) - 0.14; hi = np.maximum(a[1], b[1]) + 0.14
    assert (pl >= lo - 1e-12).all() and (pl <= hi + 1e-12).all()
    P = np.zeros((len(pl), 12)); P[:, [0, 4, 8]] = 1; P[:, 9:] = pl
    free = c_oracle.scene_distance(table_c, scene_c, None, P, mode=2) > 0
    P = P[free][:48]
    _, ok, _ = c_oracle.solve_success(table_c, scene_c, np.zeros((len(P), 15)), P)
    assert abs(100.0 * ok.mean() - res[0][1]) < 1e-9


def test_project_edges_batch_scene_tests_match_single_edge_dropin(solver, golden):
    # batched cut-at-first-collision == the per-edge drop-in project_path with the scene tests
    import gik_b200
    rng = np.random.default_rng(8)
    q0 = np.array(golden["cases"][0]["q"])
    a = np.array([1, 0, 0, 0, 1, 0, 0, 0, 1, 0.33, -0.3, 0.93], float)
    E = 12
    B = np.tile(a, (E, 1)); B[:, 9:] = rng.uniform([0.3, -0.3, 0.9], [0.5, 0.1, 1.3], size=(E, 3))
    B[0, 9:] = [0.43, -0.1, 0.95]                                    # straight into the obstacle
    A = np.tile(a, (E, 1)); Q0 = np.tile(q0, (E, 1))
    path, nv = gik_b200.project_edges_batch(solver, torch.from_numpy(Q0).cuda(), torch.from_numpy(A).cuda(),
                                            torch.from_numpy(B).cuda(), dtype=torch.float64, scene_tests=True)
    path0, nv0 = gik_b200.project_edges_batch(solver, torch.from_numpy(Q0).cuda(), torch.from_numpy(A).cuda(),
                                              torch.from_numpy(B).cuda(), dtype=torch.float64)
    assert (nv <= nv0).all() and (nv < nv0).any()                    # some edge is cut by a collision
    for e in range(E):
        rp, cp = gik_b200.project_path(solver, None, q0, A[e], B[e], cube_collision="scene", collision="scene")
        assert len(rp) - 1 == int(nv[e])
        for k in range(int(nv[e])):
            assert np.abs(rp[k + 1] - path[e, k].cpu().numpy()).max() < 1e-12
        assert path[e, int(nv[e]):].abs().max().item() == 0 if int(nv[e]) < path.shape[1] else True


def test_planner_trials_experiment(solver):
    # path_TESTS.py:910-990 in small: random start / goal placements, planning statistics
    from gik_b200 import experiments
    a = (np.eye(3), np.array([0.33, -0.3, 0.93])); b = (np.eye(3), np.array([0.4, 0.11, 0.93]))
    res = experiments.rrt_connect_trials(solver, a, b, std_devs=[(0.1, 0.1, 0.1)], trials=3,
                                         generator=torch.Generator(device="cuda:0").manual_seed(4), rng=np.random.default_rng(4))
    r = res[0]
    assert r["std_dev"] == (0.1, 0.1, 0.1) and 0.0 <= r["success_rate"] <= 100.0
    assert r["success_rate"] >= 66.0 and r["min_iterations"] >= 1 and r["avg_time"] < 30.0


def test_collision_on_a_column_subset(solver, table):
    # gik_collision_sel_*: only the listed columns are tested (the predicate's short-circuit), the rest stay 0
    Q, P = _inputs(table, 5000, 21)
    qs, ps = _t(Q, torch.float32).t().contiguous(), _t(P, torch.float32).t().contiguous()
    full = solver.collision_soa(qs, ps)
    sel = torch.nonzero(torch.arange(5000, device="cuda:0") % 3 == 1).flatten()
    part = solver.collision_soa(qs, ps, sel=sel)
    assert torch.equal(part[sel], full[sel])
    mask = torch.ones(5000, dtype=torch.bool, device="cuda:0"); mask[sel] = False
    assert part[mask].sum().item() == 0
    assert solver.collision_soa(qs, ps, sel=sel[:0]).sum().item() == 0


def test_solve_success_call_edge_cases(solver):
    # gik_solve_success_*: ragged sizes, nothing converged, empty batch
    from conftest import make_poses
    for n in (1, 33, 1000):
        far = make_poses(n, 5); far[:, 9] += 3.0
        q, succ, conv, it, res = solver.solve_success_soa(torch.zeros((15, n), device="cuda:0"),
                                                          _t(far, torch.float32).t().contiguous(), descend_while_colliding=False)
        assert succ.sum().item() == 0 and conv.sum().item() == 0 and (it == 1000).all()
    P = make_poses(777, 6)
    pose = _t(P, torch.float64).t().contiguous(); q0 = torch.zeros((15, 777), dtype=torch.float64, device="cuda:0")
    q, succ, conv, it, res = solver.solve_success_soa(q0, pose, descend_while_colliding=False)
    q2, conv2, it2, res2 = solver.solve_soa(q0, pose)
    assert torch.equal(q, q2) and torch.equal(conv, conv2) and torch.equal(it, it2)
    col = solver.collision_soa(q2, pose).bool()
    assert torch.equal(succ.bool(), conv2.bool() & ~col)
    q, succ, conv, it, res = solver.solve_success_soa(torch.zeros((15, 0), device="cuda:0"), torch.zeros((12, 0), device="cuda:0"),
                                                      descend_while_colliding=False)
    assert succ.numel() == 0


def test_tools_module_dropins(solver, table, table_c, scene_c, c_oracle, golden):
    # tools.py helpers with the reference's names (tools.py:11-68) on the GPU scene
    from gik_b200 import tools
    q0 = np.array(golden["cases"][0]["q"]); place = (np.eye(3), np.array(golden["cases"][0]["cube_p"]))
    assert tools.collision(solver, np.zeros(15)) is True                       # lab_instructions.ipynb:252
    tools.setcubeplacement(solver, None, place)
    assert np.abs(tools.getcubeplacement(solver)[9:] - place[1]).max() == 0
    assert np.abs(tools.getcubeplacement(solver, "LARM_HOOK")[9:] - (place[1] + [0, 0.05, 0])).max() < 1e-15
    assert tools.collision(solver, q0) is False
    P = np.concatenate([np.eye(3).reshape(9), place[1]])[None]
    d_ref = c_oracle.scene_distance(table_c, scene_c, q0[None], P, mode=1)[0]
    d = tools.distanceToObstacle(solver, q0)
    assert abs(d - d_ref) < 1e-5 and d > 0
    assert tools.distanceToObstacle(solver, np.zeros(15)) == 0.0               # hands inside the table at q0
    q_bad = q0.copy(); q_bad[3] = 2.0
    assert tools.jointlimitsviolated(solver, q_bad) and not tools.jointlimitsviolated(solver, q0)
    assert abs(tools.jointlimitscost(solver, q_bad) - (2.0 - table.upper[3])) < 1e-12
    assert np.array_equal(tools.projecttojointlimits(solver, q_bad), np.minimum(np.maximum(table.lower, q_bad), table.upper))


def test_success_flag_agreement_fp32(solver, table_c, scene_c, c_oracle):
    # north_star: success flags agree on >= 99.9 % with collision() applied identically to both outputs.  fp32 GPU
    # (solve + collision on the device) against the fp64 oracle of the whole predicate, 384 workspace problems;
    # one borderline problem is 0.26 %, so the assertion allows a single disagreement
    from conftest import make_poses
    n = 384
    P = make_poses(n, 314)
    _, oko, _ = c_oracle.solve_success(table_c, scene_c, np.zeros((n, 15)), P)
    pose = _t(P, torch.float32).t().contiguous(); q0 = torch.zeros((15, n), device="cuda:0")
    for mode in (False, True):
        _, succ, _, _, _ = solver.solve_success_soa(q0, pose, descend_while_colliding=mode)
        agree = (succ.bool().cpu().numpy() == oko).sum()
        assert agree >= n - 1, (mode, agree)
    assert 0.2 < oko.mean() < 0.7


@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-8), (torch.float32, 2e-3)])
def test_bezier_fit_kernel_matches_the_host_fit(solver, dtype, tol):
    # maketraj's least-squares fit (control.py:63-195) for many paths in one launch (gik_bezier_fit_*) against the numpy
    # closed form of trajectory.maketraj: control points, the pinned ends, the residual cost and the acceptance flag
    from gik_b200.trajectory import maketraj, maketraj_batch, fit_operands
    rng = np.random.default_rng(2)
    N, n_points, dim = 301, 37, 15                                      # not a multiple of the warps per block
    q0 = rng.normal(size=(N, dim)) * 0.2; q1 = rng.normal(size=(N, dim)) * 0.2
    t = np.linspace(0, 1, n_points)[None, :, None]
    paths = q0[:, None, :] * (1 - t) + q1[:, None, :] * t + 0.05 * np.sin(3 * np.pi * t) * rng.normal(size=(N, 1, dim))
    paths[:, 0], paths[:, -1] = q0, q1
    P, cost = maketraj_batch(_t(q0, dtype), _t(q1, dtype), _t(paths, dtype), solver=solver)
    assert P.shape == (N, 21, dim) and cost.shape == (N,) and P.is_cuda
    P = P.double().cpu().numpy(); cost = cost.double().cpu().numpy()
    assert np.abs(P[:, :3] - q0[:, None]).max() < 1e-6 and np.abs(P[:, -3:] - q1[:, None]).max() < 1e-6   # P0 = P1 = P2 = q0, ...
    for i in range(0, N, 7):
        (q, _, _), ok = maketraj(q0[i], q1[i], paths[i], 15.0)
        ref = np.array(q.control_points_)                                  # the Bernstein design matrix is ill-conditioned
        assert np.abs(P[i] - ref).max() < tol * max(1.0, np.abs(ref).max())
        pinv, basis, w0, w1 = fit_operands(20, n_points)
        rhs = paths[i] - w0[:, None] * q0[i] - w1[:, None] * q1[i]
        c_ref = ((basis @ ref[3:-3] - rhs) ** 2).sum()
        assert abs(cost[i] - c_ref) < max(tol, 1e-6) * max(1.0, c_ref)
        assert ok == bool(c_ref < 0.15)
    # other sizes: a short path, a lower degree, an empty batch
    P2, c2 = maketraj_batch(_t(q0[:5], dtype), _t(q1[:5], dtype), _t(paths[:5, ::4], dtype), degree=8, solver=solver)
    (q, _, _), _ = maketraj(q0[0], q1[0], paths[0, ::4], 1.0, degree=8)
    assert P2.shape == (5, 9, dim) and np.abs(P2[0].double().cpu().numpy() - np.array(q.control_points_)).max() < tol
    P3, c3 = maketraj_batch(_t(q0[:0], dtype), _t(q1[:0], dtype), _t(paths[:0], dtype), solver=solver)
    assert P3.shape == (0, 21, dim) and c3.shape == (0,)


def test_restarts_with_the_collision_term(solver):
    # computeqgrasppose_batch(restarts=R, collision=True): every candidate gets the full predicate, the selection runs over
    # the SUCCESSFUL candidates -- a returned success is converged and collision-free, and a placement whose restart 0
    # (the caller's q_init) succeeds is never lost to a colliding restart with a smaller residual
    import gik_b200
    from conftest import make_poses
    n, R = 96, 6
    P = _t(make_poses(n, 77), torch.float64)
    g = torch.Generator(device="cuda:0").manual_seed(3)
    q1, ok1 = gik_b200.computeqgrasppose_batch(solver, torch.zeros(15), P, dtype=torch.float64, collision=True)
    qR, okR, info = gik_b200.computeqgrasppose_batch(solver, torch.zeros(15), P, dtype=torch.float64, collision=True, restarts=R,
                                                     generator=g, return_info=True)
    assert qR.shape == (n, 15) and okR.shape == (n,) and info.which.shape == (n,)
    assert (okR | ~ok1).all() and okR.sum() >= ok1.sum()                 # restart 0 is the single-start problem
    idx = torch.nonzero(okR).flatten()
    assert idx.numel() >= 10
    assert (info.resid[idx] < 1e-3).all()
    col = solver.collision_soa(qR[idx].t().contiguous(), P[idx].t().contiguous()).bool()
    assert not col.any()
    # without the collision term more placements "succeed" (converged but colliding ones): the term is really applied
    _, okc = gik_b200.computeqgrasppose_batch(solver, torch.zeros(15), P, dtype=torch.float64, restarts=R,
                                              generator=torch.Generator(device="cuda:0").manual_seed(3))
    assert okc.sum() > okR.sum()
