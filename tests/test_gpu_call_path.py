"""The call path from GraspIK to the kernels: `solver.launches` (gik_launch_count) counts exactly the library kernels a
call puts on the GPU, as the profiler sees them, and every tensor check of ops.py raises before anything is launched."""
import json

import pytest
import torch

from conftest import make_poses

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
F64 = torch.float64


@pytest.fixture(scope="module")
def solver(table):
    import gik_b200
    s = gik_b200.GraspIK(table, DEV).attach_scene()
    yield s
    s.close()


@pytest.fixture(scope="module")
def inp(solver):
    """Small valid inputs of every GraspIK method that launches (fp64)."""
    from gik_b200 import trajectory
    g = torch.Generator(device=DEV).manual_seed(3)
    d = dict(n=256, n_place=64, n_restart=4, E=32, S=4)
    d["q"] = torch.zeros((15, d["n"]), dtype=F64, device=DEV)
    d["pose"] = torch.as_tensor(make_poses(d["n"], 5), dtype=F64, device=DEV).t().contiguous()
    d["q_rows"], d["pose_rows"] = torch.zeros(15, dtype=F64), torch.as_tensor(make_poses(d["n"], 5))
    d["sel"] = torch.arange(0, d["n"], 3, device=DEV)
    d["res"] = solver.solve_soa(d["q"], d["pose"])
    E = d["E"]
    d["edge"] = (d["q"][:, :E].contiguous(), d["pose"][:, :E].contiguous(), d["pose"][:, E:2 * E].contiguous(),
                 torch.full((E,), 3, dtype=torch.int32, device=DEV))
    d["dests"] = [torch.zeros((15, 2 * d["n"]), dtype=F64, device=DEV) for _ in range(2)]
    d["conv_dests"] = [torch.zeros((2 * d["n"],), dtype=torch.uint8, device=DEV) for _ in range(2)]
    # Bezier fit, check and refinement: degree-20 curves through noisy paths of 50 points
    N, n_points = 16, 50
    d["fit_ops"] = trajectory.fit_operands(20, n_points)
    d["path"] = 0.1 * torch.rand((N, n_points, 15), dtype=F64, device=DEV, generator=g)
    d["ctrl"] = solver.bezier_fit(d["path"][:, 0], d["path"][:, -1], d["path"], *d["fit_ops"])[0]
    d["weights"] = trajectory.sample_weights(21, 64)
    # four trees (two queries) of 8 vertices in a chain 0 <- 1 <- ... <- 7
    T, cap = 4, 16
    d["tree"] = (torch.rand((T, 15, cap), dtype=F64, device=DEV, generator=g),
                 torch.rand((T, 12, cap), dtype=F64, device=DEV, generator=g),
                 (torch.arange(cap, dtype=torch.int32, device=DEV) - 1).repeat(T, 1).contiguous(),
                 torch.full((T,), 8, dtype=torch.int32, device=DEV))
    d["targets"] = torch.rand((10, 15), dtype=F64, device=DEV, generator=g)
    d["target_tree"] = torch.arange(10, dtype=torch.int32, device=DEV) % T
    d["grow"] = (torch.arange(T, dtype=torch.int32, device=DEV), torch.full((T,), 7, dtype=torch.int32, device=DEV),
                 d["q"][:, :T].contiguous(), d["pose"][:, :T].contiguous(), d["pose"][:, T:2 * T].contiguous(),
                 torch.full((T,), 3, dtype=torch.int32, device=DEV), torch.full((T,), 2, dtype=torch.int32, device=DEV),
                 torch.rand((3, 15, T), dtype=F64, device=DEV, generator=g))
    d["ends"] = (torch.tensor([3, 2], dtype=torch.int32, device=DEV), torch.tensor([1, 4], dtype=torch.int32, device=DEV))
    verts, cubes, parent, n_verts = d["tree"]
    d["paths"] = solver.tree_paths(verts, cubes, parent, n_verts, *d["ends"])      # rows 6 and 8
    i32 = lambda a: torch.tensor(a, dtype=torch.int32, device=DEV)             # noqa: E731
    d["cands"] = (i32([[0, 1], [0, 2]]), i32([[3, 4], [4, 6]]), i32([[2, 2], [2, 2]]), i32([[2, 0], [2, 2]]),
                  torch.rand((3, 15, 4), dtype=F64, device=DEV, generator=g))
    torch.cuda.synchronize()
    return d


def _tree_grow(solver, d, **bad):
    verts, cubes, parent, n_verts = (bad.get(k, v) for k, v in zip(("verts", "cubes", "parent", "n_verts"), d["tree"]))
    overflow = bad.get("overflow", torch.zeros(4, dtype=torch.uint8, device=DEV))
    grow = [bad.get(k, v) for k, v in zip(("edge_tree", "near", "q_start", "pose_a", "pose_b", "num_steps", "n_valid",
                                           "q_path"), d["grow"])]
    return solver.tree_grow(verts.clone(), cubes.clone(), parent.clone(), n_verts.clone(), overflow, *grow)


def _shortcut(solver, d, **bad):
    q, cube, off = (bad.get(k, v) for k, v in zip(("q", "cube", "offsets"), d["paths"]))
    cands = [bad.get(k, v) for k, v in zip(("pair_i", "pair_j", "num_steps", "n_valid", "q_path"), d["cands"])]
    return solver.path_shortcut(q, cube, off, *cands, join_tol=0.5)


def _scatter(solver, d, out=None, pose=None):
    return solver.solve_scatter_soa(d["q"], d["pose"] if pose is None else pose, [t.data_ptr() for t in d["dests"]],
                                    [t.data_ptr() for t in d["conv_dests"]], 2 * d["n"], d["n"], out=out)


CALLS = {
    "fk_soa": lambda s, d: s.fk_soa(d["q"]),
    "jac_soa": lambda s, d: s.jac_soa(d["q"]),
    "solve_soa": lambda s, d: s.solve_soa(d["q"], d["pose"]),
    "solve_host": lambda s, d: s.solve_host(d["q_rows"], d["pose_rows"], dtype=F64),
    "solve_scatter_soa": _scatter,
    "best_of_soa": lambda s, d: s.best_of_soa(d["res"][0], d["res"][1], d["res"][3], d["n_place"], d["n_restart"]),
    "project_edges_soa": lambda s, d: s.project_edges_soa(*d["edge"], d["S"]),
    "collision_soa": lambda s, d: s.collision_soa(d["q"], d["pose"]),
    "collision_soa_sel": lambda s, d: s.collision_soa(d["q"], d["pose"], sel=d["sel"]),
    "clearance_soa": lambda s, d: s.clearance_soa(d["q"], d["pose"]),
    "obstacle_distance_soa": lambda s, d: s.obstacle_distance_soa(d["q"]),
    "cube_collision_soa": lambda s, d: s.cube_collision_soa(d["pose"]),
    "solve_success_soa": lambda s, d: s.solve_success_soa(d["q"], d["pose"]),
    "solve_success_soa_no_descend": lambda s, d: s.solve_success_soa(d["q"], d["pose"], descend_while_colliding=False),
    "bezier_fit": lambda s, d: s.bezier_fit(d["path"][:, 0], d["path"][:, -1], d["path"], *d["fit_ops"]),
    "check_trajectories": lambda s, d: s.check_trajectories(d["ctrl"], d["weights"], limit_tol=1e-6, grasp_tol=1e-2),
    "refine_trajectories": lambda s, d: s.refine_trajectories(d["ctrl"], d["weights"], max_iters=2, tol=5e-3, damping=1e-3),
    "tree_nearest": lambda s, d: s.tree_nearest(d["tree"][0], d["tree"][3], d["targets"], d["target_tree"]),
    "tree_grow": _tree_grow,
    "tree_paths": lambda s, d: s.tree_paths(*d["tree"][:4], *d["ends"]),
    "path_shortcut": _shortcut,
}


@pytest.mark.parametrize("call", sorted(CALLS))
def test_launch_count_matches_the_profiler(solver, inp, call, tmp_path):
    from torch.profiler import ProfilerActivity, profile
    before = solver.launches
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        CALLS[call](solver, inp)
        torch.cuda.synchronize()
    counted = solver.launches - before
    trace = tmp_path / "trace.json"
    prof.export_chrome_trace(str(trace))
    kernels = [e["name"] for e in json.load(open(trace))["traceEvents"] if e.get("cat") == "kernel" and "gik_" in e["name"]]
    assert len(kernels) >= 1, call
    assert counted == len(kernels), (call, kernels)


def _nc(t):
    """The same values, not contiguous."""
    return torch.empty((*t.shape[:-1], 2 * t.shape[-1]), dtype=t.dtype, device=t.device)[..., ::2].copy_(t)


def _bad_calls(d):
    """(name, call, exception): one wrong shape, dtype, device or layout per tensor check of ops.py."""
    q, pose, n = d["q"], d["pose"], d["n"]
    f32 = lambda t: t.float()                                                   # noqa: E731
    res = d["res"]
    out = lambda **b: tuple(b.get(k, v) for k, v in zip(("q", "conv", "iters", "resid"), (torch.empty_like(q),) + res[1:]))  # noqa: E731
    best = lambda s, q_=res[0], c=res[1], r=res[3]: s.best_of_soa(q_, c, r, d["n_place"], d["n_restart"])  # noqa: E731
    edge = lambda s, i, t, **kw: s.project_edges_soa(*[t if k == i else a for k, a in enumerate(d["edge"])], d["S"], **kw)  # noqa: E731
    E, S = d["E"], d["S"]
    eout = lambda **b: tuple(b.get(k, v) for k, v in zip(("path", "nv", "itt"), (  # noqa: E731
        torch.zeros((S, 15, E), dtype=F64, device=DEV), torch.empty(E, dtype=torch.int32, device=DEV),
        torch.empty(E, dtype=torch.int32, device=DEV))))
    pinv, basis, w0, w1 = d["fit_ops"]
    P = d["path"]
    fit = lambda s, q0=P[:, 0], path=P, w=w0: s.bezier_fit(q0, P[:, -1], path, pinv, basis, w, w1)  # noqa: E731
    chk = lambda s, c=d["ctrl"], w=d["weights"]: s.check_trajectories(c, w, limit_tol=1e-6, grasp_tol=1e-2)  # noqa: E731
    ref = lambda s, c=d["ctrl"], w=d["weights"]: s.refine_trajectories(c, w, max_iters=2, tol=5e-3, damping=1e-3)  # noqa: E731
    verts, cubes, parent, n_verts = d["tree"]
    return [
        ("fk q rows", lambda s: s.fk_soa(q[:14]), ValueError),
        ("fk q on the host", lambda s: s.fk_soa(q.cpu()), ValueError),
        ("jac q 3-D", lambda s: s.jac_soa(q[None]), ValueError),
        ("solve q rows", lambda s: s.solve_soa(q[:14], pose), ValueError),
        ("solve pose columns", lambda s: s.solve_soa(q, pose[:, 1:]), ValueError),
        ("solve pose dtype", lambda s: s.solve_soa(q, f32(pose)), TypeError),
        ("solve q layout", lambda s: s.solve_soa(_nc(q), pose), ValueError),
        ("solve out q shape", lambda s: s.solve_soa(q, pose, out=out(q=torch.empty_like(q[:, 1:]))), ValueError),
        ("solve out conv dtype", lambda s: s.solve_soa(q, pose, out=out(conv=res[2])), TypeError),
        ("solve out iters shape", lambda s: s.solve_soa(q, pose, out=out(iters=res[2][1:])), ValueError),
        ("solve out resid layout", lambda s: s.solve_soa(q, pose, out=out(resid=_nc(res[3]))), ValueError),
        ("scatter pose rows", lambda s: _scatter(s, d, pose=pose[:11]), ValueError),
        ("scatter out iters dtype", lambda s: _scatter(s, d, out=(res[1], res[3])), TypeError),
        ("scatter out resid shape", lambda s: _scatter(s, d, out=(res[2], res[3][:1])), ValueError),
        ("best_of q columns", lambda s: best(s, q_=res[0][:, 1:]), ValueError),
        ("best_of conv dtype", lambda s: best(s, c=res[2]), TypeError),
        ("best_of resid shape", lambda s: best(s, r=res[3][0]), ValueError),
        ("edges q_start rows", lambda s: edge(s, 0, d["edge"][0][:14]), ValueError),
        ("edges pose_a columns", lambda s: edge(s, 1, d["edge"][1][:, 1:]), ValueError),
        ("edges pose_b dtype", lambda s: edge(s, 2, f32(d["edge"][2])), TypeError),
        ("edges num_steps dtype", lambda s: edge(s, 3, d["edge"][3].long()), TypeError),
        ("edges out q_path shape", lambda s: edge(s, 3, d["edge"][3], out=eout(path=torch.zeros((S, 15, E + 1), dtype=F64, device=DEV))), ValueError),
        ("edges out n_valid dtype", lambda s: edge(s, 3, d["edge"][3], out=eout(nv=torch.empty(E, dtype=torch.int64, device=DEV))), TypeError),
        ("collision q rows", lambda s: s.collision_soa(q[:14]), ValueError),
        ("collision cube columns", lambda s: s.collision_soa(q, pose[:, 1:]), ValueError),
        ("collision sel 2-D", lambda s: s.collision_soa(q, pose, sel=d["sel"][None]), ValueError),
        ("clearance cube rows", lambda s: s.clearance_soa(q, pose[:11]), ValueError),
        ("distance q on the host", lambda s: s.obstacle_distance_soa(q.cpu()), ValueError),
        ("cube collision rows", lambda s: s.cube_collision_soa(pose[:11]), ValueError),
        ("success pose columns", lambda s: s.solve_success_soa(q, pose[:, 1:]), ValueError),
        ("success pose dtype", lambda s: s.solve_success_soa(q, f32(pose)), TypeError),
        ("bezier w0 length", lambda s: fit(s, w=w0[1:]), ValueError),
        ("bezier q0 dtype", lambda s: fit(s, q0=f32(P[:, 0])), TypeError),
        ("bezier path 2-D", lambda s: fit(s, path=P[0]), ValueError),
        ("check ctrl joints", lambda s: chk(s, c=d["ctrl"][..., :14]), ValueError),
        ("check weights columns", lambda s: chk(s, w=d["weights"][:, 1:]), ValueError),
        ("refine ctrl on the host", lambda s: ref(s, c=d["ctrl"].cpu()), ValueError),
        ("refine weights columns", lambda s: ref(s, w=d["weights"][:, 1:]), ValueError),
        ("nearest n_verts dtype", lambda s: s.tree_nearest(verts, n_verts.long(), d["targets"], d["target_tree"]), TypeError),
        ("nearest targets joints", lambda s: s.tree_nearest(verts, n_verts, d["targets"][:, 1:], d["target_tree"]), ValueError),
        ("nearest verts layout", lambda s: s.tree_nearest(_nc(verts), n_verts, d["targets"], d["target_tree"]), ValueError),
        ("grow overflow dtype", lambda s: _tree_grow(s, d, overflow=torch.zeros(4, dtype=torch.int32, device=DEV)), TypeError),
        ("grow q_path edges", lambda s: _tree_grow(s, d, q_path=d["grow"][7][..., 1:]), ValueError),
        ("grow parent shape", lambda s: _tree_grow(s, d, parent=parent[:, 1:]), ValueError),
        ("grow near dtype", lambda s: _tree_grow(s, d, near=d["grow"][1].long()), TypeError),
        ("paths start_end shape", lambda s: s.tree_paths(verts, cubes, parent, n_verts, d["ends"][0][:1], d["ends"][1]), ValueError),
        ("paths cubes dtype", lambda s: s.tree_paths(verts, f32(cubes), parent, n_verts, *d["ends"]), TypeError),
        ("shortcut offsets dtype", lambda s: _shortcut(s, d, offsets=d["paths"][2].int()), TypeError),
        ("shortcut cube rows", lambda s: _shortcut(s, d, cube=d["paths"][1][1:]), ValueError),
        ("shortcut pair_j shape", lambda s: _shortcut(s, d, pair_j=d["cands"][1][:, :1]), ValueError),
        ("shortcut q_path candidates", lambda s: _shortcut(s, d, q_path=d["cands"][4][..., :3]), ValueError),
    ]


def test_bad_tensors_raise_before_any_launch(solver, inp):
    for name, call, exc in _bad_calls(inp):
        before = solver.launches
        with pytest.raises(exc):
            call(solver)
        torch.cuda.synchronize()
        assert solver.launches == before, name
