"""Batched counterparts of the two IK call sites in the reference's `path.py`:

  * `sample_cube_placement` (path.py:27-67): uniform placement in a box, IK from `robot.q0`   -> `sample_grasp_poses_batch`
  * `project_path`         (path.py:125-163): warm-started IK along an interpolated cube edge -> `project_edges_batch`

plus `project_path`, a drop-in with the reference's signature and return value for ONE edge, and `computepath`, the
RRT-connect driver (path.py:186-278) with the reference's tree logic on the host and its two IK call sites batched:
samples come from a pool validated `sample_batch` at a time, and `expand` tree extensions per iteration go through ONE
launch of the edge kernel.  The cube-vs-scene collision test (path.py:51-54, 144-149), the robot collision term of the
grasp predicate and the obstacle-distance filter (path.py:61-62) run in the collision kernels on the attached scene
("scene"), or as host callables the caller passes in.

Deliberate differences from the reference loop (never unsafe: every returned vertex passed every reference test):
  * an edge is marched to the first NON-CONVERGED step and THEN cut at the first step whose cube or robot collides.  The
    reference tests the cube before the IK of each step and, for a converged-but-colliding iterate, keeps descending
    (inverse_geometry.py:70) -- it may find a free q there and carry on with it as the next warm start, so its edges
    can be longer than the ones returned here, never shorter;
  * the sampler abandons stalled descents early (GIK_F_EARLY_STOP) and skips the extra descent on colliding samples:
    accepted samples satisfy the reference's acceptance rule; which candidates are accepted can differ;
  * the batched planner (planner.computepath_batch) draws a fixed number of candidates (16) per extension slot and
    iteration instead of rejecting until a valid sample turns up: a slot whose candidates all fail stays idle for that
    iteration -- no edge, and no connect test for that slot."""
from __future__ import annotations

import numpy as np
import torch

from .inverse_geometry import _pose_to_array, solver_for
from .ops import DT, EPSILON, MAX_ITERS, as_pose12

Z_MIN, Z_MAX = 1.05, 1.4          # path.py:37
STEP_SIZE = 0.025                 # path.py:125, 203-206


def sample_cube_placements(n, p0, p1, *, z_range=(Z_MIN, Z_MAX), device="cuda", dtype=torch.float32, generator=None):
    """n translations uniform in the box of path.py:35-45: x, y between the two given cube translations, z in
    `z_range`; identity rotation (path.py:47).  `p0` / `p1` are one placement each (translation last), or per-row
    placements [n,3|12] (tensors or arrays): row i is then drawn from its own box.  Returns [n,3]."""
    if getattr(p0, "ndim", 1) == 2:
        a = torch.as_tensor(p0, device=device)[:, -3:].to(dtype)
        b = torch.as_tensor(p1, device=device)[:, -3:].to(dtype)
        z = torch.tensor(z_range, dtype=dtype, device=device).expand(a.shape[0], 2)
        lo = torch.cat([torch.minimum(a[:, :2], b[:, :2]), z[:, :1]], dim=1)
        hi = torch.cat([torch.maximum(a[:, :2], b[:, :2]), z[:, 1:]], dim=1)
    else:
        p0 = np.asarray(p0, float).reshape(-1)[-3:]
        p1 = np.asarray(p1, float).reshape(-1)[-3:]
        lo = torch.tensor([min(p0[0], p1[0]), min(p0[1], p1[1]), z_range[0]], dtype=dtype, device=device)
        hi = torch.tensor([max(p0[0], p1[0]), max(p0[1], p1[1]), z_range[1]], dtype=dtype, device=device)
    u = torch.rand((n, 3), dtype=dtype, device=device, generator=generator)
    return lo + u * (hi - lo)


MIN_OBSTACLE_DISTANCE = 0.04      # path.py:32


def sample_grasp_poses_batch(robot, n, cubeplacementq0, cubeplacementqgoal, *, q0=None, dtype=torch.float32,
                             generator=None, cube_collision="scene", collision="scene",
                             min_obstacle_distance=MIN_OBSTACLE_DISTANCE, eps=EPSILON, dt=DT, max_iters=MAX_ITERS,
                             damping=0.0):
    """n candidate samples of path.sample_cube_placement (path.py:27-67) evaluated at once, every filter on the GPU:
      1. placement uniform in the box of path.py:35-45, identity rotation (:47);
      2. reject if the cube collides with the table / obstacle (:50-54)          -> gik_cube_collision_*
      3. IK from `q0` (robot.q0 = zeros, :57) with the reference's success flag  -> gik_solve_* + gik_collision_*
      4. reject if distanceToObstacle(robot, q) < min_obstacle_distance (:61-62) -> gik_clearance_*
    Returns (q [n,nq], placements [n,3], ok bool [n]).  `cube_collision` / `collision`: "scene" = the attached
    collision scene, None = skip that filter, or a callable (placements [n,3] -> bool [n]) / (q ndarray -> bool)."""
    solver = solver_for(robot)
    a = _pose_to_array(cubeplacementq0)
    b = _pose_to_array(cubeplacementqgoal)
    pl = sample_cube_placements(n, a[9:], b[9:], device=solver.device, dtype=dtype, generator=generator)
    qi = torch.zeros(solver.nq, dtype=dtype, device=solver.device) if q0 is None else torch.as_tensor(q0, device=solver.device).to(dtype)
    q, ok = _grasp_filter(solver, pl, qi, dtype, cube_collision=cube_collision, collision=collision,
                          min_obstacle_distance=min_obstacle_distance, eps=eps, dt=dt, max_iters=max_iters, damping=damping)
    return q, pl, ok


def _grasp_filter(solver, pl, qi, dtype, *, cube_collision="scene", collision="scene",
                  min_obstacle_distance=MIN_OBSTACLE_DISTANCE, eps=EPSILON, dt=DT, max_iters=MAX_ITERS, damping=0.0):
    """Steps 2-4 of sample_grasp_poses_batch on the placements pl [n,3] with IK from qi [nq]: cube collision, IK with
    the success predicate, clearance.  Returns (q [n,nq], ok bool [n]).  Shared with the batched planner's sampler."""
    n = pl.shape[0]
    p12 = as_pose12(pl, dtype=dtype, device=solver.device)
    pose_soa = p12.t().contiguous()
    if collision == "scene":
        # a failed sample is rejected either way: the reference's extra descent on converged-but-colliding samples is
        # skipped and stalled solves are abandoned early (GIK_F_EARLY_STOP).  Every ACCEPTED sample satisfies the
        # reference's acceptance rule with the reference's q; a few candidates the reference would still have accepted
        # (late convergers at the rim of the workspace: 2 in 10^6 measured; collisions freed by further descent) are
        # rejected here -- the planner only needs an i.i.d. stream of valid samples
        q_soa, succ, _, _, _ = solver.solve_success_soa(qi.unsqueeze(1).expand(solver.nq, n).contiguous(), pose_soa, eps=eps,
                                                        dt=dt, max_iters=max_iters, damping=damping,
                                                        descend_while_colliding=False, early_stop=True)
        ok = succ.bool()
        if min_obstacle_distance is not None and min_obstacle_distance > 0:
            ok &= solver.clearance_soa(q_soa, pose_soa, min_obstacle_distance).bool()
        q = q_soa.t()
    else:
        q, ok = solver.solve(qi, pl, dtype=dtype, eps=eps, dt=dt, max_iters=max_iters, damping=damping)
        if callable(collision):
            from .inverse_geometry import apply_collision
            ok = apply_collision(q, ok, collision)
    if cube_collision == "scene":
        ok = ok & ~solver.cube_collision_soa(pose_soa).bool()
    elif callable(cube_collision):
        ok = ok & ~torch.as_tensor(cube_collision(pl), device=solver.device).bool()
    return q, ok


def edge_num_steps(cube_a12: torch.Tensor, cube_b12: torch.Tensor, step_size=STEP_SIZE) -> torch.Tensor:
    """num_steps = int(||p_a - p_b|| / step_size) + 1   (path.py:129-130)."""
    d = (cube_a12[:, 9:].double() - cube_b12[:, 9:].double()).norm(dim=1)
    return (torch.floor(d / step_size).to(torch.int32) + 1)


def project_edges_batch(robot, q_start, cube_a, cube_b, *, num_steps=None, step_size=STEP_SIZE, max_steps=None,
                        dtype=torch.float32, eps=EPSILON, dt=DT, max_iters=MAX_ITERS, damping=0.0,
                        return_info=False, scene_tests=False):
    """E edges marched at once.  q_start [E,nq]; cube_a / cube_b [E,12|4x4|7|3]; num_steps int [E] (default from
    `step_size` as in the reference).  Returns (q_path [E,S,nq], n_valid int32 [E]) where q_path[e, k] is the
    configuration for placement Interpolate(a, b, (k+1)/num_steps[e]) and n_valid[e] counts the steps before the
    first failure (path.py:153-156); entries beyond n_valid are zero.  `scene_tests=True` also applies, for every edge at
    once, the two collision tests of the reference loop -- the cube against the table / obstacle at each interpolated
    placement (path.py:144-149) and the robot collision term of the grasp predicate -- and cuts each edge at its first
    failing step."""
    solver = solver_for(robot)
    dev = solver.device
    a12 = as_pose12(cube_a, dtype=dtype, device=dev)
    b12 = as_pose12(cube_b, dtype=dtype, device=dev, batch=a12.shape[0])
    E = a12.shape[0]
    qs = torch.as_tensor(q_start, device=dev).to(dtype)
    if qs.dim() == 1:
        qs = qs.unsqueeze(0).expand(E, solver.nq)
    if num_steps is None:
        ns = edge_num_steps(a12, b12, step_size)
    else:
        ns = torch.as_tensor(num_steps, device=dev).to(torch.int32).reshape(-1)
        if ns.numel() == 1:
            ns = ns.expand(E).contiguous()
    if max_steps is None:
        max_steps = int(ns.max().item()) if E else 0     # host sync: pass max_steps to avoid it
    path, nv, itt = solver.project_edges_soa(qs.t().contiguous(), a12.t().contiguous(), b12.t().contiguous(),
                                             ns.contiguous(), max_steps, eps=eps, dt=dt, max_iters=max_iters,
                                             damping=damping)
    if scene_tests and E and max_steps:
        nv = _cut_at_first_collision(solver, path, nv, a12, b12, ns, max_steps)
    out = (path.permute(2, 0, 1), nv)
    if return_info:
        out = out + (itt,)
    return out


def _cut_at_first_collision(solver, path, nv, a12, b12, ns, S, dense=False):
    """path [S][nq][E] (zero beyond n_valid), nv [E] -> nv cut at the first step whose cube placement or robot
    configuration collides with the attached scene; rows beyond the new nv are zeroed.  `dense=True` tests all S steps
    of every edge and masks the result instead of gathering the valid ones first: more collision work, no host
    synchronisation (the gather sizes its output); same result."""
    solver._need_scene()
    E = a12.shape[0]
    dev = a12.device
    k = torch.arange(S, device=dev)
    valid = k[None, :] < nv[:, None]                                            # [E,S]
    if dense:
        e_idx = torch.arange(E, device=dev).repeat_interleave(S)
        k_idx = k.repeat(E)
    else:
        e_idx, k_idx = torch.nonzero(valid, as_tuple=True)
    bad = torch.zeros((E, S), dtype=torch.bool, device=dev)
    if e_idx.numel():
        # (dense: the clamps keep the unused steps' placements finite; a valid step's alpha is unchanged)
        alpha = ((k_idx + 1).to(a12.dtype) / ns[e_idx].clamp_min(1).to(a12.dtype)).clamp(max=1.0)
        poses = se3_interpolate(a12[e_idx], b12[e_idx], alpha).t().contiguous()   # [12][M]
        q = path[k_idx, :, e_idx].t().contiguous()                                # [nq][M]
        hit = solver.cube_collision_soa(poses).bool() | solver.collision_soa(q, poses).bool()
        if dense:
            bad = hit.reshape(E, S) & valid
        else:
            bad[e_idx, k_idx] = hit
    first_bad = torch.where(bad.any(dim=1), bad.to(torch.int32).argmax(dim=1), torch.full((E,), S, device=dev)).to(nv.dtype)
    nv_new = torch.minimum(nv, first_bad)
    path.mul_((k[None, :] < nv_new[:, None]).t()[:, None, :].to(path.dtype))      # zero the rows that were cut
    return nv_new


def project_path(robot, cube, q_curr, cube_curr, cube_rand, step_size=STEP_SIZE, viz=None, *, cube_collision=None,
                 collision=None, dtype=torch.float64):
    """Drop-in for path.project_path (path.py:125-163), one edge: returns (robot_path, cube_path), both starting
    with the given q / placement.  The march itself (SE3.Interpolate, warm-started IK, stop at the first non-converged
    step) is ONE launch of the edge kernel; the two collision tests of the reference loop -- the cube against the
    table / obstacle (path.py:144-149) and the robot (the collision term of computeqgrasppose's predicate) -- are then
    applied to all steps at once and the path is cut at the first step that fails either.
    `cube_collision` / `collision`: None = no test, "scene" = the GPU kernels on the attached scene, or host callables
    (pose12 -> bool) / (q -> bool)."""
    solver = solver_for(robot, cube)
    a = _pose_to_array(cube_curr)
    b = _pose_to_array(cube_rand)
    num_steps = int(np.linalg.norm(a[9:] - b[9:]) / step_size) + 1
    q_path, nv, = project_edges_batch(solver, np.asarray(q_curr, float), a[None], b[None], num_steps=[num_steps],
                                      max_steps=num_steps, dtype=dtype)
    n_ok = int(nv[0].item())
    qs = q_path[0].double().cpu().numpy()
    robot_path, cube_path = [q_curr], [cube_curr]
    if n_ok == 0:
        return robot_path, cube_path
    # placements along the edge, same interpolation as the kernel, for the returned cube_path
    A = torch.from_numpy(a)[None].expand(n_ok, 12)
    B = torch.from_numpy(b)[None].expand(n_ok, 12)
    alphas = torch.arange(1, n_ok + 1, dtype=torch.float64) / num_steps
    poses = se3_interpolate(A, B, alphas)
    bad = np.zeros(n_ok, bool)
    if cube_collision == "scene" or collision == "scene":
        pd = poses.to(solver.device, dtype).t().contiguous()
        if cube_collision == "scene":
            bad |= solver.cube_collision_soa(pd).bool().cpu().numpy()
        if collision == "scene":
            qd = q_path[0, :n_ok].to(dtype).t().contiguous()
            bad |= solver.collision_soa(qd, pd).bool().cpu().numpy()
    poses = poses.numpy()
    for k in range(n_ok):
        if bad[k] or (callable(cube_collision) and cube_collision(poses[k])) or (callable(collision) and collision(qs[k])):
            break
        robot_path.append(qs[k].copy())
        cube_path.append(_like(cube_curr, poses[k]))
    return robot_path, cube_path


# ------------------------------------------------------------------------------------------------------
# RRT-connect driver (path.computepath, path.py:194-278): the reference's tree logic, with its two IK call sites
# replaced by the batched sampler (a pool of pre-validated samples) and the edge kernel.
# ------------------------------------------------------------------------------------------------------
GOAL_TOLERANCE = 0.5        # path.py:202
GOAL_BIAS = 0.1             # path.py:224
MAX_ITERATIONS = 250        # path.py:199
MAX_RETRIES = 10            # path.py:200


class _SamplePool:
    """Stream of valid (q, placement) samples of path.sample_cube_placement, drawn `batch` candidates at a time on the
    GPU.  Taking the next valid sample of an i.i.d. candidate stream is what the reference's rejection loop does."""

    def __init__(self, solver, a, b, dtype, batch, generator, scene):
        self.args = (solver, a, b, dtype, batch, generator, scene)
        self.q, self.pl = [], []

    def next(self):
        solver, a, b, dtype, batch, generator, scene = self.args
        while not self.q:
            q, pl, ok = sample_grasp_poses_batch(solver, batch, a, b, dtype=dtype, generator=generator,
                                                 cube_collision="scene" if scene else None,
                                                 collision="scene" if scene else None)
            idx = torch.nonzero(ok).flatten()
            self.q = list(q[idx].double().cpu().numpy())
            self.pl = list(pl[idx].double().cpu().numpy())
        return self.q.pop(0), self.pl.pop(0)


def _get_path(G, node=-1):
    """path.get_path (path.py:174-183), from any vertex of the tree (the reference always starts at the last one)."""
    path, node = [], G[node]
    while node[0] is not None:
        path.insert(0, node[1])
        node = G[node[0]]
    path.insert(0, G[0][1])
    return path


def _project_batch(solver, q_start, cube_a, cube_b, step_size, dtype, scene):
    """K edges of path.project_path (path.py:125-163) in ONE launch of the edge kernel + one batched pass of the two
    collision tests.  q_start [K][nq], cube_a / cube_b [K][12] (numpy).  Returns per edge (q_seg [m+1,nq], cube_seg
    [m+1,12]): the start vertex followed by the m valid steps, like the reference's (robot_path, cube_path)."""
    q_start = np.asarray(q_start, float); a = np.asarray(cube_a, float); b = np.asarray(cube_b, float)
    K = a.shape[0]
    ns = (np.floor(np.linalg.norm(a[:, 9:] - b[:, 9:], axis=1) / step_size).astype(np.int32) + 1)   # path.py:129-130
    S = int(ns.max())
    q_path, nv = project_edges_batch(solver, q_start, a, b, num_steps=ns, max_steps=S, dtype=dtype, scene_tests=scene)
    qp = q_path.double().cpu().numpy()
    nv = nv.cpu().numpy()
    A = torch.from_numpy(a)[:, None, :].expand(K, S, 12).reshape(-1, 12)
    B = torch.from_numpy(b)[:, None, :].expand(K, S, 12).reshape(-1, 12)
    alpha = (torch.arange(1, S + 1, dtype=torch.float64)[None, :] / torch.from_numpy(ns.astype(np.float64))[:, None]).clamp(max=1.0)
    poses = se3_interpolate(A, B, alpha.reshape(-1)).reshape(K, S, 12).numpy()
    return [(np.vstack([q_start[k][None], qp[k, :nv[k]]]), np.vstack([a[k][None], poses[k, :nv[k]]])) for k in range(K)]


def computepath(qinit, qgoal, cubeplacementq0, cubeplacementqgoal, robot=None, cube=None, *, step_size=STEP_SIZE,
                goal_tolerance=GOAL_TOLERANCE, max_iterations=MAX_ITERATIONS, max_retries=MAX_RETRIES, rng=None,
                generator=None, dtype=torch.float64, sample_batch=512, scene=True, expand=8, return_stats=False):
    """Drop-in for path.computepath (path.py:194-278): bidirectional RRT over cube placements, each new vertex a grasp
    configuration.  Same rules as the reference -- goal bias 0.1, nearest vertex in configuration space, project_path
    towards the sample from the start tree and towards the goal placement from the goal tree, connect when the two new
    configurations are closer than goal_tolerance -- with `expand` extensions per iteration instead of one: `expand`
    targets are drawn, their nearest start-tree vertices are found in one vectorised query, and all `expand` edges (then
    all `expand` goal-tree edges) are projected by ONE launch of the edge kernel each.  An edge's time is the latency of
    its own warm-started chain, so `expand` edges cost what one costs and a query needs ~1/expand of the iterations.
    `expand=1` is the reference loop step for step.  The first extension (lowest index) that connects ends the search.
    `max_iterations` stays the reference's budget of start-tree EXTENSIONS per retry (250), i.e. ceil(250 / expand)
    iterations: this planner connects early in a retry or not at all (the vertex nearest to qgoal in configuration space
    keeps being the one whose straight cube path is blocked), so a retry must not become `expand` times more expensive.
    `robot`: pinocchio RobotWrapper / KinematicTable / GraspIK / None (built-in Nextage); `cube` is unused unless
    `robot` is a pinocchio wrapper.  Returns the list of configurations (empty on failure), like the reference."""
    solver = solver_for(robot, cube)
    if scene:
        solver._need_scene()
    rng = rng if rng is not None else np.random.default_rng()
    qinit, qgoal = np.asarray(qinit, float), np.asarray(qgoal, float)
    a12, b12 = _pose_to_array(cubeplacementq0), _pose_to_array(cubeplacementqgoal)
    pool = _SamplePool(solver, a12, b12, dtype, sample_batch, generator, scene)
    K = max(int(expand), 1)
    stats = {"iterations": 0, "retries": 0, "edges": 0, "vertices": 0, "expand": K}

    def nearest(points, targets):           # KDTree.query of the reference (path.py:186-192): exact nearest neighbours
        P, T = np.asarray(points), np.asarray(targets)
        return ((P[None, :, :] - T[:, None, :]) ** 2).sum(axis=2).argmin(axis=1)

    def grow(G, C, near, segs):             # path.py:241-244: the segment's first vertex is re-added too
        ends = []
        for k, (sq, sc) in enumerate(segs):
            for j in range(len(sq)):
                G.append((len(G) - 1 if j > 0 else int(near[k]), sq[j]))
                C.append(sc[j])
            ends.append(len(G) - 1)
        return ends

    for retry in range(max_retries):
        G_start, G_goal = [(None, qinit)], [(None, qgoal)]
        C_start, C_goal = [a12], [b12]
        for i in range(-(-max_iterations // K)):
            stats["iterations"] += 1
            q_rand, cube_rand = [], []
            for _ in range(K):
                if rng.random() < GOAL_BIAS:
                    q_rand.append(qgoal); cube_rand.append(b12)
                else:
                    q, p = pool.next()
                    q_rand.append(q); cube_rand.append(np.concatenate([np.eye(3).reshape(9), p]))
            ns = nearest([g[1] for g in G_start], q_rand)
            segs = _project_batch(solver, [G_start[j][1] for j in ns], [C_start[j] for j in ns], cube_rand, step_size,
                                  dtype, scene)
            ends_s = grow(G_start, C_start, ns, segs)
            q_new = [sq[-1] for sq, _ in segs]
            ng = nearest([g[1] for g in G_goal], q_new)
            segs2 = _project_batch(solver, [G_goal[j][1] for j in ng], [C_goal[j] for j in ng], [b12] * K, step_size,
                                   dtype, scene)
            ends_g = grow(G_goal, C_goal, ng, segs2)
            stats["edges"] += 2 * K
            for k in range(K):
                if np.linalg.norm(segs2[k][0][-1] - q_new[k]) < goal_tolerance:
                    path = _get_path(G_start, ends_s[k]) + _get_path(G_goal, ends_g[k])[::-1]
                    stats["vertices"] = len(G_start) + len(G_goal)
                    return (path, stats) if return_stats else path
        stats["retries"] += 1
    return ([], stats) if return_stats else []


def _like(template, pose12):
    """Return the placement in the caller's own type when it is a pinocchio SE3, else the 12-vector."""
    if hasattr(template, "rotation") and hasattr(template, "translation"):
        try:
            return type(template)(pose12[:9].reshape(3, 3).copy(), pose12[9:].copy())
        except Exception:
            pass
    return pose12


def se3_interpolate(a12: torch.Tensor, b12: torch.Tensor, alpha) -> torch.Tensor:
    """pin.SE3.Interpolate(A, B, alpha) = A exp6(alpha log6(A^-1 B)) on [B,12] host/device tensors; alpha a float or a
    [B] tensor (bookkeeping for the returned cube paths and the scene tests; the kernel has its own copy in
    gik_core.cuh).  log3 follows pinocchio, including its form for rotations within 1e-2 of pi: |w_i| from the
    diagonal, the sign of w_i from the antisymmetric part.  At exactly pi about an axis that is not a coordinate axis
    the signs are rounding noise in pinocchio too.  log6(A^-1 B) is evaluated in fp64 whatever the input dtype (an
    fp32 log3 cannot resolve the axis near pi) and rounded to the input dtype; exp6 and the product with A run in the
    input dtype, so that an edge without rotation gives the kernel's placements bit for bit.  Returned on the input's
    device."""
    dtype = a12.dtype
    alpha = torch.as_tensor(alpha, dtype=dtype, device=a12.device).reshape(-1, 1)
    Ra, pa = a12[:, :9].reshape(-1, 3, 3), a12[:, 9:]
    Ra64, pa64 = Ra.to(torch.float64), pa.to(torch.float64)
    Rb64, pb64 = b12[:, :9].reshape(-1, 3, 3).to(torch.float64), b12[:, 9:].to(torch.float64)
    R = Ra64.transpose(1, 2) @ Rb64
    p = (Ra64.transpose(1, 2) @ (pb64 - pa64).unsqueeze(-1)).squeeze(-1)
    # log3
    v = torch.stack([R[:, 2, 1] - R[:, 1, 2], R[:, 0, 2] - R[:, 2, 0], R[:, 1, 0] - R[:, 0, 1]], dim=1)
    c = ((R.diagonal(dim1=1, dim2=2).sum(1) - 1) * 0.5).clamp(-1, 1)
    s = 0.5 * v.norm(dim=1)
    th = torch.atan2(s, c)
    fac = torch.where(s > 1e-12, 0.5 * th / s.clamp_min(1e-300), torch.full_like(s, 0.5))
    w = fac.unsqueeze(1) * v
    # near pi, v = 2 sin(theta) u loses the axis to rounding: pinocchio's form, selected without a host synchronisation
    near_pi = (th >= np.pi - 1e-2).unsqueeze(1)
    w_pi = ((R.diagonal(dim1=1, dim2=2) - c.unsqueeze(1)) * (th * th / (1 - c).clamp_min(1)).unsqueeze(1)).clamp_min(0).sqrt()
    w = torch.where(near_pi, torch.where(v > 0, w_pi, -w_pi), w)
    t2 = th * th
    small = t2 < 1e-8
    # (theta/2) cot(theta/2) = (theta/2) (1 + c) / s = (theta/2) s / (1 - c): the second form keeps its accuracy near pi
    half_cot = torch.where(small, torch.ones_like(th),
                           0.5 * th * torch.where(c >= 0, (1 + c) / s.clamp_min(1e-300), s / (1 - c).clamp_min(1e-300)))
    alpha_c = torch.where(small, 1 - t2 / 12, half_cot)
    beta_c = torch.where(small, torch.full_like(th, 1.0 / 12), (1 - alpha_c) / t2.clamp_min(1e-300))
    lin = alpha_c.unsqueeze(1) * p - 0.5 * torch.cross(w, p, dim=1) + (beta_c * (w * p).sum(1)).unsqueeze(1) * w
    # exp6(alpha * [lin; w]) in the input dtype
    lv, lw = alpha * lin.to(dtype), alpha * w.to(dtype)
    t2 = (lw * lw).sum(1)
    t = t2.sqrt()
    # series below the kernel's threshold (se3_advance): in fp32 (t - sin t) / t^3 cancels up to t^2 = 0.25
    small = t2 < (1e-8 if dtype == torch.float64 else 0.25)
    ts = t.clamp_min(torch.finfo(dtype).tiny)
    ca = torch.where(small, 1 - t2 * (1 / 6 - t2 * (1 / 120 - t2 * (1 / 5040 - t2 / 362880))), torch.sin(t) / ts)
    cb = torch.where(small, 0.5 - t2 * (1 / 24 - t2 * (1 / 720 - t2 * (1 / 40320 - t2 / 3628800))),
                     (1 - torch.cos(t)) / ts ** 2)
    cc = torch.where(small, 1 / 6 - t2 * (1 / 120 - t2 * (1 / 5040 - t2 * (1 / 362880 - t2 / 39916800))),
                     (t - torch.sin(t)) / ts ** 3)
    W = torch.zeros((lw.shape[0], 3, 3), dtype=lw.dtype, device=lw.device)
    W[:, 0, 1], W[:, 0, 2], W[:, 1, 0] = -lw[:, 2], lw[:, 1], lw[:, 2]
    W[:, 1, 2], W[:, 2, 0], W[:, 2, 1] = -lw[:, 0], -lw[:, 1], lw[:, 0]
    W2 = W @ W
    eye = torch.eye(3, dtype=lw.dtype, device=lw.device)
    E = eye + ca[:, None, None] * W + cb[:, None, None] * W2
    V = eye + cb[:, None, None] * W + cc[:, None, None] * W2
    Ro = Ra @ E
    po = pa + (Ra @ (V @ lv.unsqueeze(-1))).squeeze(-1)
    return torch.cat([Ro.reshape(-1, 9), po], dim=1)
