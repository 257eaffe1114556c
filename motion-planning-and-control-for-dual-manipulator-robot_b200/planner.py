"""RRT-connect for many queries per call: `computepath_batch` plans Q independent queries of path.computepath
(path.py:194-278) in lockstep, with their trees in device memory (csrc/gik_tree.cuh).  Each iteration, the K
extensions of every still-active query go through ONE launch of the edge kernel for the start trees and one for the
goal trees; nearest-vertex search, tree growth, the connect test and the retry bookkeeping are device work, so the
loop reads back one thing per iteration: which queries are still active."""
from __future__ import annotations

import numpy as np
import torch

from .inverse_geometry import solver_for
from .ops import as_pose12
from .path import (GOAL_BIAS, GOAL_TOLERANCE, MAX_ITERATIONS, MAX_RETRIES, STEP_SIZE, Z_MAX, Z_MIN,
                   _cut_at_first_collision, _grasp_filter, sample_cube_placements)

CANDIDATES = 16     # sample candidates drawn and validated per extension slot and iteration


def _num_steps(a12, b12, step_size):
    """int(||p_a - p_b|| / step_size) + 1 (path.py:129-130), summed in numpy's order so that the step count is the one
    path.computepath computes."""
    d = a12[:, 9:] - b12[:, 9:]
    sq = d * d
    return torch.floor(torch.sqrt((sq[:, 0] + sq[:, 1]) + sq[:, 2]) / step_size).to(torch.int32) + 1


def _draw_targets(solver, query, retry, iteration, K, q_goal, cube_start, cube_goal, dtype, generator):
    """Targets of the K extension slots of each active query: with probability GOAL_BIAS the goal (q_goal, cube_goal),
    else the first valid one of CANDIDATES samples of path.sample_cube_placement drawn in the query's own box (the
    filters of sample_grasp_poses_batch).  query / retry / iteration [A] identify each active query and where it is in
    its search (unused here: a scripted replacement can key on them).  -> (q [A,K,nq], cube [A,K,12], has bool [A,K]);
    has = False when every candidate failed: the slot stays idle this iteration."""
    A, dev, C = q_goal.shape[0], q_goal.device, CANDIDATES
    coin = torch.rand((A, K), dtype=torch.float64, device=dev, generator=generator) < GOAL_BIAS
    pl = sample_cube_placements(A * K * C, cube_start.repeat_interleave(K * C, 0), cube_goal.repeat_interleave(K * C, 0),
                                device=dev, dtype=dtype, generator=generator)
    q, ok = _grasp_filter(solver, pl, torch.zeros(solver.nq, dtype=dtype, device=dev), dtype)
    ok = ok.reshape(A, K, C)
    first = ok.to(torch.int8).argmax(dim=2)                                          # first valid candidate
    q = q.reshape(A, K, C, -1).gather(2, first[:, :, None, None].expand(A, K, 1, solver.nq)).squeeze(2)
    pl = pl.reshape(A, K, C, 3).gather(2, first[:, :, None, None].expand(A, K, 1, 3)).squeeze(2)
    cube = as_pose12(pl.reshape(-1, 3), dtype=dtype, device=dev).reshape(A, K, 12)
    q = torch.where(coin[:, :, None], q_goal[:, None, :], q)
    cube = torch.where(coin[:, :, None], cube_goal[:, None, :], cube)
    return q, cube, coin | ok.any(dim=2)


def _extend(solver, trees, tree, near, cube_b, has, S, step_size):
    """One extension per slot: project_path (path.py:125-163) from vertex near[e] of tree[e] towards cube_b[e] (edge
    kernel + scene cut), appended to the trees.  Idle slots (has = False) march nothing and append nothing.
    -> seg_end int32 [E] (-1: no segment)."""
    verts, cubes, parent, n_verts, overflow = trees
    t, v = tree.long(), near.clamp_min(0).long()
    qs, ca = verts[t, :, v], cubes[t, :, v]                                          # [E,nq], [E,12]
    ns = torch.where(has, _num_steps(ca, cube_b, step_size).clamp(max=S), 0)      # (S bounds every edge in the boxes)
    q_soa, pa, pb = qs.t().contiguous(), ca.t().contiguous(), cube_b.t().contiguous()
    path, nv, _ = solver.project_edges_soa(q_soa, pa, pb, ns, S)
    nv = _cut_at_first_collision(solver, path, nv, ca, cube_b, ns, S, dense=True)
    nv = torch.where(has, nv, -1)
    return solver.tree_grow(verts, cubes, parent, n_verts, overflow, tree, near, q_soa, pa, pb, ns, nv, path)


def computepath_batch(qinit, qgoal, cube0, cube1, robot=None, cube=None, *, step_size=STEP_SIZE,
                      goal_tolerance=GOAL_TOLERANCE, max_iterations=MAX_ITERATIONS, max_retries=MAX_RETRIES,
                      generator=None, dtype=torch.float64, expand=8):
    """path.computepath for Q independent queries in one call: qinit / qgoal [Q,nq], cube0 / cube1 [Q,12|4x4|7|3].

    Each query follows computepath's rules: goal bias 0.1, K = `expand` extensions per iteration (start-tree extension
    towards the target, then a goal-tree extension from the goal tree's vertex nearest to the new configuration
    towards the goal placement), the first connecting extension (lowest k) ends the query, ceil(max_iterations / K)
    iterations per retry, then the trees are reset, `max_retries` retries in all.  Targets are drawn per slot from
    CANDIDATES samples validated at once; a slot whose candidates all fail stays idle for that iteration (see path.py).

    Returns (q [total,nq], cube [total,12], offsets int64 [Q+1], stats): the path of query i is
    q[offsets[i]:offsets[i+1]] with its cube placements aligned, empty when the query failed.  stats holds int32 [Q]
    tensors iterations, retries, edges (edges projected), vertices (both trees at the connection, 0 on failure) and
    overflows (retries ended by a full tree) -- computepath(return_stats=True)'s counts.

    Memory: 2Q trees of capacity cap = 1 + ceil(max_iterations / K) * K * (max_steps + 1), the worst case of one retry,
    so a tree cannot overflow with the defaults; max_steps = int(box diagonal / step_size) + 1 for the box spanning
    both placements and the sample box.  That is 2 * Q * cap * (nq + 12) * sizeof(dtype) bytes: for fp64, Q = 1024,
    K = 8 and the reference's boxes (max_steps about 26) about 3 GB."""
    solver = solver_for(robot, cube)
    solver._need_scene()
    dev, nq = solver.device, solver.nq
    qi = torch.as_tensor(qinit, device=dev).to(dtype).reshape(-1, nq)
    qg = torch.as_tensor(qgoal, device=dev).to(dtype).reshape(-1, nq)
    Q = qi.shape[0]
    a12 = as_pose12(cube0, dtype=dtype, device=dev, batch=Q).contiguous()
    b12 = as_pose12(cube1, dtype=dtype, device=dev, batch=Q).contiguous()
    if qg.shape[0] != Q or a12.shape[0] != Q or b12.shape[0] != Q:
        raise ValueError("computepath_batch: qinit, qgoal, cube0 and cube1 must have one row per query")
    K = max(int(expand), 1)
    per_retry = -(-max_iterations // K)
    i32 = dict(dtype=torch.int32, device=dev)
    stats = {k: torch.zeros(Q, **i32) for k in ("iterations", "retries", "edges", "vertices", "overflows")}
    if Q == 0:
        return (torch.empty((0, nq), dtype=dtype, device=dev), torch.empty((0, 12), dtype=dtype, device=dev),
                torch.zeros(1, dtype=torch.int64, device=dev), stats)
    # host-side bound on the steps of any edge, from the query boxes (one read before the loop)
    pa, pb = a12[:, 9:].double().cpu().numpy(), b12[:, 9:].double().cpu().numpy()
    lo, hi = np.minimum(pa, pb), np.maximum(pa, pb)
    lo[:, 2], hi[:, 2] = np.minimum(lo[:, 2], Z_MIN), np.maximum(hi[:, 2], Z_MAX)
    S = int(np.linalg.norm(hi - lo, axis=1).max() * (1 + 1e-9) / step_size) + 1
    cap = 1 + per_retry * K * (S + 1)

    verts = torch.empty((2 * Q, nq, cap), dtype=dtype, device=dev)
    cubes = torch.empty((2 * Q, 12, cap), dtype=dtype, device=dev)
    parent = torch.empty((2 * Q, cap), **i32)
    verts[:Q, :, 0], verts[Q:, :, 0] = qi, qg
    cubes[:Q, :, 0], cubes[Q:, :, 0] = a12, b12
    parent[:, 0] = -1
    n_verts = torch.ones(2 * Q, **i32)
    overflow = torch.zeros(2 * Q, dtype=torch.uint8, device=dev)
    trees = (verts, cubes, parent, n_verts, overflow)

    active = torch.ones(Q, dtype=torch.bool, device=dev)
    retry, it_r = torch.zeros(Q, **i32), torch.zeros(Q, **i32)
    start_end, goal_end = torch.full((Q,), -1, **i32), torch.full((Q,), -1, **i32)
    while True:
        idx = torch.nonzero(active).flatten()                     # the loop's one host synchronisation
        A = idx.numel()
        if A == 0:
            break
        gidx = idx + Q
        q_t, c_t, has = _draw_targets(solver, idx, retry[idx], it_r[idx], K, qg[idx], a12[idx], b12[idx], dtype, generator)
        E = A * K
        has = has.reshape(E)
        tree_s = idx.to(torch.int32).repeat_interleave(K)         # the edges of one tree are consecutive
        near_s = solver.tree_nearest(verts, n_verts, q_t.reshape(E, nq), tree_s)
        seg_s = _extend(solver, trees, tree_s, near_s, c_t.reshape(E, 12), has, S, step_size)
        q_new = verts[tree_s.long(), :, seg_s.clamp_min(0).long()]
        tree_g = tree_s + Q
        near_g = solver.tree_nearest(verts, n_verts, q_new, tree_g)
        seg_g = _extend(solver, trees, tree_g, near_g, b12[idx].repeat_interleave(K, 0), has, S, step_size)
        q_goal_new = verts[tree_g.long(), :, seg_g.clamp_min(0).long()]

        ovf = (overflow[idx] | overflow[gidx]).bool()
        conn = (has & (seg_s >= 0) & (seg_g >= 0) &
                (torch.linalg.vector_norm(q_goal_new - q_new, dim=1) < goal_tolerance)).reshape(A, K) & ~ovf[:, None]
        hit = conn.any(dim=1)
        k0 = conn.to(torch.int8).argmax(dim=1, keepdim=True)       # first connecting extension
        start_end[idx] = torch.where(hit, seg_s.reshape(A, K).gather(1, k0).squeeze(1), start_end[idx])
        goal_end[idx] = torch.where(hit, seg_g.reshape(A, K).gather(1, k0).squeeze(1), goal_end[idx])
        stats["vertices"][idx] = torch.where(hit, n_verts[idx] + n_verts[gidx], 0)
        stats["iterations"][idx] += 1
        stats["edges"][idx] += 2 * has.reshape(A, K).sum(dim=1, dtype=torch.int32)
        stats["overflows"][idx] += ovf.to(torch.int32)

        it_r[idx] += 1
        end = ~hit & ((it_r[idx] >= per_retry) | ovf)             # retry over: trees back to their roots
        retry[idx] += end.to(torch.int32)
        it_r[idx] = torch.where(end, 0, it_r[idx])
        n_verts[idx] = torch.where(end, 1, n_verts[idx])
        n_verts[gidx] = torch.where(end, 1, n_verts[gidx])
        overflow[idx] = torch.where(end, 0, overflow[idx])
        overflow[gidx] = torch.where(end, 0, overflow[gidx])
        active[idx] = ~hit & (retry[idx] < max_retries)
    stats["retries"] = retry
    q, cube_rows, offsets = solver.tree_paths(verts, cubes, parent, n_verts, start_end, goal_end)
    return q, cube_rows, offsets, stats


# ------------------------------------------------------------------------------------------------ path shortcutting
SHORTCUT_ROUNDS = 16        # defaults chosen from the length-per-round curve of tools/bench_shortcut.py: DESIGN.md
SHORTCUT_CANDIDATES = 16    # "Path shortcutting"


def _draw_pairs(n, K, generator):
    """K candidate pairs per path: n int64 [Q] path lengths -> (i, j) int32 [Q, K], uniform over the pairs with
    0 <= i and i + 2 <= j <= n - 1 (two distinct slots x != y of n - 1, i = min, j = max + 1); -1 for a path with fewer
    than 3 vertices.  Drawn on n's device from `generator`."""
    Q, dev = n.shape[0], n.device
    u = torch.rand((Q, K, 2), dtype=torch.float64, device=dev, generator=generator)
    m = (n - 1).clamp_min(2)[:, None]
    x = torch.minimum((u[..., 0] * m).long(), m - 1)                                # [0, n-1)
    y = torch.minimum((u[..., 1] * (m - 1)).long(), m - 2)                          # [0, n-2)
    y = y + (y >= x).long()
    i, j = torch.minimum(x, y), torch.maximum(x, y) + 1
    ok = (n >= 3)[:, None]
    return torch.where(ok, i, -1).to(torch.int32), torch.where(ok, j, -1).to(torch.int32)


def shortcut_paths_batch(q, cube, offsets, robot=None, *, rounds=SHORTCUT_ROUNDS, candidates=SHORTCUT_CANDIDATES,
                         step_size=STEP_SIZE, join_tol=GOAL_TOLERANCE, generator=None):
    """Shortcut CSR paths as computepath_batch returns them: q [total, nq], cube [total, 12], offsets int64 [Q+1].

    Each round draws `candidates` (K <= 32) pairs (i, j), j >= i + 2, per path of at least 3 vertices (_draw_pairs),
    marches each as one edge from (q_i, cube_i) towards cube_j in _num_steps(cube_i, cube_j) steps (all Q·K edges in
    one edge launch, cut at the first collision), and accepts a candidate when every step converged collision-free,
    the last step lands within join_tol of q_j and the joint-space length strictly drops.  Per path the accepted
    candidate with the largest gain (ties: the lowest index) replaces vertices i+1 .. j-1 with the edge's steps but
    the last, each stored with the placement it was solved for (gik_path_shortcut_*, semantics in include/gik.h).
    The end rows of every path are kept bit for bit; lengths never increase; no cube move above step_size is added.

    Returns (q, cube, offsets, stats) in the same form; stats holds shortcuts int32 [Q] (splices accepted) and
    length float64 [Q] (joint-space length after the last round).  Host synchronisations: one before the loop (the
    step bound S, from the largest cube-translation bounding-box diagonal of a path) and one per round (the new row
    count).  A candidate needing more than S steps (possible only when a path rotates the cube) is dropped: it
    marches no step."""
    solver = solver_for(robot, None)
    solver._need_scene()
    dev = solver.device
    q = torch.as_tensor(q, device=dev)
    cube = torch.as_tensor(cube, device=dev).to(q.dtype)
    offsets = torch.as_tensor(offsets, device=dev).to(torch.int64)
    K = int(candidates)
    if not 0 <= K <= 32:
        raise ValueError("shortcut_paths_batch: candidates must be in [0, 32]")
    Q, total = offsets.shape[0] - 1, q.shape[0]
    stats = {"shortcuts": torch.zeros(Q, dtype=torch.int32, device=dev),
             "length": torch.zeros(Q, dtype=torch.float64, device=dev)}
    if Q == 0 or total == 0:
        return q, cube, offsets, stats
    # step bound: the largest bounding-box diagonal of a path's cube translations (the one read before the loop)
    pid = torch.searchsorted(offsets[1:], torch.arange(total, device=dev), right=True)[:, None].expand(total, 3)
    p = cube[:, 9:].double()
    lo = torch.zeros((Q, 3), dtype=torch.float64, device=dev).scatter_reduce(0, pid, p, "amin", include_self=False)
    hi = torch.zeros((Q, 3), dtype=torch.float64, device=dev).scatter_reduce(0, pid, p, "amax", include_self=False)
    S = int(torch.linalg.vector_norm(hi - lo, dim=1).max().item() * (1 + 1e-6) / step_size) + 1
    i32 = dict(dtype=torch.int32, device=dev)
    if rounds <= 0 or K == 0:                               # lengths only
        none = torch.zeros((Q, 0), **i32)
        q, cube, offsets, _, stats["length"] = solver.path_shortcut(
            q, cube, offsets, none, none, none, none, torch.zeros((0, solver.nq, 0), dtype=q.dtype, device=dev),
            join_tol=join_tol)
        return q, cube, offsets, stats
    for _ in range(int(rounds)):
        n = offsets[1:] - offsets[:-1]
        pi, pj = _draw_pairs(n, K, generator)
        has = (pi >= 0).reshape(-1)
        last = q.shape[0] - 1
        ri = (offsets[:-1, None] + pi.long()).clamp(0, last).reshape(-1)
        rj = (offsets[:-1, None] + pj.long()).clamp(0, last).reshape(-1)
        ca, cb = cube[ri], cube[rj]
        ns = _num_steps(ca, cb, step_size)
        ns = torch.where(has & (ns <= S), ns, 0)
        path, nv, _ = solver.project_edges_soa(q[ri].t().contiguous(), ca.t().contiguous(), cb.t().contiguous(), ns, S)
        nv = _cut_at_first_collision(solver, path, nv, ca, cb, ns, S, dense=True)
        q, cube, offsets, chosen, stats["length"] = solver.path_shortcut(
            q, cube, offsets, pi, pj, ns.reshape(Q, K), nv.reshape(Q, K), path, join_tol=join_tol)
        stats["shortcuts"] += (chosen >= 0).to(torch.int32)
    return q, cube, offsets, stats
