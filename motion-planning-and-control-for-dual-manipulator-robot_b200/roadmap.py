"""A grasp roadmap for many planning queries in one static scene: `build_roadmap` samples grasp vertices once and joins
each to its k nearest neighbours with projected grasp edges; `query_roadmap_batch` then answers a batch of queries with
one attachment edge launch, one shortest-path launch and one path launch -- no IK sampling at query time, and no query
waits for another's RRT iterations.  Its output has computepath_batch's (q, cube, offsets, stats) form, so the fit,
check, refine and shortcut calls take it unchanged.  Kernels in csrc/gik_roadmap.cuh, rules in include/gik.h.

A query the roadmap cannot connect gets an empty path (stats["connected"] == 0); to plan those, pass their rows to
computepath_batch."""
from __future__ import annotations

from dataclasses import dataclass

import torch

from .inverse_geometry import _pose_to_array, solver_for
from .ops import as_pose12
from .path import GOAL_TOLERANCE, STEP_SIZE, Z_MAX, Z_MIN, _cut_at_first_collision, _grasp_filter, sample_cube_placements
from .planner import _num_steps

OVERSAMPLE = 4          # placements drawn per vertex still needed, as experiments.random_endpoints draws them


@dataclass
class Roadmap:
    """Device tensors of a grasp roadmap and its build parameters.  Edges are CSR by source: the edges of vertex i are
    row_ptr[i] .. row_ptr[i+1]-1, nearest target first; edge e's steps 1 .. ns[e]-1 (the step at the target is
    replaced by the target's q) are steps[step_ptr[e]:step_ptr[e+1]].  torch.save(vars(roadmap), f) and
    Roadmap(**torch.load(f)) round-trip it."""
    q: torch.Tensor             # [N, nq] vertex grasps
    cube: torch.Tensor          # [N, 12] their placements (identity rotation)
    row_ptr: torch.Tensor       # int64 [N+1]
    dst: torch.Tensor           # int32 [E]
    weight: torch.Tensor        # float64 [E] joint-space length of q_i, the steps, q_j
    ns: torch.Tensor            # int32 [E] steps of the edge
    step_ptr: torch.Tensor      # int64 [E+1]
    steps: torch.Tensor         # [rows, nq]
    k: int                      # neighbours per vertex
    join_tol: float
    step_size: float
    box: tuple                  # ((x, y, z) low, (x, y, z) high) the vertices were drawn in
    drawn: int                  # placements drawn until the N-th vertex was found


def _march(solver, q_from, c_from, c_to, q_to, ns, S, join_tol):
    """Edges from (q_from, c_from) towards c_to in ns steps (one edge launch, the dense scene cut), judged against
    q_to.  -> (weight float64 [E] (+inf: rejected), q_path [S][nq][E])."""
    path, nv, _ = solver.project_edges_soa(q_from.t().contiguous(), c_from.t().contiguous(), c_to.t().contiguous(), ns, S)
    nv = _cut_at_first_collision(solver, path, nv, c_from, c_to, ns, S, dense=True)
    return solver.roadmap_edges(q_from, q_to, ns, nv, path, join_tol=join_tol), path


def _check_k(k, N, name):
    if not 1 <= int(k) <= min(32, N - 1):
        raise ValueError(f"{name} must be in [1, min(32, N - 1)] with N = {N}, got {k}")
    return int(k)


def build_roadmap(cube0, cube1, n_vertices, *, k=16, box=None, join_tol=GOAL_TOLERANCE, step_size=STEP_SIZE,
                  dtype=torch.float64, generator=None, robot=None) -> Roadmap:
    """A roadmap of n_vertices grasps and their edges.

    Vertices: placements uniform in `box` with identity rotation (sample_cube_placements), validated by the planner's
    sample filters (cube collision-free, IK from zeros passes the success predicate, clearance >= 0.04 m), kept in draw
    order.  The default box is path.sample_cube_placement's for cube0 / cube1: x and y between them, z in [Z_MIN, Z_MAX];
    box=(low, high) overrides it.
    Edges: i -> j for each of the k nearest vertices j of i by cube translation (gik_knn_*), marched from (q_i, cube_i)
    towards cube_j in _num_steps(cube_i, cube_j) steps (all N k edges in one edge launch, cut at the first collision),
    accepted when every step converged collision-free and the last lies within join_tol of q_j (gik_roadmap_edges_*).
    1 <= k <= min(32, N - 1).

    Host reads: one per draw of the vertex loop (the valid count), the step bound S (the largest neighbour edge's step
    count) and the accepted-edge and step-row totals of the compaction."""
    solver = solver_for(robot)
    solver._need_scene()
    dev, nq, N = solver.device, solver.nq, int(n_vertices)
    k = _check_k(k, N, "k")
    if box is None:
        a, b = _pose_to_array(cube0)[9:], _pose_to_array(cube1)[9:]
        box = ((min(a[0], b[0]), min(a[1], b[1]), Z_MIN), (max(a[0], b[0]), max(a[1], b[1]), Z_MAX))
    box = (tuple(float(x) for x in box[0]), tuple(float(x) for x in box[1]))
    lo, hi = box
    zero = torch.zeros(nq, dtype=dtype, device=dev)
    qs, ps, need, drawn = [], [], N, 0
    while need > 0:
        m = max(need * OVERSAMPLE, 256)
        pl = sample_cube_placements(m, lo, hi, z_range=(lo[2], hi[2]), device=dev, dtype=dtype, generator=generator)
        q, ok = _grasp_filter(solver, pl, zero, dtype)
        idx = torch.nonzero(ok).flatten()[:need]
        if idx.numel() == need:
            drawn += int(idx[-1]) + 1
        else:
            drawn += m
            if idx.numel() == 0 and drawn >= (1 << 22):
                raise RuntimeError(f"build_roadmap: no valid grasp among {drawn} placements drawn in the box {box}")
        qs.append(q[idx]); ps.append(pl[idx])
        need -= idx.numel()
    q = torch.cat(qs).contiguous()
    cube = as_pose12(torch.cat(ps), dtype=dtype, device=dev).contiguous()

    nbr = solver.knn(cube, k)
    src = torch.arange(N, device=dev).repeat_interleave(k)
    dst = nbr.reshape(-1).long()
    ca, cb = cube[src], cube[dst]
    ns = _num_steps(ca, cb, step_size)
    S = int(ns.max().item())
    weight, path = _march(solver, q[src], ca, cb, q[dst], ns, S, join_tol)

    keep = torch.nonzero(torch.isfinite(weight)).flatten()          # host read: the accepted edges
    E = keep.numel()
    rows = (ns[keep] - 1).long()
    step_ptr = torch.zeros(E + 1, dtype=torch.int64, device=dev)
    step_ptr[1:] = torch.cumsum(rows, 0)
    R = int(step_ptr[-1].item())                                   # host read: the step rows
    e_row = keep.repeat_interleave(rows, output_size=R)
    m_row = torch.arange(R, device=dev) - step_ptr[:-1].repeat_interleave(rows, output_size=R)
    row_ptr = torch.zeros(N + 1, dtype=torch.int64, device=dev)
    row_ptr[1:] = torch.cumsum(torch.bincount(src[keep], minlength=N), 0)
    return Roadmap(q=q, cube=cube, row_ptr=row_ptr, dst=dst[keep].to(torch.int32), weight=weight[keep].contiguous(),
                   ns=ns[keep].contiguous(), step_ptr=step_ptr, steps=path[m_row, :, e_row].contiguous(), k=k,
                   join_tol=float(join_tol), step_size=float(step_size), box=box, drawn=drawn)


def query_roadmap_batch(roadmap: Roadmap, q_init, q_goal, cube0, cube1, *, k_attach=None, robot=None):
    """Shortest roadmap paths for Q queries: q_init / q_goal [Q,nq], cube0 / cube1 [Q,12|4x4|7|3] (any rotation).

    Each query attaches (q_init, cube0) to its k_attach nearest vertices a (landing within join_tol of q_a), the
    k_attach vertices b nearest cube1 to (q_goal, cube1), and tries the direct edge start -> goal: all Q (2 k_attach + 1)
    attachments in one edge launch, cut and judged by the roadmap's rules (k_attach defaults to roadmap.k).  One
    gik_roadmap_sssp launch finds each query's shortest path: the exact fp64 minimum of left-to-right length sums, as
    Dijkstra gives it, ties broken deterministically (include/gik.h).  The output is the same whether a query runs alone
    or in a batch.

    Returns (q [total,nq], cube [total,12], offsets int64 [Q+1], stats) in computepath_batch's form: query i's path is
    q_init, the start attachment's steps, then per roadmap edge its steps and the next vertex, the goal attachment's
    steps and q_goal; each step row carries the placement it was solved for, vertex rows the vertex's placement, the
    first and last rows cube0 and cube1.  No cube move exceeds step_size.  An unconnected query has no rows.  stats:
    connected int32 [Q], length float64 [Q] (+inf when unconnected), vertices int32 [Q] (roadmap vertices on the path),
    attach_start / attach_goal int32 [Q] (accepted attachments).

    Host reads: two (the attachment step bound and the total row count).  Memory: the per-query distances and
    predecessors take 12 Q N bytes (N = roadmap vertices)."""
    solver = solver_for(robot)
    solver._need_scene()
    rm = roadmap
    dev, nq, dtype = solver.device, solver.nq, rm.q.dtype
    N = rm.q.shape[0]
    ka = _check_k(rm.k if k_attach is None else k_attach, N, "k_attach")
    qi = torch.as_tensor(q_init, device=dev).to(dtype).reshape(-1, nq)
    qg = torch.as_tensor(q_goal, device=dev).to(dtype).reshape(-1, nq)
    Q = qi.shape[0]
    a12 = as_pose12(cube0, dtype=dtype, device=dev, batch=Q).contiguous()
    b12 = as_pose12(cube1, dtype=dtype, device=dev, batch=Q).contiguous()
    if qg.shape[0] != Q or a12.shape[0] != Q or b12.shape[0] != Q:
        raise ValueError("query_roadmap_batch: q_init, q_goal, cube0 and cube1 must have one row per query")
    i32 = dict(dtype=torch.int32, device=dev)
    if Q == 0:
        stats = {k: torch.zeros(0, **i32) for k in ("connected", "vertices", "attach_start", "attach_goal")}
        stats["length"] = torch.zeros(0, dtype=torch.float64, device=dev)
        return (torch.empty((0, nq), dtype=dtype, device=dev), torch.empty((0, 12), dtype=dtype, device=dev),
                torch.zeros(1, dtype=torch.int64, device=dev), stats)

    nbr = solver.knn(rm.cube, ka, torch.cat([a12, b12]))
    sv, gv = nbr[:Q].long(), nbr[Q:].long()
    A = 2 * ka + 1
    att_vertex = torch.cat([nbr[:Q], nbr[Q:], torch.full((Q, 1), -1, **i32)], 1).contiguous()

    # slots per query: ka start attachments, ka goal attachments, the direct edge
    q_from = torch.cat([qi[:, None].expand(Q, ka, nq), rm.q[gv], qi[:, None]], 1).reshape(Q * A, nq)
    c_from = torch.cat([a12[:, None].expand(Q, ka, 12), rm.cube[gv], a12[:, None]], 1).reshape(Q * A, 12)
    c_to = torch.cat([rm.cube[sv], b12[:, None].expand(Q, ka, 12), b12[:, None]], 1).reshape(Q * A, 12)
    q_to = torch.cat([rm.q[sv], qg[:, None].expand(Q, ka, nq), qg[:, None]], 1).reshape(Q * A, nq)
    ns = _num_steps(c_from, c_to, rm.step_size)
    S = int(ns.max().item())                                        # host read: the attachment step bound
    att_w, att_path = _march(solver, q_from, c_from, c_to, q_to, ns, S, rm.join_tol)
    att_w = att_w.reshape(Q, A)
    _, pred, goal_pred, length, a_s, a_g = solver.roadmap_sssp(rm.row_ptr, rm.dst, rm.weight, att_vertex, att_w)
    q, cube, offsets, verts = solver.roadmap_paths(rm.q, rm.cube, rm.row_ptr, rm.dst, rm.ns, rm.step_ptr, rm.steps, qi, qg,
                                                   a12, b12, att_vertex, att_w, ns.reshape(Q, A), att_path, pred,
                                                   goal_pred)
    stats = {"connected": (goal_pred != -2).to(torch.int32), "length": length, "vertices": verts, "attach_start": a_s,
             "attach_goal": a_g}
    return q, cube, offsets, stats
