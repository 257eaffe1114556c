"""Grasp roadmap (build_roadmap / query_roadmap_batch) on one GPU: prints one JSON line and writes it to --out.

  * build: wall time (ending in a device synchronise), placements drawn against vertices kept, edges accepted, step
    rows, and the roadmap's strongly connected components, for N in --sizes x k in --ks x join_tol in --tols, fp64,
    the default box (path.sample_cube_placement's: x, y between the reference's two cube placements, z in
    [Z_MIN, Z_MAX]);
  * queries on the planner experiment's endpoints (experiments.random_endpoints, spreads 0.1 .. 0.4, --queries per
    spread and call) against the roadmap of N = --query-n, k = --query-k at each join_tol: success rate, time per call
    (median of --reps calls after a warm-up, each ending in a device synchronise), queries/s next to computepath_batch
    on the same endpoints in the same process, joint-space length and vertices per path;
  * downstream at 100 queries per spread: maketraj_paths -> check -> refine -> check valid counts of the roadmap's
    paths and of computepath_batch's on the same endpoints (an unconnected query counts as invalid).
The endpoints reach below Z_MIN (the experiment clips them to the placements' box +- 0.14 m), so the attachments have
to bridge from them into the vertex box.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import gik_b200                                                    # noqa: E402
from gik_b200 import experiments                                   # noqa: E402

A = (np.eye(3), np.array([0.33, -0.3, 0.93]))                     # config.py:36-37
B = (np.eye(3), np.array([0.4, 0.11, 0.93]))
SPREADS = (0.1, 0.2, 0.3, 0.4)


def _card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "not read"
    return name, out


def _timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0


def _components(rm):
    from scipy.sparse import csr_matrix
    from scipy.sparse.csgraph import connected_components
    N = rm.q.shape[0]
    G = csr_matrix((np.ones(rm.dst.numel()), rm.dst.cpu().numpy(), rm.row_ptr.cpu().numpy()), shape=(N, N))
    n, lab = connected_components(G, directed=True, connection="strong")
    return {"strong_components": int(n), "largest_strong_component": int(np.bincount(lab).max())}


def _downstream(solver, qi, qg, q, off):
    ctrl, _ = gik_b200.maketraj_paths(qi, qg, q, off, solver=solver)
    ok = off[1:] > off[:-1]
    ctrl = ctrl[ok]
    before = gik_b200.check_trajectories_batch(ctrl, solver=solver)
    ref = gik_b200.refine_trajectories_batch(ctrl, solver=solver)
    after = gik_b200.check_trajectories_batch(ref["ctrl"], solver=solver)
    return {"paths": int(ok.sum().item()), "valid_fitted": int(before["valid"].sum().item()),
            "valid_refined": int(after["valid"].sum().item())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="4096,16384")
    ap.add_argument("--ks", default="8,16")
    ap.add_argument("--tols", default="0.5,0.05")
    ap.add_argument("--query-n", type=int, default=16384)
    ap.add_argument("--query-k", type=int, default=16)
    ap.add_argument("--queries", default="100,1024")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join("profiles", "roadmap.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_roadmap needs a GPU")
    solver = gik_b200.GraspIK(gik_b200.nextage_table(), "cuda:0").attach_scene()
    name, power = _card()
    tols = [float(x) for x in args.tols.split(",")]

    # warm-up of every kernel the timed calls use (module load, first launches)
    g = torch.Generator(device="cuda:0").manual_seed(0)
    small = gik_b200.build_roadmap(A, B, 256, k=8, robot=solver, generator=g)
    q, pl = experiments.random_endpoints(solver, A, B, (0.1,) * 3, 16, generator=g)
    gik_b200.query_roadmap_batch(small, q[:8], q[8:], pl[:8], pl[8:], robot=solver)
    gik_b200.computepath_batch(q[:8], q[8:], pl[:8], pl[8:], robot=solver, generator=g)

    builds, roadmaps = [], {}
    for tol in tols:
        for N in [int(x) for x in args.sizes.split(",")]:
            for k in [int(x) for x in args.ks.split(",")]:
                g = torch.Generator(device="cuda:0").manual_seed(1)
                rm, t = _timed(lambda: gik_b200.build_roadmap(A, B, N, k=k, join_tol=tol, robot=solver, generator=g))
                builds.append({"n_vertices": N, "k": k, "join_tol": tol, "build_s": t, "drawn": rm.drawn, "kept": N,
                               "edges_tried": N * k, "edges_accepted": int(rm.dst.numel()),
                               "step_rows": int(rm.steps.shape[0]), **_components(rm)})
                print(json.dumps(builds[-1]), file=sys.stderr)
                if N == args.query_n and k == args.query_k:
                    roadmaps[tol] = rm
                else:
                    del rm

    queries, downstream = [], []
    for sd in SPREADS:
        for Q in [int(x) for x in args.queries.split(",")]:
            g = torch.Generator(device="cuda:0").manual_seed(int(sd * 100) + Q)
            q, pl = experiments.random_endpoints(solver, A, B, (sd, sd, sd), 2 * Q, generator=g)
            qi, qg, ci, cg = q[:Q], q[Q:], pl[:Q], pl[Q:]
            (rq, _, roff, _), t_rrt = _timed(lambda: gik_b200.computepath_batch(qi, qg, ci, cg, robot=solver, generator=g))
            rrt_ok = float((roff[1:] > roff[:-1]).double().mean().item())
            for tol, rm in roadmaps.items():
                out, ts = None, []
                for _ in range(args.reps):
                    out, t = _timed(lambda: gik_b200.query_roadmap_batch(rm, qi, qg, ci, cg, robot=solver))
                    ts.append(t)
                qq, _, off, st = out
                ok = st["connected"].bool()
                t = float(np.median(ts))
                row = {"std_dev": sd, "queries": Q, "join_tol": tol, "success_rate": float(ok.double().mean().item()),
                       "call_s": t, "queries_per_s": Q / t, "rrt_call_s": t_rrt, "rrt_queries_per_s": Q / t_rrt,
                       "rrt_success_rate": rrt_ok,
                       "length_mean": float(st["length"][ok].mean().item()) if ok.any() else None,
                       "vertices_mean": float(st["vertices"][ok].double().mean().item()) if ok.any() else None,
                       "rows_mean": float((off[1:] - off[:-1])[ok].double().mean().item()) if ok.any() else None,
                       "attach_start_mean": float(st["attach_start"].double().mean().item()),
                       "attach_goal_mean": float(st["attach_goal"].double().mean().item())}
                queries.append(row)
                print(json.dumps(row), file=sys.stderr)
                if Q == 100:
                    downstream.append({"std_dev": sd, "queries": Q, "join_tol": tol, "planner": "roadmap",
                                       **_downstream(solver, qi, qg, qq, off)})
                    print(json.dumps(downstream[-1]), file=sys.stderr)
            if Q == 100:
                downstream.append({"std_dev": sd, "queries": Q, "planner": "computepath_batch",
                                   **_downstream(solver, qi, qg, rq, roff)})
                print(json.dumps(downstream[-1]), file=sys.stderr)

    totals = {}
    for d in downstream:
        key = d["planner"] + ("" if "join_tol" not in d else f"@join_tol={d['join_tol']}")
        t = totals.setdefault(key, {"queries": 0, "paths": 0, "valid_fitted": 0, "valid_refined": 0})
        for f in t:
            t[f] += d[f]
    box = roadmaps[tols[0]].box if roadmaps else None
    res = {"metric": "roadmap", "gpu": name, "power_limit": power, "dtype": "float64", "box": box,
           "query_roadmap": {"n_vertices": args.query_n, "k": args.query_k, "k_attach": args.query_k},
           "builds": builds, "queries": queries, "downstream": downstream, "downstream_totals": totals,
           "note": "times: host clock around one call ending in a device synchronise (queries: median of reps after a "
                   "warm-up; computepath_batch: one call after a warm-up call); downstream: maketraj_paths -> "
                   "check_trajectories_batch -> refine_trajectories_batch -> check, valid counts out of the queries"}
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
