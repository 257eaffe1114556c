"""Batched RRT-connect against the sequential planner on one GPU: prints one JSON line and writes it to --out.

  * the planner experiment of path_TESTS.py:910-990 (spreads 0.1 .. 0.4, --trials queries each): the SAME endpoint
    pairs planned one query at a time by computepath(expand=8) and in one computepath_batch(expand=8) call; wall time
    per spread (device-synchronised), success rate, mean iterations;
  * a sweep over the batch size Q (spread 0.1): queries/s, planner iterations (= loop iterations of the call, the
    slowest query's count) and edge-kernel launches per call (two per iteration).
Every shape is warmed up first.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gik_b200                                                    # noqa: E402
from gik_b200 import experiments                                   # noqa: E402

A = (np.eye(3), np.array([0.33, -0.3, 0.93]))                     # config.py:36-37
B = (np.eye(3), np.array([0.4, 0.11, 0.93]))


def _card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "not read"
    return name, out


def _sync_time(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def _batch(solver, q, pl, Q, g, K):
    return gik_b200.computepath_batch(q[:Q], q[Q:2 * Q], pl[:Q], pl[Q:2 * Q], robot=solver, generator=g, expand=K)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--trials", type=int, default=100)
    ap.add_argument("--sweep", default="1,16,128,1024")
    ap.add_argument("--expand", type=int, default=8)
    ap.add_argument("--out", default=os.path.join("profiles", "planner_batch.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_planner needs a GPU")
    K = args.expand
    solver = gik_b200.GraspIK(gik_b200.nextage_table(), "cuda:0").attach_scene()
    g = torch.Generator(device="cuda:0").manual_seed(0)
    name, power = _card()
    sweep = [int(x) for x in args.sweep.split(",")]

    # warm-up: both planners, every batch size of the run
    q, pl = experiments.random_endpoints(solver, A, B, (0.1, 0.1, 0.1), 2 * max(sweep + [args.trials]), generator=g)
    gik_b200.computepath(q[0].cpu().numpy(), q[1].cpu().numpy(), (np.eye(3), pl[0].cpu().numpy()),
                         (np.eye(3), pl[1].cpu().numpy()), robot=solver, generator=g, expand=K)
    for Q in sorted(set(sweep + [args.trials])):
        _batch(solver, q, pl, Q, g, K)

    spreads = []
    for sd in (0.1, 0.2, 0.3, 0.4):
        q, pl = experiments.random_endpoints(solver, A, B, (sd, sd, sd), 2 * args.trials, generator=g)
        qn, pn = q.double().cpu().numpy(), pl.double().cpu().numpy()
        n = args.trials
        rng = np.random.default_rng(int(sd * 10))
        seq_ok, seq_it = [], []

        def run_seq():
            for i in range(n):
                path, st = gik_b200.computepath(qn[i], qn[n + i], (np.eye(3), pn[i]), (np.eye(3), pn[n + i]), robot=solver,
                                                rng=rng, generator=g, expand=K, return_stats=True)
                seq_ok.append(bool(path)); seq_it.append(st["iterations"])
        t_seq, _ = _sync_time(run_seq)
        t_bat, (_, _, off, st) = _sync_time(lambda: _batch(solver, q, pl, n, g, K))
        off = off.cpu().numpy()
        it = st["iterations"].cpu().numpy()
        spreads.append({"std_dev": sd, "queries": n,
                        "sequential": {"wall_s": round(t_seq, 4), "per_query_s": round(t_seq / n, 5),
                                       "success_rate": 100.0 * np.mean(seq_ok), "mean_iterations": float(np.mean(seq_it))},
                        "batch": {"wall_s": round(t_bat, 4), "per_query_s": round(t_bat / n, 5),
                                  "success_rate": 100.0 * float(np.mean(off[1:] > off[:-1])),
                                  "mean_iterations": float(it.mean()), "loop_iterations": int(it.max())},
                        "speedup": round(t_seq / t_bat, 2)})
        print(json.dumps(spreads[-1]), file=sys.stderr)

    rows = []
    q, pl = experiments.random_endpoints(solver, A, B, (0.1, 0.1, 0.1), 2 * max(sweep), generator=g)
    for Q in sweep:
        t, (_, _, off, st) = _sync_time(lambda: _batch(solver, q, pl, Q, g, K))
        loops = int(st["iterations"].max().item())
        rows.append({"Q": Q, "wall_s": round(t, 4), "queries_per_s": round(Q / t, 1), "loop_iterations": loops,
                     "edge_launches": 2 * loops,
                     "success_rate": 100.0 * float((off[1:] > off[:-1]).double().mean().item())})
        print(json.dumps(rows[-1]), file=sys.stderr)

    res = {"metric": "rrt_connect_batch", "gpu": name, "power_limit": power, "expand": K, "dtype": "float64",
           "spreads": spreads, "sweep_sigma_0.1": rows,
           "note": "wall times device-synchronised; sequential = computepath one query at a time on the same endpoint pairs"}
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
