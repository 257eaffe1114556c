"""The trajectory check (gik_traj_check_*) on one GPU: prints one JSON line and writes it to --out.

  * kernel time: N in {1, 64, 1024, 8192} trajectories x 1501 samples (the controller's 1500 steps plus the end
    point), fp32 and fp64, CUDA events around --reps launches after a warm-up of every shape; samples/s.  The
    trajectories are the fitted planner trajectories of the experiment below, repeated to N, so the mix of valid and
    invalid ones (and so the share of samples whose pair tests are skipped after the first bad sample) is the
    planner's.  Per-sample flags are not written, as in production use.
  * the CPU oracle (numpy Bernstein sum, C oracle FK and pair distances, numpy log6; tests/traj_oracle.py) on a subset
    of --oracle-traj trajectories, single process: samples/s.
  * the grasp-error distribution behind the policy default grasp_tol = 1e-2: the planner experiment of
    path_TESTS.py:910-990 (spreads 0.1 .. 0.4, --queries queries each: experiments.random_endpoints +
    computepath_batch + maketraj_paths), every fitted trajectory checked in fp64; quantiles of grasp_err and the
    counts of each reason.
The card's name and power limit are read in the same run."""
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
sys.path.insert(0, os.path.join(ROOT, "tests"))
import gik_b200                                                    # noqa: E402
from gik_b200 import experiments                                   # noqa: E402
from gik_b200.trajectory import CHECK_SAMPLES, GRASP_TOL, LIMIT_TOL, sample_weights   # noqa: E402

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


def _quantiles(x):
    qs = (0.0, 0.5, 0.9, 0.99, 1.0)
    return {f"q{int(100 * q)}": float(np.quantile(x, q)) for q in qs} if len(x) else {}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1,64,1024,8192")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--queries", type=int, default=100)
    ap.add_argument("--oracle-traj", type=int, default=4)
    ap.add_argument("--out", default=os.path.join("profiles", "traj_check.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_traj_check needs a GPU")
    solver = gik_b200.GraspIK(gik_b200.nextage_table(), "cuda:0").attach_scene()
    g = torch.Generator(device="cuda:0").manual_seed(0)
    name, power = _card()

    # ---- the planner experiment: fitted trajectories and their grasp error
    spreads, fitted = [], []
    for sd in (0.1, 0.2, 0.3, 0.4):
        Q = args.queries
        q, pl = experiments.random_endpoints(solver, A, B, (sd, sd, sd), 2 * Q, generator=g)
        qp, _, off, _ = gik_b200.computepath_batch(q[:Q], q[Q:], pl[:Q], pl[Q:], robot=solver, generator=g)
        ctrl, cost = gik_b200.maketraj_paths(q[:Q], q[Q:], qp, off, solver=solver)
        has = (off[1:] > off[:-1])
        ctrl, cost = ctrl[has], cost[has]
        r = gik_b200.check_trajectories_batch(ctrl, solver=solver)
        ge = r["grasp_err"].cpu().numpy()
        reason = r["reason"].cpu().numpy()
        fitted.append(ctrl)
        spreads.append({"std_dev": sd, "queries": Q, "fitted": int(has.sum().item()),
                        "fit_ok": int((cost < 0.15).sum().item()),
                        "valid": int(r["valid"].sum().item()),
                        "first_bad_reason_limits": int(((reason & 1) != 0).sum()),
                        "first_bad_reason_grasp": int(((reason & 2) != 0).sum()),
                        "first_bad_reason_collision": int(((reason & 4) != 0).sum()),
                        "grasp_err": _quantiles(ge),
                        "grasp_err_above": {str(t): int((ge > t).sum()) for t in (1e-3, 3e-3, 1e-2, 3e-2, 1e-1)}})
        print(json.dumps(spreads[-1]), file=sys.stderr)
    pool = torch.cat(fitted)

    # ---- kernel time
    rows = []
    sizes = [int(x) for x in args.sizes.split(",")]
    M = CHECK_SAMPLES
    for dtype in (torch.float32, torch.float64):
        W = torch.as_tensor(sample_weights(pool.shape[1], M), dtype=dtype, device="cuda:0")
        for N in sizes:
            ctrl = pool[torch.arange(N, device=pool.device) % pool.shape[0]].to(dtype).contiguous()
            run = lambda: solver.check_trajectories(ctrl, W, limit_tol=LIMIT_TOL, grasp_tol=GRASP_TOL)
            for _ in range(3):
                run()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.reps):
                out = run()
            e1.record()
            torch.cuda.synchronize()
            t = e0.elapsed_time(e1) / 1e3 / args.reps
            rows.append({"dtype": str(dtype).split(".")[-1], "trajectories": N, "samples": N * M,
                         "call_s": t, "samples_per_s": N * M / t,
                         "valid_fraction": float(out[0].double().mean().item())})
            print(json.dumps(rows[-1]), file=sys.stderr)

    # ---- CPU oracle rate on a subset
    from oracle import c_oracle
    from traj_oracle import oracle_samples
    sub = pool[:args.oracle_traj].double().cpu().numpy()
    t0 = time.perf_counter()
    oracle_samples(c_oracle, solver.table, solver.scene, sub, M, LIMIT_TOL)
    t_or = time.perf_counter() - t0
    oracle = {"trajectories": len(sub), "samples": len(sub) * M, "wall_s": t_or, "samples_per_s": len(sub) * M / t_or,
              "threads": c_oracle.max_threads()}

    res = {"metric": "traj_check", "gpu": name, "power_limit": power, "samples_per_trajectory": M,
           "grasp_tol": GRASP_TOL, "limit_tol": LIMIT_TOL, "kernel": rows, "cpu_oracle": oracle,
           "planner_experiment": spreads,
           "note": "kernel time = CUDA events around the three launches of one gik_traj_check call (init, check, "
                   "finish), averaged over reps after warm-up; trajectories = the fitted planner trajectories, repeated"}
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
