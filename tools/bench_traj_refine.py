"""Trajectory refinement (refine_trajectories_batch) on one GPU: prints one JSON line and writes it to --out.

  * the planner experiment of path_TESTS.py:910-990 (spreads 0.1 .. 0.4, --queries queries each, fp64:
    experiments.random_endpoints + computepath_batch), raw paths and paths shortcut with the defaults (the seeds of
    tools/bench_shortcut.py), through maketraj_paths -> check -> refine (defaults) -> check: valid counts before and
    after, the reason of the first bad sample, grasp_err quantiles, the share of right-arm free control points outside
    the joint limits before refinement, and how many valid trajectories become invalid (and the reverse);
  * the table behind the defaults: every fitted trajectory of the experiment (raw and shortcut) refined with max_iters
    in {1, 2, 4, 8, 16, 32} and n_samples in {301, 1501}, then checked at 1501 samples: mean and max grasp_err, valid
    count;
  * time per call: CUDA events around --reps calls after a warm-up of every shape, N in {1, 64, 1024, 8192}
    trajectories (the experiment's raw and shortcut trajectories repeated), fp32 and fp64, 1501 samples, for each
    max_iters of --speed-iters, with the mean number of trial steps.
The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import gik_b200                                                    # noqa: E402
from gik_b200 import experiments, trajectory                       # noqa: E402

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
    return {"q50": float(np.quantile(x, 0.5)), "q90": float(np.quantile(x, 0.9)), "max": float(np.max(x))} if len(x) else {}


def _verdict(r):
    reason, ge = r["reason"].cpu().numpy(), r["grasp_err"].cpu().numpy()
    return {"valid": int(r["valid"].sum().item()),
            "first_bad_reason_limits": int(((reason & 1) != 0).sum()),
            "first_bad_reason_grasp": int(((reason & 2) != 0).sum()),
            "first_bad_reason_collision": int(((reason & 4) != 0).sum()),
            "grasp_err": _quantiles(ge)}


def _right_arm(table):
    chain, k = [], int(table.hand_joint[1])
    while k >= 0:
        chain.append(k); k = int(table.parent[k])
    return chain[::-1][1:]


def _pipeline(ctrl, solver, table):
    """check -> refine (defaults) -> check on fitted trajectories ctrl [N, 21, 15]."""
    arm = _right_arm(table)
    x = ctrl[:, 3:-3][:, :, arm].cpu().numpy()
    lo, hi = np.asarray(table.lower)[arm], np.asarray(table.upper)[arm]
    outside = float(((x < lo) | (x > hi)).mean())
    before = gik_b200.check_trajectories_batch(ctrl, solver=solver)
    ref = gik_b200.refine_trajectories_batch(ctrl, solver=solver)
    after = gik_b200.check_trajectories_batch(ref["ctrl"], solver=solver)
    vb, va = before["valid"].cpu().numpy(), after["valid"].cpu().numpy()
    return {"fitted": int(ctrl.shape[0]), "right_arm_free_ctrl_outside_limits": outside,
            "before": _verdict(before), "after": _verdict(after),
            "valid_to_invalid": int((vb & ~va).sum()), "invalid_to_valid": int((~vb & va).sum()),
            "iters_mean": float(ref["iters"].double().mean().item()),
            "accepted_mean": float(ref["accepted"].double().mean().item())}


def _sum(rows, side):
    out = {k: sum(r[side][k] for r in rows) for k in ("valid", "first_bad_reason_limits", "first_bad_reason_grasp",
                                                      "first_bad_reason_collision")}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=100)
    ap.add_argument("--sizes", default="1,64,1024,8192")
    ap.add_argument("--speed-iters", default="4,8,16")
    ap.add_argument("--table-iters", default="1,2,4,8,16,32")
    ap.add_argument("--table-samples", default="301,1501")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join("profiles", "traj_refine.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_traj_refine needs a GPU")
    solver = gik_b200.GraspIK(gik_b200.nextage_table(), "cuda:0").attach_scene()
    table = solver.table
    g = torch.Generator(device="cuda:0").manual_seed(0)
    name, power = _card()

    # ---- the planner experiment (fp64), raw and shortcut
    exp = {"raw": [], "shortcut": []}
    pools = {"raw": [], "shortcut": []}
    for sd in (0.1, 0.2, 0.3, 0.4):
        Q = args.queries
        q, pl = experiments.random_endpoints(solver, A, B, (sd, sd, sd), 2 * Q, generator=g)
        qp, cp, off, _ = gik_b200.computepath_batch(q[:Q], q[Q:], pl[:Q], pl[Q:], robot=solver, generator=g)
        gs = torch.Generator(device="cuda:0").manual_seed(1)
        qs, _, offs, _ = gik_b200.shortcut_paths_batch(qp, cp, off, robot=solver, generator=gs)
        for kind, (qq, oo) in (("raw", (qp, off)), ("shortcut", (qs, offs))):
            ctrl, _ = gik_b200.maketraj_paths(q[:Q], q[Q:], qq, oo, solver=solver)
            ctrl = ctrl[oo[1:] > oo[:-1]]
            pools[kind].append(ctrl)
            exp[kind].append({"std_dev": sd, "queries": Q, **_pipeline(ctrl, solver, table)})
            print(json.dumps({"kind": kind, **exp[kind][-1]}), file=sys.stderr)
    totals = {k: {"before": _sum(v, "before"), "after": _sum(v, "after"),
                  "valid_to_invalid": sum(r["valid_to_invalid"] for r in v),
                  "invalid_to_valid": sum(r["invalid_to_valid"] for r in v)} for k, v in exp.items()}
    pools = {k: torch.cat(v) for k, v in pools.items()}

    # ---- the table behind the defaults
    grid = []
    for kind, ctrl in pools.items():
        for M in [int(x) for x in args.table_samples.split(",")]:
            for it in [int(x) for x in args.table_iters.split(",")]:
                r = gik_b200.refine_trajectories_batch(ctrl, n_samples=M, max_iters=it, solver=solver)
                c = gik_b200.check_trajectories_batch(r["ctrl"], solver=solver)
                ge = c["grasp_err"].cpu().numpy()
                grid.append({"kind": kind, "n_samples": M, "max_iters": it, "grasp_err_mean": float(ge.mean()),
                             "grasp_err_max": float(ge.max()), "valid": int(c["valid"].sum().item()),
                             "trajectories": int(ctrl.shape[0]),
                             "iters_mean": float(r["iters"].double().mean().item())})
                print(json.dumps(grid[-1]), file=sys.stderr)

    # ---- time per call
    pool = torch.cat([pools["raw"], pools["shortcut"]])
    W = trajectory.sample_weights(pool.shape[1], trajectory.CHECK_SAMPLES)
    speed = []
    for dtype in (torch.float32, torch.float64):
        Wd = torch.as_tensor(W, dtype=dtype, device="cuda:0")
        for it in [int(x) for x in args.speed_iters.split(",")]:
            for N in [int(x) for x in args.sizes.split(",")]:
                ctrl = pool[torch.arange(N, device=pool.device) % pool.shape[0]].to(dtype).contiguous()
                run = lambda: solver.refine_trajectories(ctrl, Wd, max_iters=it, tol=trajectory.REFINE_TOL,   # noqa: E731
                                                         damping=trajectory.REFINE_DAMPING)
                out = run()
                torch.cuda.synchronize()
                reps = max(1, min(args.reps, (8 * args.reps * 64) // max(N, 64)))
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(reps):
                    out = run()
                e1.record()
                torch.cuda.synchronize()
                t = e0.elapsed_time(e1) / 1e3 / reps
                speed.append({"dtype": str(dtype).split(".")[-1], "max_iters": it, "trajectories": N, "reps": reps,
                              "call_s": t, "trajectories_per_s": N / t,
                              "iters_mean": float(out[4].double().mean().item())})
                print(json.dumps(speed[-1]), file=sys.stderr)

    res = {"metric": "traj_refine", "gpu": name, "power_limit": power, "dtype_experiment": "float64",
           "defaults": {"max_iters": trajectory.REFINE_ITERS, "tol": trajectory.REFINE_TOL,
                        "damping": trajectory.REFINE_DAMPING, "n_samples": trajectory.CHECK_SAMPLES},
           "planner_experiment": exp, "totals": totals, "defaults_table": grid, "speed": speed,
           "note": "check = check_trajectories_batch defaults (1501 samples, grasp_tol 1e-2); refine = "
                   "refine_trajectories_batch defaults unless stated; speed = CUDA events around reps calls of one "
                   "gik_traj_refine launch after a warm-up call, 1501 samples, tol = REFINE_TOL; trajectories = the "
                   "experiment's raw and shortcut fitted trajectories, repeated"}
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
