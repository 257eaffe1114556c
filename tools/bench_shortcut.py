"""Path shortcutting (shortcut_paths_batch) on one GPU: prints one JSON line and writes it to --out.

  * the planner experiment of path_TESTS.py:910-990 (spreads 0.1 .. 0.4, --queries queries each, fp64:
    experiments.random_endpoints + computepath_batch), before and after shortcutting with the defaults: path vertices,
    joint-space length, cube moves above step_size; then maketraj_paths + check_trajectories_batch: valid count, the
    reason of the first bad sample, grasp_err quantiles;
  * the length-per-round curve behind the defaults: the 4 x --queries paths shortcut one round at a time (the same
    draws as one call of that many rounds), for K in --curve-k: per round the share of paths (with >= 3 vertices) that
    accepted a shortcut and the mean length;
  * wall time of one call with the defaults, device-synchronised (host clock around the call and a synchronise,
    median of --reps after a warm-up call), at Q = 100 and Q = 1024 (the experiment's paths repeated), with the number
    of edge launches;
  * all of the above at join_tol 0.5 (GOAL_TOLERANCE) and 0.05.
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
import gik_b200                                                    # noqa: E402
from gik_b200 import experiments, planner                          # noqa: E402
from gik_b200.path import STEP_SIZE                                # noqa: E402

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


def _cat(parts):
    """Concatenate CSR path sets [(q, cube, offsets)]."""
    qs, cs, offs, base = [], [], [torch.zeros(1, dtype=torch.int64, device="cuda:0")], 0
    for q, c, o in parts:
        qs.append(q); cs.append(c); offs.append(o[1:] + base)
        base += q.shape[0]
    return torch.cat(qs), torch.cat(cs), torch.cat(offs)


def _geometry(q, cube, off, solver):
    o = off.cpu().numpy()
    n = np.diff(o)
    cn = cube.double().cpu().numpy()
    big = 0
    for p in range(len(n)):
        if n[p] > 1:
            big += int((np.linalg.norm(np.diff(cn[o[p]:o[p + 1], 9:], axis=0), axis=1) > STEP_SIZE * (1 + 1e-9)).sum())
    _, _, _, st = gik_b200.shortcut_paths_batch(q, cube, off, solver, rounds=0)   # the kernel's length of each path
    L = st["length"].cpu().numpy()
    has = n > 0
    return {"paths": int(has.sum()), "vertices": int(n.sum()), "vertices_mean": float(n[has].mean()),
            "length_sum": float(L[has].sum()), "length_mean": float(L[has].mean()), "cube_moves_above_step": big}


def _check(q0, q1, q, off, solver):
    ctrl, cost = gik_b200.maketraj_paths(q0, q1, q, off, solver=solver)
    has = off[1:] > off[:-1]
    r = gik_b200.check_trajectories_batch(ctrl[has], solver=solver)
    reason, ge = r["reason"].cpu().numpy(), r["grasp_err"].cpu().numpy()
    return {"fitted": int(has.sum().item()), "fit_ok": int((cost[has] < 0.15).sum().item()),
            "valid": int(r["valid"].sum().item()),
            "first_bad_reason_limits": int(((reason & 1) != 0).sum()),
            "first_bad_reason_grasp": int(((reason & 2) != 0).sum()),
            "first_bad_reason_collision": int(((reason & 4) != 0).sum()),
            "grasp_err": _quantiles(ge)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=100)
    ap.add_argument("--curve-rounds", type=int, default=32)
    ap.add_argument("--curve-k", default="8,16,32")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join("profiles", "shortcut.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_shortcut needs a GPU")
    solver = gik_b200.GraspIK(gik_b200.nextage_table(), "cuda:0").attach_scene()
    g = torch.Generator(device="cuda:0").manual_seed(0)
    name, power = _card()

    # ---- the planner experiment's paths (fp64)
    plans = []
    for sd in (0.1, 0.2, 0.3, 0.4):
        Q = args.queries
        q, pl = experiments.random_endpoints(solver, A, B, (sd, sd, sd), 2 * Q, generator=g)
        qp, cp, off, _ = gik_b200.computepath_batch(q[:Q], q[Q:], pl[:Q], pl[Q:], robot=solver, generator=g)
        plans.append((sd, q[:Q], q[Q:], qp, cp, off))
    q_all, c_all, off_all = _cat([(qp, cp, off) for _, _, _, qp, cp, off in plans])

    res = {"metric": "shortcut", "gpu": name, "power_limit": power, "dtype": "float64", "step_size": STEP_SIZE,
           "defaults": {"rounds": planner.SHORTCUT_ROUNDS, "candidates": planner.SHORTCUT_CANDIDATES}, "join_tol": {}}
    for tol in (0.5, 0.05):
        rec = {"spreads": [], "curve": {}, "timing": []}
        # ---- before / after, per spread
        for sd, q0, q1, qp, cp, off in plans:
            gs = torch.Generator(device="cuda:0").manual_seed(1)
            qs, cs, offs, st = gik_b200.shortcut_paths_batch(qp, cp, off, robot=solver, join_tol=tol, generator=gs)
            rec["spreads"].append({"std_dev": sd, "queries": int(off.numel() - 1),
                                   "before": {**_geometry(qp, cp, off, solver), **_check(q0, q1, qp, off, solver)},
                                   "after": {**_geometry(qs, cs, offs, solver), **_check(q0, q1, qs, offs, solver),
                                             "shortcuts_mean": float(st["shortcuts"].double().mean().item())}})
            print(json.dumps({"join_tol": tol, **rec["spreads"][-1]}), file=sys.stderr)
        # ---- length per round
        n_all = np.diff(off_all.cpu().numpy())
        elig0 = n_all > 0
        for K in [int(k) for k in args.curve_k.split(",")]:
            gs = torch.Generator(device="cuda:0").manual_seed(2)
            q, c, o = q_all, c_all, off_all
            _, _, _, st = gik_b200.shortcut_paths_batch(q, c, o, robot=solver, rounds=0)
            rows = [{"round": 0, "length_mean": float(st["length"].cpu().numpy()[elig0].mean())}]
            for r in range(args.curve_rounds):
                elig = np.diff(o.cpu().numpy()) >= 3
                q, c, o, st = gik_b200.shortcut_paths_batch(q, c, o, robot=solver, rounds=1, candidates=K,
                                                            join_tol=tol, generator=gs)
                acc = st["shortcuts"].cpu().numpy() > 0
                rows.append({"round": r + 1, "accept_rate": float(acc[elig].mean()) if elig.any() else 0.0,
                             "length_mean": float(st["length"].cpu().numpy()[elig0].mean()),
                             "vertices": int(o[-1].item())})
            # the same draws in one call: the per-round loop above is that call, round by round
            gs = torch.Generator(device="cuda:0").manual_seed(2)
            one = gik_b200.shortcut_paths_batch(q_all, c_all, off_all, robot=solver, rounds=args.curve_rounds,
                                                candidates=K, join_tol=tol, generator=gs)
            same = bool(torch.equal(one[0], q) and torch.equal(one[2], o))
            rec["curve"][str(K)] = {"rounds": rows, "equals_one_call": same}
            print(json.dumps({"join_tol": tol, "K": K, "curve": [(x["round"], round(x["length_mean"], 4),
                                                                  x.get("accept_rate")) for x in rows]}), file=sys.stderr)
        # ---- wall time per call with the defaults
        for Q in (100, 1024):
            idx = torch.arange(Q, device="cuda:0") % (off_all.numel() - 1)
            o = off_all.cpu()
            parts = [(q_all[o[i]:o[i + 1]], c_all[o[i]:o[i + 1]],
                      torch.tensor([0, int(o[i + 1] - o[i])], device="cuda:0")) for i in idx.tolist()]
            qq, cc, oo = _cat(parts)
            run = lambda: gik_b200.shortcut_paths_batch(qq, cc, oo, robot=solver, join_tol=tol,     # noqa: E731
                                                        generator=torch.Generator(device="cuda:0").manual_seed(3))
            run()
            torch.cuda.synchronize()
            ts = []
            for _ in range(args.reps):
                l0 = solver.launches
                t0 = time.perf_counter()
                out = run()
                torch.cuda.synchronize()
                ts.append(time.perf_counter() - t0)
                launches = solver.launches - l0
            rec["timing"].append({"paths": Q, "vertices_in": int(qq.shape[0]), "vertices_out": int(out[0].shape[0]),
                                  "call_s": float(np.median(ts)), "call_s_all": ts,
                                  "edge_launches": planner.SHORTCUT_ROUNDS, "library_launches": launches})
            print(json.dumps({"join_tol": tol, **rec["timing"][-1]}), file=sys.stderr)
        res["join_tol"][str(tol)] = rec

    res["note"] = ("fp64 planner paths (computepath_batch defaults); lengths are the kernel's fp64 joint-space path "
                   "lengths; timing = host clock around one shortcut_paths_batch call and a device synchronise, median "
                   "of reps after a warm-up call; Q = 1024 repeats the experiment's paths")
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
