"""The reference's IK robustness experiment (inverse_geometry_TESTS.py:474-561) at batch scale: for each Gaussian
spread, sample cube placements around the point 0.3 m above the obstacle (clipped to the box spanned by the two cube
placements +- 0.14 m, identity rotation), discard placements where the cube itself collides (:500-505), solve the grasp
IK from robot.q0 with the full success predicate (:508) and report the success rate.  The reference runs 300 trials per
spread one solve at a time; here every spread is one batched solve + one batched collision test."""
from __future__ import annotations

import numpy as np
import torch

from .inverse_geometry import _pose_to_array, solver_for
from .ops import as_pose12

OBSTACLE_POSITION = (0.43, -0.1, 0.94)       # inverse_geometry_TESTS.py:480
GAUSSIAN_OFFSET = (0.0, 0.0, 0.3)            # :481
MARGIN = 0.14                                # :484
STD_DEVS = tuple((s, s, s) for s in (0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7))    # :530


def sample_gaussian_placements(n, cubeplacementq0, cubeplacementqgoal, std_dev, *, device, dtype=torch.float64,
                               generator=None):
    """n clipped-Gaussian translations (inverse_geometry_TESTS.py:480-495) -> [n,3]."""
    a, b = _pose_to_array(cubeplacementq0)[9:], _pose_to_array(cubeplacementqgoal)[9:]
    lo = torch.tensor(np.minimum(a, b) - MARGIN, dtype=dtype, device=device)
    hi = torch.tensor(np.maximum(a, b) + MARGIN, dtype=dtype, device=device)
    centre = torch.tensor(np.add(OBSTACLE_POSITION, GAUSSIAN_OFFSET), dtype=dtype, device=device)
    sd = torch.tensor(std_dev, dtype=dtype, device=device)
    x = centre + sd * torch.randn((n, 3), dtype=dtype, device=device, generator=generator)
    return torch.minimum(torch.maximum(x, lo), hi)


def grasp_success_rate(robot, cubeplacementq0, cubeplacementqgoal, std_devs=STD_DEVS, trials=300, *, dtype=torch.float64,
                       generator=None, oversample=4, descend_while_colliding=True):
    """Returns [(std_dev, success_rate_percent, trials)] like the table the reference prints (:556-561)."""
    solver = solver_for(robot)
    solver._need_scene()
    out = []
    for sd in std_devs:
        kept = []
        need = trials
        while need > 0:
            pl = sample_gaussian_placements(max(need * oversample, 64), cubeplacementq0, cubeplacementqgoal, sd,
                                            device=solver.device, dtype=dtype, generator=generator)
            p12 = as_pose12(pl, dtype=dtype, device=solver.device)
            free = ~solver.cube_collision_soa(p12.t().contiguous()).bool()      # resample while the cube collides
            good = p12[free][:need]
            kept.append(good)
            need -= good.shape[0]
        P = torch.cat(kept, 0)
        q0 = torch.zeros((solver.nq, P.shape[0]), dtype=dtype, device=solver.device)
        _, succ, _, _, _ = solver.solve_success_soa(q0, P.t().contiguous(), descend_while_colliding=descend_while_colliding)
        out.append((tuple(sd), 100.0 * float(succ.double().mean().item()), int(P.shape[0])))
    return out


def _random_endpoint(solver, a, b, sd, dtype, generator, batch=256):
    """path_TESTS.sample_random_cube_placement: a clipped-Gaussian cube placement with a valid, collision-free grasp
    configuration that keeps the 0.04 m clearance (the same acceptance rule as path.sample_cube_placement)."""
    while True:
        pl = sample_gaussian_placements(batch, a, b, sd, device=solver.device, dtype=dtype, generator=generator)
        p12 = as_pose12(pl, dtype=dtype, device=solver.device).t().contiguous()
        q0 = torch.zeros((solver.nq, batch), dtype=dtype, device=solver.device)
        q, succ, _, _, _ = solver.solve_success_soa(q0, p12, descend_while_colliding=False, early_stop=True)
        ok = succ.bool() & ~solver.cube_collision_soa(p12).bool() & solver.clearance_soa(q, p12, 0.04).bool()
        idx = torch.nonzero(ok).flatten()
        if idx.numel():
            i = int(idx[0])
            return q[:, i].double().cpu().numpy(), (np.eye(3), pl[i].double().cpu().numpy())


def rrt_connect_trials(robot, cubeplacementq0, cubeplacementqgoal, std_devs=STD_DEVS[:4], trials=100, *,
                       dtype=torch.float64, generator=None, rng=None, expand=8):
    """The reference's planner experiment (path_TESTS.py:910-990): for each spread, `trials` planning queries between
    two random valid cube placements; success rate, wall time and RRT iteration statistics per spread."""
    import time
    from .path import computepath
    solver = solver_for(robot)
    solver._need_scene()
    rng = rng if rng is not None else np.random.default_rng()
    results = []
    for sd in std_devs:
        times, iters, wins = [], [], 0
        for _ in range(trials):
            q_init, c0 = _random_endpoint(solver, cubeplacementq0, cubeplacementqgoal, sd, dtype, generator)
            q_goal, c1 = _random_endpoint(solver, cubeplacementq0, cubeplacementqgoal, sd, dtype, generator)
            t0 = time.perf_counter()
            path, stats = computepath(q_init, q_goal, c0, c1, robot=solver, rng=rng, generator=generator, dtype=dtype,
                                      expand=expand, return_stats=True)
            times.append(time.perf_counter() - t0)
            iters.append(stats["iterations"])
            wins += bool(path)
        results.append({"std_dev": tuple(sd), "success_rate": 100.0 * wins / trials,
                        "avg_time": float(np.mean(times)), "max_time": float(np.max(times)), "min_time": float(np.min(times)),
                        "std_time": float(np.std(times)), "avg_iterations": float(np.mean(iters)),
                        "max_iterations": int(np.max(iters)), "min_iterations": int(np.min(iters)),
                        "std_iterations": float(np.std(iters))})
    return results


def random_endpoints(robot, cubeplacementq0, cubeplacementqgoal, std_dev, n, *, dtype=torch.float64, generator=None,
                     oversample=4):
    """n endpoints of path_TESTS.sample_random_cube_placement drawn in batch with the acceptance rule of
    `_random_endpoint` (valid grasp, cube and robot collision-free, 0.04 m clearance): candidates are drawn and
    validated `oversample * n` at a time and the valid ones are taken in draw order.  -> (q [n,nq], placements [n,3])."""
    solver = solver_for(robot)
    solver._need_scene()
    qs, ps, need = [], [], n
    while need > 0:
        m = max(need * oversample, 256)
        pl = sample_gaussian_placements(m, cubeplacementq0, cubeplacementqgoal, std_dev, device=solver.device, dtype=dtype,
                                        generator=generator)
        p12 = as_pose12(pl, dtype=dtype, device=solver.device).t().contiguous()
        q0 = torch.zeros((solver.nq, m), dtype=dtype, device=solver.device)
        q, succ, _, _, _ = solver.solve_success_soa(q0, p12, descend_while_colliding=False, early_stop=True)
        ok = succ.bool() & ~solver.cube_collision_soa(p12).bool() & solver.clearance_soa(q, p12, 0.04).bool()
        idx = torch.nonzero(ok).flatten()[:need]
        qs.append(q.t()[idx]); ps.append(pl[idx])
        need -= idx.numel()
    return torch.cat(qs), torch.cat(ps)


def rrt_connect_trials_batch(robot, cubeplacementq0, cubeplacementqgoal, std_devs=STD_DEVS[:4], trials=100, *,
                             dtype=torch.float64, generator=None, expand=8):
    """`rrt_connect_trials` with every query of a spread in ONE computepath_batch call: the same dict keys per spread.
    Times are AMORTISED per query -- the device-synchronised wall time of the batched call divided by `trials` -- so
    avg_time = max_time = min_time and std_time = 0; the iteration statistics are per query."""
    import time
    from .planner import computepath_batch
    solver = solver_for(robot)
    solver._need_scene()
    results = []
    for sd in std_devs:
        q, pl = random_endpoints(solver, cubeplacementq0, cubeplacementqgoal, sd, 2 * trials, dtype=dtype,
                                 generator=generator)
        torch.cuda.synchronize(solver.device)
        t0 = time.perf_counter()
        _, _, offsets, stats = computepath_batch(q[:trials], q[trials:], pl[:trials], pl[trials:], robot=solver,
                                                 generator=generator, dtype=dtype, expand=expand)
        torch.cuda.synchronize(solver.device)
        t = (time.perf_counter() - t0) / trials
        wins = int((offsets[1:] > offsets[:-1]).sum().item())
        iters = stats["iterations"].cpu().numpy()
        results.append({"std_dev": tuple(sd), "success_rate": 100.0 * wins / trials,
                        "avg_time": t, "max_time": t, "min_time": t, "std_time": 0.0,
                        "avg_iterations": float(np.mean(iters)), "max_iterations": int(np.max(iters)),
                        "min_iterations": int(np.min(iters)), "std_iterations": float(np.std(iters))})
    return results
