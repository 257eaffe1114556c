#!/usr/bin/env python
"""The reference's three mains in one script, on the GPU and without pinocchio:

  inverse_geometry.py:105-120  -> grasp poses q0 / qe for CUBE_PLACEMENT / CUBE_PLACEMENT_TARGET
  path.py:282-303              -> RRT-connect path that carries the cube over the obstacle
  control.py:431-452           -> Bezier trajectory through the path (closed-form fit)
  control.py:416-463           -> can the trajectory be executed?  (checked at the controller's 1501 sample times)

    python examples/grasp_and_plan.py            (needs a CUDA device)
"""
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gik_b200  # noqa: E402

CUBE_PLACEMENT = (np.eye(3), np.array([0.33, -0.3, 0.93]))           # config.py:36
CUBE_PLACEMENT_TARGET = (np.eye(3), np.array([0.4, 0.11, 0.93]))     # config.py:37


def main():
    robot = cube = None                                  # None = the built-in Nextage table + the packaged scene
    q = np.zeros(15)                                     # robot.q0
    t0 = time.perf_counter()
    q0, successinit = gik_b200.computeqgrasppose(robot, q, cube, CUBE_PLACEMENT)
    qe, successend = gik_b200.computeqgrasppose(robot, q, cube, CUBE_PLACEMENT_TARGET)
    t1 = time.perf_counter()
    print(f"grasp poses: success {successinit}, {successend}  ({(t1 - t0) * 1e3:.1f} ms)")
    if not (successinit and successend):
        print("error: invalid initial or end configuration")
        return 1
    path = gik_b200.computepath(q0, qe, CUBE_PLACEMENT, CUBE_PLACEMENT_TARGET, robot=robot, cube=cube,
                                rng=np.random.default_rng(0), generator=torch.Generator(device="cuda").manual_seed(0))
    t2 = time.perf_counter()
    print(f"path: {len(path)} configurations  ({(t2 - t1) * 1e3:.1f} ms)")
    if not path:
        return 1
    trajs, ok = gik_b200.maketraj(q0, qe, np.array(path), total_time=15.0)
    t3 = time.perf_counter()
    q_of_t, vq_of_t, vvq_of_t = trajs
    print(f"trajectory: degree {q_of_t.degree_}, fit accepted {ok}  ({(t3 - t2) * 1e3:.1f} ms); "
          f"|v(0)| {np.abs(vq_of_t(0.0)).max():.1e}, |a(T)| {np.abs(vvq_of_t(15.0)).max():.1e}")
    verdict = gik_b200.check_trajectory(q_of_t)
    t4 = time.perf_counter()
    print(f"check: valid {verdict['valid']}, first bad sample {verdict['first_bad']} (reason {verdict['reason']}: "
          f"1 limits, 2 grasp, 4 collision), max grasp error {verdict['grasp_err']:.2e}  ({(t4 - t3) * 1e3:.1f} ms)")
    P = np.array(q_of_t.control_points_)[None]
    refined = gik_b200.refine_trajectories_batch(torch.as_tensor(P))
    P[0] = refined["ctrl"][0].cpu().numpy()
    verdict = gik_b200.check_trajectory(gik_b200.Bezier(list(P[0]), t_min=q_of_t.T_min_, t_max=q_of_t.T_max_))
    t5 = time.perf_counter()
    print(f"refined: {int(refined['accepted'][0])} steps, check: valid {verdict['valid']}, first bad sample "
          f"{verdict['first_bad']} (reason {verdict['reason']}), max grasp error {verdict['grasp_err']:.2e}  "
          f"({(t5 - t4) * 1e3:.1f} ms)")
    return 0


if __name__ == "__main__":
    sys.exit(main())
