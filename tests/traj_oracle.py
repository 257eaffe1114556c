"""Oracle of the trajectory check (include/gik.h, gik_traj_check_*), built from independent pieces: numpy Bernstein
evaluation in fp64, the C oracle's FK and pair distances (oracle/c_oracle.py) and the numpy log6 of oracle/grasp_ik_np.py.
Shared by tests/test_traj_check_cpu.py, tests/test_gpu_traj_check.py and tools/bench_traj_check.py."""
import copy

import numpy as np

from oracle import grasp_ik_np


def list3_pairs(scene, hand_joints):
    """Restatement of list 3 (gik_scene_attach): the scene's pairs without the cube's pairs with a geometry on either
    hand joint, plus the cube's pairs with the table and the obstacle that the scene does not list.  -> [n, 2]."""
    on_hand = {g for g, geom in enumerate(scene.geoms) if geom.joint in hand_joints}
    out = [(int(a), int(b)) for a, b in scene.pairs
           if not ((a == scene.cube and b in on_hand) or (b == scene.cube and a in on_hand))]
    have = {frozenset(p) for p in out}
    for env in (scene.table, scene.obstacle):
        if env >= 0 and scene.cube >= 0 and frozenset((env, scene.cube)) not in have:
            out.append((env, scene.cube))
    return np.array(out, np.int64).reshape(-1, 2)


def sample_weights(n_ctrl, n_samples):
    from math import comb
    u = np.arange(n_samples) / (n_samples - 1)
    d = n_ctrl - 1
    return np.stack([comb(d, i) * u ** i * (1 - u) ** (d - i) for i in range(n_ctrl)], axis=1)


def se3_inv(R, p):
    return R.T, -R.T @ p


def cubes_from_hands(table, hand_R, hand_p):
    """hand frames [2] (R, p) -> the cube placement each implies, C_h = H_h hook_h^-1."""
    out = []
    for h in range(2):
        hR = np.array(table.hook_R[h]).reshape(3, 3)
        hp = np.array(table.hook_p[h])
        iR, ip = se3_inv(hR, hp)
        out.append((hand_R[h] @ iR, hand_p[h] + hand_R[h] @ ip))
    return out


def grasp_error(CL, CR):
    """||log6(C_L^-1 C_R)||_2 with the numpy log6."""
    R = CL[0].T @ CR[0]
    p = CL[0].T @ (CR[1] - CL[1])
    return float(np.linalg.norm(grasp_ik_np.log6(R, p)))


def oracle_samples(c_oracle, table, scene, ctrl, n_samples, limit_tol=1e-6):
    """Per-sample oracle of ctrl [N, n_ctrl, nq] (fp64 numpy) -> dict of [N, M] arrays: q [N, M, nq], the limit
    margin (min over joints of the distance inside the widened limits; < 0 = outside), the grasp error g, the
    collision distance (min of list 3 pairs: mode 0 on the scene with the cube-hand pairs removed, and mode 2), the
    cube placement C_L [N, M, 12]."""
    N, n_ctrl, nq = ctrl.shape
    W = sample_weights(n_ctrl, n_samples)
    q = np.einsum("mi,nij->nmj", W, ctrl).reshape(-1, nq)
    lo = np.asarray(table.lower) - limit_tol
    hi = np.asarray(table.upper) + limit_tol
    margin = np.minimum(q - lo, hi - q).min(axis=1)
    tc = table.to_c()
    HR, Hp = c_oracle.fk(tc, q)
    g = np.empty(len(q))
    CL12 = np.empty((len(q), 12))
    for s in range(len(q)):
        CL, CR = cubes_from_hands(table, HR[s], Hp[s])
        g[s] = grasp_error(CL, CR)
        CL12[s, :9] = CL[0].reshape(9); CL12[s, 9:] = CL[1]
    sc = copy.copy(scene)
    hands = tuple(int(j) for j in table.hand_joint)
    on_hand = {gi for gi, geom in enumerate(scene.geoms) if geom.joint in hands}
    sc.pairs = np.array([(a, b) for a, b in scene.pairs
                         if not ((a == scene.cube and b in on_hand) or (b == scene.cube and a in on_hand))],
                        np.int64).reshape(-1, 2)
    d0 = c_oracle.scene_distance(tc, sc.to_c(), q, CL12, mode=0, cull=0.05)
    d2 = c_oracle.scene_distance(tc, sc.to_c(), None, CL12, mode=2, cull=0.05)
    M = n_samples
    return {"q": q.reshape(N, M, nq), "margin": margin.reshape(N, M), "g": g.reshape(N, M),
            "dist": np.minimum(d0, d2).reshape(N, M), "cube": CL12.reshape(N, M, 12)}


def oracle_flags(o, grasp_tol):
    return ((o["margin"] < 0).astype(np.uint8) | ((o["g"] > grasp_tol).astype(np.uint8) << 1) |
            ((o["dist"] == 0).astype(np.uint8) << 2))


def reduce_flags(flags):
    """sample_flags [N, M] -> (valid, first_bad, reason) as gik_traj_check_* reduces them."""
    bad = flags != 0
    valid = ~bad.any(axis=1)
    first = np.where(valid, -1, bad.argmax(axis=1))
    reason = np.where(valid, 0, flags[np.arange(len(flags)), np.maximum(first, 0)])
    return valid, first.astype(np.int32), reason.astype(np.uint8)
