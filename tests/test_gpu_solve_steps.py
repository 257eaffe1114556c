"""The solve kernels one update at a time: k = 1 or 3 updates of every one of the 18 batch-mode instantiations
(fp32 packed lane / scalar lane / pair, fp64 lane / pair / large-batch pair; each in the spherical-wrist form, the
Nextage-pattern Cholesky form and the generic-table form) against the C oracle's k updates of the same inputs
(fp32-rounded, see cubes_for), problem by problem, within a bound built from the conditioning of each update; the residual the kernels
report, and their stopping decision next to eps, against an fp64 / longdouble recomputation; bit-identical results
at any batch size and column; and short edge marches.

A 1000-iteration descent corrects errors in its own step, so the end-of-solve parity tests (test_gpu_parity.py,
test_gpu_rotations.py) cannot see a step or Jacobian that is slightly wrong; a few updates from the same inputs can.

Bound of q after k updates, per problem (u: unit roundoff of the kernel's type; J_j, Delta_j: the oracle's 12 x 13
active Jacobian and step at its iterate q_j; L = 1 m):
    B = C u sum_{j<k} [1 + dt (L g(J_j) + kappa_j^p |Delta_j|)],   g = max_i s_i / (s_i^2 + lambda) (= 1 / s_min at 0)
kappa is the condition number of the matrices the kernels actually solve with: the 6 x 6 arm blocks A of J (the
chest column enters through a Sherman-Morrison correction), the worse of the two hands.  p = 1 for the wrist form,
whose solves see cond(A), and 2 for the Cholesky normal-equation form, which squares it; with damping kappa^p is
cond(A A^T + lambda I).  (cond(J) itself is no bound: on warm starts where one arm is near a singularity that the
chest column makes up for, J is well conditioned and the measured error of the wrist form is 150 u cond(J) |Delta|.)
C is one constant per dtype and form (STEP_C)."""
import copy
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT, make_poses, rot_rpy
from test_gpu_device_functions import LD, NEAR_PI_SWITCH, exp6_ld, log6_ref, log6_sweep

pytestmark = pytest.mark.gpu
U = {torch.float32: 2.0 ** -24, torch.float64: 2.0 ** -53}
F32, F64 = torch.float32, torch.float64
ACTIVE = [0] + list(range(3, 15))                      # chest + two arms (1, 2: head, passive)

# (dtype, family, form): the 18 batch-mode instantiations.  family -> the kernel argument that selects it
FAMILIES = {F32: {"lane2": "lane", "lane1": "lane1", "pair": "pair"},
            F64: {"lane": "lane", "pair": "pair", "pair_large": "pair"}}
FORMS = ("wrist", "nx", "generic")
INSTANTIATIONS = [(dt, fam, form) for dt in (F32, F64) for fam in FAMILIES[dt] for form in FORMS]
KERNEL_PREFIX = {"lane2": "gik_solve_lane2_kernel", "lane1": "gik_solve_kernel<float", "pair": "gik_solve_pair_kernel<",
                 "lane": "gik_solve_kernel<double", "pair_large": "gik_solve_pair_kernel<double"}
EXERCISED = {}                                         # (dtype, family, form) -> what the step test measured

# Step-bound constant per dtype and form, set so that the largest err / B measured on an NVIDIA B200 (1000 W) is at
# most 0.25; the test asserts err <= B, a margin of 4 for other rounding of the same arithmetic (a rewritten kernel, the
# oracle built for another host CPU -- the fp64 comparison includes the oracle's own Jacobi-SVD rounding).  The worst
# cases are at dt = 1 on warm starts.  Measured C for 0.25: fp32 9.75 / 8.52 / 8.25, fp64 25.6 / 126 / 125 (wrist / nx /
# generic).
STEP_C = {(F32, "wrist"): 10.0, (F32, "nx"): 9.0, (F32, "generic"): 9.0,
          (F64, "wrist"): 26.0, (F64, "nx"): 128.0, (F64, "generic"): 128.0}
# eps of the k-update runs: eps^2 underflows to 0, so no problem stops early (fp64 reaches eps = 1e-12 within three
# full steps from the near-converged starts)
EPS_NEVER = 1e-200
# B holds for every problem but is loose for the typical one: its kappa^p |Delta| term is the worst case over step
# directions.  Median fp32 B measured on the B200: at dt = 1e-2 1.9e-6 (wrist) / 5.6e-6 (nx) / 5.1e-6 (generic), at dt = 1
# 4.8e-5 / 3.2e-4 / 3.3e-4 -- per problem, but for the Cholesky form only 3x below the 1e-3 of the end-of-solve tests.  What makes the dt = 1 runs tight is
# the MEDIAN of err / B, which a wrong constant in every step moves (measured fp32 1.9e-2 / 4.6e-3 / 4.3e-3, fp64 6.0e-3 /
# 2.6e-4 / 3.0e-4): the test holds it at 4x its measured value.
MEDIAN_RATIO = {(F32, "wrist"): 0.08, (F32, "nx"): 0.02, (F32, "generic"): 0.018,
                (F64, "wrist"): 0.024, (F64, "nx"): 1.1e-3, (F64, "generic"): 1.2e-3}


def _iid(x):
    return f"{'f32' if x[0] == F32 else 'f64'}-{x[1]}-{x[2]}"


# ------------------------------------------------------------------------------------------------------ fp64 model
def hook_targets(table, P):
    """cube placements [n, 12] -> hook frames of both hands: R [n, 2, 3, 3], p [n, 2, 3]"""
    Rc = P[:, :9].reshape(-1, 3, 3)
    R = np.stack([Rc @ table.hook_R[h] for h in (0, 1)], 1)
    p = np.stack([P[:, 9:] + Rc @ table.hook_p[h] for h in (0, 1)], 1)
    return R, p


def hand_errors(c_oracle, table, tc, q, P, series_t2=0.0):
    """e_h = log6(hand_h^-1 hook_h) with fp64 FK and the longdouble log6 -> e [n, 2, 6], theta [n, 2].  series_t2: the
    kernel's Num<T>::kSeriesT2 -- on fp32-rounded cubes (rotations orthonormal to 6e-8 only) the series and the closed
    forms of alpha / beta are different functions of the inputs at that level, so the reference takes the kernel's"""
    Rh, ph = c_oracle.fk(tc, q)
    Rt, pt = hook_targets(table, P)
    M = np.einsum("nhji,nhjk->nhik", Rh, Rt)
    d = np.einsum("nhji,nhj->nhi", Rh, pt - ph)
    e, th = log6_ref(M.reshape(-1, 9), d.reshape(-1, 3), series_t2)
    return e.reshape(-1, 2, 6), th.reshape(-1, 2)


# kSeriesT2 of each kernel's log6 (the packed fp32 kernel has no series)
def series_t2(dtype, family):
    return 1e-4 if dtype == F64 else (0.0 if family == "lane2" else 0.25)


def step_terms(c_oracle, table, tc, q, P, lam):
    """at q: (gain g, max_h cond(A_h), max_h cond(A_h A_h^T + lambda I), |Delta|) with the oracle's step Delta = J^T (J J^T
    + lambda I)^-1 e, from the SVDs of the active Jacobian and of its arm blocks"""
    J = c_oracle.jac(tc, q).reshape(len(q), 12, -1)[:, :, ACTIVE]
    e = hand_errors(c_oracle, table, tc, q, P)[0].reshape(-1, 12).astype(np.float64)
    Uu, s, Vt = np.linalg.svd(J, full_matrices=False)
    f = s / (s * s + lam)
    delta = np.einsum("nji,nj->ni", Vt, f * np.einsum("nji,nj->ni", Uu, e))
    sa = np.stack([np.linalg.svd(J[:, 6 * h:6 * h + 6, 1 + 6 * h:7 + 6 * h], compute_uv=False) for h in (0, 1)], 1)
    kap = (sa[:, :, 0] / sa[:, :, -1]).max(1)
    kap2 = ((sa[:, :, 0] ** 2 + lam) / (sa[:, :, -1] ** 2 + lam)).max(1)
    return f.max(1), kap, kap2, np.linalg.norm(delta, axis=1)


def step_bound(c_oracle, table, tc, Q0, P, k, dt, lam, form):
    """sum_{j<k} [1 + dt (L g + kappa^p |Delta|)] at the oracle's iterates (B / (C u)) and the oracle's q_k"""
    S = np.zeros(len(Q0))
    q = Q0
    for j in range(k):
        g, kap, kap2, dn = step_terms(c_oracle, table, tc, q, P, lam)
        S += 1 + dt * (g + (kap if form == "wrist" else kap2) * dn)
        q = c_oracle.solve(tc, Q0, P, eps=EPS_NEVER, dt=dt, max_iters=j + 1, damping=lam)[0]
    return S, q


def clamp_aware_err(q, qo, lo, hi):
    """max_i |q_i - qo_i| of both clamped to the limits: an update that ends just beyond a limit in one and just inside
    it in the other differs by no more than its error, and a limit hides nothing larger"""
    return np.abs(np.clip(q, lo, hi) - np.clip(qo, lo, hi)).max(1)


# ------------------------------------------------------------------------------------------------------ inputs
def r32(a):
    """rounded to fp32, held in fp64: the same values reach the fp32 kernel, the fp64 kernel and the oracle"""
    return np.asarray(a, np.float32).astype(np.float64)


def cubes_for(dtype, P):
    """The cube placements a k-update comparison runs on: fp32-rounded for the fp32 kernels.  The fp64 kernels and their
    oracle run get the fp64 placements: a rounded rotation is orthonormal to 6e-8 only, and there the oracle's log3
    (pinocchio's acos form) and the kernels' atan2 form are different functions at the 1e-8 level -- far above the fp64
    bound, and not an error of either."""
    return r32(P) if dtype == F32 else P


def generic_table(table):
    """a table of the Nextage topology without its zero pattern or tip-aligned hands (test_gpu_parity.
    test_other_robot_tables_generic_instantiation): the TZ = 0 instantiations"""
    rng = np.random.default_rng(17)
    t = copy.deepcopy(table)
    t.joint_p = t.joint_p + rng.uniform(0.004, 0.02, size=t.joint_p.shape) * np.sign(rng.normal(size=t.joint_p.shape))
    t.hand_R = np.array([rot_rpy(0.1, -0.05, 1.2), rot_rpy(-0.08, 0.03, 1.9)])
    t.hand_p = t.hand_p + rng.normal(scale=0.01, size=(2, 3))
    t.hook_R = np.array([rot_rpy(0.02, 0.0, 0.1), rot_rpy(0.0, 0.03, -3.0)])
    t.lower = t.lower * 0.9; t.upper = t.upper * 0.9
    t.meta = {"source": "test"}
    return t


def probe_inputs(c_oracle, table, tc, seed, m=96):
    """Three sets of m problems -> (Q0 [3m, 15] fp32-rounded, P [3m, 12] in fp64, set index [3m]):
    0: zero start over the workspace box, a third of the cubes yawed by up to 0.6 rad, a sixth near a half turn;
    1: warm starts uniform in the limits, with joints at and beyond a limit and joint angles beyond +-pi;
    2: an fp64 solution plus a perturbation of 1e-4 ... 1e-2 (the small-angle path of log6)."""
    rng = np.random.default_rng(seed)
    P0 = make_poses(m, seed)
    for i in range(0, m, 3):
        P0[i, :9] = rot_rpy(0, 0, rng.uniform(-0.6, 0.6)).reshape(9)
    for i in range(1, m, 6):
        P0[i, :9] = rot_rpy(0, 0, np.pi - rng.uniform(1e-3, 0.05) * rng.choice([-1, 1])).reshape(9)
    lo, hi = table.lower, table.upper
    Q1 = rng.uniform(lo, hi, size=(m, 15))
    j = rng.integers(0, 15, size=m)
    Q1[np.arange(0, m, 4), j[::4]] = hi[j[::4]]                          # at the upper limit
    Q1[np.arange(1, m, 4), j[1::4]] = lo[j[1::4]] - 0.05                 # beyond the lower limit
    big = np.flatnonzero(np.minimum(lo, -np.pi) < -np.pi)                # joints whose range passes -pi
    Q1[np.arange(2, m, 4)[:, None], big] = lo[big] + rng.uniform(0, 0.3, (len(np.arange(2, m, 4)), len(big)))
    P1 = make_poses(m, seed + 1)
    Ps = make_poses(8 * m, seed + 2, "sampler")
    qs, oks, _, _ = c_oracle.solve(tc, np.zeros((len(Ps), 15)), Ps)
    take = np.flatnonzero(oks)[:m]
    assert len(take) == m
    Q2 = qs[take] + rng.choice([-1, 1], (m, 15)) * np.exp(rng.uniform(np.log(1e-4), np.log(1e-2), (m, 15)))
    Q2 = np.clip(Q2, lo, hi)
    P2 = Ps[take]
    Q0 = np.concatenate([np.zeros((m, 15)), Q1, Q2]); P = np.concatenate([P0, P1, P2])
    return r32(Q0), P, np.repeat([0, 1, 2], m)


@pytest.fixture(scope="module")
def robots(table, c_oracle):
    import gik_b200
    gt = generic_table(table)
    out = {}
    for name, t in (("nextage", table), ("generic", gt)):
        s = gik_b200.GraspIK(t, "cuda:0")
        tc = t.to_c()
        Q0, P, sets = probe_inputs(c_oracle, t, tc, 11 if name == "nextage" else 12)
        out[name] = (s, t, tc, Q0, P, sets)
    yield out
    for s, *_ in out.values():
        s.close()


def _soa(a, dtype):
    return torch.as_tensor(np.ascontiguousarray(np.asarray(a).T), dtype=dtype, device="cuda:0")


def _np(t):
    return t.double().cpu().numpy() if t.is_floating_point() else t.cpu().numpy()


def f64_hoist_warps():
    """kF64HoistWarps, read from gik_kernels.cu: choose_launch runs the fp64 pair kernel with register-resident constants
    up to 16 * kF64HoistWarps * SMs problems and its large-batch instantiation above"""
    src = open(os.path.join(ROOT, "motion-planning-and-control-for-dual-manipulator-robot_b200", "csrc",
                            "gik_kernels.cu")).read()
    w = int(re.search(r"constexpr int kF64HoistWarps = (\d+);", src).group(1))
    assert re.search(r"k->hoist = sizeof\(T\) == 4 \|\| n <= \(int64_t\)16 \* kF64HoistWarps \* h->sm_count;", src)
    return w


def large_n():
    """the smallest fp64 batch that runs the large-batch pair instantiation"""
    return 16 * f64_hoist_warps() * torch.cuda.get_device_properties(0).multi_processor_count + 1


def kernel_arg(family, form, lam):
    base = FAMILIES[F32].get(family) or FAMILIES[F64][family]
    return base + "+chol" if form == "nx" and lam == 0.0 else base


def run_kernel(s, dtype, family, form, lam, Q0, P, **kw):
    """solve_soa through the instantiation (dtype, family, form); the fp64 large-batch pair instantiation runs the
    problems tiled to more than 16 * kF64HoistWarps * SMs columns -> results of the first copy, and all copies"""
    n = len(Q0)
    reps = -(-large_n() // n) if family == "pair_large" else 1
    q0, pose = _soa(np.tile(Q0, (reps, 1)), dtype), _soa(np.tile(P, (reps, 1)), dtype)
    kern = kernel_arg(family, form, lam)
    # kernel_name reports the undamped launch: a damped one takes the Cholesky form like "+chol" (use_wrist)
    name = s.kernel_name(reps * n, dtype, kern if lam == 0.0 else kern + "+chol")
    assert name.startswith(KERNEL_PREFIX[family]), (family, name)
    assert ("wrist" in name) == (form == "wrist"), (form, lam, name)
    if form == "generic":                   # a table without the Nextage pattern never runs the wrist form
        assert "wrist" not in s.kernel_name(reps * n, dtype, kern.replace("+chol", ""))
    out = s.solve_soa(q0, pose, damping=lam, kernel=kern, **kw)
    full = [_np(x) for x in out]
    first = [x[..., :n] for x in full]
    return first, full, reps


# ------------------------------------------------------------------------------------------------------ A: k updates
ORACLE_CACHE = {}


def oracle_k(c_oracle, rob, name, k, dt, lam, form, dtype):
    key = (name, k, dt, lam, form, dtype)
    if key not in ORACLE_CACHE:
        s, t, tc, Q0, P, _ = rob
        S, qk = step_bound(c_oracle, t, tc, Q0, cubes_for(dtype, P), k, dt, lam, form)
        ORACLE_CACHE[key] = (S, qk)
    return ORACLE_CACHE[key]


@pytest.mark.parametrize("inst", INSTANTIATIONS, ids=_iid)
def test_k_updates_match_oracle(robots, c_oracle, inst):
    dtype, family, form = inst
    name = "generic" if form == "generic" else "nextage"
    rob = robots[name]
    s, t, tc, Q0, P, sets = rob
    P = cubes_for(dtype, P)
    u = U[dtype]
    C = STEP_C[(dtype, form)]
    lams = (0.0,) if form == "wrist" else (0.0, 1e-6, 1e-2)
    ratios, Bs, dts, worst, rk, rpi = [], [], [], [], [], []
    for k in (1, 3):
        for dt in (1e-2, 1.0):
            for lam in lams:
                S, qo = oracle_k(c_oracle, rob, name, k, dt, lam, form, dtype)
                B = C * u * S
                (q, conv, it, res), full, reps = run_kernel(s, dtype, family, form, lam, Q0, P, eps=EPS_NEVER,
                                                            dt=dt, max_iters=k)
                assert (it == k).all() and (conv == 0).all()
                for r in range(1, reps):                                 # every copy of the tiled batch: the same bits
                    assert np.array_equal(full[0][:, r * len(Q0):(r + 1) * len(Q0)], q)
                err = clamp_aware_err(q.T, qo, t.lower, t.upper)
                w = int(np.argmax(err / B))
                worst.append((err[w] / B[w], k, dt, lam, int(sets[w]), err[w], B[w]))
                ratios.append(err / B); Bs.append(B); dts.append(dt)
                # resid: the kernel evaluates the residual again at it == max_iters, so it is that of the RETURNED q
                # (the numpy reference reports its previous iterate's); checked against fp64 at the kernel's q
                e, th = hand_errors(c_oracle, t, tc, q.T, P, series_t2(dtype, family))
                ref = np.sqrt((e.astype(np.float64) ** 2).sum(2)).T
                far = (th < NEAR_PI_SWITCH).T
                rerr = np.abs(res - ref)
                rk.append((rerr[far] / (u * (1 + ref[far]))).max())
                rpi.append(rerr[~far].max(initial=0.0))
    med_B = {d: np.median(np.concatenate([b for b, x in zip(Bs, dts) if x == d])) for d in (1e-2, 1.0)}
    ratios = np.concatenate(ratios); Bs = np.concatenate(Bs)
    EXERCISED[inst] = (ratios.max(), np.median(ratios), med_B[1e-2], med_B[1.0])
    print(f"{_iid(inst)}: err/B max {ratios.max():.3f}, median {np.median(ratios):.2e}, quantiles 0.9/0.99 "
          f"{np.quantile(ratios, 0.9):.2e}/{np.quantile(ratios, 0.99):.2e}; median B {np.median(Bs):.2e} "
          f"(dt = 1e-2: {med_B[1e-2]:.2e}, dt = 1: {med_B[1.0]:.2e}); C for err/B <= 0.25: {4 * C * ratios.max():.3g}; "
          f"worst (ratio, k, dt, lambda, set, err, B) {max(worst)}; "
          f"resid: max err / (u (1 + |e|)) {max(rk):.2f}, near pi {max(rpi):.2e}")
    assert ratios.max() <= 1.0, max(worst)
    assert np.median(ratios) <= MEDIAN_RATIO[(dtype, form)]
    assert max(rk) <= RESID_K[dtype] and max(rpi) <= RESID_NEAR_PI[dtype]
    if dtype == F32:
        assert med_B[1e-2] <= 1e-5, med_B[1e-2]


# ------------------------------------------------------------------------------------------------------ B: residual
# Bars of the residual the kernels report, |resid - ||e||_fp64| <= K u (1 + ||e||) away from pi (the hand pose's
# rounding through FK, of order u times the reach of the arm); near pi, pinocchio's diagonal form: RESID_NEAR_PI.
# Measured on an NVIDIA B200 (1000 W): K = 14.2 (fp32, after k updates; 9.5 at q0) and 4.0 (fp64); near pi 7.5e-7
# (fp32) and 8.9e-16 (fp64).
RESID_K = {F32: 16.0, F64: 8.0}
RESID_NEAR_PI = {F32: 1e-6, F64: 2e-15}


def xi_cubes(c_oracle, table, tc, q_star, xi):
    """cube = FK_L(q*) exp6(xi) hook_L^-1: the left hand's error at q* is xi (up to rounding) -> P [n, 12]"""
    Rh, ph = c_oracle.fk(tc, q_star)
    Re, pe = exp6_ld(xi)
    Re = Re.astype(np.float64).reshape(-1, 3, 3); pe = pe.astype(np.float64)
    RL, pL = Rh[:, 0], ph[:, 0]
    Rg = RL @ Re; pg = pL + np.einsum("nij,nj->ni", RL, pe)                  # hook frame of the left hand
    HR, hp = table.hook_R[0], table.hook_p[0]
    Rc = Rg @ HR.T; pc = pg - np.einsum("nij,j->ni", Rc, hp)
    return np.concatenate([Rc.reshape(-1, 9), pc], 1)


@pytest.fixture(scope="module")
def q_stars(robots, c_oracle):
    """per robot: tightly converged grasps (fp32-rounded), both hands' residual ~1e-12 there"""
    out = {}
    for name, (s, t, tc, *_ ) in robots.items():
        P = make_poses(64, 77, "sampler")
        q, ok, _, _ = c_oracle.solve(tc, np.zeros((len(P), 15)), P)
        q, ok, _, _ = c_oracle.solve(tc, q[ok], P[ok], eps=1e-13, dt=1.0, max_iters=50)
        out[name] = r32(q[ok][:16])
    return out


@pytest.mark.parametrize("inst", INSTANTIATIONS, ids=_iid)
def test_residual_at_q0(robots, q_stars, c_oracle, inst):
    # max_iters = 0: the kernel evaluates the residual at q0 through the real instantiation, q0 returned as is
    dtype, family, form = inst
    name = "generic" if form == "generic" else "nextage"
    s, t, tc, *_ = robots[name]
    xi, theta = log6_sweep(21, per=1)
    qs = q_stars[name][np.arange(len(xi)) % len(q_stars[name])]
    P = r32(xi_cubes(c_oracle, t, tc, qs, xi))
    lam = 1e-6 if form == "nx" else 0.0
    (q, conv, it, res), _, _ = run_kernel(s, dtype, family, form, lam, qs, P, max_iters=0)
    assert (it == 0).all() and (conv == 0).all() and np.array_equal(q.T, qs)
    e, th = hand_errors(c_oracle, t, tc, qs, P, series_t2(dtype, family))
    ref = np.sqrt((e.astype(np.float64) ** 2).sum(2)).T
    u = U[dtype]
    far = (th < NEAR_PI_SWITCH).T
    rerr = np.abs(res - ref)
    k_far = (rerr[far] / (u * (1 + ref[far]))).max()
    print(f"{_iid(inst)}: resid at q0, max err / (u (1 + |e|)) {k_far:.2f} away from pi, max abs err near pi "
          f"{rerr[~far].max(initial=0):.2e} ({(~far).sum()} hands)")
    assert (~far).sum() >= 10
    assert k_far <= RESID_K[dtype]
    assert rerr[~far].max() <= RESID_NEAR_PI[dtype]


@pytest.mark.parametrize("inst", INSTANTIATIONS, ids=_iid)
def test_stopping_next_to_eps(robots, q_stars, c_oracle, inst):
    # max_iters = 1, max(||e_L||, ||e_R||) at eps (1 +- 1e-3) and eps (1 +- 1e-5): every problem further than the
    # residual bound from eps stops with iters = 0, conv = 1 and q returned bit for bit, or takes exactly one update,
    # as its side of eps says; problems within the bound may do either, but nothing else
    dtype, family, form = inst
    name = "generic" if form == "generic" else "nextage"
    s, t, tc, *_ = robots[name]
    eps = 1e-3
    qs = q_stars[name]
    rng = np.random.default_rng(31)
    rel = np.array([1 - 1e-3, 1 + 1e-3, 1 - 1e-5, 1 + 1e-5])
    m = len(qs)
    d = rng.standard_normal((4 * m, 6)); d /= np.linalg.norm(d, axis=1)[:, None]
    Q = np.tile(qs, (4, 1)); target = eps * np.repeat(rel, m)
    scale = target.copy()
    for _ in range(4):                                                   # the max residual of both hands onto target
        Pr = xi_cubes(c_oracle, t, tc, Q, d * scale[:, None])
        e, _ = hand_errors(c_oracle, t, tc, Q, Pr)
        r = np.sqrt((e.astype(np.float64) ** 2).sum(2)).max(1)
        scale *= target / r
    P = r32(xi_cubes(c_oracle, t, tc, Q, d * scale[:, None]))
    e, _ = hand_errors(c_oracle, t, tc, Q, P, series_t2(dtype, family))
    r = np.sqrt((e.astype(np.float64) ** 2).sum(2)).max(1)
    u = U[dtype]
    tol = RESID_K[dtype] * u * (1 + r)
    lam = 1e-6 if form == "nx" else 0.0
    (q, conv, it, res), _, _ = run_kernel(s, dtype, family, form, lam, Q, P, eps=eps, max_iters=1)
    stopped = (it == 0) & (conv == 1) & np.all(q.T == Q, axis=1)
    stepped = (it == 1) & (conv == 0) & np.any(q.T != Q, axis=1)
    assert (stopped | stepped).all()
    below, above = r < eps - tol, r > eps + tol
    print(f"{_iid(inst)}: {below.sum()} below / {above.sum()} above eps beyond the bound, "
          f"{(~below & ~above).sum()} within it")
    assert stopped[below].all() and stepped[above].all()
    assert below.sum() >= m and above.sum() >= m
    if dtype == F64:
        assert (below | above).all()                                   # fp64 resolves eps (1 +- 1e-5)


# ------------------------------------------------------------------------------------------------------ batch position
def _switch_n(s, dtype, pred, kernel=None):
    """smallest n with pred(kernel_name(n)) (monotone in n), by bisection (as __graft_entry__.smoke finds the lane2 size)"""
    lo, hi = 1, 1 << 22
    assert pred(s.kernel_name(hi, dtype, kernel)) and not pred(s.kernel_name(lo, dtype, kernel))
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if pred(s.kernel_name(mid, dtype, kernel)):
            hi = mid
        else:
            lo = mid
    return hi


@pytest.mark.parametrize("dtype", [F32, F64], ids=["f32", "f64"])
def test_batch_size_and_column_do_not_change_results(robots, c_oracle, dtype):
    # a fixed set of probe problems at random columns inside batches whose sizes straddle each launch choice: the same
    # instantiation gives the same bits at any size or column; different instantiations agree within the step bound
    s, t, tc, Q0, P, _ = robots["nextage"]
    P = r32(P)
    probes = np.arange(0, len(Q0), 9)
    sw64 = large_n()
    assert s.kernel_name(sw64 - 1, F64).startswith("gik_solve_pair_kernel<double")
    rng = np.random.default_rng(55)
    filler = r32(make_poses(1 << 17, 56))
    by_family = {}
    for lam in (0.0, 1e-6):
        # the fp32 pair <-> lane2 switch depends on the occupancy of the form's lane2 kernel: a damped launch is a
        # "+chol" one (kernel_name reports undamped launches)
        karg = None if lam == 0.0 else "auto+chol"
        sw32 = _switch_n(s, F32, lambda nm: nm.startswith("gik_solve_lane2"), karg)
        sizes = [1, 31, 33] + ([sw32 - 1, sw32] if dtype == F32 else [sw64 - 1, sw64, sw64 + 1])
        for n in sizes:
            pr = probes[:n]
            cols = np.sort(rng.choice(n, size=len(pr), replace=False))
            Qb = np.zeros((n, 15)); Pb = filler[:n].copy()
            Qb[cols] = Q0[pr]; Pb[cols] = P[pr]
            nm = s.kernel_name(n, dtype, karg)
            fam = ("lane2" if "lane2" in nm else "pair") if dtype == F32 else \
                ("pair_large" if n >= sw64 else "pair")
            out = s.solve_soa(_soa(Qb, dtype), _soa(Pb, dtype), eps=EPS_NEVER, dt=1.0, max_iters=3, damping=lam)
            q = _np(out[0])[:, cols]; res = _np(out[3])[:, cols]
            key = (fam, lam)
            ref = by_family.setdefault(key, {})
            for j, p in enumerate(pr):
                if p in ref:
                    assert np.array_equal(ref[p][0], q[:, j]) and np.array_equal(ref[p][1], res[:, j]), (key, n, p)
                else:
                    ref[p] = (q[:, j], res[:, j])
    fams = sorted({f for f, _ in by_family})
    assert fams == (["lane2", "pair"] if dtype == F32 else ["pair", "pair_large"])
    for lam in (0.0, 1e-6):
        a, b = by_family[(fams[0], lam)], by_family[(fams[1], lam)]
        common = sorted(set(a) & set(b))
        assert common
        d = np.array([np.abs(a[p][0] - b[p][0]).max() for p in common])
        if dtype == F64:
            assert (d == 0).all()                              # fp64 families run the same operations: the same bits
        else:                                                  # each within B / 4 of the oracle: within B / 2 of each other
            form = "wrist" if lam == 0.0 else "nx"
            B = STEP_C[(F32, form)] * U[F32] * oracle_k(c_oracle, robots["nextage"], "nextage", 3, 1.0, lam, form, F32)[0]
            assert (d <= 0.5 * B[common]).all(), (d / B[common]).max()
        print(f"{'f32' if dtype == F32 else 'f64'} lambda {lam}: {fams} agree to {d.max():.2e} on {len(common)} probes")


# ------------------------------------------------------------------------------------------------------ edge mode
EDGE_FAMILIES = [(F32, "lane"), (F32, "pair"), (F32, "lane1"), (F64, "lane"), (F64, "pair")]
# (margin of a stopping decision from eps, |q_path - oracle|); measured on an NVIDIA B200 (1000 W): 5.7e-7 / 6.7e-16
EDGE_TOL = {F32: (1e-6, 2e-6), F64: (1e-9, 1e-14)}


@pytest.fixture(scope="module")
def edge_case(robots, c_oracle):
    """64 edges from converged starts, 1-3 steps of ~0.4 mm each, and the oracle's march; per edge the smallest
    distance |max(||e_L||, ||e_R||) - eps| over the oracle's stopping decisions (replayed step by step)"""
    s, t, tc, *_ = robots["nextage"]
    rng = np.random.default_rng(61)
    E = 64
    A = make_poses(4 * E, 62, "sampler")
    q, ok, _, _ = c_oracle.solve(tc, np.zeros((len(A), 15)), A)
    A, q0 = A[ok][:E], q[ok][:E]
    ns = rng.integers(1, 4, size=E).astype(np.int32)
    B = A.copy()
    B[:, 9:] += rng.uniform(-1, 1, (E, 3)) * 4e-4 * ns[:, None]
    A, B, q0 = r32(A), r32(B), r32(q0)
    path, nv, itt = c_oracle.project_edges(tc, q0, A, B, ns, 3)
    margin = np.full(E, np.inf)
    qcur = q0.copy()
    for st in range(3):
        live = np.flatnonzero(nv > st)
        if not len(live):
            break
        cube = c_oracle.interpolate(A[live], B[live], (st + 1) / ns[live])
        done = np.zeros(len(live), bool)
        for j in range(1001):
            qj = c_oracle.solve(tc, qcur[live], cube, eps=1e-12, max_iters=j)[0]
            e, _ = hand_errors(c_oracle, t, tc, qj, cube)
            r = np.sqrt((e.astype(np.float64) ** 2).sum(2)).max(1)
            margin[live[~done]] = np.minimum(margin[live[~done]], np.abs(r - 1e-3)[~done])
            done |= r < 1e-3
            if done.all():
                break
        qcur[live] = path[live, st]
    return A, B, q0, ns, path, nv, itt, margin


@pytest.mark.parametrize("dtype,kern", EDGE_FAMILIES, ids=lambda x: x if isinstance(x, str) else str(x)[6:])
def test_edge_marches_match_oracle(robots, edge_case, dtype, kern):
    s = robots["nextage"][0]
    A, B, q0, ns, path_o, nv_o, it_o, margin = edge_case
    m_tol, q_tol = EDGE_TOL[dtype]
    path, nv, itt = s.project_edges_soa(_soa(q0, dtype), _soa(A, dtype), _soa(B, dtype),
                                        torch.as_tensor(ns, device="cuda:0"), 3, kernel=kern)
    path = _np(path).transpose(2, 0, 1); nv = _np(nv); itt = _np(itt)
    clear = margin > m_tol
    assert clear.sum() >= len(A) // 2 and (nv_o[clear] >= 1).all()
    assert np.array_equal(nv[clear], nv_o[clear]) and np.array_equal(itt[clear], it_o[clear])
    d = max(np.abs(path[e, :nv[e]] - path_o[e, :nv[e]]).max(initial=0) for e in np.flatnonzero(clear))
    print(f"edges {dtype} {kern}: {clear.sum()} of {len(A)} clear of eps, {it_o[clear].mean():.1f} iterations per edge, "
          f"max |q_path - oracle| {d:.2e}")
    assert d <= q_tol
    EXERCISED[("edges", dtype, kern)] = d


# ------------------------------------------------------------------------------------------------------ completeness
def test_every_instantiation_was_exercised(request):
    # reads what the step and edge tests of this module recorded: meaningful only when they ran in this session
    names = {it.originalname for it in request.session.items}
    if not {"test_k_updates_match_oracle", "test_edge_marches_match_oracle"} <= names:
        pytest.skip("the step and edge tests of this module were not selected in this session")
    missing = [_iid(x) for x in INSTANTIATIONS if x not in EXERCISED]
    assert len(INSTANTIATIONS) == 18 and not missing, missing
    assert all(("edges", dt, k) in EXERCISED for dt, k in EDGE_FAMILIES)
    for x in INSTANTIATIONS:
        mx, med, mb, mb1 = EXERCISED[x]
        print(f"{_iid(x):22s} err/B max {mx:.3f} median {med:.2e}  median B dt = 1e-2 {mb:.2e}, dt = 1 {mb1:.2e}")
