"""Bezier trajectory through a planned path: the reference's `control.Bezier` / `maketraj` (control.py:18-195) with
the fit done in closed form.

The reference minimises  sum_k ||B(t_k) - q_k||^2  over the 21 control points of a degree-20 Bezier curve with SLSQP
under six equality constraints: position, velocity and acceleration at both ends (control.py:110-158).  For a Bezier
curve those constraints are LINEAR in the control points and decouple completely:
    B(0) = P0 = q0,  B'(0) = n (P1 - P0) / T = 0,  B''(0) = n (n-1) (P2 - 2 P1 + P0) / T^2 = 0   =>  P0 = P1 = P2 = q0
and likewise P_n = P_{n-1} = P_{n-2} = q1 (the reference's own saved results, trajectory*.json, show exactly that).  What
is left is an unconstrained linear least-squares problem in the free control points P3 .. P_{n-3} with the Bernstein
matrix as design matrix, identical for every joint: one small `lstsq`, deterministic, instead of an iterative solver
that "works 90 percent of the time ... pretty slow" (control.py:192).  `maketraj_batch` fits many paths at once
(SURVEY 8f-4): the design matrix is the same for every path with the same number of points, so it is factored ONCE on the
host in fp64 (`fit_operands`: Bernstein basis of the free control points and its pseudo-inverse) and CUDA tensors go
through one launch of `gik_bezier_fit_*` (csrc/gik_bezier.cuh: a warp per path, operands in shared memory, the path read
once); CPU tensors / numpy take the same two matrix products in numpy.  `maketraj` (one path, the reference's call) is the
numpy form."""
from __future__ import annotations

import json
from math import comb

import numpy as np

DEGREE = 20              # control.py:87
COST_OK = 0.15           # control.py:185: the fit is accepted when the residual cost is below this


class Bezier:
    """Same interface as control.Bezier (control.py:18-60): callable on t in [t_min, t_max], `derivative(order)`."""

    def __init__(self, pointlist, t_min=0.0, t_max=1.0, mult_t=1.0):
        self.control_points_ = [np.asarray(p, dtype=float) for p in pointlist]
        self.dim_ = self.control_points_[0].shape[0]
        self.T_min_, self.T_max_, self.mult_T_ = float(t_min), float(t_max), float(mult_t)
        self.size_ = self.degree_ = len(self.control_points_) - 1
        if self.size_ < 1 or self.T_max_ <= self.T_min_:
            raise ValueError(f"Bezier: needs at least two control points and t_min < t_max (got {len(self.control_points_)} points, [{self.T_min_}, {self.T_max_}])")

    def __call__(self, t):
        if not (self.T_min_ <= t <= self.T_max_):
            raise ValueError(f"Bezier: t = {t} is outside [{self.T_min_}, {self.T_max_}]")
        u = (t - self.T_min_) / (self.T_max_ - self.T_min_)
        pts = np.array(self.control_points_)
        for _ in range(self.degree_):                      # de Casteljau
            pts = (1.0 - u) * pts[:-1] + u * pts[1:]
        return self.mult_T_ * pts[0]

    def derivative(self, order):
        if order == 0:
            return self
        d = [self.degree_ * (b - a) for a, b in zip(self.control_points_[:-1], self.control_points_[1:])]
        return Bezier(d, self.T_min_, self.T_max_, self.mult_T_ / (self.T_max_ - self.T_min_)).derivative(order - 1)


def bernstein_matrix(degree: int, u: np.ndarray) -> np.ndarray:
    """[len(u), degree+1] Bernstein basis values."""
    u = np.asarray(u, float)[:, None]
    i = np.arange(degree + 1)[None, :]
    c = np.array([comb(degree, k) for k in range(degree + 1)], float)[None, :]
    return c * u ** i * (1.0 - u) ** (degree - i)


def _fit(q0, q1, path_points, degree, xp):
    """Closed-form constrained fit; xp = numpy or torch namespace.  path_points [..., n_points, dim]."""
    n_points = path_points.shape[-2]
    B = bernstein_matrix(degree, np.linspace(0.0, 1.0, n_points))           # times = linspace(0, T, n_points), control.py:95
    fixed0, fixed1, free = slice(0, 3), slice(degree - 2, degree + 1), slice(3, degree - 2)
    w0, w1 = B[:, fixed0].sum(1), B[:, fixed1].sum(1)
    if xp is np:
        rhs = path_points - w0[:, None] * q0[..., None, :] - w1[:, None] * q1[..., None, :]
        Pf = np.linalg.lstsq(B[:, free], rhs, rcond=None)[0] if rhs.ndim == 2 else np.linalg.pinv(B[:, free]) @ rhs
        cost = ((B[:, free] @ Pf - rhs) ** 2).sum(axis=(-2, -1))
        return Pf, cost
    import torch
    Bt = torch.as_tensor(B, dtype=path_points.dtype, device=path_points.device)
    rhs = path_points - Bt[:, fixed0].sum(1)[:, None] * q0[..., None, :] - Bt[:, fixed1].sum(1)[:, None] * q1[..., None, :]
    Pf = torch.linalg.pinv(Bt[:, free]) @ rhs                                # one batched solve for every path and joint
    cost = ((Bt[:, free] @ Pf - rhs) ** 2).sum(dim=(-2, -1))
    return Pf, cost


def maketraj(q0, q1, path_points, total_time, degree=DEGREE):
    """Drop-in for control.maketraj (control.py:63-195): returns ([q_of_t, vq_of_t, vvq_of_t], ok) with ok = the
    residual cost is below 0.15 (control.py:185-195)."""
    q0, q1 = np.asarray(q0, float), np.asarray(q1, float)
    path_points = np.asarray(path_points, float)
    if degree < 6:
        raise ValueError("degree must be at least 6 (three control points are pinned at each end)")
    Pf, cost = _fit(q0, q1, path_points, degree, np)
    P = [q0.copy() for _ in range(3)] + [p for p in Pf] + [q1.copy() for _ in range(3)]
    q_of_t = Bezier(P, t_min=0.0, t_max=total_time)
    return [q_of_t, q_of_t.derivative(1), q_of_t.derivative(2)], bool(cost < COST_OK)


def fit_operands(degree: int, n_points: int):
    """The factored design matrix of the fit for paths of `n_points` points (fp64 numpy):
    (pinv [n_free, n_points], basis [n_points, n_free], w0 [n_points], w1 [n_points]) -- Bernstein values of the free
    control points 3 .. degree-3 at times linspace(0, 1, n_points) (control.py:95), their pseudo-inverse, and the summed
    basis values of the three pinned control points at each end."""
    if degree < 6:
        raise ValueError("degree must be at least 6 (three control points are pinned at each end)")
    B = bernstein_matrix(degree, np.linspace(0.0, 1.0, n_points))
    Bf = B[:, 3:degree - 2]
    return np.linalg.pinv(Bf), Bf.copy(), B[:, :3].sum(1), B[:, degree - 2:].sum(1)


def maketraj_batch(q0, q1, path_points, degree=DEGREE, solver=None):
    """Many paths at once: q0, q1 [N, dim], path_points [N, n_points, dim] -> (control points [N, degree+1, dim],
    cost [N]).  CUDA tensors: one launch of gik_bezier_fit_* (`solver`: a GraspIK on that device; default: the built-in
    Nextage solver -- the kernel only uses its device).  CPU tensors: the same products through torch on the host."""
    import torch
    if path_points.is_cuda:
        from .ops import default_solver
        s = solver if solver is not None else default_solver(path_points.device)
        pinv, basis, w0, w1 = fit_operands(degree, path_points.shape[-2])
        lead = path_points.shape[:-2]
        n_points, dim = path_points.shape[-2:]
        ctrl, cost = s.bezier_fit(q0.reshape(-1, dim), q1.reshape(-1, dim), path_points.reshape(-1, n_points, dim),
                                  pinv, basis, w0, w1)
        return ctrl.reshape(*lead, degree + 1, dim), cost.reshape(lead)
    Pf, cost = _fit(q0, q1, path_points, degree, torch)
    rep0 = q0.unsqueeze(-2).expand(*q0.shape[:-1], 3, q0.shape[-1])
    rep1 = q1.unsqueeze(-2).expand(*q1.shape[:-1], 3, q1.shape[-1])
    return torch.cat([rep0, Pf, rep1], dim=-2), cost


def maketraj_paths(q0, q1, q, offsets, degree=DEGREE, solver=None):
    """Fit CSR-packed paths, e.g. computepath_batch's (q [total, nq], offsets [Q+1]): path i is
    q[offsets[i]:offsets[i+1]].  q0, q1 [Q, nq].  One host read of `offsets`, then one maketraj_batch per distinct path
    length (one gik_bezier_fit_* launch for CUDA tensors).  -> (control points [Q, degree+1, nq], cost [Q]); a query
    without a path gets NaN control points and cost +inf."""
    import torch
    off = offsets.cpu().numpy() if torch.is_tensor(offsets) else np.asarray(offsets)
    Q, nq = len(off) - 1, q.shape[-1]
    lens = np.diff(off)
    ctrl = torch.full((Q, degree + 1, nq), float("nan"), dtype=q.dtype, device=q.device)
    cost = torch.full((Q,), float("inf"), dtype=q.dtype, device=q.device)
    for n in np.unique(lens[lens > 0]):
        rows = np.nonzero(lens == n)[0]
        idx = torch.as_tensor(off[rows][:, None] + np.arange(n)[None, :], device=q.device)
        r = torch.as_tensor(rows, device=q.device)
        c, k = maketraj_batch(q0[r], q1[r], q[idx], degree, solver)
        ctrl[r], cost[r] = c, k
    return ctrl, cost


CHECK_SAMPLES = 1501     # the controller's 1500 steps of 0.01 s over T = 15 s (control.py:416-463), plus the end point
GRASP_TOL = 1e-2         # policy default, not derived from the controller: see DESIGN.md "Trajectory check"
LIMIT_TOL = 1e-6         # rad: round-off of the weights on a curve that lies on a joint limit


def sample_weights(n_ctrl: int, n_samples: int) -> np.ndarray:
    """Bernstein weights [n_samples, n_ctrl] (fp64) of the parameters u_k = k / (n_samples - 1)."""
    return bernstein_matrix(n_ctrl - 1, np.arange(n_samples) / (n_samples - 1))


def check_trajectories_batch(ctrl, *, n_samples=CHECK_SAMPLES, grasp_tol=GRASP_TOL, limit_tol=LIMIT_TOL, per_sample=False,
                             solver=None):
    """Can these fitted trajectories be executed?  ctrl [N, n_ctrl, nq] Bezier control points (maketraj_batch /
    maketraj_paths), checked at u_k = k / (n_samples - 1) in one gik_traj_check_* call (semantics in include/gik.h):
    joint limits (flag 1), grasp error between the cube placements the two hands imply (flag 2), collisions with the
    carried cube at the left hand's placement (flag 4).  `solver`: a GraspIK (default: the built-in Nextage solver on
    ctrl's CUDA device, or the current one); ctrl is moved to its device.  -> dict of tensors on that device: valid
    bool [N], first_bad int32 [N] (-1 = none), reason uint8 [N] (flags of the first bad sample), grasp_err [N] (max over
    the samples) and, with per_sample, sample_flags uint8 [N, n_samples]."""
    import torch
    from .ops import default_solver
    ctrl = torch.as_tensor(ctrl)
    s = solver if solver is not None else default_solver(ctrl.device if ctrl.is_cuda else None)
    ctrl = ctrl.to(s.device)
    W = sample_weights(ctrl.shape[-2], int(n_samples))
    valid, first_bad, reason, grasp_err, flags = s.check_trajectories(ctrl, W, limit_tol=limit_tol, grasp_tol=grasp_tol,
                                                                       per_sample=per_sample)
    out = {"valid": valid.bool(), "first_bad": first_bad, "reason": reason, "grasp_err": grasp_err}
    if per_sample:
        out["sample_flags"] = flags
    return out


REFINE_ITERS = 8         # Levenberg-Marquardt trial steps: see DESIGN.md "Trajectory refinement" for the table behind it
REFINE_TOL = 0.5 * GRASP_TOL   # stop once max_k ||r_k|| <= this: half the check's grasp tolerance (the pinned end
                               # points alone leave ~2e-3 on planned trajectories, so a tighter tol only adds steps)
REFINE_DAMPING = 1e-3    # initial lambda of (H + lambda diag H)


def refine_trajectories_batch(ctrl, *, n_samples=CHECK_SAMPLES, max_iters=REFINE_ITERS, tol=REFINE_TOL, solver=None):
    """Refine fitted trajectories onto the grasp: the left hand leads, the right arm follows.  ctrl [N, n_ctrl, nq]
    (maketraj_batch / maketraj_paths; 7 <= n_ctrl <= 26).  One gik_traj_refine_* call (semantics in include/gik.h)
    moves only the right-arm columns of the free control points so that the grasp error check_trajectories_batch
    measures at u_k = k / (n_samples - 1) drops: Levenberg-Marquardt on sum_k ||log6(C_L^-1 C_R)||^2, every step kept
    inside the joint limits (a control point already outside them never moves further out).  Collisions are not
    considered: check the output.  `solver` as in check_trajectories_batch.  -> dict of tensors on the solver's
    device: ctrl (the refined control points), obj_before / obj_after fp64 [N] (the objective at input and output),
    grasp_err [N] (max over the samples at the output), iters int32 [N] (trial steps), accepted int32 [N]."""
    import torch
    from .ops import default_solver
    ctrl = torch.as_tensor(ctrl)
    s = solver if solver is not None else default_solver(ctrl.device if ctrl.is_cuda else None)
    ctrl = ctrl.to(s.device)
    W = sample_weights(ctrl.shape[-2], int(n_samples))
    out, before, after, grasp_err, iters, accepted = s.refine_trajectories(ctrl, W, max_iters=max_iters, tol=tol,
                                                                            damping=REFINE_DAMPING)
    return {"ctrl": out, "obj_before": before, "obj_after": after, "grasp_err": grasp_err, "iters": iters,
            "accepted": accepted}


def check_trajectory(q_of_t, *, n_samples=CHECK_SAMPLES, grasp_tol=GRASP_TOL, limit_tol=LIMIT_TOL, per_sample=False,
                     solver=None, dtype=None):
    """check_trajectories_batch for one reference-style Bezier (maketraj's q_of_t): sampled at n_samples evenly spaced
    times over [t_min, t_max].  -> dict with valid (bool), first_bad (int), reason (int), grasp_err (float) and, with
    per_sample, sample_flags (uint8 tensor [n_samples])."""
    import torch
    P = np.array(q_of_t.control_points_, dtype=float) * q_of_t.mult_T_
    ctrl = torch.as_tensor(P[None], dtype=dtype if dtype is not None else torch.float64)
    r = check_trajectories_batch(ctrl, n_samples=n_samples, grasp_tol=grasp_tol, limit_tol=limit_tol,
                                 per_sample=per_sample, solver=solver)
    out = {"valid": bool(r["valid"][0]), "first_bad": int(r["first_bad"][0]), "reason": int(r["reason"][0]),
           "grasp_err": float(r["grasp_err"][0])}
    if per_sample:
        out["sample_flags"] = r["sample_flags"][0]
    return out


def save_trajectory_to_json(filename, q_of_t, vq_of_t, vvq_of_t):
    """control.save_trajectory_to_json (control.py:203-216), same file format."""
    data = {"q_control_points": [p.tolist() for p in q_of_t.control_points_],
            "vq_control_points": [p.tolist() for p in vq_of_t.control_points_],
            "vvq_control_points": [p.tolist() for p in vvq_of_t.control_points_],
            "t_min": q_of_t.T_min_, "t_max": q_of_t.T_max_, "mult_t": q_of_t.mult_T_}
    with open(filename, "w") as f:
        json.dump(data, f, indent=4)


def load_trajectory_from_json(filename):
    """control.load_trajectory_from_json (control.py:220-240).  The derivative curves are rebuilt from the position
    control points (their stored control points are exactly degree * differences of those).  Note: the reference
    reloads the stored derivative curves with the POSITION curve's mult_t, i.e. without the 1 / T factors of a time
    derivative (control.py:229-237); here vq / vvq are the true time derivatives."""
    d = json.load(open(filename))
    q = Bezier([np.array(p) for p in d["q_control_points"]], t_min=d["t_min"], t_max=d["t_max"], mult_t=d["mult_t"])
    return q, q.derivative(1), q.derivative(2)
