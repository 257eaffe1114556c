"""Torch-facing wrapper of the C ABI: device memory, streams and layout conversion only -- every number is
produced by the CUDA kernels in csrc/.  Tensors must live on the handle's CUDA device; launches go to the
current torch stream and never synchronise."""
from __future__ import annotations

import ctypes
import threading
from dataclasses import dataclass

import numpy as np
import torch

from . import _cabi
from .model import KinematicTable, nextage_table
from .scene import CollisionScene, nextage_scene

# Reference literals: EPSILON (config.py:22), DT / max_iters (inverse_geometry.py:53-54)
EPSILON = 1e-3
DT = 1e-2
MAX_ITERS = 1000


@dataclass
class SolveInfo:
    iters: torch.Tensor     # [B] int32, updates applied
    resid: torch.Tensor     # [B,2] residual norms (left, right) at the returned q


def _sfx(dtype) -> str:
    if dtype == torch.float32:
        return "f32"
    if dtype == torch.float64:
        return "f64"
    raise TypeError(f"dtype must be torch.float32 or torch.float64, got {dtype}")


def as_pose12(pose, *, dtype, device, batch=None) -> torch.Tensor:
    """Normalise a cube placement batch to [B,12] (rotation row-major, translation).
    Accepts [B,12], [B,4,4], [B,7] (x y z qx qy qz qw, pinocchio XYZQUAT order) or [B,3] (identity rotation,
    the only case path.py samples: path.py:47)."""
    t = torch.as_tensor(pose, dtype=dtype, device=device) if not torch.is_tensor(pose) else pose.to(device=device, dtype=dtype)
    if t.dim() == 1 or (t.dim() == 2 and t.shape == (4, 4)):
        t = t.unsqueeze(0)
    if t.dim() == 3 and t.shape[1:] == (4, 4):
        out = torch.cat([t[:, :3, :3].reshape(-1, 9), t[:, :3, 3]], dim=1)
    elif t.dim() == 2 and t.shape[1] == 12:
        out = t
    elif t.dim() == 2 and t.shape[1] == 3:
        eye = torch.eye(3, dtype=dtype, device=device).reshape(1, 9).expand(t.shape[0], 9)
        out = torch.cat([eye, t], dim=1)
    elif t.dim() == 2 and t.shape[1] == 7:
        x, y, z, w = t[:, 3], t[:, 4], t[:, 5], t[:, 6]
        R = torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                         2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                         2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], dim=1)
        out = torch.cat([R, t[:, :3]], dim=1)
    else:
        raise ValueError(f"unsupported pose shape {tuple(t.shape)}")
    if batch is not None and out.shape[0] == 1 and batch != 1:
        out = out.expand(batch, 12)
    return out


class GraspIK:
    """Handle on the flattened kinematic model living on one GPU (gik_create / gik_destroy)."""

    def __init__(self, table: KinematicTable | None = None, device=None):
        if not torch.cuda.is_available():
            raise RuntimeError("GraspIK needs a CUDA device: there is no CPU fallback")
        self.table = table if table is not None else nextage_table()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.type != "cuda":
            raise ValueError("device must be a CUDA device")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self._lib = _cabi.lib()
        self._h = ctypes.c_void_p()
        ct = self.table.to_c()
        _cabi.check(self._lib.gik_create(ctypes.byref(ct), self.device.index, ctypes.byref(self._h)), "gik_create")
        self.nq = self.table.nq

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.gik_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ helpers
    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    @property
    def launches(self) -> int:
        """Kernels of this library launched through this handle (gik_launch_count)."""
        count = ctypes.c_int64()
        _cabi.check(self._lib.gik_launch_count(self._h, ctypes.byref(count)), "gik_launch_count")
        return count.value

    def _call(self, entry: str, dtype, *args):
        """Call gik_<entry>_f32 / _f64 (chosen by dtype; None: gik_<entry>, an entry without a storage type) with the
        handle first and the current stream last; raise on an error code."""
        f = getattr(self._lib, f"gik_{entry}" if dtype is None else f"gik_{entry}_{_sfx(dtype)}")
        _cabi.check(f(self._h, *args, self._stream()), f"gik_{entry}")

    def _arg(self, t, shape, dtype, name, *, copy=False) -> torch.Tensor:
        """A tensor handed to an entry: on this handle's device, of `dtype`, exactly `shape` (None: any size) and
        contiguous -- or, with `copy`, made contiguous.  TypeError for the dtype, ValueError otherwise."""
        if not torch.is_tensor(t) or not t.is_cuda or t.device != self.device:
            raise ValueError(f"{name}: expected a tensor on {self.device}, got {getattr(t, 'device', type(t).__name__)}")
        if t.dtype != dtype:
            raise TypeError(f"{name}: expected {dtype}, got {t.dtype}")
        if t.dim() != len(shape) or any(s is not None and s != d for s, d in zip(shape, t.shape)):
            want = "[" + "][".join("*" if s is None else str(s) for s in shape) + "]"
            raise ValueError(f"{name}: expected shape {want}, got {list(t.shape)}")
        if not t.is_contiguous():
            if not copy:
                raise ValueError(f"{name} must be contiguous")
            t = t.contiguous()
        return t

    def _q_cube(self, q_soa, cube_pose_soa):
        """q [nq][n] and the optional cube_pose [12][n] (converted to q's dtype) of the collision entries."""
        q = self._arg(q_soa, (self.nq, None), q_soa.dtype, "q", copy=True)
        if cube_pose_soa is None:
            return q, None
        return q, self._arg(cube_pose_soa.to(q.dtype), (12, q.shape[1]), q.dtype, "cube_pose", copy=True)

    # GIK_F_LANE_KERNEL / GIK_F_PAIR_KERNEL / GIK_F_SCALAR_LANE (fp32: "lane" = packed FFMA2 kernel, "lane1" = scalar)
    _KERNEL_FLAGS = {None: 0, "auto": 0, "lane": 2, "pair": 4, "lane1": 2 | 8}

    # Step form: by default an undamped step on a spherical-wrist table (Nextage) runs as two 3x3 solves per hand
    # (gik_core.cuh "Spherical-wrist form"); `force_cholesky` (a solver attribute, or the "+chol" kernel suffix) keeps the
    # general block-Cholesky form for A/B runs and tests.  GIK_F_CHOLESKY = 32.
    force_cholesky = False

    def _params(self, eps, dt, max_iters, damping, kernel=None, early_stop=False) -> _cabi.GikParams:
        chol = self.force_cholesky
        if isinstance(kernel, str) and kernel.endswith("+chol"):
            chol, kernel = True, (kernel[:-5] or None)
        if kernel not in self._KERNEL_FLAGS:
            raise ValueError(f"kernel must be one of {list(self._KERNEL_FLAGS)} (optionally with the suffix '+chol')")
        flags = self._KERNEL_FLAGS[kernel] | (16 if early_stop else 0) | (32 if chol else 0)   # GIK_F_EARLY_STOP, GIK_F_CHOLESKY
        return _cabi.GikParams(float(eps), float(dt), float(damping), int(max_iters), flags)

    def kernel_name(self, n, dtype=torch.float32, kernel=None) -> str:
        """Kernel the batch solve launches for n problems (gik_solve_kernel_name); for reports."""
        esz = 4 if dtype == torch.float32 else 8
        flags = self._params(1e-3, 1e-2, 1, 0.0, kernel).flags
        return self._lib.gik_solve_kernel_name(self._h, esz, int(n), flags).decode()

    @staticmethod
    def _ptr(t):
        return ctypes.c_void_p(0 if t is None else t.data_ptr())

    def limits(self, dtype=torch.float64):
        return (torch.as_tensor(self.table.lower, dtype=dtype, device=self.device),
                torch.as_tensor(self.table.upper, dtype=dtype, device=self.device))

    # ------------------------------------------------------------------ SoA entry points (no copies)
    def fk_soa(self, q_soa: torch.Tensor) -> torch.Tensor:
        """q [nq][n] -> frames [2][12][n]  (gik_fk_*)."""
        q = self._arg(q_soa, (self.nq, None), q_soa.dtype, "q", copy=True)
        out = torch.empty((2, 12, q.shape[1]), dtype=q.dtype, device=self.device)
        self._call("fk", q.dtype, q.shape[1], self._ptr(q), self._ptr(out))
        return out

    def jac_soa(self, q_soa: torch.Tensor) -> torch.Tensor:
        """q [nq][n] -> jac [2][6][nq][n]  (gik_jac_*)."""
        q = self._arg(q_soa, (self.nq, None), q_soa.dtype, "q", copy=True)
        out = torch.empty((2, 6, self.nq, q.shape[1]), dtype=q.dtype, device=self.device)
        self._call("jac", q.dtype, q.shape[1], self._ptr(q), self._ptr(out))
        return out

    def solve_soa(self, q_init: torch.Tensor, pose: torch.Tensor, *, eps=EPSILON, dt=DT, max_iters=MAX_ITERS,
                  damping=0.0, out=None, kernel=None, early_stop=False):
        """q_init [nq][n], pose [12][n] (contiguous) -> (q [nq][n], converged u8 [n], iters i32 [n], resid [2][n]).
        `out` may carry preallocated (q, converged, iters, resid) to keep the call allocation-free.
        `kernel`: None = launcher's choice by batch size, "lane" / "pair" force a thread mapping (same results).
        `early_stop`: fast preset (GIK_F_EARLY_STOP) -- stalled problems are abandoned early; flags and converged q
        are unchanged, the q / iters of FAILED problems are not the reference's."""
        ft = q_init.dtype
        q_init = self._arg(q_init, (self.nq, None), ft, "q_init")
        n = q_init.shape[1]
        pose = self._arg(pose, (12, n), ft, "pose")
        if out is None:
            q = torch.empty_like(q_init)
            conv = torch.empty((n,), dtype=torch.uint8, device=self.device)
            iters = torch.empty((n,), dtype=torch.int32, device=self.device)
            resid = torch.empty((2, n), dtype=ft, device=self.device)
        else:
            q, conv, iters, resid = out
            self._arg(q, (self.nq, n), ft, "out q")
            self._arg(conv, (n,), torch.uint8, "out converged")
            self._arg(iters, (n,), torch.int32, "out iters")
            self._arg(resid, (2, n), ft, "out resid")
        prm = self._params(eps, dt, max_iters, damping, kernel, early_stop)
        self._call("solve", ft, n, self._ptr(q_init), self._ptr(pose), ctypes.byref(prm), self._ptr(q), self._ptr(conv),
                   self._ptr(iters), self._ptr(resid))
        return q, conv, iters, resid

    def solve_scatter_soa(self, q_init: torch.Tensor, pose: torch.Tensor, q_ptrs, conv_ptrs, n_total: int, offset: int,
                          *, eps=EPSILON, dt=DT, max_iters=MAX_ITERS, damping=0.0, kernel=None, out=None):
        """K3 fused with its all-gather (gik_solve_scatter_*): solve this rank's slab and store every result into the
        result arrays of ALL ranks.  `q_ptrs` / `conv_ptrs`: device addresses (ints) of each rank's [nq][n_total] q
        array and [n_total] flag array as mapped on THIS device (see dist.SymmetricResults).  Returns the local
        (iters [n], resid [2][n]); the caller runs the cross-rank barrier."""
        ft = q_init.dtype
        q_init = self._arg(q_init, (self.nq, None), ft, "q_init")
        n = q_init.shape[1]
        pose = self._arg(pose, (12, n), ft, "pose")
        if len(q_ptrs) != len(conv_ptrs) or not q_ptrs:
            raise ValueError("need one q and one flag pointer per rank")
        if out is None:
            iters = torch.empty((n,), dtype=torch.int32, device=self.device)
            resid = torch.empty((2, n), dtype=ft, device=self.device)
        else:
            iters, resid = out
            self._arg(iters, (n,), torch.int32, "out iters")
            self._arg(resid, (2, n), ft, "out resid")
        P = len(q_ptrs)
        qa = (ctypes.c_void_p * P)(*[int(p) for p in q_ptrs])
        ca = (ctypes.c_void_p * P)(*[int(p) for p in conv_ptrs])
        prm = self._params(eps, dt, max_iters, damping, kernel)
        self._call("solve_scatter", ft, n, self._ptr(q_init), self._ptr(pose), ctypes.byref(prm), P, qa, ca, int(n_total),
                   int(offset), self._ptr(iters), self._ptr(resid))
        return iters, resid

    def best_of_soa(self, q, conv, resid, n_place: int, n_restart: int):
        """Problem (p, r) at column p * n_restart + r.  -> (q_best [nq][n_place], conv u8, which i32)."""
        N = n_place * n_restart
        q = self._arg(q, (self.nq, N), q.dtype, "q", copy=True)
        conv = self._arg(conv, (N,), torch.uint8, "converged", copy=True)
        resid = self._arg(resid, (2, N), q.dtype, "resid", copy=True)
        qb = torch.empty((self.nq, n_place), dtype=q.dtype, device=self.device)
        cb = torch.empty((n_place,), dtype=torch.uint8, device=self.device)
        wh = torch.empty((n_place,), dtype=torch.int32, device=self.device)
        self._call("best_of", q.dtype, n_place, n_restart, self._ptr(q), self._ptr(conv), self._ptr(resid), self._ptr(qb),
                   self._ptr(cb), self._ptr(wh))
        return qb, cb, wh

    def project_edges_soa(self, q_start, pose_a, pose_b, num_steps, max_steps: int, *, eps=EPSILON, dt=DT,
                          max_iters=MAX_ITERS, damping=0.0, kernel=None, out=None):
        """q_start [nq][E], pose_a/b [12][E], num_steps i32 [E] -> (q_path [max_steps][nq][E], n_valid i32 [E],
        iters_total i32 [E]).  Rows >= n_valid[e] of q_path are zero."""
        ft = q_start.dtype
        q_start = self._arg(q_start, (self.nq, None), ft, "q_start", copy=True)
        E = q_start.shape[1]
        pose_a = self._arg(pose_a, (12, E), ft, "pose_a", copy=True)
        pose_b = self._arg(pose_b, (12, E), ft, "pose_b", copy=True)
        num_steps = self._arg(num_steps, (E,), torch.int32, "num_steps", copy=True)
        if out is None:
            path = torch.zeros((max_steps, self.nq, E), dtype=ft, device=self.device)
            nv = torch.empty((E,), dtype=torch.int32, device=self.device)
            itt = torch.empty((E,), dtype=torch.int32, device=self.device)
        else:
            path, nv, itt = out
            self._arg(path, (max_steps, self.nq, E), ft, "out q_path")
            self._arg(nv, (E,), torch.int32, "out n_valid")
            self._arg(itt, (E,), torch.int32, "out iters_total")
        prm = self._params(eps, dt, max_iters, damping, kernel)
        self._call("project_edges", ft, E, max_steps, self._ptr(q_start), self._ptr(pose_a), self._ptr(pose_b),
                   self._ptr(num_steps), ctypes.byref(prm), self._ptr(path), self._ptr(nv), self._ptr(itt))
        return path, nv, itt

    # ------------------------------------------------------------------ collision predicate (SURVEY 8f-1)
    def attach_scene(self, scene: CollisionScene | None = None) -> "GraspIK":
        """Upload the flattened collision model (gik_scene_attach).  Default: the reference's scene."""
        self.scene = scene if scene is not None else nextage_scene()
        sc = self.scene.to_c()
        _cabi.check(self._lib.gik_scene_attach(self._h, ctypes.byref(sc)), "gik_scene_attach")
        return self

    def _need_scene(self):
        """Attach a collision scene on first use.  Only two cases are automatic: the built-in Nextage table gets the
        packaged reference scene, and a solver built from a pinocchio RobotWrapper flattens that robot's OWN
        `collision_model` (scene_from_pinocchio: its geometries, placements and pair list, whatever they are).  Any
        other table (a URDF, a hand-made KinematicTable) needs an explicit attach_scene(scene): a silently wrong
        collision model is worse than an error."""
        if getattr(self, "scene", None) is None:
            src = self.table.meta.get("source")
            robot = getattr(self, "_robot", None)
            if src == "builtin-nextage":
                self.attach_scene()
            elif robot is not None and hasattr(robot, "collision_model"):
                from .scene import scene_from_pinocchio
                self.attach_scene(scene_from_pinocchio(robot))
            else:
                raise RuntimeError("no collision scene attached: call GraspIK.attach_scene(scene) for this robot "
                                   "(scene_from_urdf / scene_from_pinocchio build one)")

    def collision_soa(self, q_soa: torch.Tensor, cube_pose_soa: torch.Tensor | None = None, sel: torch.Tensor | None = None) -> torch.Tensor:
        """tools.collision(robot, q) for every column: q [nq][n], cube_pose [12][n] (None = scene's cube placement)
        -> colliding u8 [n].  `sel` (int64 [m], device): test only those columns (gik_collision_sel_*); the other
        entries of the result are 0."""
        self._need_scene()
        q, cp = self._q_cube(q_soa, cube_pose_soa)
        n = q.shape[1]
        if sel is not None:
            sel = self._arg(sel.to(torch.int64), (None,), torch.int64, "sel", copy=True)
            out = torch.zeros((n,), dtype=torch.uint8, device=self.device)
            if sel.numel():
                self._call("collision_sel", q.dtype, n, sel.numel(), self._ptr(sel), self._ptr(q), self._ptr(cp),
                           self._ptr(out))
            return out
        out = torch.empty((n,), dtype=torch.uint8, device=self.device)
        self._call("collision", q.dtype, n, self._ptr(q), self._ptr(cp), self._ptr(out))
        return out

    def clearance_soa(self, q_soa: torch.Tensor, cube_pose_soa: torch.Tensor | None = None, threshold: float = 0.04) -> torch.Tensor:
        """distanceToObstacle(robot, q) >= threshold (tools.py:38-51, path.py:61-62) -> clear u8 [n]."""
        self._need_scene()
        q, cp = self._q_cube(q_soa, cube_pose_soa)
        out = torch.empty((q.shape[1],), dtype=torch.uint8, device=self.device)
        self._call("clearance", q.dtype, q.shape[1], self._ptr(q), self._ptr(cp), float(threshold), self._ptr(out))
        return out

    def obstacle_distance_soa(self, q_soa: torch.Tensor, cube_pose_soa: torch.Tensor | None = None, d_max: float = 2.0) -> torch.Tensor:
        """distanceToObstacle(robot, q) (tools.py:38-51) as a value -> dist [n] in q's dtype: smallest distance between
        the robot (and cube) and the table / obstacle, capped at d_max, 0 on intersection (gik_obstacle_distance_*)."""
        self._need_scene()
        q, cp = self._q_cube(q_soa, cube_pose_soa)
        out = torch.empty((q.shape[1],), dtype=q.dtype, device=self.device)
        self._call("obstacle_distance", q.dtype, q.shape[1], self._ptr(q), self._ptr(cp), float(d_max), self._ptr(out))
        return out

    def bezier_fit(self, q0: torch.Tensor, q1: torch.Tensor, path: torch.Tensor, pinv, basis, w0, w1):
        """The least-squares fit of `maketraj` (control.py:63-195) for many paths in one launch (gik_bezier_fit_*).
        q0, q1 [N, dim], path [N, n_points, dim] on this device; pinv [n_free, n_points], basis [n_points, n_free],
        w0 / w1 [n_points]: the factored design matrix (trajectory.fit_operands).  -> (ctrl [N, n_free + 6, dim], cost [N])."""
        ft = path.dtype
        path = self._arg(path, (None, None, None), ft, "path", copy=True)
        N, n_points, dim = path.shape
        q0 = self._arg(q0, (N, dim), ft, "q0", copy=True)
        q1 = self._arg(q1, (N, dim), ft, "q1", copy=True)
        n_free = int(pinv.shape[0])
        ops = [self._arg(torch.as_tensor(x, dtype=ft, device=self.device), shape, ft, name, copy=True)
               for x, shape, name in ((pinv, (n_free, n_points), "pinv"), (basis, (n_points, n_free), "basis"),
                                      (w0, (n_points,), "w0"), (w1, (n_points,), "w1"))]
        ctrl = torch.empty((N, n_free + 6, dim), dtype=ft, device=self.device)
        cost = torch.empty((N,), dtype=ft, device=self.device)
        self._call("bezier_fit", ft, N, n_points, dim, n_free + 6, *[self._ptr(x) for x in ops], self._ptr(q0), self._ptr(q1),
                   self._ptr(path), self._ptr(ctrl), self._ptr(cost))
        return ctrl, cost

    def _traj_args(self, ctrl, weights):
        """ctrl [N, n_ctrl, nq] and weights [M, n_ctrl] (converted to ctrl's dtype) of the trajectory entries."""
        ctrl = self._arg(ctrl, (None, None, self.nq), ctrl.dtype, "ctrl", copy=True)
        W = torch.as_tensor(weights, dtype=ctrl.dtype, device=self.device)
        return ctrl, self._arg(W, (None, ctrl.shape[1]), ctrl.dtype, "weights", copy=True)

    def check_trajectories(self, ctrl: torch.Tensor, weights, *, limit_tol: float, grasp_tol: float, per_sample=False):
        """Validity of many Bezier trajectories at the sample times of `weights` (gik_traj_check_*, semantics in
        include/gik.h): joint limits, grasp error between the cube placements the two hands imply, collisions with the
        carried cube at the left hand's placement.  ctrl [N, n_ctrl, nq] on this device; weights [M, n_ctrl]: Bernstein
        weights of the samples (trajectory.sample_weights).  -> (valid u8 [N], first_bad i32 [N] (-1 = none), reason u8
        [N] (flags of the first bad sample: 1 limits | 2 grasp | 4 collision), grasp_err [N] (max over the samples),
        sample_flags u8 [N, M] or None)."""
        self._need_scene()
        ctrl, W = self._traj_args(ctrl, weights)
        (N, n_ctrl, _), M = ctrl.shape, W.shape[0]
        valid = torch.empty((N,), dtype=torch.uint8, device=self.device)
        first_bad = torch.empty((N,), dtype=torch.int32, device=self.device)
        reason = torch.empty((N,), dtype=torch.uint8, device=self.device)
        grasp_err = torch.empty((N,), dtype=ctrl.dtype, device=self.device)
        flags = torch.empty((N, M), dtype=torch.uint8, device=self.device) if per_sample else None
        self._call("traj_check", ctrl.dtype, N, n_ctrl, M, self._ptr(W), self._ptr(ctrl), float(limit_tol), float(grasp_tol),
                   self._ptr(valid), self._ptr(first_bad), self._ptr(reason), self._ptr(grasp_err), self._ptr(flags))
        return valid, first_bad, reason, grasp_err, flags

    def refine_trajectories(self, ctrl: torch.Tensor, weights, *, max_iters: int, tol: float, damping: float):
        """Refine many Bezier trajectories onto the grasp (gik_traj_refine_*, semantics in include/gik.h): the right
        arm's free control points follow the left hand.  ctrl [N, n_ctrl, nq] on this device; weights [M, n_ctrl]:
        Bernstein weights of the samples (trajectory.sample_weights).  -> (ctrl_out [N, n_ctrl, nq], obj_before f64 [N],
        obj_after f64 [N], grasp_err [N] (max over the samples at the output), iters i32 [N], accepted i32 [N])."""
        ctrl, W = self._traj_args(ctrl, weights)
        N, n_ctrl, _ = ctrl.shape
        out = torch.empty_like(ctrl)
        f64 = lambda: torch.empty((N,), dtype=torch.float64, device=self.device)       # noqa: E731
        i32 = lambda: torch.empty((N,), dtype=torch.int32, device=self.device)         # noqa: E731
        obj_before, obj_after, iters, accepted = f64(), f64(), i32(), i32()
        grasp_err = torch.empty((N,), dtype=ctrl.dtype, device=self.device)
        self._call("traj_refine", ctrl.dtype, N, n_ctrl, W.shape[0], self._ptr(W), self._ptr(ctrl), int(max_iters),
                   float(tol), float(damping), self._ptr(out), self._ptr(obj_before), self._ptr(obj_after),
                   self._ptr(grasp_err), self._ptr(iters), self._ptr(accepted))
        return out, obj_before, obj_after, grasp_err, iters, accepted

    # ------------------------------------------------------------------ RRT-connect trees on the device (csrc/gik_tree.cuh)
    # verts [n_trees][nq][cap], cubes [n_trees][12][cap], parent i32 [n_trees][cap], n_verts i32 [n_trees]; the trees
    # are updated in place, so these are checked, never copied
    def _tree(self, verts, n_verts, cubes=None, parent=None):
        self._arg(verts, (None, self.nq, None), verts.dtype, "verts")
        n_trees, _, cap = verts.shape
        self._arg(n_verts, (n_trees,), torch.int32, "n_verts")
        if cubes is not None:
            self._arg(cubes, (n_trees, 12, cap), verts.dtype, "cubes")
        if parent is not None:
            self._arg(parent, (n_trees, cap), torch.int32, "parent")
        return n_trees, cap

    def tree_nearest(self, verts, n_verts, targets, target_tree) -> torch.Tensor:
        """Nearest vertex of tree target_tree[t] to each row of targets [n,nq] (gik_tree_nearest_*): squared distances
        in fp64, numpy's sum order and argmin's tie rule (lowest index).  -> nearest int32 [n] (-1: empty tree)."""
        n_trees, cap = self._tree(verts, n_verts)
        tg = self._arg(targets.to(verts.dtype), (None, self.nq), verts.dtype, "targets", copy=True)
        n = tg.shape[0]
        tt = self._arg(target_tree.to(torch.int32), (n,), torch.int32, "target_tree", copy=True)
        out = torch.empty((n,), dtype=torch.int32, device=self.device)
        self._call("tree_nearest", verts.dtype, n_trees, cap, self._ptr(verts), self._ptr(n_verts), n, self._ptr(tg),
                   self._ptr(tt), self._ptr(out))
        return out

    def tree_grow(self, verts, cubes, parent, n_verts, overflow, edge_tree, near, q_start, pose_a, pose_b, num_steps,
                  n_valid, q_path) -> torch.Tensor:
        """Append the output of one edge launch to the trees in place (gik_tree_grow_*; grow() of computepath).
        Edge e (the edges of one tree consecutive) belongs to tree edge_tree[e] and starts at vertex near[e];
        q_start [nq][E], pose_a / pose_b [12][E], num_steps i32 [E] and q_path [S][nq][E] are project_edges_soa's
        inputs and output, n_valid i32 [E] its step counts (< 0: no segment).  overflow u8 [n_trees] is set for a tree
        that would exceed its capacity (left unchanged).  -> seg_end int32 [E] (tree index of each segment's last
        vertex, -1 without a segment)."""
        n_trees, cap = self._tree(verts, n_verts, cubes, parent)
        ft = verts.dtype
        self._arg(overflow, (n_trees,), torch.uint8, "overflow")
        q_start = self._arg(q_start, (self.nq, None), ft, "q_start", copy=True)
        E = q_start.shape[1]
        pose_a = self._arg(pose_a, (12, E), ft, "pose_a", copy=True)
        pose_b = self._arg(pose_b, (12, E), ft, "pose_b", copy=True)
        q_path = self._arg(q_path, (None, self.nq, E), ft, "q_path", copy=True)
        edge_tree, near, num_steps, n_valid = [self._arg(t, (E,), torch.int32, name, copy=True) for t, name in
                                               ((edge_tree, "edge_tree"), (near, "near"), (num_steps, "num_steps"),
                                                (n_valid, "n_valid"))]
        seg_end = torch.empty((E,), dtype=torch.int32, device=self.device)
        self._call("tree_grow", ft, n_trees, cap, self._ptr(verts), self._ptr(cubes), self._ptr(parent), self._ptr(n_verts),
                   self._ptr(overflow), E, q_path.shape[0],
                   *[self._ptr(x) for x in (edge_tree, near, q_start, pose_a, pose_b, num_steps, n_valid, q_path)],
                   self._ptr(seg_end))
        return seg_end

    def tree_paths(self, verts, cubes, parent, n_verts, start_end, goal_end):
        """Paths of Q queries (2Q trees: start tree i, goal tree Q + i) that connected at (start_end[i], goal_end[i])
        (-1 = did not connect): get_path(start) + get_path(goal)[::-1] (path.py:226-233, 317) as packed rows
        (gik_tree_paths_*).  -> (q [total][nq], cube [total][12], offsets int64 [Q+1]); query i owns rows
        offsets[i]:offsets[i+1].  One host synchronisation (reading the total)."""
        n_trees, cap = self._tree(verts, n_verts, cubes, parent)
        Q = n_trees // 2
        if n_trees != 2 * Q:
            raise ValueError("tree_paths: expected 2Q trees")
        se = self._arg(start_end.to(torch.int32), (Q,), torch.int32, "start_end", copy=True)
        ge = self._arg(goal_end.to(torch.int32), (Q,), torch.int32, "goal_end", copy=True)
        offsets = torch.zeros((Q + 1,), dtype=torch.int64, device=self.device)
        tree = [self._ptr(x) for x in (verts, cubes, parent, n_verts, se, ge)]
        self._call("tree_paths", verts.dtype, Q, cap, *tree, self._ptr(offsets), None, None)
        total = int(offsets[-1].item()) if Q else 0
        q = torch.empty((total, self.nq), dtype=verts.dtype, device=self.device)
        cube = torch.empty((total, 12), dtype=verts.dtype, device=self.device)
        if total:
            self._call("tree_paths", verts.dtype, Q, cap, *tree, self._ptr(offsets), self._ptr(q), self._ptr(cube))
        return q, cube, offsets

    def path_shortcut(self, q, cube, offsets, pair_i, pair_j, num_steps, n_valid, q_path, *, join_tol: float):
        """One shortcut round for CSR paths (gik_path_shortcut_*, semantics in include/gik.h): q [total][nq], cube
        [total][12], offsets int64 [Q+1] (tree_paths' form); candidate k of path p is edge p * K + k of one
        project_edges_soa launch: pair_i / pair_j / num_steps / n_valid int32 [Q, K] and q_path [S][nq][Q*K].
        -> (q [total'][nq], cube [total'][12], offsets int64 [Q+1], chosen int32 [Q] (-1 = none), length float64 [Q]
        (joint-space length of each output path)).  One host synchronisation (reading the new total)."""
        ft = q.dtype
        q = self._arg(q, (None, self.nq), ft, "q", copy=True)
        cube = self._arg(cube, (q.shape[0], 12), ft, "cube", copy=True)
        offsets = self._arg(offsets, (None,), torch.int64, "offsets", copy=True)
        Q = offsets.shape[0] - 1
        pair_i = self._arg(pair_i, (Q, None), torch.int32, "pair_i", copy=True)
        K = pair_i.shape[1]
        pair_j, num_steps, n_valid = [self._arg(t, (Q, K), torch.int32, name, copy=True) for t, name in
                                      ((pair_j, "pair_j"), (num_steps, "num_steps"), (n_valid, "n_valid"))]
        q_path = self._arg(q_path, (None, self.nq, Q * K), ft, "q_path", copy=True)
        chosen = torch.empty((Q,), dtype=torch.int32, device=self.device)
        length = torch.empty((Q,), dtype=torch.float64, device=self.device)
        off_out = torch.empty((Q + 1,), dtype=torch.int64, device=self.device)
        head = [self._ptr(x) for x in (offsets, q, cube, pair_i, pair_j, num_steps, n_valid, q_path)]
        tail = [self._ptr(chosen), self._ptr(length), self._ptr(off_out)]
        self._call("path_shortcut", ft, Q, K, q_path.shape[0], *head, float(join_tol), *tail, None, None)
        total = int(off_out[-1].item()) if Q else 0
        q_out = torch.empty((total, self.nq), dtype=ft, device=self.device)
        cube_out = torch.empty((total, 12), dtype=ft, device=self.device)
        if total:
            self._call("path_shortcut", ft, Q, K, q_path.shape[0], *head, float(join_tol), *tail, self._ptr(q_out),
                       self._ptr(cube_out))
        return q_out, cube_out, off_out, chosen, length

    # ------------------------------------------------------------------ grasp roadmap (csrc/gik_roadmap.cuh)
    def knn(self, cube, k: int, points=None) -> torch.Tensor:
        """The k vertices nearest each point by the fp64 distance of cube translations, nearest first, ties to the lower
        index (gik_knn_*, semantics in include/gik.h).  cube [N,12] vertex placements; points [P,12] (converted to
        cube's dtype), None: the vertices themselves, each excluding itself.  -> nbr int32 [P,k]."""
        cube = self._arg(cube, (None, 12), cube.dtype, "cube", copy=True)
        N = cube.shape[0]
        if not 1 <= int(k) <= min(32, N - 1):
            raise ValueError(f"knn: k must be in [1, min(32, N - 1)] with N = {N}, got {k}")
        if points is not None:
            points = self._arg(points.to(cube.dtype), (None, 12), cube.dtype, "points", copy=True)
        P = N if points is None else points.shape[0]
        nbr = torch.empty((P, int(k)), dtype=torch.int32, device=self.device)
        self._call("knn", cube.dtype, N, int(k), self._ptr(cube), P, self._ptr(points), self._ptr(nbr))
        return nbr

    def roadmap_edges(self, q_from, q_to, num_steps, n_valid, q_path, *, join_tol: float) -> torch.Tensor:
        """Acceptance and fp64 weight of the E edges of one project_edges_soa launch (gik_roadmap_edges_*, semantics in
        include/gik.h): edge e from q_from[e] towards q_to[e] ([E,nq]), num_steps / n_valid int32 [E], q_path
        [S][nq][E].  -> weight float64 [E], +inf for a rejected edge."""
        ft = q_path.dtype
        q_path = self._arg(q_path, (None, self.nq, None), ft, "q_path", copy=True)
        E = q_path.shape[2]
        q_from = self._arg(q_from, (E, self.nq), ft, "q_from", copy=True)
        q_to = self._arg(q_to, (E, self.nq), ft, "q_to", copy=True)
        num_steps = self._arg(num_steps, (E,), torch.int32, "num_steps", copy=True)
        n_valid = self._arg(n_valid, (E,), torch.int32, "n_valid", copy=True)
        weight = torch.empty((E,), dtype=torch.float64, device=self.device)
        self._call("roadmap_edges", ft, E, q_path.shape[0], self._ptr(q_from), self._ptr(q_to), self._ptr(num_steps),
                   self._ptr(n_valid), self._ptr(q_path), float(join_tol), self._ptr(weight))
        return weight

    def _csr(self, row_ptr, dst, weight=None, ns=None):
        row_ptr = self._arg(row_ptr, (None,), torch.int64, "row_ptr", copy=True)
        dst = self._arg(dst, (None,), torch.int32, "dst", copy=True)
        E = dst.shape[0]
        out = [row_ptr, dst]
        if weight is not None:
            out.append(self._arg(weight, (E,), torch.float64, "weight", copy=True))
        if ns is not None:
            out.append(self._arg(ns, (E,), torch.int32, "ns", copy=True))
        return out

    def roadmap_sssp(self, row_ptr, dst, weight, att_vertex, att_weight):
        """Shortest paths of Q queries over one roadmap, one CTA per query (gik_roadmap_sssp, semantics in
        include/gik.h).  row_ptr int64 [N+1], dst int32 [E], weight float64 [E]; att_vertex int32 [Q, 2ka+1] and
        att_weight float64 [Q, 2ka+1]: the attachment slots.  -> (dist float64 [Q,N], pred int32 [Q,N], goal_pred int32
        [Q], length float64 [Q], attach_start int32 [Q], attach_goal int32 [Q]).  dist and pred take 12 Q N bytes."""
        row_ptr, dst, weight = self._csr(row_ptr, dst, weight)
        N, E = row_ptr.shape[0] - 1, dst.shape[0]
        att_vertex = self._arg(att_vertex, (None, None), torch.int32, "att_vertex", copy=True)
        Q, A = att_vertex.shape
        if A % 2 != 1:
            raise ValueError(f"att_vertex: expected 2 * k_attach + 1 slots per query, got {A}")
        att_weight = self._arg(att_weight, (Q, A), torch.float64, "att_weight", copy=True)
        dist = torch.empty((Q, N), dtype=torch.float64, device=self.device)
        pred = torch.empty((Q, N), dtype=torch.int32, device=self.device)
        goal_pred, a_s, a_g = [torch.empty((Q,), dtype=torch.int32, device=self.device) for _ in range(3)]
        length = torch.empty((Q,), dtype=torch.float64, device=self.device)
        self._call("roadmap_sssp", None, Q, N, (A - 1) // 2, E, *[self._ptr(x) for x in (
            row_ptr, dst, weight, att_vertex, att_weight, dist, pred, goal_pred, length, a_s, a_g)])
        return dist, pred, goal_pred, length, a_s, a_g

    def roadmap_paths(self, vq, vcube, row_ptr, dst, ns, step_ptr, steps, q_init, q_goal, cube0, cube1, att_vertex,
                      att_weight, att_ns, att_path, pred, goal_pred):
        """The paths of a query batch from roadmap_sssp's pred / goal_pred (gik_roadmap_paths_*, semantics in
        include/gik.h): roadmap vq [N,nq], vcube [N,12], row_ptr / dst / ns / step_ptr / steps [rows,nq]; queries q_init /
        q_goal [Q,nq], cube0 / cube1 [Q,12]; attachment slots att_vertex / att_ns int32 and att_weight float64 [Q, A],
        att_path [S][nq][Q*A].  -> (q [total,nq], cube [total,12], offsets int64 [Q+1], vertices int32 [Q]).  One host
        synchronisation (reading the total)."""
        ft = vq.dtype
        vq = self._arg(vq, (None, self.nq), ft, "vq", copy=True)
        N = vq.shape[0]
        vcube = self._arg(vcube, (N, 12), ft, "vcube", copy=True)
        row_ptr, dst, ns = self._csr(row_ptr, dst, ns=ns)
        if row_ptr.shape[0] != N + 1:
            raise ValueError(f"row_ptr: expected shape [{N + 1}], got {list(row_ptr.shape)}")
        E = dst.shape[0]
        step_ptr = self._arg(step_ptr, (E + 1,), torch.int64, "step_ptr", copy=True)
        steps = self._arg(steps, (None, self.nq), ft, "steps", copy=True)
        q_init = self._arg(q_init, (None, self.nq), ft, "q_init", copy=True)
        Q = q_init.shape[0]
        q_goal = self._arg(q_goal, (Q, self.nq), ft, "q_goal", copy=True)
        cube0 = self._arg(cube0, (Q, 12), ft, "cube0", copy=True)
        cube1 = self._arg(cube1, (Q, 12), ft, "cube1", copy=True)
        att_vertex = self._arg(att_vertex, (Q, None), torch.int32, "att_vertex", copy=True)
        A = att_vertex.shape[1]
        if A % 2 != 1:
            raise ValueError(f"att_vertex: expected 2 * k_attach + 1 slots per query, got {A}")
        att_weight = self._arg(att_weight, (Q, A), torch.float64, "att_weight", copy=True)
        att_ns = self._arg(att_ns, (Q, A), torch.int32, "att_ns", copy=True)
        att_path = self._arg(att_path, (None, self.nq, Q * A), ft, "att_path", copy=True)
        pred = self._arg(pred, (Q, N), torch.int32, "pred", copy=True)
        goal_pred = self._arg(goal_pred, (Q,), torch.int32, "goal_pred", copy=True)
        offsets = torch.zeros((Q + 1,), dtype=torch.int64, device=self.device)
        vertices = torch.zeros((Q,), dtype=torch.int32, device=self.device)
        head = [Q, N, (A - 1) // 2, att_path.shape[0], E] + [self._ptr(x) for x in (
            vq, vcube, row_ptr, dst, ns, step_ptr, steps if steps.numel() else None, q_init, q_goal, cube0, cube1,
            att_vertex, att_weight, att_ns, att_path, pred, goal_pred, offsets, vertices)]
        self._call("roadmap_paths", ft, *head, None, None)
        total = int(offsets[-1].item()) if Q else 0
        q = torch.empty((total, self.nq), dtype=ft, device=self.device)
        cube = torch.empty((total, 12), dtype=ft, device=self.device)
        if total:
            self._call("roadmap_paths", ft, *head, self._ptr(q), self._ptr(cube))
        return q, cube, offsets, vertices

    def cube_collision_soa(self, cube_pose_soa: torch.Tensor) -> torch.Tensor:
        """The cube's own collision test (cube vs table / obstacle, path.py:51-52): cube_pose [12][n] -> u8 [n]."""
        self._need_scene()
        cp = self._arg(cube_pose_soa, (12, None), cube_pose_soa.dtype, "cube_pose", copy=True)
        out = torch.empty((cp.shape[1],), dtype=torch.uint8, device=self.device)
        self._call("cube_collision", cp.dtype, cp.shape[1], self._ptr(cp), self._ptr(out))
        return out

    def collision(self, q, cube_pose=None, *, dtype=None) -> torch.Tensor:
        """Row-major convenience: q [B,nq] (or [nq]), cube_pose [B,12|4x4|7|3] or None -> colliding bool [B]."""
        qt = torch.as_tensor(q, device=self.device)
        dtype = dtype or (qt.dtype if qt.dtype in (torch.float32, torch.float64) else torch.float64)
        qt = qt.to(dtype)
        if qt.dim() == 1:
            qt = qt.unsqueeze(0)
        cp = None
        if cube_pose is not None:
            cp = as_pose12(cube_pose, dtype=dtype, device=self.device, batch=qt.shape[0]).t().contiguous()
        return self.collision_soa(qt.t().contiguous(), cp).bool()

    def solve_success_soa(self, q_init, pose, *, eps=EPSILON, dt=DT, max_iters=MAX_ITERS, damping=0.0, kernel=None,
                          descend_while_colliding=True, early_stop=False, return_stats=False):
        """The reference's FULL success predicate on the device: `success = converged and not collision(q)`
        (inverse_geometry.py:70, 97-98), including its behaviour on converged-but-colliding iterates -- the loop keeps
        descending and re-tests collision(q) after every update until an iterate is free or max_iters is reached.
        ONE stream-ordered C call (gik_solve_success_*), no host synchronisation: the batched solve, the collision test
        of the converged problems, a continuation launch that runs the converged-but-colliding ones to the cap, and a
        warp-per-problem kernel that decides each of them (persistent collision, or a replay that tests the undecided
        pairs on every iterate).  `descend_while_colliding=False` (GIK_F_NO_DESCEND) evaluates the collision term once,
        at the configuration the descent stopped at: differs only where further descent would have freed a collision,
        and in the q returned for failed problems.
        -> (q [nq][n], success u8 [n], converged u8 [n], iters i32 [n], resid [2][n][, stats]); stats (device int64 [4]):
        problems decided as persistent collisions, problems replayed, replayed iterations, replays that succeeded."""
        self._need_scene()
        ft = q_init.dtype
        q_init = self._arg(q_init, (self.nq, None), ft, "q_init", copy=True)
        n = q_init.shape[1]
        pose = self._arg(pose, (12, n), ft, "pose", copy=True)
        q = torch.empty_like(q_init)
        succ = torch.empty((n,), dtype=torch.uint8, device=self.device)
        conv = torch.empty((n,), dtype=torch.uint8, device=self.device)
        iters = torch.empty((n,), dtype=torch.int32, device=self.device)
        resid = torch.empty((2, n), dtype=ft, device=self.device)
        esz = 4 if ft == torch.float32 else 8
        nbytes = int(self._lib.gik_solve_success_scratch_bytes(self._h, n, esz))
        scratch = torch.empty((max(nbytes, 8),), dtype=torch.uint8, device=self.device)
        prm = self._params(eps, dt, max_iters, damping, kernel, early_stop)
        if not descend_while_colliding:
            prm.flags |= 64                                                  # GIK_F_NO_DESCEND
        self._call("solve_success", ft, n, self._ptr(q_init), self._ptr(pose), ctypes.byref(prm), self._ptr(q),
                   self._ptr(succ), self._ptr(conv), self._ptr(iters), self._ptr(resid), self._ptr(scratch))
        if return_stats:
            stats = scratch[nbytes - 256 + 8:nbytes - 256 + 40].view(torch.int64).clone() if n else torch.zeros(4, dtype=torch.int64, device=self.device)
            return q, succ, conv, iters, resid, stats
        return q, succ, conv, iters, resid

    # ------------------------------------------------------------------ row-major convenience ([B, ...])
    def fk(self, q: torch.Tensor):
        """q [B,nq] -> (R [B,2,3,3], p [B,2,3]) world placements of LARM_EFF / RARM_EFF."""
        fr = self.fk_soa(q.t().contiguous())              # [2][12][B]
        fr = fr.permute(2, 0, 1)                          # [B,2,12]
        return fr[:, :, :9].reshape(-1, 2, 3, 3), fr[:, :, 9:]

    def jacobians(self, q: torch.Tensor):
        """q [B,nq] -> J [B,2,6,nq] (LOCAL frame, rows [linear; angular])."""
        return self.jac_soa(q.t().contiguous()).permute(3, 0, 1, 2)

    def solve(self, q_init, pose, *, dtype=torch.float32, eps=EPSILON, dt=DT, max_iters=MAX_ITERS, damping=0.0,
              return_info=False, kernel=None):
        """q_init [B,nq] (or [nq], broadcast), pose [B,12|4x4|7|3] -> (q [B,nq], converged bool [B][, SolveInfo])."""
        p12 = as_pose12(pose, dtype=dtype, device=self.device)
        B = p12.shape[0]
        qi = torch.as_tensor(q_init, device=self.device).to(dtype)
        if qi.dim() == 1:
            qi = qi.unsqueeze(0)
        if qi.shape[0] == 1 and B != 1:
            qi = qi.expand(B, self.nq)
        elif B == 1 and qi.shape[0] != 1:
            B = qi.shape[0]
            p12 = p12.expand(B, 12)
        q, conv, iters, resid = self.solve_soa(qi.t().contiguous(), p12.t().contiguous(), eps=eps, dt=dt,
                                               max_iters=max_iters, damping=damping, kernel=kernel)
        res = (q.t(), conv.bool())
        if return_info:
            res = res + (SolveInfo(iters, resid.t()),)
        return res


def _pinned(cache, key, shape, dtype):
    t = cache.get(key)
    if t is None or tuple(t.shape) != tuple(shape) or t.dtype != dtype:
        t = torch.empty(shape, dtype=dtype).pin_memory()
        cache[key] = t
    return t


def _slab_bounds(B: int, slabs: int, align: int = 32):
    """Slab boundaries of the streamed host path: a small first slab so the kernel starts early, the rest in equal
    parts, every interior boundary a multiple of `align` rows (rows are 60 / 48 B: a multiple of 32 rows is a multiple
    of 128 B, so no cache line ever holds rows of two slabs)."""
    slabs = max(1, int(slabs))
    if slabs == 1 or B <= (1 << 16):                 # small batches: one slab, nothing to overlap
        return [0, B]
    first = min(B, max(1 << 16, B // 16))
    first -= first % align
    if first <= 0 or first >= B:
        return [0, B]
    bounds = [0, first]
    for k in range(1, slabs):
        b = first + ((B - first) * k) // (slabs - 1)
        if k < slabs - 1:
            b -= b % align
        if b > bounds[-1]:
            bounds.append(b)
    bounds[-1] = B
    return bounds


def solve_host(self, q_init, pose, *, dtype=torch.float32, eps=EPSILON, dt=DT, max_iters=MAX_ITERS, damping=0.0,
               slabs=4, return_info=False, kernel=None, out=None):
    """Host-buffer entry: q_init [B,nq] (or [nq]) and pose [B,12|4x4|7|3] are CPU tensors / arrays (pageable or pinned);
    returns CPU tensors (q [B,nq], converged bool [B][, SolveInfo]).

    Ownership: by default the results are FRESH pinned tensors owned by the caller (one pinned allocation per call).
    `out=(q [B,nq], converged uint8 [B][, iters int32 [B], resid [B,2]])` -- pinned, contiguous CPU tensors -- makes the
    call allocation-free: the kernel stores straight into them (the zero-copy path bench.py's e2e leg uses).  The
    device staging buffers are cached on the solver and guarded by a lock: concurrent calls on one solver serialise.

    ONE solve launch (gik_solve_rows_*), overlapped with its own transfers:
      * inputs: the copy engine streams the row-major host arrays into device staging buffers slab by slab on a copy
        stream and advances a device counter after each slab; the kernel is launched as soon as the first (small) slab
        is in, and a lane refill only waits if it runs ahead of the copies (copies deliver ~20x faster than the solver
        consumes, so in practice never);
      * outputs: the kernel stores q / converged (/ iters / resid) of each finished problem straight into the pinned
        host arrays (UVA stores over PCIe), so no device-to-host copy follows the kernel."""
    dev = self.device
    p12 = as_pose12(pose, dtype=dtype, device="cpu")
    B = p12.shape[0]
    qi = torch.as_tensor(q_init).to(dtype)
    if qi.dim() == 1:
        qi = qi.unsqueeze(0)
    if qi.shape[0] == 1 and B != 1:
        qi = qi.expand(B, self.nq)
    if out is not None:
        q_out, c_out = out[0], out[1]
        it_out = out[2] if len(out) > 2 else None
        r_out = out[3] if len(out) > 3 else None
        if return_info and (it_out is None or r_out is None):
            raise ValueError("return_info=True needs out=(q, converged, iters, resid)")
        want = [(q_out, (B, self.nq), dtype), (c_out, (B,), torch.uint8)]
        if it_out is not None:
            want.append((it_out, (B,), torch.int32))
        if r_out is not None:
            want.append((r_out, (B, 2), dtype))
        for t, shape, dt_ in want:
            if tuple(t.shape) != shape or t.dtype != dt_ or not t.is_contiguous() or t.is_cuda or (B and not t.is_pinned()):
                raise ValueError(f"out tensors must be pinned contiguous CPU tensors; expected {shape} {dt_}")
    else:
        q_out = torch.empty((B, self.nq), dtype=dtype, pin_memory=True) if B else torch.empty((0, self.nq), dtype=dtype)
        c_out = torch.empty((B,), dtype=torch.uint8, pin_memory=True) if B else torch.empty((0,), dtype=torch.uint8)
        it_out = (torch.empty((B,), dtype=torch.int32, pin_memory=True) if B else torch.empty((0,), dtype=torch.int32)) if return_info else None
        r_out = (torch.empty((B, 2), dtype=dtype, pin_memory=True) if B else torch.empty((0, 2), dtype=dtype)) if return_info else None
    if B == 0:
        return (q_out, c_out.view(torch.bool)) + ((SolveInfo(it_out, r_out),) if return_info else ())
    lock = self.__dict__.setdefault("_host_lock", threading.Lock())
    with lock:
        cache = self.__dict__.setdefault("_host_cache", {})
        # pageable inputs are staged through cached pinned buffers (a host memcpy); pinned inputs are used in place
        q_in = qi if (qi.is_pinned() and qi.is_contiguous()) else _pinned(cache, "q_in", (B, self.nq), dtype).copy_(qi)
        p_in = p12 if (p12.is_pinned() and p12.is_contiguous()) else _pinned(cache, "p_in", (B, 12), dtype).copy_(p12)
        key = (B, dtype)
        if cache.get("stage_key") != key:
            cache["stage_key"] = key
            cache["dq"] = torch.empty((B, self.nq), dtype=dtype, device=dev)
            cache["dp"] = torch.empty((B, 12), dtype=dtype, device=dev)
            cache["ready"] = torch.zeros((1,), dtype=torch.int64, device=dev)
        dq, dp, ready = cache["dq"], cache["dp"], cache["ready"]
        if self.__dict__.get("_poison_staging"):          # test hook: stale staging contents must never be read
            dq.fill_(float("nan")); dp.fill_(float("nan"))
        copy_stream = cache.get("copy_stream")
        if copy_stream is None:
            copy_stream = cache["copy_stream"] = torch.cuda.Stream(device=dev)
        bounds = _slab_bounds(B, slabs)
        marks = _pinned(cache, "marks", (len(bounds) - 1,), torch.int64)
        marks.copy_(torch.tensor(bounds[1:], dtype=torch.int64))
        cur = torch.cuda.current_stream(dev)
        copy_stream.wait_stream(cur)                      # staging buffers may still be read by a previous launch
        first_in = torch.cuda.Event()
        with torch.cuda.stream(copy_stream):
            ready.zero_()
            for k in range(len(bounds) - 1):
                lo, hi = bounds[k], bounds[k + 1]
                dq[lo:hi].copy_(q_in[lo:hi], non_blocking=True)
                dp[lo:hi].copy_(p_in[lo:hi], non_blocking=True)
                ready.copy_(marks[k:k + 1], non_blocking=True)
                if k == 0:
                    first_in.record(copy_stream)
        cur.wait_event(first_in)
        prm = self._params(eps, dt, max_iters, damping, kernel)
        self._call("solve_rows", dtype, B, self._ptr(dq), self._ptr(dp), ctypes.byref(prm), self._ptr(q_out),
                   self._ptr(c_out), self._ptr(it_out), self._ptr(r_out), self._ptr(ready))
        cur.synchronize()          # results are host memory: the call returns when the kernel has stored them
        copy_stream.synchronize()
    return (q_out, c_out.view(torch.bool)) + ((SolveInfo(it_out, r_out),) if return_info else ())


GraspIK.solve_host = solve_host

_default = {}


def default_solver(device=None) -> GraspIK:
    """Process-wide GraspIK for the built-in Nextage table on `device` (current CUDA device by default)."""
    if not torch.cuda.is_available():
        raise RuntimeError("no CUDA device: the batched grasp IK has no CPU fallback")
    idx = torch.cuda.current_device() if device is None else torch.device(device).index
    if idx is None:
        idx = torch.cuda.current_device()
    if idx not in _default:
        _default[idx] = GraspIK(nextage_table(), torch.device("cuda", idx))
    return _default[idx]


def fma_peak_tflops(device_index: int, elem_size: int, repeats: int = 5) -> float:
    out = ctypes.c_double(0.0)
    _cabi.check(_cabi.lib().gik_measure_fma_peak(device_index, elem_size, repeats, ctypes.byref(out)), "gik_measure_fma_peak")
    return out.value


def flops_per_iter() -> int:
    return int(_cabi.lib().gik_flops_per_iter())


def flops_per_iter_executed(elem_size: int, wrist: bool) -> int:
    return int(_cabi.lib().gik_flops_per_iter_executed(int(elem_size), 1 if wrist else 0))


def bytes_per_solve(elem_size: int) -> int:
    return int(_cabi.lib().gik_bytes_per_solve(elem_size))
