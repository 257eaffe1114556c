"""ctypes loader for the C oracle (oracle/grasp_ik_oracle.c) -- TEST INFRASTRUCTURE ONLY.
Row-major numpy in/out, fp64.  The table argument is any ctypes struct laid out like gik_table_t."""
from __future__ import annotations

import atexit
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))


def _cpu_tag():
    """The oracle is compiled with -march=native, so the artefact is keyed by the host CPU's model and ISA flags:
    a library built in the build container is not reused on a GPU box with a different CPU."""
    import hashlib
    key = ""
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith(("model name", "flags")):
                key += line
            if line.startswith("flags"):
                break
    except OSError:
        pass
    return hashlib.sha1(key.encode()).hexdigest()[:10]


LIB = os.path.join(_HERE, "_build", f"liboracle-{_cpu_tag()}.so")
_lib = None


def _writable(d):
    try:
        os.makedirs(d, exist_ok=True)
    except OSError:
        return False
    return os.access(d, os.W_OK)


def build(force=False):
    """Builds the library when it is missing or older than its sources.  Where oracle/_build cannot be written (a
    read-only checkout), it goes to a temporary directory that is removed when the process exits: bench.py's CPU
    baseline and smoke() then run from such a checkout.  The test suite still needs a writable one (it also builds
    tests/hostsim/_build)."""
    global LIB
    srcs = [os.path.join(_HERE, f) for f in ("grasp_ik_oracle.c", "collision_oracle.inc")]
    if force or not os.path.exists(LIB) or os.path.getmtime(LIB) < max(os.path.getmtime(s) for s in srcs):
        if not _writable(os.path.dirname(LIB)):
            d = tempfile.mkdtemp(prefix="gik-oracle-")
            atexit.register(shutil.rmtree, d, True)
            LIB = os.path.join(d, os.path.basename(LIB))
        subprocess.run(["make", "-C", _HERE, "-B" if force else "-s", f"OUT={LIB}"], check=True, capture_output=True)
    return LIB


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = ctypes.CDLL(LIB)
    return _lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _c(a, dt=np.float64):
    return np.ascontiguousarray(a, dtype=dt)


def fk(table_c, q):
    q = _c(q); n = q.shape[0]
    out = np.empty((n, 2, 12))
    lib().orc_fk(ctypes.byref(table_c), ctypes.c_int64(n), _p(q), _p(out))
    return out[:, :, :9].reshape(n, 2, 3, 3), out[:, :, 9:]


def jac(table_c, q):
    q = _c(q); n, nq = q.shape
    out = np.empty((n, 2, 6, nq))
    lib().orc_jac(ctypes.byref(table_c), ctypes.c_int64(n), _p(q), _p(out))
    return out


def solve(table_c, q_init, pose12, eps=1e-3, dt=1e-2, max_iters=1000, threads=0, damping=0.0):
    """damping = 0: the reference's pinv step; > 0: J^T (J J^T + damping I)^-1 e (BASELINE config 3's setting)."""
    q_init = _c(q_init); pose12 = _c(pose12); n, nq = q_init.shape
    q = np.empty((n, nq)); conv = np.empty(n, np.uint8); it = np.empty(n, np.int32); res = np.empty((n, 2))
    lib().orc_solve(ctypes.byref(table_c), ctypes.c_int64(n), _p(q_init), _p(pose12), ctypes.c_double(eps),
                    ctypes.c_double(dt), ctypes.c_int(max_iters), ctypes.c_double(damping), ctypes.c_int(threads), _p(q),
                    _p(conv), _p(it), _p(res))
    return q, conv.astype(bool), it, res


def set_step_method(method: int):
    """0 = pinv through the Jacobi SVD (the restatement every parity test uses); 1 = Cholesky of the normal equations
    (bench.py's `cpu_baseline.strong` timing only)."""
    lib().orc_set_step_method(ctypes.c_int(int(method)))


def interpolate(A12, B12, alpha):
    A12 = _c(A12); B12 = _c(B12); alpha = _c(alpha); n = A12.shape[0]
    out = np.empty((n, 12))
    lib().orc_interpolate(ctypes.c_int64(n), _p(A12), _p(B12), _p(alpha), _p(out))
    return out


def project_edges(table_c, q_start, pose_a, pose_b, num_steps, max_steps, eps=1e-3, dt=1e-2, max_iters=1000, threads=0,
                  damping=0.0):
    q_start = _c(q_start); pose_a = _c(pose_a); pose_b = _c(pose_b); ns = _c(num_steps, np.int32)
    n, nq = q_start.shape
    path = np.zeros((n, max_steps, nq)); nv = np.empty(n, np.int32); itt = np.empty(n, np.int32)
    lib().orc_project_edges(ctypes.byref(table_c), ctypes.c_int64(n), ctypes.c_int(max_steps), _p(q_start), _p(pose_a),
                            _p(pose_b), _p(ns), ctypes.c_double(eps), ctypes.c_double(dt), ctypes.c_int(max_iters),
                            ctypes.c_double(damping), ctypes.c_int(threads), _p(path), _p(nv), _p(itt))
    return path, nv, itt


def scene_distance(table_c, scene_c, q, cube_pose=None, mode=0, cull=0.0, threads=0):
    """Minimum pair distance per configuration (0 = collision).  mode 0: all pairs (tools.collision), 1: table/obstacle
    pairs (tools.distanceToObstacle), 2: cube vs table/obstacle (path.py:51-52; q may be None)."""
    if q is not None:
        q = _c(q); n = q.shape[0]
    else:
        cube_pose = _c(cube_pose); n = cube_pose.shape[0]
    cp = _c(cube_pose) if cube_pose is not None else None
    out = np.empty(n)
    L = lib()
    L.orc_scene_distance(ctypes.byref(table_c), ctypes.byref(scene_c), ctypes.c_int64(n), _p(q) if q is not None else None,
                         _p(cp) if cp is not None else None, ctypes.c_int(mode), ctypes.c_double(cull),
                         ctypes.c_int(threads), _p(out))
    return out


def solve_success(table_c, scene_c, q_init, pose12, eps=1e-3, dt=1e-2, max_iters=1000, threads=0, damping=0.0,
                  return_ever=False):
    """computeqgrasppose with the collision term of the predicate (inverse_geometry.py:70, 97-98).
    return_ever: also return whether both residuals ever passed (i.e. the plain solve would have converged)."""
    q_init = _c(q_init); pose12 = _c(pose12); n, nq = q_init.shape
    q = np.empty((n, nq)); ok = np.empty(n, np.uint8); it = np.empty(n, np.int32); ever = np.empty(n, np.uint8)
    lib().orc_solve_success(ctypes.byref(table_c), ctypes.byref(scene_c), ctypes.c_int64(n), _p(q_init), _p(pose12),
                            ctypes.c_double(eps), ctypes.c_double(dt), ctypes.c_int(max_iters), ctypes.c_double(damping),
                            ctypes.c_int(threads), _p(q), _p(ok), _p(it), _p(ever))
    if return_ever:
        return q, ok.astype(bool), it, ever.astype(bool)
    return q, ok.astype(bool), it


def pair_distance(type_a, Ra, pa, sa, type_b, Rb, pb, sb):
    L = lib()
    L.orc_pair_distance.restype = ctypes.c_double
    a = [_c(np.asarray(x, float).reshape(-1)) for x in (Ra, pa, sa, Rb, pb, sb)]
    return L.orc_pair_distance(ctypes.c_int(type_a), _p(a[0]), _p(a[1]), _p(a[2]), ctypes.c_int(type_b), _p(a[3]), _p(a[4]), _p(a[5]))


def max_threads():
    return int(lib().orc_max_threads())
