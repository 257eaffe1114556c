"""ctypes binding of libgik.so (include/gik.h).  No CPU fallback: if the library is missing or a call fails,
this module raises."""
from __future__ import annotations

import ctypes
import os
import shutil
import subprocess

from .model import GikTable

_HERE = os.path.dirname(os.path.abspath(__file__))
# GIK_LIB overrides the library path (A/B runs of differently tuned builds of the SAME sources; still no fallback)
LIB_PATH = os.environ.get("GIK_LIB") or os.path.join(_HERE, "libgik.so")
CSRC = os.path.join(_HERE, "csrc")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O3", "-lineinfo",
              "-shared", "-Xcompiler", "-fPIC"]


class GikParams(ctypes.Structure):
    """ctypes mirror of gik_params_t."""
    _fields_ = [("eps", ctypes.c_double), ("dt", ctypes.c_double), ("damping", ctypes.c_double),
                ("max_iters", ctypes.c_int32), ("flags", ctypes.c_int32)]


class GikError(RuntimeError):
    def __init__(self, code: int, msg: str, where: str):
        super().__init__(f"{where}: {msg} (code {code})")
        self.code = code


def _sources():
    return [os.path.join(CSRC, f) for f in ("gik_kernels.cu", "gik_core.cuh", "gik_table.h", "gik_collide.cuh",
                                            "gik_collide_impl.cuh", "gik_bezier.cuh", "gik_tree.cuh",
                                            "gik_shortcut.cuh", "gik_traj.cuh")] + \
           [os.path.join(_HERE, "..", "include", "gik.h")]


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/gik_kernels.cu for sm_100a into libgik.so next to this file (nvcc cross-compiles
    without a GPU).  Rebuilds when a source is newer than the library."""
    srcs = _sources()
    if os.environ.get("GIK_LIB"):
        return LIB_PATH
    if not force and os.path.exists(LIB_PATH):
        t = os.path.getmtime(LIB_PATH)
        if all(os.path.getmtime(s) <= t for s in srcs if os.path.exists(s)):
            return LIB_PATH
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: cannot build libgik.so")
    tmp = LIB_PATH + ".tmp"
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", tmp, srcs[0]]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    os.replace(tmp, LIB_PATH)
    return LIB_PATH


_lib = None

_P = ctypes.c_void_p
_I64 = ctypes.c_int64
_I32 = ctypes.c_int32


def lib() -> ctypes.CDLL:
    """Load libgik.so (once).  Fails loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: the CUDA library has not been built "
            "(run `python -c 'import __graft_entry__ as g; g.build()'`).  There is no CPU fallback.")
    L = ctypes.CDLL(LIB_PATH)
    PP = ctypes.POINTER(GikParams)
    L.gik_default_params.argtypes = [PP]; L.gik_default_params.restype = None
    L.gik_create.argtypes = [ctypes.POINTER(GikTable), ctypes.c_int, ctypes.POINTER(_P)]
    L.gik_destroy.argtypes = [_P]
    for sfx in ("f32", "f64"):
        getattr(L, f"gik_fk_{sfx}").argtypes = [_P, _I64, _P, _P, _P]
        getattr(L, f"gik_jac_{sfx}").argtypes = [_P, _I64, _P, _P, _P]
        getattr(L, f"gik_solve_{sfx}").argtypes = [_P, _I64, _P, _P, PP, _P, _P, _P, _P, _P]
        getattr(L, f"gik_solve_rows_{sfx}").argtypes = [_P, _I64, _P, _P, PP, _P, _P, _P, _P, _P, _P]
        getattr(L, f"gik_solve_scatter_{sfx}").argtypes = [_P, _I64, _P, _P, PP, _I32, ctypes.POINTER(_P),
                                                            ctypes.POINTER(_P), _I64, _I64, _P, _P, _P]
        getattr(L, f"gik_best_of_{sfx}").argtypes = [_P, _I64, _I32, _P, _P, _P, _P, _P, _P, _P]
        getattr(L, f"gik_project_edges_{sfx}").argtypes = [_P, _I64, _I32, _P, _P, _P, _P, PP, _P, _P, _P, _P]
    from .scene import GikScene
    L.gik_scene_attach.argtypes = [_P, ctypes.POINTER(GikScene)]
    for sfx in ("f32", "f64"):
        getattr(L, f"gik_collision_{sfx}").argtypes = [_P, _I64, _P, _P, _P, _P]
        getattr(L, f"gik_collision_sel_{sfx}").argtypes = [_P, _I64, _I64, _P, _P, _P, _P, _P]
        getattr(L, f"gik_solve_success_{sfx}").argtypes = [_P, _I64, _P, _P, PP, _P, _P, _P, _P, _P, _P, _P]
        getattr(L, f"gik_clearance_{sfx}").argtypes = [_P, _I64, _P, _P, ctypes.c_double, _P, _P]
        getattr(L, f"gik_cube_collision_{sfx}").argtypes = [_P, _I64, _P, _P, _P]
        getattr(L, f"gik_obstacle_distance_{sfx}").argtypes = [_P, _I64, _P, _P, ctypes.c_double, _P, _P]
        getattr(L, f"gik_bezier_fit_{sfx}").argtypes = [_P, _I64, _I32, _I32, _I32] + [_P] * 10
        getattr(L, f"gik_tree_nearest_{sfx}").argtypes = [_P, _I64, _I32, _P, _P, _I64, _P, _P, _P, _P]
        getattr(L, f"gik_tree_grow_{sfx}").argtypes = [_P, _I64, _I32, _P, _P, _P, _P, _P, _I64, _I32] + [_P] * 10
        getattr(L, f"gik_tree_paths_{sfx}").argtypes = [_P, _I64, _I32] + [_P] * 10
        getattr(L, f"gik_path_shortcut_{sfx}").argtypes = [_P, _I64, _I32, _I32] + [_P] * 8 + [ctypes.c_double] + [_P] * 6
        getattr(L, f"gik_traj_check_{sfx}").argtypes = [_P, _I64, _I32, _I32, _P, _P, ctypes.c_double, ctypes.c_double] + [_P] * 6
    L.gik_solve_success_scratch_bytes.argtypes = [_P, _I64, ctypes.c_int]
    L.gik_solve_success_scratch_bytes.restype = ctypes.c_size_t
    L.gik_flops_per_iter.restype = ctypes.c_size_t
    L.gik_flops_per_iter_executed.argtypes = [ctypes.c_int, ctypes.c_int]
    L.gik_flops_per_iter_executed.restype = ctypes.c_size_t
    L.gik_bytes_per_solve.argtypes = [ctypes.c_int]; L.gik_bytes_per_solve.restype = ctypes.c_size_t
    L.gik_measure_fma_peak.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_double)]
    L.gik_solve_launch_dims.argtypes = [_P, ctypes.c_int, _I64, ctypes.POINTER(_I32), ctypes.POINTER(_I32)]
    L.gik_solve_kernel_name.argtypes = [_P, ctypes.c_int, _I64, ctypes.c_int]
    L.gik_solve_kernel_name.restype = ctypes.c_char_p
    L.gik_strerror.argtypes = [ctypes.c_int]; L.gik_strerror.restype = ctypes.c_char_p
    L.gik_version.restype = ctypes.c_char_p
    _lib = L
    return L


EXPORTS = [
    "gik_default_params", "gik_create", "gik_destroy",
    "gik_fk_f32", "gik_fk_f64", "gik_jac_f32", "gik_jac_f64", "gik_solve_f32", "gik_solve_f64",
    "gik_solve_rows_f32", "gik_solve_rows_f64", "gik_solve_scatter_f32", "gik_solve_scatter_f64", "gik_best_of_f32", "gik_best_of_f64", "gik_project_edges_f32", "gik_project_edges_f64",
    "gik_scene_attach", "gik_collision_f32", "gik_collision_f64", "gik_collision_sel_f32", "gik_collision_sel_f64", "gik_solve_success_f32", "gik_solve_success_f64", "gik_solve_success_scratch_bytes", "gik_clearance_f32", "gik_clearance_f64",
    "gik_cube_collision_f32", "gik_cube_collision_f64", "gik_obstacle_distance_f32", "gik_obstacle_distance_f64",
    "gik_bezier_fit_f32", "gik_bezier_fit_f64",
    "gik_tree_nearest_f32", "gik_tree_nearest_f64", "gik_tree_grow_f32", "gik_tree_grow_f64",
    "gik_tree_paths_f32", "gik_tree_paths_f64", "gik_path_shortcut_f32", "gik_path_shortcut_f64", "gik_traj_check_f32", "gik_traj_check_f64",
    "gik_flops_per_iter", "gik_flops_per_iter_executed", "gik_bytes_per_solve", "gik_measure_fma_peak", "gik_solve_launch_dims",
    "gik_solve_kernel_name",
    "gik_strerror", "gik_version",
]


def check(code: int, where: str) -> None:
    if code != 0:
        raise GikError(code, lib().gik_strerror(code).decode(), where)
