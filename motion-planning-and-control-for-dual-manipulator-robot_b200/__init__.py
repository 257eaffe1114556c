"""B200-native batched dual-arm grasp-pose IK: drop-in for the hot path of the reference's
`inverse_geometry.computeqgrasppose` (Ulixes-8/Motion-Planning-and-Control-for-Dual-Manipulator-Robot).

    from gik_b200 import computeqgrasppose, computeqgrasppose_batch, GraspIK

The arithmetic lives in csrc/ (CUDA, sm_100a) behind the C ABI of include/gik.h; nothing here falls back to
the CPU."""
from .model import KinematicTable, from_pinocchio, from_urdf, nextage_table          # noqa: F401
from .scene import CollisionScene, nextage_scene, scene_from_pinocchio, scene_from_urdf                               # noqa: F401
from .ops import (DT, EPSILON, MAX_ITERS, GraspIK, SolveInfo, as_pose12, bytes_per_solve,  # noqa: F401
                  default_solver, flops_per_iter, flops_per_iter_executed, fma_peak_tflops)
from .inverse_geometry import apply_collision, computeqgrasppose, computeqgrasppose_batch, solver_for  # noqa: F401
from .path import (computepath, edge_num_steps, project_edges_batch, project_path, sample_cube_placements,  # noqa: F401
                   sample_grasp_poses_batch, se3_interpolate)
from .planner import computepath_batch, shortcut_paths_batch                          # noqa: F401
from .roadmap import Roadmap, build_roadmap, query_roadmap_batch                      # noqa: F401
from .trajectory import (Bezier, check_trajectories_batch, check_trajectory, maketraj, maketraj_batch,  # noqa: F401
                         maketraj_paths, refine_trajectories_batch)
from . import tools                                                                   # noqa: F401
from . import experiments                                                             # noqa: F401
from . import dist                                                                     # noqa: F401
from ._cabi import GikError, build                                                     # noqa: F401

__version__ = "0.1.0"
