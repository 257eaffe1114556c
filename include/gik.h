/* gik.h -- C ABI of the B200-native batched dual-arm grasp-pose IK library (libgik.so).
 *
 * The reference (Ulixes-8/Motion-Planning-and-Control-for-Dual-Manipulator-Robot) is pure Python and
 * has no FFI layer of its own; its boundary for this path is the Python function
 *     computeqgrasppose(robot, qcurrent, cube, cubetarget, viz=None) -> (q, success)
 * (inverse_geometry.py:17,100).  The entry points below are what a reference-side binding (ctypes, see
 * INTEGRATION.md) calls to replace the body of that function and of its two batch callers
 * (path.py:57 sampling, path.py:125-163 edge projection).  Each entry cites the reference code it replaces.
 *
 * Conventions
 *   - Plain C, no CUDA or torch types.  `stream` is a cudaStream_t passed as void* (NULL = default stream).
 *   - All data pointers are DEVICE pointers owned by the caller.  The handle owns only the constant
 *     kinematic table.  Launches are asynchronous on `stream`; the caller synchronises.
 *   - Return value: 0 = ok, negative = invalid argument / unsupported model (GIK_E_*),
 *     positive = a cudaError_t value.  No exceptions cross the ABI.
 *   - A handle is immutable after gik_create: concurrent calls on different streams are safe.
 *   - Batch layout is structure-of-arrays, component-major: element (c, i) of a [C][n] array lives at
 *     ptr[c * n + i], so consecutive problems are consecutive addresses.
 *       q      : [nq][n]           joint configuration, pinocchio order (q index = joint id - 1)
 *       pose   : [12][n]           cube placement: rows 0-8 rotation row-major, rows 9-11 translation
 *       frames : [2][12][n]        LARM_EFF, RARM_EFF world placements, same 12-row layout
 *       jac    : [2][6][nq][n]     LOCAL frame Jacobians, rows [linear(3); angular(3)]
 *       resid  : [2][n]            ||log6(hand^-1 * hook)|| for left, right
 */
#ifndef GIK_H_
#define GIK_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GIK_MAX_NQ 32

/* error codes (negative); positive return values are cudaError_t */
#define GIK_OK                 0
#define GIK_E_NULL            -1   /* null pointer argument */
#define GIK_E_SIZE            -2   /* negative / oversized count */
#define GIK_E_MODEL           -3   /* kinematic table is not a tree of 1-dof revolute joints */
#define GIK_E_TOPOLOGY        -4   /* table does not match the compiled torso + two 6R-arm fast path */
#define GIK_E_PARAM           -5   /* bad solver parameter (eps<=0, dt<=0, max_iters<0, damping<0) */
#define GIK_E_HANDLE          -6   /* bad or destroyed handle */
#define GIK_E_NOSCENE         -7   /* collision entry called before gik_scene_attach */

/* Host-side flattened kinematic model: what the reference obtains from
 * RobotWrapper.BuildFromURDF + translaterobot (setup_pinocchio.py:28-32,73-75) and from the cube's
 * hook frames (setup_pinocchio.py:44-50, tools.py:54-59).  All joints are 1-dof revolute about a
 * coordinate axis (pinocchio JointModelRX/RY/RZ), listed in q order with parents first. */
typedef struct gik_table_s {
  int32_t nq;                        /* number of joints = size of q (15 for Nextage) */
  int32_t parent[GIK_MAX_NQ];        /* parent q index, -1 = universe */
  int32_t axis[GIK_MAX_NQ];          /* 0 = x, 1 = y, 2 = z */
  double  joint_R[GIK_MAX_NQ][9];    /* model.jointPlacements[i+1].rotation, row-major */
  double  joint_p[GIK_MAX_NQ][3];    /* model.jointPlacements[i+1].translation */
  double  lower[GIK_MAX_NQ];         /* model.lowerPositionLimit */
  double  upper[GIK_MAX_NQ];         /* model.upperPositionLimit */
  int32_t hand_joint[2];             /* q index of the joint carrying LARM_EFF / RARM_EFF (config.py:25-26) */
  double  hand_R[2][9];              /* model.frames[getFrameId(hand)].placement.rotation */
  double  hand_p[2][3];
  double  hook_R[2][9];              /* cube.data.oMf[getFrameId(LARM_HOOK / RARM_HOOK)] (config.py:28-29) */
  double  hook_p[2][3];
} gik_table_t;

/* Solver parameters.  Defaults reproduce the reference literals:
 * eps = EPSILON = 1e-3 (config.py:22), dt = DT = 1e-2 and max_iters = 1000 (inverse_geometry.py:53-54),
 * damping = 0 (undamped pseudo-inverse, inverse_geometry.py:83). */
typedef struct gik_params_s {
  double  eps;        /* per-hand convergence tolerance on ||log6||_2 */
  double  dt;         /* step length: q <- clamp(q + dt * J^+ e) */
  double  damping;    /* lambda in J^T (J J^T + lambda I)^-1 e; 0 = pseudo-inverse */
  int32_t max_iters;  /* iteration cap */
  int32_t flags;      /* 0, or GIK_F_* bits: scheduling overrides (results unaffected) and GIK_F_EARLY_STOP */
} gik_params_t;

/* gik_params_t.flags: by default the launcher picks the kernel mapping from the batch size -- one problem per lane
 * when the batch can occupy at least half of the lanes of every resident warp, one problem per lane PAIR (one hand
 * per lane) below that.  These force one mapping (A/B measurements, tests). */
#define GIK_F_LANE_KERNEL 2
#define GIK_F_PAIR_KERNEL 4
#define GIK_F_SCALAR_LANE 8   /* fp32 lane mapping with scalar FFMA instead of the packed FFMA2 kernel (A/B only) */
/* NOT the reference semantics for failed problems -- a separately reported fast preset: stop a problem as soon as the
 * sum of its two squared residuals has fallen by less than 10 % over the last 64 iterations (a converging problem
 * shrinks it by 72 % over 64 iterations at dt = 1e-2; a problem pinned at its joint limits plateaus).  The problem is
 * reported non-converged with iters = iterations done and q = the iterate reached.  The q of converged problems is
 * unchanged; success flags agree on 99.9997 % (fp32) / 99.993 % (fp64) of 2^20 workspace problems -- the exceptions
 * are late convergers (850-1000 iterations) that are given up on; there are no false successes (DESIGN.md). */
#define GIK_F_EARLY_STOP 16
/* Form of the step.  By default an UNDAMPED step (damping = 0) on a table with a spherical wrist (the Nextage arms: the
 * axes of the last three joints of each arm meet in one point) is computed as dq_arm = u - kappa w with u = A^-1 e,
 * w = A^-1 c through two 3x3 solves per hand at the wrist centre -- algebraically the same pinv(J) e as the reference's
 * (inverse_geometry.py:83) wherever J has full row rank.  This flag keeps the general form (6x6 block Cholesky of
 * A A^T + lambda I and Sherman-Morrison), which damping > 0 and other tables always use.  For A/B runs and tests. */
#define GIK_F_CHOLESKY 32

typedef struct gik_handle_s* gik_handle_t;

/* Fills `p` with the reference defaults above. */
void gik_default_params(gik_params_t* p);

/* Validates `host_table`, derives the fast-path constants and uploads them to `device`. */
int gik_create(const gik_table_t* host_table, int device, gik_handle_t* out);
int gik_destroy(gik_handle_t h);

/* K1. Replaces pin.framesForwardKinematics + data.oMf[LARM_EFF / RARM_EFF]
 * (inverse_geometry.py:58,62-63).  q [nq][n] -> frames [2][12][n]. */
int gik_fk_f32(gik_handle_t h, int64_t n, const float* q, float* frames, void* stream);
int gik_fk_f64(gik_handle_t h, int64_t n, const double* q, double* frames, void* stream);

/* K2. Replaces pin.computeFrameJacobian(model, data, q, frame_id) for both hands, LOCAL reference
 * frame (inverse_geometry.py:75-76).  q [nq][n] -> jac [2][6][nq][n]. */
int gik_jac_f32(gik_handle_t h, int64_t n, const float* q, float* jac, void* stream);
int gik_jac_f64(gik_handle_t h, int64_t n, const double* q, double* jac, void* stream);

/* K3. Replaces the descent loop of computeqgrasppose (inverse_geometry.py:49-94) for n independent
 * problems, without the collision() term of the predicate at :70 (applied by the caller, see
 * INTEGRATION.md).  q_init [nq][n], pose [12][n] -> q_out [nq][n], converged [n] (1 = the loop broke
 * with both residuals < eps), iters [n] (updates applied), resid [2][n] (residuals at q_out).
 * `iters` and `resid` may be NULL. */
int gik_solve_f32(gik_handle_t h, int64_t n, const float* q_init, const float* pose,
                  const gik_params_t* params, float* q_out, uint8_t* converged, int32_t* iters,
                  float* resid, void* stream);
int gik_solve_f64(gik_handle_t h, int64_t n, const double* q_init, const double* pose,
                  const gik_params_t* params, double* q_out, uint8_t* converged, int32_t* iters,
                  double* resid, void* stream);

/* K3 with ROW-MAJOR I/O and streamed input, for host-resident batches (the layout of the Python API: q [n][nq],
 * pose [n][12]).  q_init / pose are DEVICE staging buffers; `ready` (device, may be NULL = everything resident) counts
 * the leading problems already copied in -- the caller advances it on its copy stream after each slab, so the copy
 * engine fills the staging buffers while the kernel is already solving (a lane refill waits only if it runs ahead of
 * the copies).  q_out [n][nq], converged [n], iters [n] and resid [n][2] (iters / resid may be NULL) may be PINNED
 * HOST memory (UVA): results are stored straight over PCIe from the kernel, so no device-to-host copy follows it. */
int gik_solve_rows_f32(gik_handle_t h, int64_t n, const float* q_init, const float* pose, const gik_params_t* params,
                       float* q_out, uint8_t* converged, int32_t* iters, float* resid,
                       const unsigned long long* ready, void* stream);
int gik_solve_rows_f64(gik_handle_t h, int64_t n, const double* q_init, const double* pose, const gik_params_t* params,
                       double* q_out, uint8_t* converged, int32_t* iters, double* resid,
                       const unsigned long long* ready, void* stream);

/* K3 fused with its all-gather (multi-GPU, SURVEY.md 8e): the same solve, and the SAME launch fills the result arrays
 * of ALL ranks through peer-mapped pointers -- lanes store into the array that lives on this device, pusher warps of
 * the kernel copy finished 1024-problem chunks into the others with coalesced 16-byte NVLink / NVSwitch P2P stores while
 * the remaining blocks keep solving, and a tail kernel (same stream) copies the chunks still in flight at the end -- so
 * no collective follows.  Results are bit-identical to gik_solve_*.  q_all[p] / conv_all[p] are HOST arrays of n_peers
 * device pointers, valid on this handle's device (this rank's own buffer and the peer mappings of the others, e.g.
 * CUDA IPC or torch symmetric memory): rank p's q array [nq][n_total] and flag array [n_total].  This rank's problem i
 * lands in column offset + i of every array.  iters [n] / resid [2][n] stay local and may be NULL.  The caller
 * provides the cross-rank barrier after the launch (results are visible to a peer once this stream has passed it). */
#define GIK_MAX_PEERS 16
int gik_solve_scatter_f32(gik_handle_t h, int64_t n, const float* q_init, const float* pose,
                          const gik_params_t* params, int32_t n_peers, float* const* q_all,
                          uint8_t* const* conv_all, int64_t n_total, int64_t offset, int32_t* iters, float* resid,
                          void* stream);
int gik_solve_scatter_f64(gik_handle_t h, int64_t n, const double* q_init, const double* pose,
                          const gik_params_t* params, int32_t n_peers, double* const* q_all,
                          uint8_t* const* conv_all, int64_t n_total, int64_t offset, int32_t* iters, double* resid,
                          void* stream);

/* K4. Best-of-restarts reduction (new; BASELINE config 3).  Problem (p, r) of a [n_place x n_restart]
 * solve is stored at index p * n_restart + r.  Picks, per placement, the converged candidate with the
 * smallest max(resid_L, resid_R); ties -> lowest restart index; if none converged, the smallest
 * residual overall with converged = 0.  q [nq][n_place*n_restart] -> q_best [nq][n_place],
 * conv_best [n_place], which [n_place] (restart index chosen; may be NULL). */
int gik_best_of_f32(gik_handle_t h, int64_t n_place, int32_t n_restart, const float* q,
                    const uint8_t* converged, const float* resid, float* q_best, uint8_t* conv_best,
                    int32_t* which, void* stream);
int gik_best_of_f64(gik_handle_t h, int64_t n_place, int32_t n_restart, const double* q,
                    const uint8_t* converged, const double* resid, double* q_best, uint8_t* conv_best,
                    int32_t* which, void* stream);

/* K5. Replaces the loop of project_path (path.py:137-160) for n_edges independent edges: for
 * step = 1..num_steps[e] the cube placement is SE3.Interpolate(pose_a, pose_b, step / num_steps[e])
 * (path.py:139-141) and the IK is warm-started from the previous step's q (path.py:152);
 * the march stops at the first non-converged step (path.py:153-156).
 * q_start [nq][E], pose_a / pose_b [12][E], num_steps [E] (1..max_steps) ->
 * q_path [max_steps][nq][E] (rows >= n_valid[e] are left untouched), n_valid [E] (converged steps),
 * iters_total [E] (descent iterations executed on the edge; may be NULL). */
int gik_project_edges_f32(gik_handle_t h, int64_t n_edges, int32_t max_steps, const float* q_start,
                          const float* pose_a, const float* pose_b, const int32_t* num_steps,
                          const gik_params_t* params, float* q_path, int32_t* n_valid,
                          int32_t* iters_total, void* stream);
int gik_project_edges_f64(gik_handle_t h, int64_t n_edges, int32_t max_steps, const double* q_start,
                          const double* pose_a, const double* pose_b, const int32_t* num_steps,
                          const gik_params_t* params, double* q_path, int32_t* n_valid,
                          int32_t* iters_total, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Collision predicate (SURVEY.md 8f-1).  The reference's success flag is `converged and not collision(robot, q)`
 * (inverse_geometry.py:70,97-98); path.py additionally filters samples on distanceToObstacle(robot, q) >= 0.04
 * (path.py:61-62) and on the cube's own collisions with the table / obstacle (path.py:51-52, 145-146).
 * gik_scene_t is the flattened collision model that setup_pinocchio.py:44-83 assembles: convex primitives attached
 * to joints, plus the pair list after addAllCollisionPairs / SRDF removal / the extra obstacle-cube pair.
 * ------------------------------------------------------------------------------------------------------- */
#define GIK_MAX_GEOMS 64
#define GIK_MAX_PAIRS 1024
#define GIK_GEOM_BOX      0   /* size = half extents */
#define GIK_GEOM_SPHERE   1   /* size[0] = radius */
#define GIK_GEOM_CYLINDER 2   /* size[0] = radius, size[1] = half length, axis = local z */

typedef struct gik_geom_s {
  int32_t type;       /* GIK_GEOM_* */
  int32_t joint;      /* q index of the parent joint, -1 = universe (GeometryObject.parentJoint - 1) */
  double  R[9];       /* GeometryObject.placement in the parent joint frame, row-major */
  double  p[3];
  double  size[3];
} gik_geom_t;

typedef struct gik_scene_s {
  int32_t n_geoms, n_pairs;
  int32_t cube_geom;      /* geometry whose placement is replaced per problem (tools.setcubeplacement) */
  int32_t table_geom;     /* 'baseLink_0' */
  int32_t obstacle_geom;  /* 'obstaclebase_0' */
  int32_t reserved;
  gik_geom_t geoms[GIK_MAX_GEOMS];
  uint8_t pair_a[GIK_MAX_PAIRS], pair_b[GIK_MAX_PAIRS];   /* robot.collision_model.collisionPairs */
} gik_scene_t;

/* Uploads the scene to the handle's device (replaces a previous one).  Returns GIK_E_SIZE / GIK_E_MODEL on a bad scene. */
int gik_scene_attach(gik_handle_t h, const gik_scene_t* scene);

/* Replaces tools.collision(robot, q) (tools.py:25-35) for n configurations: q [nq][n]; cube_pose [12][n] = placement
 * of the cube geometry for each problem (what setcubeplacement wrote before the reference's call; NULL = the scene's
 * own) -> colliding [n] (1 = at least one collision pair intersects). */
int gik_collision_f32(gik_handle_t h, int64_t n, const float* q, const float* cube_pose, uint8_t* colliding, void* stream);
int gik_collision_f64(gik_handle_t h, int64_t n, const double* q, const double* cube_pose, uint8_t* colliding, void* stream);

/* Same test on a SUBSET of the columns: sel [n_sel] (device, int64) lists the columns of the [.][n] arrays to test;
 * colliding[sel[k]] is written, the other entries are left untouched.  This is the predicate's short-circuit
 * (inverse_geometry.py:70 evaluates collision() only where both residuals pass) without gathering the columns. */
int gik_collision_sel_f32(gik_handle_t h, int64_t n, int64_t n_sel, const int64_t* sel, const float* q,
                          const float* cube_pose, uint8_t* colliding, void* stream);
int gik_collision_sel_f64(gik_handle_t h, int64_t n, int64_t n_sel, const int64_t* sel, const double* q,
                          const double* cube_pose, uint8_t* colliding, void* stream);

/* K3 + the collision term: the reference's FULL success predicate (inverse_geometry.py:70, 97-98) in ONE stream-ordered
 * call without host synchronisation.
 *   1. the descent loop (as gik_solve_*), stopping at the first iterate with both residuals < eps;
 *   2. success[i] = converged[i] && !collision(q_out[:, i]), collision() evaluated only on the converged problems
 *      (device-side compaction: the predicate's short-circuit);
 *   3. the reference KEEPS DESCENDING while a converged iterate collides, re-testing collision() after every update
 *      until an iterate is free (success, that q, that iteration count) or max_iters is reached (failure, q after
 *      max_iters updates).  The converged-but-colliding problems are continued to the cap by a second launch of the
 *      solve kernel, and a warp-per-problem kernel then decides each one: a pair of solids that still intersects after
 *      erosion by the (bounded) displacement of the remaining descent collides on every iterate -- the problem fails
 *      with the final q, as in the reference; otherwise the descent is replayed from the converged iterate with the
 *      undecided pairs tested on every iterate.  Same decisions as the reference's loop.
 * params.flags & GIK_F_NO_DESCEND stops after step 2 (the predicate evaluated once, at the configuration the descent
 * stopped at: differs only where further descent would have freed a collision, and in the q of failed problems).
 * On return converged[i] = 1 iff the loop broke at q_out[:, i] (so converged == success except with GIK_F_NO_DESCEND,
 * where converged keeps step 1's flag); iters / resid describe q_out.  success, converged, iters, resid must not be
 * NULL.  scratch: device memory of gik_solve_success_scratch_bytes(h, n, elem_size) bytes. */
#define GIK_F_NO_DESCEND 64
size_t gik_solve_success_scratch_bytes(gik_handle_t h, int64_t n, int elem_size);
int gik_solve_success_f32(gik_handle_t h, int64_t n, const float* q_init, const float* pose, const gik_params_t* params,
                          float* q_out, uint8_t* success, uint8_t* converged, int32_t* iters, float* resid,
                          void* scratch, void* stream);
int gik_solve_success_f64(gik_handle_t h, int64_t n, const double* q_init, const double* pose, const gik_params_t* params,
                          double* q_out, uint8_t* success, uint8_t* converged, int32_t* iters, double* resid,
                          void* scratch, void* stream);

/* Replaces `distanceToObstacle(robot, q) >= threshold` (tools.py:38-51 with path.py:61-62): clear [n] = 1 when every
 * pair whose second geometry is the table or the obstacle is at least `threshold` apart. */
int gik_clearance_f32(gik_handle_t h, int64_t n, const float* q, const float* cube_pose, double threshold, uint8_t* clear, void* stream);
int gik_clearance_f64(gik_handle_t h, int64_t n, const double* q, const double* cube_pose, double threshold, uint8_t* clear, void* stream);

/* Replaces `distanceToObstacle(robot, q)` itself (tools.py:38-51) as a value: dist [n] = the smallest distance over the
 * pairs whose second geometry is the table or the obstacle, capped at d_max (> 0); 0 when such a pair intersects
 * (hpp-fcl returns the negative penetration depth there -- every caller in the reference only compares the value with
 * a positive threshold, path.py:61-62).  One launch: each pair's distance is bracketed by bisection on the margin of
 * the same boolean GJK, to d_max / 2^20 (f32) or d_max / 2^40 (f64). */
int gik_obstacle_distance_f32(gik_handle_t h, int64_t n, const float* q, const float* cube_pose, double d_max, float* dist, void* stream);
int gik_obstacle_distance_f64(gik_handle_t h, int64_t n, const double* q, const double* cube_pose, double d_max, double* dist, void* stream);

/* Replaces the cube's own collision test of path.py:51-52 / 145-146 (cube vs table, cube vs obstacle):
 * cube_pose [12][n] -> colliding [n]. */
int gik_cube_collision_f32(gik_handle_t h, int64_t n, const float* cube_pose, uint8_t* colliding, void* stream);
int gik_cube_collision_f64(gik_handle_t h, int64_t n, const double* cube_pose, uint8_t* colliding, void* stream);

/* Measurement helpers (bench.py). */
/* Algorithmic FLOPs of ONE descent iteration of ONE dual-arm problem (SURVEY.md 8d breakdown). */
size_t gik_flops_per_iter(void);
/* FLOPs the solve kernels actually EXECUTE per descent iteration of one problem, from the executed opcode mix of the
 * committed ncu captures (FMA = 2, MUL / ADD = 1): elem_size 4 / 8, wrist = 1 for the spherical-wrist step, 0 for the
 * block-Cholesky step.  Reported by bench.py beside the algorithmic count (roofline.frac_executed). */
size_t gik_flops_per_iter_executed(int elem_size, int wrist);
/* Algorithmic bytes moved per solve (inputs + outputs), elem_size = 4 or 8. */
size_t gik_bytes_per_solve(int elem_size);
/* Runs a register-resident FMA chain on every SM and returns the achieved TFLOP/s (FMA = 2 FLOP) of the
 * FP32 (elem_size 4) or FP64 (elem_size 8) CUDA-core pipe in *tflops; synchronous. */
int gik_measure_fma_peak(int device, int elem_size, int repeats, double* tflops);
/* Grid the solver launches for n problems on the handle's device (for gpu_launches / occupancy reports). */
int gik_solve_launch_dims(gik_handle_t h, int elem_size, int64_t n, int32_t* blocks, int32_t* threads);
/* Name of the kernel gik_solve_* launches for n problems with params.flags = flags (static string; "" on bad
 * arguments).  For reports: bench.py's roofline.kernel. */
const char* gik_solve_kernel_name(gik_handle_t h, int elem_size, int64_t n, int flags);

const char* gik_strerror(int code);
const char* gik_version(void);

/* Replaces the least-squares fit inside `maketraj` (control.py:63-195: degree-n Bezier curve through the planned path
 * with position / velocity / acceleration constraints at both ends) for MANY paths at once.  The constraints pin three
 * control points at each end; the free ones are a linear least-squares problem whose design matrix -- Bernstein basis at
 * n_points uniform times -- is the same for every path, so the caller factors it once on the host:
 *   basis [n_points][n_free]  Bernstein values of the free control points 3 .. n_ctrl-4   (n_free = n_ctrl - 6)
 *   pinv  [n_free][n_points]  its pseudo-inverse
 *   w0, w1 [n_points]         summed basis values of the three pinned control points at the start / end
 * q0, q1 [n_paths][dim], path [n_paths][n_points][dim] (row-major, as the reference passes a path: a list of q)
 * -> ctrl [n_paths][n_ctrl][dim] (rows 0-2 = q0, last three = q1), cost [n_paths] = squared residual of the fit
 * (the reference accepts a fit when it is below 0.15, control.py:185).  All pointers are device pointers. */
int gik_bezier_fit_f32(gik_handle_t h, int64_t n_paths, int32_t n_points, int32_t dim, int32_t n_ctrl, const float* pinv,
                       const float* basis, const float* w0, const float* w1, const float* q0, const float* q1,
                       const float* path, float* ctrl, float* cost, void* stream);
int gik_bezier_fit_f64(gik_handle_t h, int64_t n_paths, int32_t n_points, int32_t dim, int32_t n_ctrl, const double* pinv,
                       const double* basis, const double* w0, const double* w1, const double* q0, const double* q1,
                       const double* path, double* ctrl, double* cost, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * RRT-connect trees on the device (computepath, path.py:186-278, for many queries at once).  n_trees trees of capacity
 * cap share one set of arrays, component-major like every batch array above:
 *   verts  [n_trees][nq][cap]   vertex configurations (nq = the handle's table)
 *   cubes  [n_trees][12][cap]   cube placement each configuration was solved for
 *   parent [n_trees][cap]       int32, -1 = root
 *   n_verts[n_trees]            int32, vertices in use (a tree is reset by setting it back to 1: its root stays at 0)
 * A planner of Q queries uses tree i as the start tree and tree Q + i as the goal tree of query i.
 * ------------------------------------------------------------------------------------------------------- */

/* Replaces the nearest-vertex query of computepath (the reference's KDTree query, path.py:186-192): for each of the
 * n_targets rows of targets [n_targets][nq] (row-major), nearest[t] = the vertex of tree target_tree[t] with the
 * smallest squared distance, ties to the lowest index (numpy's argmin).  Distances are fp64 whatever the storage
 * type, summed in numpy's order for nq = 15 so that the choice is numpy's bit for bit.  nearest[t] = -1 when the tree
 * id is out of range or the tree is empty. */
int gik_tree_nearest_f32(gik_handle_t h, int64_t n_trees, int32_t cap, const float* verts, const int32_t* n_verts,
                         int64_t n_targets, const float* targets, const int32_t* target_tree, int32_t* nearest, void* stream);
int gik_tree_nearest_f64(gik_handle_t h, int64_t n_trees, int32_t cap, const double* verts, const int32_t* n_verts,
                         int64_t n_targets, const double* targets, const int32_t* target_tree, int32_t* nearest, void* stream);

/* Replaces grow() of computepath (path.py:241-244): appends the output of one gik_project_edges_* launch to the trees.
 * Edge e belongs to tree edge_tree[e] (the edges of one tree are consecutive and are appended in edge order) and
 * starts at vertex near[e]; q_start [nq][E], pose_a / pose_b [12][E], num_steps [E] and q_path [max_steps][nq][E] are
 * the edge launch's inputs and output, n_valid [E] its step counts after any cut (path.py:144-156).  Each segment
 * appends q_start[:, e] again as a child of near[e], then its n_valid[e] steps, each the child of the previous one.
 * The placement of step j is computed as in the edge kernel (SE3 interpolation at alpha = (j+1) / num_steps[e]), so it
 * is the placement the step was solved for.  n_valid[e] < 0 = no segment for this edge.  seg_end [E] = tree index of
 * the segment's last vertex (-1: no segment, or its tree overflowed).  A tree whose vertices would exceed cap is left
 * unchanged and overflow[tree] is set to 1 (never cleared here).  q_path may be NULL only when max_steps = 0. */
int gik_tree_grow_f32(gik_handle_t h, int64_t n_trees, int32_t cap, float* verts, float* cubes, int32_t* parent,
                      int32_t* n_verts, uint8_t* overflow, int64_t n_edges, int32_t max_steps, const int32_t* edge_tree,
                      const int32_t* near, const float* q_start, const float* pose_a, const float* pose_b,
                      const int32_t* num_steps, const int32_t* n_valid, const float* q_path, int32_t* seg_end,
                      void* stream);
int gik_tree_grow_f64(gik_handle_t h, int64_t n_trees, int32_t cap, double* verts, double* cubes, int32_t* parent,
                      int32_t* n_verts, uint8_t* overflow, int64_t n_edges, int32_t max_steps, const int32_t* edge_tree,
                      const int32_t* near, const double* q_start, const double* pose_a, const double* pose_b,
                      const int32_t* num_steps, const int32_t* n_valid, const double* q_path, int32_t* seg_end,
                      void* stream);

/* The returned path of computepath (path.py:226-233, 317) for n_queries queries (2 * n_queries trees): query i
 * connected at vertex start_end[i] of tree i and goal_end[i] of tree n_queries + i (-1 = did not connect); its path
 * is get_path(start tree, start_end) followed by get_path(goal tree, goal_end) reversed, packed as CSR rows
 * offsets [n_queries + 1] (int64), q [total][nq], cube [total][12] (row-major); an unconnected query has no rows.
 * Two calls: with q = cube = NULL the lengths are computed and offsets written (offsets[n_queries] = total, the one
 * value the caller reads back to size q / cube); then, with q and cube, the rows are written at those offsets. */
int gik_tree_paths_f32(gik_handle_t h, int64_t n_queries, int32_t cap, const float* verts, const float* cubes,
                       const int32_t* parent, const int32_t* n_verts, const int32_t* start_end, const int32_t* goal_end,
                       int64_t* offsets, float* q, float* cube, void* stream);
int gik_tree_paths_f64(gik_handle_t h, int64_t n_queries, int32_t cap, const double* verts, const double* cubes,
                       const int32_t* parent, const int32_t* n_verts, const int32_t* start_end, const int32_t* goal_end,
                       int64_t* offsets, double* q, double* cube, void* stream);

/* Shortcutting of planned paths, one round for n_paths paths (what gik_tree_paths_* returns: CSR rows offsets
 * [n_paths + 1] int64, q [total][nq], cube [total][12], row-major).  Path p has n = offsets[p+1] - offsets[p] rows and
 * K = n_cand candidates; candidate k is edge e = p * K + k of one gik_project_edges_* launch of E = n_paths * K edges
 * (max_steps, q_path [max_steps][nq][E]) from (q_i, cube_i) towards cube_j, (i, j) = (pair_i[e], pair_j[e]), with
 * num_steps[e] = ns steps and n_valid[e] = nv its converged, collision-free steps.  Let s_m be the q of step m and
 * ||.|| the fp64 norm of the fp64 difference, squares summed left to right.  Candidate k is accepted when
 *   0 <= i, i + 2 <= j <= n - 1, 1 <= ns <= max_steps, nv == ns, ||s_ns - q_j|| < join_tol, and
 *   gain = L_old - L_new > 0, where L_old = sum_{k=i}^{j-1} ||q_{k+1} - q_k|| and
 *   L_new = ||s_1 - q_i|| + sum_{m=1}^{ns-2} ||s_{m+1} - s_m|| + ||q_j - s_{ns-1}||  (ns = 1: ||q_j - q_i||),
 * every sum in fp64, left to right, without contraction.  Of the accepted candidates the one with the largest gain is
 * chosen, ties to the lowest k; chosen[p] = k, or -1.  The chosen candidate replaces rows i+1 .. j-1 with steps
 * 1 .. ns-1 (s_ns is dropped, q_j kept); the placement stored with step m is cube_i * exp6((m / ns) xi),
 * xi = log6(cube_i^-1 cube_j): the placement the edge kernel solved it for.  length[p] = joint-space length of the
 * output path (sum of ||q_{r+1} - q_r|| over its rows, left to right).  K <= 32; K = 0 computes lengths only.
 * Two calls: with q_out = cube_out = NULL, chosen, length and offsets_out [n_paths + 1] are written (offsets_out[n_paths]
 * = the new total, the one value the caller reads back to size q_out / cube_out); then, with q_out and cube_out, the
 * rows are written at offsets_out.
 * Errors: GIK_E_SIZE (n_paths < 0, n_cand < 0 or > 32, max_steps < 0), GIK_E_PARAM (join_tol negative or NaN),
 * GIK_E_NULL (a required pointer is NULL and n_paths > 0; the candidate arrays are required when n_cand > 0, q_path
 * when also max_steps > 0; q_out without cube_out or the reverse), GIK_E_HANDLE; n_paths = 0 is a no-op. */
int gik_path_shortcut_f32(gik_handle_t h, int64_t n_paths, int32_t n_cand, int32_t max_steps, const int64_t* offsets,
                          const float* q, const float* cube, const int32_t* pair_i, const int32_t* pair_j,
                          const int32_t* num_steps, const int32_t* n_valid, const float* q_path, double join_tol,
                          int32_t* chosen, double* length, int64_t* offsets_out, float* q_out, float* cube_out,
                          void* stream);
int gik_path_shortcut_f64(gik_handle_t h, int64_t n_paths, int32_t n_cand, int32_t max_steps, const int64_t* offsets,
                          const double* q, const double* cube, const int32_t* pair_i, const int32_t* pair_j,
                          const int32_t* num_steps, const int32_t* n_valid, const double* q_path, double join_tol,
                          int32_t* chosen, double* length, int64_t* offsets_out, double* q_out, double* cube_out,
                          void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Trajectory check: can a fitted trajectory be executed?  The reference finds out only by running its 1500 pybullet
 * control steps (control.py:416-463): between the path vertices the least-squares curve lies on no grasp manifold, and
 * its free control points are unconstrained.  This checks the curve itself at the controller's sample times.
 *
 * Input: n_traj trajectories as Bezier control points ctrl [n_traj][n_ctrl][nq] (row-major, what gik_bezier_fit_*
 * writes) and the Bernstein weights of n_samples parameters u_k = k / (n_samples - 1): weights [n_samples][n_ctrl],
 * weights[k][i] = C(n_ctrl - 1, i) u_k^i (1 - u_k)^(n_ctrl - 1 - i), computed by the caller (in fp64, then rounded to
 * the kernel's type).  The controller runs 1500 steps of 0.01 s over T = 15 s, so 1501 samples cover every step and the
 * end point; time only rescales u, so positions need no T.  For every sample (n, k):
 *   1. q = sum_i weights[k][i] * ctrl[n][i]  (i ascending).
 *   2. bit 0 (joint limits): some q_j < lower_j - limit_tol or q_j > upper_j + limit_tol (a NaN q_j counts).  limit_tol
 *      absorbs the round-off of the weights on a curve that lies on a limit.
 *   3. bit 1 (grasp): hand frames H_h = oMi[hand_joint[h]] * hand offset (LARM_EFF / RARM_EFF), the cube placement each
 *      hand implies C_h = H_h * hook_h^-1, and the grasp error g = ||log6(C_L^-1 * C_R)||_2 -- zero exactly when both
 *      hands sit on the hooks of one rigid cube; the same norm as the IK residual, and the same log6, near-pi form
 *      included.  The bit is set when g > grasp_tol (or g is NaN).
 *   4. bit 2 (collisions): the carried cube is placed at C_L (the left hand carries the pose; the right hand's deviation
 *      is g) and some pair of "list 3" intersects.  List 3, built by gik_scene_attach, is every pair of the scene except
 *      the pairs of the cube with a geometry attached to hand_joint[0] or hand_joint[1] (that contact is what bit 1
 *      judges: the cube sits about a millimetre from the finger faces), plus the cube's own pairs with the table and
 *      the obstacle (gik_cube_collision_*) when the scene does not list them.
 * Outputs per trajectory: valid [n_traj] u8 = no sample has a bit set; first_bad [n_traj] i32 = the first sample with
 * a bit set, -1 if none; reason [n_traj] u8 = the bits of that sample (0 if none); grasp_err [n_traj] = max of g over
 * all samples (+inf where g is NaN).  sample_flags [n_traj][n_samples] u8 (may be NULL = not written): every sample's
 * bits.  Every output is a min / max reduction: independent of the launch configuration, identical between runs.
 * Errors: GIK_E_SIZE (n_traj < 0, n_ctrl < 2, n_samples < 2 or > 2^28 - 1), GIK_E_PARAM (a negative or NaN
 * tolerance), GIK_E_NULL (a required pointer is NULL and n_traj > 0), GIK_E_HANDLE, GIK_E_NOSCENE; n_traj = 0 is a
 * no-op. */
int gik_traj_check_f32(gik_handle_t h, int64_t n_traj, int32_t n_ctrl, int32_t n_samples, const float* weights,
                       const float* ctrl, double limit_tol, double grasp_tol, uint8_t* valid, int32_t* first_bad,
                       uint8_t* reason, float* grasp_err, uint8_t* sample_flags, void* stream);
int gik_traj_check_f64(gik_handle_t h, int64_t n_traj, int32_t n_ctrl, int32_t n_samples, const double* weights,
                       const double* ctrl, double limit_tol, double grasp_tol, uint8_t* valid, int32_t* first_bad,
                       uint8_t* reason, double* grasp_err, uint8_t* sample_flags, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GIK_H_ */
