// gik_tree.cuh -- RRT-connect trees kept in device memory for many planning queries at once (included at the end of
// gik_kernels.cu: one translation unit, one library).  The tree logic is the reference's (path.py:174-278, computepath
// in path.py here); what changes is where it lives: the trees of Q queries are device arrays, and the nearest-vertex
// search, the append of projected edges and the final path assembly are kernels, so a planning iteration of all Q
// queries needs no host round trip.
//
// Storage, component-major like every batch array of the library (n_trees trees of capacity cap):
//   verts  [n_trees][nq][cap]   configurations
//   cubes  [n_trees][12][cap]   cube placement of each vertex (the one its configuration was solved for)
//   parent [n_trees][cap]       int32, -1 = root
//   n_verts[n_trees]            int32
//
// The per-target scan, the per-tree append and the path walk are GIK_HD functions: tests/test_tree_cpu.py compiles
// them with g++ against Python restatements of the reference loop.  The kernels below are thin around them.
#pragma once

namespace gik {

// Correctly rounded products and sums without contraction into FMAs: the nearest-vertex search must reproduce
// numpy's distances bit for bit (ties and near-ties decide which vertex an edge starts from).
GIK_HD double tree_mul(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dmul_rn(a, b);
#else
  return a * b;
#endif
}
GIK_HD double tree_add(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dadd_rn(a, b);
#else
  return a + b;
#endif
}

// Squared distance in fp64 between vertex `v` of a tree ([nq][cap], column stride cap) and a target row [nq].  For
// nq = 15 the terms are summed in the order of numpy's pairwise sum over a 15-long row (eight partial terms
// ((t0+t1)+(t2+t3))+((t4+t5)+(t6+t7)), then t8 .. t14 one at a time), so that the result equals
// ((P[None]-T[:,None])**2).sum(axis=2) of path.computepath bit for bit; other nq sum left to right.
template <typename T>
GIK_HD double tree_sqdist(const T* tree, int64_t cap, int64_t v, const T* target, int nq) {
  if (nq == 15) {
    double t[8];
    for (int c = 0; c < 8; ++c) {
      const double d = (double)tree[c * cap + v] - (double)target[c];
      t[c] = tree_mul(d, d);
    }
    double s = tree_add(tree_add(tree_add(t[0], t[1]), tree_add(t[2], t[3])),
                        tree_add(tree_add(t[4], t[5]), tree_add(t[6], t[7])));
    for (int c = 8; c < 15; ++c) {
      const double d = (double)tree[c * cap + v] - (double)target[c];
      s = tree_add(s, tree_mul(d, d));
    }
    return s;
  }
  double s = 0.0;
  for (int c = 0; c < nq; ++c) {
    const double d = (double)tree[c * cap + v] - (double)target[c];
    s = tree_add(s, tree_mul(d, d));
  }
  return s;
}

// (distance, index) order of argmin: smaller distance first, then the lower index.
GIK_HD bool tree_better(double d, int i, double bd, int bi) { return d < bd || (d == bd && i < bi); }

// Scan of vertices v0, v0 + stride, ... < nv of one tree: the (distance, index)-smallest one is merged into
// (best_d, best_i).  stride = 1 is the whole scan; the kernel gives each lane of a warp one residue class.
template <typename T>
GIK_HD void tree_scan_nearest(const T* tree, int64_t cap, int nv, const T* target, int nq, int v0, int stride,
                              double& best_d, int& best_i) {
  for (int v = v0; v < nv; v += stride) {
    const double d = tree_sqdist(tree, cap, v, target, nq);
    if (tree_better(d, v, best_d, best_i)) { best_d = d; best_i = v; }
  }
}

// grow() of path.computepath (path.py:241-244) for the edges [e0, e1) of ONE tree (in edge order).  Edge e appends
// its start configuration q_start[:, e] again, with placement pose_a[:, e], as a child of near[e], then its
// n_valid[e] steps q_path[j][:, e], each the child of the previous vertex; step j stores edge_placement of step j + 1,
// the placement the edge kernel solved that step for.
// n_valid[e] < 0 marks an edge that was not projected: it appends nothing and seg_end[e] = -1.  Otherwise seg_end[e]
// is the index of the segment's last vertex.  If the vertices would exceed cap, the tree is left unchanged, every
// seg_end of the range is -1 and the function returns false.  q_path is [max_steps][nq][E]; a step count above
// max_steps is read as max_steps.
template <typename T>
GIK_HD bool tree_append(int nq, int64_t cap, int max_steps, int64_t E, int64_t e0, int64_t e1, T* verts, T* cubes, int32_t* parent,
                        int32_t* n_verts, const int32_t* near, const T* q_start, const T* pose_a, const T* pose_b,
                        const int32_t* num_steps, const int32_t* n_valid, const T* q_path, int32_t* seg_end) {
  int64_t n = *n_verts, need = 0;
  for (int64_t e = e0; e < e1; ++e)
    if (n_valid[e] >= 0) need += 1 + (n_valid[e] < max_steps ? n_valid[e] : max_steps);
  if (n + need > cap) {
    for (int64_t e = e0; e < e1; ++e) seg_end[e] = -1;
    return false;
  }
  for (int64_t e = e0; e < e1; ++e) {
    const int m = n_valid[e] < max_steps ? n_valid[e] : max_steps;
    if (m < 0) { seg_end[e] = -1; continue; }
    T a[12], b[12], xi[6], cube[12];
    for (int c = 0; c < 12; ++c) { a[c] = pose_a[c * E + e]; b[c] = pose_b[c * E + e]; }
    for (int c = 0; c < nq; ++c) verts[c * cap + n] = q_start[c * E + e];
    for (int c = 0; c < 12; ++c) cubes[c * cap + n] = a[c];
    parent[n] = near[e];
    ++n;
    if (m > 0) se3_delta(a, b, xi);
    for (int j = 0; j < m; ++j) {
      edge_placement(a, xi, j + 1, num_steps[e], cube);
      for (int c = 0; c < nq; ++c) verts[c * cap + n] = q_path[((int64_t)j * nq + c) * E + e];
      for (int c = 0; c < 12; ++c) cubes[c * cap + n] = cube[c];
      parent[n] = (int32_t)(n - 1);
      ++n;
    }
    seg_end[e] = (int32_t)(n - 1);
  }
  *n_verts = (int32_t)n;
  return true;
}

// Number of vertices from `node` to the root of a tree (path.get_path, path.py:174-183), or 0 when node is not a
// vertex.  A parent outside [0, nv) ends the walk, so a corrupted tree cannot make it run away.
GIK_HD int64_t tree_depth(const int32_t* parent, int nv, int node) {
  if (node < 0 || node >= nv) return 0;
  int64_t len = 0;
  while (node >= 0 && node < nv && len < nv) { ++len; node = parent[node]; }
  return len;
}

// Path of one query: _get_path(G_start, s) + _get_path(G_goal, g)[::-1] (path.py:226-233, 317) written from row 0 of
// q [.][nq] / cube [.][12] (row-major).  Returns the rows written: 0 unless both ends are vertices.
template <typename T>
GIK_HD int64_t tree_write_path(int nq, int64_t cap, const T* vs, const T* cs, const int32_t* ps, int nvs, int s,
                               const T* vg, const T* cg, const int32_t* pg, int nvg, int g, T* q, T* cube) {
  const int64_t ls = tree_depth(ps, nvs, s), lg = tree_depth(pg, nvg, g);
  if (ls == 0 || lg == 0) return 0;
  int node = s;
  for (int64_t r = ls - 1; r >= 0; --r) {                 // start tree: root first
    for (int c = 0; c < nq; ++c) q[r * nq + c] = vs[c * cap + node];
    for (int c = 0; c < 12; ++c) cube[r * 12 + c] = cs[c * cap + node];
    node = ps[node];
  }
  node = g;
  for (int64_t r = ls; r < ls + lg; ++r) {                // goal tree: from the connecting vertex to its root
    for (int c = 0; c < nq; ++c) q[r * nq + c] = vg[c * cap + node];
    for (int c = 0; c < 12; ++c) cube[r * 12 + c] = cg[c * cap + node];
    node = pg[node];
  }
  return ls + lg;
}

#if defined(__CUDACC__)
constexpr int kTreeWarps = 4;

template <typename T>
__global__ void __launch_bounds__(kTreeWarps * 32)
gik_tree_nearest_kernel(int nq, int64_t n_trees, int64_t cap, const T* __restrict__ verts, const int32_t* __restrict__ n_verts,
                        int64_t n_targets, const T* __restrict__ targets, const int32_t* __restrict__ target_tree,
                        int32_t* __restrict__ nearest) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * kTreeWarps;
  for (int64_t t = (int64_t)blockIdx.x * kTreeWarps + (threadIdx.x >> 5); t < n_targets; t += warps) {
    const int32_t tree = target_tree[t];
    double bd = INFINITY;
    int bi = -1;
    if (tree >= 0 && tree < n_trees) {
      const int nv = (int)min((int64_t)n_verts[tree], cap);
      tree_scan_nearest(verts + (int64_t)tree * nq * cap, cap, nv, targets + t * nq, nq, lane, 32, bd, bi);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double od = __shfl_xor_sync(0xffffffffu, bd, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (oi >= 0 && (bi < 0 || tree_better(od, oi, bd, bi))) { bd = od; bi = oi; }
    }
    if (lane == 0) nearest[t] = bi;
  }
}

// One thread per run of consecutive edges with the same tree (the thread of the run's first edge appends them all).
// (min 1 block per SM: lets ptxas keep the fp32 instantiation's state around the accurate sincosf call in registers --
// with the default bound it spills 16 bytes.)
template <typename T>
__global__ void __launch_bounds__(128, 1)
gik_tree_grow_kernel(int nq, int64_t n_trees, int64_t cap, int max_steps, T* verts, T* cubes, int32_t* parent, int32_t* n_verts,
                     uint8_t* overflow, int64_t E, const int32_t* edge_tree, const int32_t* near, const T* q_start,
                     const T* pose_a, const T* pose_b, const int32_t* num_steps, const int32_t* n_valid,
                     const T* q_path, int32_t* seg_end) {
  const int64_t e0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e0 >= E) return;
  const int32_t tree = edge_tree[e0];
  if (e0 > 0 && edge_tree[e0 - 1] == tree) return;
  int64_t e1 = e0 + 1;
  while (e1 < E && edge_tree[e1] == tree) ++e1;
  if (tree < 0 || tree >= n_trees) {
    for (int64_t e = e0; e < e1; ++e) seg_end[e] = -1;
    return;
  }
  const int64_t off = (int64_t)tree * cap;
  if (!tree_append(nq, cap, max_steps, E, e0, e1, verts + off * nq, cubes + off * 12, parent + off, n_verts + tree, near, q_start,
                   pose_a, pose_b, num_steps, n_valid, q_path, seg_end))
    overflow[tree] = 1;
}

__global__ void __launch_bounds__(128)
gik_tree_path_len_kernel(int64_t Q, int64_t cap, const int32_t* parent, const int32_t* n_verts, const int32_t* start_end,
                         const int32_t* goal_end, int64_t* offsets) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= Q) return;
  const int nvs = (int)min((int64_t)n_verts[i], cap), nvg = (int)min((int64_t)n_verts[Q + i], cap);
  const int64_t ls = tree_depth(parent + i * cap, nvs, start_end[i]);
  const int64_t lg = tree_depth(parent + (Q + i) * cap, nvg, goal_end[i]);
  offsets[i + 1] = (ls && lg) ? ls + lg : 0;
  if (i == 0) offsets[0] = 0;
}

// Inclusive scan of offsets[1 .. Q] in place (one block: a thread sums a contiguous chunk, the chunk sums are scanned
// in shared memory, then each thread rewrites its chunk).
constexpr int kScanThreads = 1024;
__global__ void __launch_bounds__(kScanThreads) gik_tree_scan_kernel(int64_t Q, int64_t* offsets) {
  __shared__ int64_t part[kScanThreads];
  const int64_t chunk = (Q + kScanThreads - 1) / kScanThreads;
  const int64_t b = 1 + threadIdx.x * chunk, e = min(b + chunk, Q + 1);
  int64_t s = 0;
  for (int64_t i = b; i < e; ++i) s += offsets[i];
  part[threadIdx.x] = s;
  __syncthreads();
  for (int o = 1; o < kScanThreads; o <<= 1) {
    const int64_t v = threadIdx.x >= o ? part[threadIdx.x - o] : 0;
    __syncthreads();
    part[threadIdx.x] += v;
    __syncthreads();
  }
  s = threadIdx.x ? part[threadIdx.x - 1] : 0;
  for (int64_t i = b; i < e; ++i) { s += offsets[i]; offsets[i] = s; }
}

template <typename T>
__global__ void __launch_bounds__(128)
gik_tree_path_write_kernel(int nq, int64_t Q, int64_t cap, const T* verts, const T* cubes, const int32_t* parent,
                           const int32_t* n_verts, const int32_t* start_end, const int32_t* goal_end,
                           const int64_t* offsets, T* q, T* cube) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= Q || offsets[i + 1] == offsets[i]) return;
  const int64_t s = i, g = Q + i, o = offsets[i];
  tree_write_path(nq, cap, verts + s * nq * cap, cubes + s * 12 * cap, parent + s * cap, (int)min((int64_t)n_verts[s], cap),
                  start_end[i], verts + g * nq * cap, cubes + g * 12 * cap, parent + g * cap,
                  (int)min((int64_t)n_verts[g], cap), goal_end[i], q + o * nq, cube + o * 12);
}
#endif  // __CUDACC__

}  // namespace gik

#if defined(__CUDACC__)
namespace {

// Argument checks come before the handle check and before any CUDA call (sizes, then pointers, then the handle).
inline int tree_blocks(int64_t n, int per_block) { return (int)((n + per_block - 1) / per_block); }

template <typename T>
int tree_nearest_api(gik_handle_t h, int64_t n_trees, int32_t cap, const T* verts, const int32_t* n_verts, int64_t n_targets,
                     const T* targets, const int32_t* target_tree, int32_t* nearest, void* stream) {
  if (n_trees < 0 || cap < 1 || n_targets < 0) return GIK_E_SIZE;
  if (n_targets > 0 && (!verts || !n_verts || !targets || !target_tree || !nearest)) return GIK_E_NULL;
  if (bad_handle(h)) return GIK_E_HANDLE;
  if (n_targets == 0) return GIK_OK;
  DeviceGuard g(h->device);
  if (g.err != cudaSuccess) return (int)g.err;
  int64_t blocks = (n_targets + gik::kTreeWarps - 1) / gik::kTreeWarps;
  const int64_t most = (int64_t)h->sm_count * 16;
  if (blocks > most) blocks = most;
  gik::gik_tree_nearest_kernel<T><<<(int)blocks, gik::kTreeWarps * 32, 0, (cudaStream_t)stream>>>(
      h->host.nq, n_trees, cap, verts, n_verts, n_targets, targets, target_tree, nearest);
  return (int)cudaGetLastError();
}

template <typename T>
int tree_grow_api(gik_handle_t h, int64_t n_trees, int32_t cap, T* verts, T* cubes, int32_t* parent, int32_t* n_verts,
                  uint8_t* overflow, int64_t n_edges, int32_t max_steps, const int32_t* edge_tree, const int32_t* near,
                  const T* q_start, const T* pose_a, const T* pose_b, const int32_t* num_steps, const int32_t* n_valid,
                  const T* q_path, int32_t* seg_end, void* stream) {
  if (n_trees < 0 || cap < 1 || n_edges < 0 || max_steps < 0) return GIK_E_SIZE;
  if (n_edges > 0 && (!verts || !cubes || !parent || !n_verts || !overflow || !edge_tree || !near || !q_start || !pose_a ||
                      !pose_b || !num_steps || !n_valid || !seg_end || (max_steps > 0 && !q_path)))
    return GIK_E_NULL;
  if (bad_handle(h)) return GIK_E_HANDLE;
  if (n_edges == 0) return GIK_OK;
  DeviceGuard g(h->device);
  if (g.err != cudaSuccess) return (int)g.err;
  gik::gik_tree_grow_kernel<T><<<tree_blocks(n_edges, 128), 128, 0, (cudaStream_t)stream>>>(
      h->host.nq, n_trees, cap, max_steps, verts, cubes, parent, n_verts, overflow, n_edges, edge_tree, near, q_start, pose_a,
      pose_b, num_steps, n_valid, q_path, seg_end);
  return (int)cudaGetLastError();
}

template <typename T>
int tree_paths_api(gik_handle_t h, int64_t n_queries, int32_t cap, const T* verts, const T* cubes, const int32_t* parent,
                   const int32_t* n_verts, const int32_t* start_end, const int32_t* goal_end, int64_t* offsets, T* q,
                   T* cube, void* stream) {
  if (n_queries < 0 || cap < 1) return GIK_E_SIZE;
  if (n_queries > 0 && (!offsets || !verts || !cubes || !parent || !n_verts || !start_end || !goal_end || (!q) != (!cube)))
    return GIK_E_NULL;
  if (bad_handle(h)) return GIK_E_HANDLE;
  if (n_queries == 0) return GIK_OK;
  DeviceGuard g(h->device);
  if (g.err != cudaSuccess) return (int)g.err;
  cudaStream_t st = (cudaStream_t)stream;
  const int blocks = tree_blocks(n_queries, 128);
  if (!q) {
    gik::gik_tree_path_len_kernel<<<blocks, 128, 0, st>>>(n_queries, cap, parent, n_verts, start_end, goal_end, offsets);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return (int)e;
    gik::gik_tree_scan_kernel<<<1, gik::kScanThreads, 0, st>>>(n_queries, offsets);
    return (int)cudaGetLastError();
  }
  gik::gik_tree_path_write_kernel<T><<<blocks, 128, 0, st>>>(h->host.nq, n_queries, cap, verts, cubes, parent, n_verts,
                                                              start_end, goal_end, offsets, q, cube);
  return (int)cudaGetLastError();
}

}  // namespace

extern "C" {
int gik_tree_nearest_f32(gik_handle_t h, int64_t n_trees, int32_t cap, const float* verts, const int32_t* n_verts,
                         int64_t n_targets, const float* targets, const int32_t* target_tree, int32_t* nearest, void* s) {
  return tree_nearest_api<float>(h, n_trees, cap, verts, n_verts, n_targets, targets, target_tree, nearest, s);
}
int gik_tree_nearest_f64(gik_handle_t h, int64_t n_trees, int32_t cap, const double* verts, const int32_t* n_verts,
                         int64_t n_targets, const double* targets, const int32_t* target_tree, int32_t* nearest, void* s) {
  return tree_nearest_api<double>(h, n_trees, cap, verts, n_verts, n_targets, targets, target_tree, nearest, s);
}
int gik_tree_grow_f32(gik_handle_t h, int64_t n_trees, int32_t cap, float* verts, float* cubes, int32_t* parent,
                      int32_t* n_verts, uint8_t* overflow, int64_t n_edges, int32_t max_steps, const int32_t* edge_tree,
                      const int32_t* near, const float* q_start, const float* pose_a, const float* pose_b,
                      const int32_t* num_steps, const int32_t* n_valid, const float* q_path, int32_t* seg_end, void* s) {
  return tree_grow_api<float>(h, n_trees, cap, verts, cubes, parent, n_verts, overflow, n_edges, max_steps, edge_tree, near,
                              q_start, pose_a, pose_b, num_steps, n_valid, q_path, seg_end, s);
}
int gik_tree_grow_f64(gik_handle_t h, int64_t n_trees, int32_t cap, double* verts, double* cubes, int32_t* parent,
                      int32_t* n_verts, uint8_t* overflow, int64_t n_edges, int32_t max_steps, const int32_t* edge_tree,
                      const int32_t* near, const double* q_start, const double* pose_a, const double* pose_b,
                      const int32_t* num_steps, const int32_t* n_valid, const double* q_path, int32_t* seg_end, void* s) {
  return tree_grow_api<double>(h, n_trees, cap, verts, cubes, parent, n_verts, overflow, n_edges, max_steps, edge_tree, near,
                               q_start, pose_a, pose_b, num_steps, n_valid, q_path, seg_end, s);
}
int gik_tree_paths_f32(gik_handle_t h, int64_t n_queries, int32_t cap, const float* verts, const float* cubes,
                       const int32_t* parent, const int32_t* n_verts, const int32_t* start_end, const int32_t* goal_end,
                       int64_t* offsets, float* q, float* cube, void* s) {
  return tree_paths_api<float>(h, n_queries, cap, verts, cubes, parent, n_verts, start_end, goal_end, offsets, q, cube, s);
}
int gik_tree_paths_f64(gik_handle_t h, int64_t n_queries, int32_t cap, const double* verts, const double* cubes,
                       const int32_t* parent, const int32_t* n_verts, const int32_t* start_end, const int32_t* goal_end,
                       int64_t* offsets, double* q, double* cube, void* s) {
  return tree_paths_api<double>(h, n_queries, cap, verts, cubes, parent, n_verts, start_end, goal_end, offsets, q, cube, s);
}
}  // extern "C"
#endif  // __CUDACC__
