// gik_roadmap.cuh -- a grasp roadmap built once in a static scene and queried many times (included at the end of
// gik_kernels.cu, after gik_shortcut.cuh).  Semantics in include/gik.h (gik_knn_*, gik_roadmap_*).
//
// Vertex v is a grasp (q_v [nq], cube_v [12]).  Edge i -> j is an edge-kernel march from (q_i, cube_i) towards cube_j,
// accepted when every step converged collision-free and the last one landed within join_tol of q_j; its weight is the
// fp64 joint-space length of the rows q_i, steps 1 .. ns-1, q_j, summed as sc_length sums a shortcut's length.  The
// roadmap is CSR by source: row_ptr [N+1] int64, dst / ns [E] int32, weight [E] f64, step_ptr [E+1] int64 and
// steps [rows][nq] (row-major, steps 1 .. ns-1 of every edge).
// A batch of Q queries has A = 2 ka + 1 attachment edges per query; slot s of query p is edge e = p * A + s of one edge
// launch:  s < ka: (q_init, cube0) -> vertex att_vertex[e];  ka <= s < 2 ka: vertex att_vertex[e] -> (q_goal, cube1);
// s = 2 ka: the direct edge (q_init, cube0) -> (q_goal, cube1).
// The selection, judgement, relaxation, predecessor and path rules are GIK_HD functions: tests/test_roadmap_cpu.py
// compiles them with g++.
#pragma once

namespace gik {

constexpr int32_t kRmNone = 0x7fffffff;     // index of an empty kNN slot, and of a vertex without a predecessor yet

// fp64 Euclidean distance of two placements' translations (values 9..11): ((dx^2 + dy^2) + dz^2), then the root.
template <typename T>
GIK_HD double rm_dist(const T* a, const T* b) {
  double s = 0.0;
  for (int c = 9; c < 12; ++c) {
    const double d = tree_add((double)a[c], -(double)b[c]);
    s = tree_add(s, tree_mul(d, d));
  }
  return sc_sqrt(s);
}

// Slot l of a sorted kNN list (one (distance, index) entry per slot, best first, tree_better's order) after candidate
// (cd, ci) is inserted: from its own entry (d, i) and slot l - 1's (pd, pi); `first` = slot 0.
GIK_HD void rm_knn_slot(bool first, double d, int i, double pd, int pi, double cd, int ci, double& od, int& oi) {
  if (tree_better(d, i, cd, ci)) { od = d; oi = i; }
  else if (first || tree_better(pd, pi, cd, ci)) { od = cd; oi = ci; }
  else { od = pd; oi = pi; }
}

// Weight of the edge from q_from towards q_to: column e of an edge launch's q_path [max_steps][nq][E] with ns steps,
// nv of them converged and collision-free.  +inf unless 1 <= ns <= max_steps, nv == ns and ||s_ns - q_to|| < join_tol;
// otherwise ||s_1 - q_from|| + ... + ||q_to - s_{ns-1}|| (ns = 1: ||q_to - q_from||), left to right from 0.
template <typename T>
GIK_HD double rm_edge_weight(int nq, const T* q_from, const T* q_to, int ns, int nv, int max_steps, const T* q_path,
                             int64_t E, int64_t e, double join_tol) {
  if (ns < 1 || ns > max_steps || nv != ns) return INFINITY;
  const T* step = q_path + e;
  const int64_t sstride = (int64_t)nq * E;
  if (!(sc_dist(step + (int64_t)(ns - 1) * sstride, E, q_to, 1, nq) < join_tol)) return INFINITY;
  double w = 0.0;
  const T* a = q_from;
  int64_t sa = 1;
  for (int m = 1; m < ns; ++m) {
    const T* b = step + (int64_t)(m - 1) * sstride;
    w = tree_add(w, sc_dist(b, E, a, sa, nq));
    a = b; sa = E;
  }
  return tree_add(w, sc_dist(q_to, 1, a, sa, nq));
}

// Distances are kept as the bit patterns of non-negative doubles, which order like the values: atomicMin on them is a
// min on the distances.
GIK_HD uint64_t rm_bits(double x) {
#if defined(__CUDA_ARCH__)
  return (uint64_t)__double_as_longlong(x);
#else
  uint64_t b; memcpy(&b, &x, 8); return b;
#endif
}
GIK_HD double rm_val(uint64_t b) {
#if defined(__CUDA_ARCH__)
  return __longlong_as_double((long long)b);
#else
  double x; memcpy(&x, &b, 8); return x;
#endif
}
// Loads that see other threads' atomics of the same round (L2, not a stale L1 line)
GIK_HD uint64_t rm_load(const uint64_t* p) {
#if defined(__CUDA_ARCH__)
  return (uint64_t)__ldcg((const unsigned long long*)p);
#else
  return *p;
#endif
}
GIK_HD int32_t rm_load(const int32_t* p) {
#if defined(__CUDA_ARCH__)
  return __ldcg(p);
#else
  return *p;
#endif
}
// *p = min(*p, bits of v); true when it lowered *p
GIK_HD bool rm_lower(uint64_t* p, double v) {
  const uint64_t b = rm_bits(v);
#if defined(__CUDA_ARCH__)
  return b < (uint64_t)atomicMin((unsigned long long*)p, (unsigned long long)b);
#else
  if (b < *p) { *p = b; return true; }
  return false;
#endif
}
GIK_HD void rm_min(int32_t* p, int32_t v) {
#if defined(__CUDA_ARCH__)
  atomicMin(p, v);
#else
  if (v < *p) *p = v;
#endif
}

// Out-edges [e0, e1) of row u, clamped to [0, E)
GIK_HD void rm_row(const int64_t* row_ptr, int64_t E, int u, int64_t& e0, int64_t& e1) {
  e0 = row_ptr[u]; e1 = row_ptr[u + 1];
  e0 = e0 < 0 ? 0 : (e0 > E ? E : e0);
  e1 = e1 < e0 ? e0 : (e1 > E ? E : e1);
}

// One Bellman-Ford relaxation of vertex u's out-edges: dist[v] = min(dist[v], dist[u] + w(u, v)); a lowered v gets
// mark[v] = round, so that the next round relaxes it.  -> whether something was lowered.
GIK_HD bool rm_relax(int N, int64_t E, const int64_t* row_ptr, const int32_t* dst, const double* weight, uint64_t* dist,
                     int32_t* mark, int u, int round) {
  const double du = rm_val(rm_load(dist + u));
  int64_t e0, e1;
  rm_row(row_ptr, E, u, e0, e1);
  bool ch = false;
  for (int64_t e = e0; e < e1; ++e) {
    const int v = dst[e];
    if (v < 0 || v >= N) continue;
    if (rm_lower(dist + v, tree_add(du, weight[e]))) { mark[v] = round; ch = true; }
  }
  return ch;
}

// The predecessor rule for vertex u's out-edges once the distances are final: pred[v] = min(pred[v], u) when
// dist[u] + w(u, v) == dist[v].  (The virtual start, -1, is entered before: it wins ties.)
GIK_HD void rm_pred(int N, int64_t E, const int64_t* row_ptr, const int32_t* dst, const double* weight,
                    const uint64_t* dist, int32_t* pred, int u) {
  const double du = rm_val(rm_load(dist + u));
  if (!(du < INFINITY)) return;
  int64_t e0, e1;
  rm_row(row_ptr, E, u, e0, e1);
  for (int64_t e = e0; e < e1; ++e) {
    const int v = dst[e];
    if (v >= 0 && v < N && rm_bits(tree_add(du, weight[e])) == rm_load(dist + v)) rm_min(pred + v, u);
  }
}

// Slot of vertex v among att_vertex[s0 .. s1) with a finite weight, or -1
GIK_HD int rm_slot(const int32_t* att_vertex, const double* att_weight, int s0, int s1, int v) {
  for (int s = s0; s < s1; ++s)
    if (att_vertex[s] == v && att_weight[s] < INFINITY) return s;
  return -1;
}

// The answer of one query (its 2 ka + 1 attachment slots): min(w_direct, min_b dist[b] + w(b -> goal)) over the accepted
// goal slots.  -> the goal's predecessor: -1 = the direct edge (wins ties), b = the smallest b achieving the minimum,
// -2 = unconnected (length +inf).
GIK_HD int rm_goal(int N, int ka, const int32_t* att_vertex, const double* att_weight, const uint64_t* dist, double& length) {
  double best = att_weight[2 * ka];
  int gp = best < INFINITY ? -1 : -2;
  for (int s = ka; s < 2 * ka; ++s) {
    const int b = att_vertex[s];
    if (b < 0 || b >= N || !(att_weight[s] < INFINITY)) continue;
    const double db = rm_val(rm_load(dist + b));
    if (!(db < INFINITY)) continue;
    const double c = tree_add(db, att_weight[s]);
    if (c < best || (c == best && gp >= 0 && b < gp)) { best = c; gp = b; }
  }
  length = gp == -2 ? INFINITY : best;
  return gp;
}

// Edge u -> v of the CSR, or -1
GIK_HD int64_t rm_find_edge(int N, int64_t E, const int64_t* row_ptr, const int32_t* dst, int u, int v) {
  if (u < 0 || u >= N) return -1;
  int64_t e0, e1;
  rm_row(row_ptr, E, u, e0, e1);
  for (int64_t e = e0; e < e1; ++e)
    if (dst[e] == v) return e;
  return -1;
}

// Rows of one query's path (0: unconnected, or a predecessor chain that does not end at the start within N steps),
// and the roadmap vertices on it.  Rows: q_init, then per segment (start attachment, roadmap edges, goal attachment)
// its ns - 1 steps and its end row.
GIK_HD int64_t rm_path_rows(int N, int64_t E, int ka, const int64_t* row_ptr, const int32_t* dst, const int32_t* ns,
                            const int32_t* att_vertex, const double* att_weight, const int32_t* att_ns,
                            const int32_t* pred, int gp, int32_t& verts) {
  verts = 0;
  if (gp == -2) return 0;
  if (gp == -1) return 1 + att_ns[2 * ka];
  const int sg = rm_slot(att_vertex, att_weight, ka, 2 * ka, gp);
  if (sg < 0 || gp < 0 || gp >= N) return 0;
  int64_t rows = 1 + att_ns[sg];
  int v = gp;
  for (int hop = 0; hop < N; ++hop) {
    ++verts;
    const int u = pred[v];
    if (u == -1) {
      const int ss = rm_slot(att_vertex, att_weight, 0, ka, v);
      if (ss < 0) break;
      return rows + att_ns[ss];
    }
    const int64_t e = rm_find_edge(N, E, row_ptr, dst, u, v);
    if (e < 0) break;
    rows += ns[e];
    v = u;
  }
  verts = 0;
  return 0;
}

// Rows r0 .. r0 + ns - 2 of a path: steps 1 .. ns-1 of an edge from cube_from towards cube_to, step m's q at
// src + (m - 1) * sm + c * sc, its cube edge_placement(cube_from, xi, m, ns) as tree_append stores it.
template <typename T>
GIK_HD void rm_write_steps(int nq, int64_t r0, const T* src, int64_t sm, int64_t sc, int ns, const T (&cf)[12],
                           const T* cube_to, T* q, T* cube) {
  if (ns <= 1) return;
  T ct[12], xi[6], pl[12];
  for (int c = 0; c < 12; ++c) ct[c] = cube_to[c];
  se3_delta(cf, ct, xi);
  for (int m = 1; m < ns; ++m) {
    const int64_t r = r0 + m - 1;
    for (int c = 0; c < nq; ++c) q[r * nq + c] = src[(int64_t)(m - 1) * sm + c * sc];
    edge_placement(cf, xi, m, ns, pl);
    for (int c = 0; c < 12; ++c) cube[r * 12 + c] = pl[c];
  }
}

template <typename T>
GIK_HD void rm_put(int nq, int64_t r, const T* qr, const T* cr, T* q, T* cube) {
  for (int c = 0; c < nq; ++c) q[r * nq + c] = qr[c];
  for (int c = 0; c < 12; ++c) cube[r * 12 + c] = cr[c];
}

// Everything gik_roadmap_paths_* reads, for one batch
template <typename T>
struct RmPathArgs {
  int nq, N, ka, max_steps;
  int64_t Q, E;
  const T *vq, *vcube;
  const int64_t* row_ptr;
  const int32_t *dst, *ns;
  const int64_t* step_ptr;
  const T* steps;
  const T *q_init, *q_goal, *cube0, *cube1;
  const int32_t* att_vertex;
  const double* att_weight;
  const int32_t* att_ns;
  const T* att_path;                 // [max_steps][nq][Q * (2 ka + 1)]
  const int32_t *pred, *goal_pred;   // [Q][N], [Q]
};

// Writes the rows of query p from row 0 of q / cube, back to front; `rows` from rm_path_rows.
template <typename T>
GIK_HD void rm_write_path(const RmPathArgs<T>& a, int64_t p, int64_t rows, T* q, T* cube) {
  if (rows <= 0) return;
  const int nq = a.nq, A = 2 * a.ka + 1;
  const int64_t EA = a.Q * A, e_base = p * A;
  const int32_t* av = a.att_vertex + e_base;
  const double* aw = a.att_weight + e_base;
  const int32_t* pred = a.pred + p * a.N;
  const T *qi = a.q_init + p * nq, *qg = a.q_goal + p * nq, *c0 = a.cube0 + p * 12, *c1 = a.cube1 + p * 12;
  T cf[12];
  int64_t r = rows - 1;
  rm_put(nq, r, qg, c1, q, cube);
  const int gp = a.goal_pred[p];
  // an attachment slot's steps: column e_base + s of att_path
  auto att = [&](int s, const T* from, const T* to) {
    const int m = a.att_ns[e_base + s];
    for (int c = 0; c < 12; ++c) cf[c] = from[c];
    r -= m;
    rm_write_steps(nq, r + 1, a.att_path + e_base + s, (int64_t)nq * EA, EA, m, cf, to, q, cube);
  };
  if (gp == -1) {
    att(2 * a.ka, c0, c1);
  } else {
    att(rm_slot(av, aw, a.ka, 2 * a.ka, gp), a.vcube + (int64_t)gp * 12, c1);
    int v = gp;
    rm_put(nq, r, a.vq + (int64_t)v * nq, a.vcube + (int64_t)v * 12, q, cube);
    while (r > 0) {
      const int u = pred[v];
      if (u == -1) {
        att(rm_slot(av, aw, 0, a.ka, v), c0, a.vcube + (int64_t)v * 12);
        break;
      }
      const int64_t e = rm_find_edge(a.N, a.E, a.row_ptr, a.dst, u, v);
      const int m = a.ns[e];
      for (int c = 0; c < 12; ++c) cf[c] = a.vcube[(int64_t)u * 12 + c];
      r -= m;
      rm_write_steps(nq, r + 1, a.steps + a.step_ptr[e] * nq, (int64_t)nq, (int64_t)1, m, cf, a.vcube + (int64_t)v * 12, q,
                     cube);
      rm_put(nq, r, a.vq + (int64_t)u * nq, a.vcube + (int64_t)u * 12, q, cube);
      v = u;
    }
  }
  rm_put(nq, 0, qi, c0, q, cube);
}

#if defined(__CUDACC__)
constexpr int kKnnWarps = 4;
constexpr int kSsspThreads = 256;

// One warp per point: lane l holds entry l of the sorted list of the best 32 candidates seen.  Each chunk of 32
// vertices is judged against entry k - 1; the candidates that beat it are inserted one at a time, in lane order.
template <typename T>
__global__ void __launch_bounds__(kKnnWarps * 32)
gik_knn_kernel(int N, int k, const T* __restrict__ cube, int64_t P, const T* __restrict__ points, int32_t* __restrict__ nbr) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * kKnnWarps;
  for (int64_t p = (int64_t)blockIdx.x * kKnnWarps + (threadIdx.x >> 5); p < P; p += warps) {
    const T* pt = points ? points + p * 12 : cube + p * 12;
    const int self = points ? -1 : (int)p;
    double d = INFINITY;
    int i = kRmNone;
    for (int v0 = 0; v0 < N; v0 += 32) {
      const int v = v0 + lane;
      const double cd = v < N && v != self ? rm_dist(cube + (int64_t)v * 12, pt) : INFINITY;
      const double td = __shfl_sync(0xffffffffu, d, k - 1);
      const int ti = __shfl_sync(0xffffffffu, i, k - 1);
      unsigned mask = __ballot_sync(0xffffffffu, v < N && v != self && tree_better(cd, v, td, ti));
      while (mask) {
        const int src = __ffs(mask) - 1;
        mask &= mask - 1;
        const double bd = __shfl_sync(0xffffffffu, cd, src);
        const double pd = __shfl_up_sync(0xffffffffu, d, 1);
        const int pi = __shfl_up_sync(0xffffffffu, i, 1);
        rm_knn_slot(lane == 0, d, i, pd, pi, bd, v0 + src, d, i);
      }
    }
    if (lane < k) nbr[p * k + lane] = i;
  }
}

template <typename T>
__global__ void __launch_bounds__(128)
gik_roadmap_edges_kernel(int nq, int64_t E, int max_steps, const T* __restrict__ q_from, const T* __restrict__ q_to,
                         const int32_t* __restrict__ num_steps, const int32_t* __restrict__ n_valid,
                         const T* __restrict__ q_path, double join_tol, double* __restrict__ weight) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += stride)
    weight[e] = rm_edge_weight(nq, q_from + e * nq, q_to + e * nq, num_steps[e], n_valid[e], max_steps, q_path, E, e, join_tol);
}

// One CTA per query: Bellman-Ford rounds over the vertices marked in the previous round, until a round lowers nothing;
// then the predecessors, the goal's choice and the attachment counts.  mark and pred share the [N] array of the query.
__global__ void __launch_bounds__(kSsspThreads)
gik_roadmap_sssp_kernel(int64_t Q, int N, int ka, int64_t E, const int64_t* __restrict__ row_ptr,
                        const int32_t* __restrict__ dst, const double* __restrict__ weight,
                        const int32_t* __restrict__ att_vertex, const double* __restrict__ att_weight, uint64_t* dist_all,
                        int32_t* pred_all, int32_t* __restrict__ goal_pred, double* __restrict__ length,
                        int32_t* __restrict__ attach_start, int32_t* __restrict__ attach_goal) {
  const int A = 2 * ka + 1;
  for (int64_t p = blockIdx.x; p < Q; p += gridDim.x) {
    uint64_t* dist = dist_all + p * N;
    int32_t* mark = pred_all + p * N;
    const int32_t* av = att_vertex + p * A;
    const double* aw = att_weight + p * A;
    for (int v = threadIdx.x; v < N; v += blockDim.x) { dist[v] = rm_bits(INFINITY); mark[v] = -1; }
    __syncthreads();
    if (threadIdx.x < ka) {
      const int a = av[threadIdx.x];
      if (a >= 0 && a < N && aw[threadIdx.x] < INFINITY && rm_lower(dist + a, aw[threadIdx.x])) mark[a] = 0;
    }
    __syncthreads();
    for (int round = 1;; ++round) {
      bool ch = false;
      for (int u = threadIdx.x; u < N; u += blockDim.x)
        if (rm_load(mark + u) == round - 1) ch |= rm_relax(N, E, row_ptr, dst, weight, dist, mark, u, round);
      if (!__syncthreads_or(ch)) break;
    }
    int32_t* pred = mark;
    for (int v = threadIdx.x; v < N; v += blockDim.x) pred[v] = kRmNone;
    __syncthreads();
    if (threadIdx.x < ka) {
      const int a = av[threadIdx.x];
      if (a >= 0 && a < N && aw[threadIdx.x] < INFINITY && rm_bits(aw[threadIdx.x]) == rm_load(dist + a)) rm_min(pred + a, -1);
    }
    for (int u = threadIdx.x; u < N; u += blockDim.x) rm_pred(N, E, row_ptr, dst, weight, dist, pred, u);
    __syncthreads();
    for (int v = threadIdx.x; v < N; v += blockDim.x)
      if (rm_load(pred + v) == kRmNone) pred[v] = -2;
    if (threadIdx.x == 0) {
      double len;
      goal_pred[p] = rm_goal(N, ka, av, aw, dist, len);
      length[p] = len;
      int ns = 0, ng = 0;
      for (int s = 0; s < ka; ++s) ns += aw[s] < INFINITY;
      for (int s = ka; s < 2 * ka; ++s) ng += aw[s] < INFINITY;
      attach_start[p] = ns;
      attach_goal[p] = ng;
    }
    __syncthreads();
  }
}

template <typename T>
__global__ void __launch_bounds__(128)
gik_roadmap_path_len_kernel(RmPathArgs<T> a, int64_t* __restrict__ offsets, int32_t* __restrict__ vertices) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= a.Q) return;
  const int64_t e = p * (2 * a.ka + 1);
  int32_t verts;
  offsets[p + 1] = rm_path_rows(a.N, a.E, a.ka, a.row_ptr, a.dst, a.ns, a.att_vertex + e, a.att_weight + e, a.att_ns + e,
                                a.pred + p * a.N, a.goal_pred[p], verts);
  vertices[p] = verts;
  if (p == 0) offsets[0] = 0;
}

// (min 1 block per SM, as gik_tree_grow_kernel: keeps the fp32 instantiation's state around sincosf in registers)
template <typename T>
__global__ void __launch_bounds__(128, 1)
gik_roadmap_path_write_kernel(RmPathArgs<T> a, const int64_t* __restrict__ offsets, T* __restrict__ q, T* __restrict__ cube) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= a.Q) return;
  const int64_t o = offsets[p];
  rm_write_path(a, p, offsets[p + 1] - o, q + o * a.nq, cube + o * 12);
}
#endif  // __CUDACC__

}  // namespace gik

#if defined(__CUDACC__)
namespace {

template <typename T>
int knn_api(gik_handle_t h, int32_t n_vertices, int32_t k, const T* cube, int64_t n_points, const T* points, int32_t* nbr,
            void* stream) {
  if (k < 1 || k > 32 || n_vertices < k + 1 || n_points < 0 || (!points && n_points != n_vertices)) return GIK_E_SIZE;
  if (n_points > 0 && (!cube || !nbr)) return GIK_E_NULL;
  if (bad_handle(h)) return GIK_E_HANDLE;
  if (n_points == 0) return GIK_OK;
  DeviceGuard g(h->device);
  if (g.err != cudaSuccess) return (int)g.err;
  return launch(h, gik::gik_knn_kernel<T>, capped_grid(h, n_points, gik::kKnnWarps, 16), gik::kKnnWarps * 32, 0,
                (cudaStream_t)stream, n_vertices, k, cube, n_points, points, nbr);
}

template <typename T>
int roadmap_edges_api(gik_handle_t h, int64_t n_edges, int32_t max_steps, const T* q_from, const T* q_to,
                      const int32_t* num_steps, const int32_t* n_valid, const T* q_path, double join_tol, double* weight,
                      void* stream) {
  if (n_edges < 0 || max_steps < 0) return GIK_E_SIZE;
  if (!(join_tol >= 0.0)) return GIK_E_PARAM;
  if (n_edges > 0 && (!q_from || !q_to || !num_steps || !n_valid || !weight || (max_steps > 0 && !q_path))) return GIK_E_NULL;
  if (bad_handle(h)) return GIK_E_HANDLE;
  if (n_edges == 0) return GIK_OK;
  DeviceGuard g(h->device);
  if (g.err != cudaSuccess) return (int)g.err;
  return launch(h, gik::gik_roadmap_edges_kernel<T>, capped_grid(h, n_edges, 128, 16), 128, 0, (cudaStream_t)stream,
                h->host.nq, n_edges, max_steps, q_from, q_to, num_steps, n_valid, q_path, join_tol, weight);
}

template <typename T>
int roadmap_paths_api(gik_handle_t h, int64_t n_queries, int32_t n_vertices, int32_t k_attach, int32_t max_steps,
                      int64_t n_edges, const T* vq, const T* vcube, const int64_t* row_ptr, const int32_t* dst,
                      const int32_t* ns, const int64_t* step_ptr, const T* steps, const T* q_init, const T* q_goal,
                      const T* cube0, const T* cube1, const int32_t* att_vertex, const double* att_weight,
                      const int32_t* att_ns, const T* att_path, const int32_t* pred, const int32_t* goal_pred,
                      int64_t* offsets, int32_t* vertices, T* q, T* cube, void* stream) {
  if (n_queries < 0 || n_vertices < 1 || k_attach < 0 || k_attach > 32 || max_steps < 0 || n_edges < 0) return GIK_E_SIZE;
  if (n_queries > 0 && (!vq || !vcube || !row_ptr || !step_ptr || (n_edges > 0 && (!dst || !ns)) || !q_init || !q_goal ||
                        !cube0 || !cube1 || !att_vertex || !att_weight || !att_ns || (max_steps > 0 && !att_path) || !pred ||
                        !goal_pred || !offsets || !vertices || (!q) != (!cube)))
    return GIK_E_NULL;
  if (bad_handle(h)) return GIK_E_HANDLE;
  if (n_queries == 0) return GIK_OK;
  DeviceGuard g(h->device);
  if (g.err != cudaSuccess) return (int)g.err;
  cudaStream_t st = (cudaStream_t)stream;
  const gik::RmPathArgs<T> a{h->host.nq, n_vertices, k_attach, max_steps, n_queries, n_edges, vq, vcube, row_ptr, dst, ns,
                             step_ptr, steps, q_init, q_goal, cube0, cube1, att_vertex, att_weight, att_ns, att_path, pred,
                             goal_pred};
  const int blocks = (int)((n_queries + 127) / 128);
  if (!q) {
    if (int rc = launch(h, gik::gik_roadmap_path_len_kernel<T>, blocks, 128, 0, st, a, offsets, vertices)) return rc;
    return launch(h, gik::gik_tree_scan_kernel, 1, gik::kScanThreads, 0, st, n_queries, offsets);
  }
  return launch(h, gik::gik_roadmap_path_write_kernel<T>, blocks, 128, 0, st, a, (const int64_t*)offsets, q, cube);
}

}  // namespace

extern "C" {
int gik_knn_f32(gik_handle_t h, int32_t n_vertices, int32_t k, const float* cube, int64_t n_points, const float* points,
                int32_t* nbr, void* s) {
  return knn_api<float>(h, n_vertices, k, cube, n_points, points, nbr, s);
}
int gik_knn_f64(gik_handle_t h, int32_t n_vertices, int32_t k, const double* cube, int64_t n_points, const double* points,
                int32_t* nbr, void* s) {
  return knn_api<double>(h, n_vertices, k, cube, n_points, points, nbr, s);
}
int gik_roadmap_edges_f32(gik_handle_t h, int64_t n_edges, int32_t max_steps, const float* q_from, const float* q_to,
                          const int32_t* num_steps, const int32_t* n_valid, const float* q_path, double join_tol,
                          double* weight, void* s) {
  return roadmap_edges_api<float>(h, n_edges, max_steps, q_from, q_to, num_steps, n_valid, q_path, join_tol, weight, s);
}
int gik_roadmap_edges_f64(gik_handle_t h, int64_t n_edges, int32_t max_steps, const double* q_from, const double* q_to,
                          const int32_t* num_steps, const int32_t* n_valid, const double* q_path, double join_tol,
                          double* weight, void* s) {
  return roadmap_edges_api<double>(h, n_edges, max_steps, q_from, q_to, num_steps, n_valid, q_path, join_tol, weight, s);
}
int gik_roadmap_sssp(gik_handle_t h, int64_t n_queries, int32_t n_vertices, int32_t k_attach, int64_t n_edges,
                     const int64_t* row_ptr, const int32_t* dst, const double* weight, const int32_t* att_vertex,
                     const double* att_weight, double* dist, int32_t* pred, int32_t* goal_pred, double* length,
                     int32_t* attach_start, int32_t* attach_goal, void* stream) {
  if (n_queries < 0 || n_vertices < 1 || k_attach < 0 || k_attach > 32 || n_edges < 0) return GIK_E_SIZE;
  if (n_queries > 0 && (!row_ptr || (n_edges > 0 && (!dst || !weight)) || !att_vertex || !att_weight || !dist || !pred ||
                        !goal_pred || !length || !attach_start || !attach_goal))
    return GIK_E_NULL;
  if (bad_handle(h)) return GIK_E_HANDLE;
  if (n_queries == 0) return GIK_OK;
  DeviceGuard g(h->device);
  if (g.err != cudaSuccess) return (int)g.err;
  return launch(h, gik::gik_roadmap_sssp_kernel, capped_grid(h, n_queries, 1, 8), gik::kSsspThreads, 0, (cudaStream_t)stream,
                n_queries, n_vertices, k_attach, n_edges, row_ptr, dst, weight, att_vertex, att_weight, (uint64_t*)dist, pred,
                goal_pred, length, attach_start, attach_goal);
}
int gik_roadmap_paths_f32(gik_handle_t h, int64_t n_queries, int32_t n_vertices, int32_t k_attach, int32_t max_steps,
                          int64_t n_edges, const float* vq, const float* vcube, const int64_t* row_ptr, const int32_t* dst,
                          const int32_t* ns, const int64_t* step_ptr, const float* steps, const float* q_init,
                          const float* q_goal, const float* cube0, const float* cube1, const int32_t* att_vertex,
                          const double* att_weight, const int32_t* att_ns, const float* att_path, const int32_t* pred,
                          const int32_t* goal_pred, int64_t* offsets, int32_t* vertices, float* q, float* cube, void* s) {
  return roadmap_paths_api<float>(h, n_queries, n_vertices, k_attach, max_steps, n_edges, vq, vcube, row_ptr, dst, ns,
                                  step_ptr, steps, q_init, q_goal, cube0, cube1, att_vertex, att_weight, att_ns, att_path,
                                  pred, goal_pred, offsets, vertices, q, cube, s);
}
int gik_roadmap_paths_f64(gik_handle_t h, int64_t n_queries, int32_t n_vertices, int32_t k_attach, int32_t max_steps,
                          int64_t n_edges, const double* vq, const double* vcube, const int64_t* row_ptr, const int32_t* dst,
                          const int32_t* ns, const int64_t* step_ptr, const double* steps, const double* q_init,
                          const double* q_goal, const double* cube0, const double* cube1, const int32_t* att_vertex,
                          const double* att_weight, const int32_t* att_ns, const double* att_path, const int32_t* pred,
                          const int32_t* goal_pred, int64_t* offsets, int32_t* vertices, double* q, double* cube, void* s) {
  return roadmap_paths_api<double>(h, n_queries, n_vertices, k_attach, max_steps, n_edges, vq, vcube, row_ptr, dst, ns,
                                   step_ptr, steps, q_init, q_goal, cube0, cube1, att_vertex, att_weight, att_ns, att_path,
                                   pred, goal_pred, offsets, vertices, q, cube, s);
}
}  // extern "C"
#endif  // __CUDACC__
