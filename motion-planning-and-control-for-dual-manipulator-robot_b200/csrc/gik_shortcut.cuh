// gik_shortcut.cuh -- shortcutting of planned paths for many paths at once (included at the end of gik_kernels.cu,
// after gik_tree.cuh).  Semantics in include/gik.h (gik_path_shortcut_*).
//
// A round projects K candidate shortcuts (i, j) per path through one edge launch: the edge from (q_i, cube_i) towards
// cube_j.  The kernels here judge those edges and splice the best one into each path, on CSR paths:
//   offsets [Q+1] int64, q [total][nq], cube [total][12] (row-major, what gik_tree_paths_* writes),
//   edge e = p * K + k is candidate k of path p; q_path [max_steps][nq][E] is the edge launch's output.
// Lengths are fp64 sums of fp64 norms, left to right, with tree_mul / tree_add (no contraction), so that a numpy
// restatement gives the same bits.  The per-candidate judgement, the new path length and the row writer are GIK_HD
// functions: tests/test_shortcut_cpu.py compiles them with g++.
#pragma once

namespace gik {

GIK_HD double sc_sqrt(double x) {
#if defined(__CUDA_ARCH__)
  return __dsqrt_rn(x);
#else
  return sqrt(x);
#endif
}

// ||a - b|| in fp64; a and b are nq values with strides sa / sb.  Squares summed left to right.
template <typename T>
GIK_HD double sc_dist(const T* a, int64_t sa, const T* b, int64_t sb, int nq) {
  double s = 0.0;
  for (int c = 0; c < nq; ++c) {
    const double d = tree_add((double)a[c * sa], -(double)b[c * sb]);
    s = tree_add(s, tree_mul(d, d));
  }
  return sc_sqrt(s);
}

// Row r of the path after splicing candidate (i, j, ns) into path rows q [n][nq]: rows 0..i are the old ones, rows
// i+1 .. i+ns-1 are steps 1 .. ns-1 (column e of q_path [.][nq][E]), then the old rows j .. n-1.  chosen = false:
// the old row r.  -> (pointer, stride of its components).
template <typename T>
GIK_HD const T* sc_row(int64_t r, bool chosen, int nq, const T* q, int i, int j, int ns, const T* q_path, int64_t E,
                       int64_t e, int64_t& stride) {
  if (chosen && r > i) {
    if (r < i + ns) { stride = E; return q_path + (r - i - 1) * nq * E + e; }
    r += j - i - ns;
  }
  stride = 1;
  return q + r * nq;
}

// Candidate k of one path of n rows q [n][nq]: pair (i, j), edge column e with num_steps ns and n_valid nv.  It is
// accepted when 0 <= i, i + 2 <= j <= n - 1, 1 <= ns <= max_steps, nv == ns, ||s_ns - q_j|| < join_tol and
// gain = L_old - L_new > 0, with L_old = sum_{k=i}^{j-1} ||q_{k+1} - q_k|| and L_new = ||s_1 - q_i|| +
// sum_{m=1}^{ns-2} ||s_{m+1} - s_m|| + ||q_j - s_{ns-1}|| (ns = 1: ||q_j - q_i||).  Returns acceptance; gain is set
// when accepted.
template <typename T>
GIK_HD bool sc_candidate(int nq, int64_t n, const T* q, int i, int j, int ns, int nv, int max_steps, const T* q_path,
                         int64_t E, int64_t e, double join_tol, double& gain) {
  if (i < 0 || j < i + 2 || j > n - 1 || ns < 1 || ns > max_steps || nv != ns) return false;
  const T* qi = q + (int64_t)i * nq;
  const T* qj = q + (int64_t)j * nq;
  const T* step = q_path + e;                                       // step m at step + (m - 1) * nq * E
  const int64_t sstride = (int64_t)nq * E;
  if (!(sc_dist(step + (int64_t)(ns - 1) * sstride, E, qj, 1, nq) < join_tol)) return false;
  double l_old = 0.0;
  for (int k = i; k < j; ++k) l_old = tree_add(l_old, sc_dist(q + (int64_t)(k + 1) * nq, 1, q + (int64_t)k * nq, 1, nq));
  double l_new;
  if (ns == 1) {
    l_new = sc_dist(qj, 1, qi, 1, nq);
  } else {
    l_new = sc_dist(step, E, qi, 1, nq);
    for (int m = 1; m <= ns - 2; ++m) l_new = tree_add(l_new, sc_dist(step + m * sstride, E, step + (m - 1) * sstride, E, nq));
    l_new = tree_add(l_new, sc_dist(qj, 1, step + (int64_t)(ns - 2) * sstride, E, nq));
  }
  const double g = tree_add(l_old, -l_new);
  if (!(g > 0.0)) return false;
  gain = g;
  return true;
}

// (gain, candidate) order of the choice: larger gain first, then the lower candidate index.  k = -1: none.
GIK_HD bool sc_better(double g, int k, double bg, int bk) { return k >= 0 && (bk < 0 || g > bg || (g == bg && k < bk)); }

// Joint-space length of the path after the splice (chosen = false: of the path itself): sum over its rows of
// ||q_{r+1} - q_r||, left to right.
template <typename T>
GIK_HD double sc_length(int nq, int64_t n_out, bool chosen, const T* q, int i, int j, int ns, const T* q_path, int64_t E,
                        int64_t e) {
  double len = 0.0;
  int64_t sa, sb;
  const T* a = n_out > 0 ? sc_row(0, chosen, nq, q, i, j, ns, q_path, E, e, sa) : q;
  for (int64_t r = 1; r < n_out; ++r) {
    const T* b = sc_row(r, chosen, nq, q, i, j, ns, q_path, E, e, sb);
    len = tree_add(len, sc_dist(b, sb, a, sa, nq));
    a = b; sa = sb;
  }
  return len;
}

// Output row r of one path: q_out / cube_out point at the path's first output row.  A step row stores
// edge_placement(cube_i, xi, m, ns), xi = se3_delta(cube_i, cube_j), the placement the edge kernel solved it for.
template <typename T>
GIK_HD void sc_write_row(int64_t r, bool chosen, int nq, const T* q, const T* cube, int i, int j, int ns, const T* q_path,
                         int64_t E, int64_t e, const T (&cube_i)[12], const T (&xi)[6], T* q_out, T* cube_out) {
  int64_t s;
  const T* src = sc_row(r, chosen, nq, q, i, j, ns, q_path, E, e, s);
  for (int c = 0; c < nq; ++c) q_out[r * nq + c] = src[c * s];
  if (chosen && r > i && r < i + ns) {
    T pl[12];
    edge_placement(cube_i, xi, (int)(r - i), ns, pl);
    for (int c = 0; c < 12; ++c) cube_out[r * 12 + c] = pl[c];
  } else {
    const int64_t o = chosen && r > i ? r + j - i - ns : r;
    for (int c = 0; c < 12; ++c) cube_out[r * 12 + c] = cube[o * 12 + c];
  }
}

#if defined(__CUDACC__)
constexpr int kShortcutWarps = 4;

// One warp per path: lane k judges candidate k (K <= 32), the best one is merged across the warp, lane 0 writes the
// choice, the new length and the new row count.
template <typename T>
__global__ void __launch_bounds__(kShortcutWarps * 32)
gik_path_shortcut_select_kernel(int nq, int64_t Q, int K, int max_steps, const int64_t* __restrict__ offsets,
                                const T* __restrict__ q, const int32_t* __restrict__ pair_i, const int32_t* __restrict__ pair_j,
                                const int32_t* __restrict__ num_steps, const int32_t* __restrict__ n_valid,
                                const T* __restrict__ q_path, double join_tol, int32_t* __restrict__ chosen,
                                double* __restrict__ length, int64_t* __restrict__ offsets_out) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * kShortcutWarps;
  const int64_t E = Q * K;
  for (int64_t p = (int64_t)blockIdx.x * kShortcutWarps + (threadIdx.x >> 5); p < Q; p += warps) {
    const int64_t o = offsets[p], n = offsets[p + 1] - o;
    const T* qp = q + o * nq;
    double bg = 0.0;
    int bk = -1;
    if (lane < K) {
      const int64_t e = p * K + lane;
      double g;
      if (sc_candidate(nq, n, qp, pair_i[e], pair_j[e], num_steps[e], n_valid[e], max_steps, q_path, E, e, join_tol, g)) {
        bg = g; bk = lane;
      }
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
      const double og = __shfl_xor_sync(0xffffffffu, bg, s);
      const int ok = __shfl_xor_sync(0xffffffffu, bk, s);
      if (sc_better(og, ok, bg, bk)) { bg = og; bk = ok; }
    }
    if (lane == 0) {
      int64_t n_out = n;
      int i = 0, j = 0, ns = 0;
      const int64_t e = p * K + (bk < 0 ? 0 : bk);
      if (bk >= 0) {
        i = pair_i[e]; j = pair_j[e]; ns = num_steps[e];
        n_out = n - (j - i) + ns;
      }
      chosen[p] = bk;
      length[p] = sc_length(nq, n_out, bk >= 0, qp, i, j, ns, q_path, E, e);
      offsets_out[p + 1] = n_out;
      if (p == 0) offsets_out[0] = 0;
    }
  }
}

// One warp per path: the lanes write its output rows.
template <typename T>
__global__ void __launch_bounds__(kShortcutWarps * 32)
gik_path_shortcut_write_kernel(int nq, int64_t Q, int K, const int64_t* __restrict__ offsets, const T* __restrict__ q,
                               const T* __restrict__ cube, const int32_t* __restrict__ pair_i,
                               const int32_t* __restrict__ pair_j, const int32_t* __restrict__ num_steps,
                               const T* __restrict__ q_path, const int32_t* __restrict__ chosen,
                               const int64_t* __restrict__ offsets_out, T* __restrict__ q_out, T* __restrict__ cube_out) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * kShortcutWarps;
  const int64_t E = Q * K;
  for (int64_t p = (int64_t)blockIdx.x * kShortcutWarps + (threadIdx.x >> 5); p < Q; p += warps) {
    const int64_t o = offsets[p], oo = offsets_out[p], n_out = offsets_out[p + 1] - oo;
    const int k = chosen[p];
    const bool ch = k >= 0;
    const int64_t e = ch ? p * K + k : 0;
    const int i = ch ? pair_i[e] : 0, j = ch ? pair_j[e] : 0, ns = ch ? num_steps[e] : 0;
    T ci[12], xi[6] = {};
    for (int c = 0; c < 12; ++c) ci[c] = ch ? cube[(o + i) * 12 + c] : T(0);
    if (ch && ns > 1) {
      T cj[12];
      for (int c = 0; c < 12; ++c) cj[c] = cube[(o + j) * 12 + c];
      se3_delta(ci, cj, xi);
    }
    for (int64_t r = lane; r < n_out; r += 32)
      sc_write_row(r, ch, nq, q + o * nq, cube + o * 12, i, j, ns, q_path, E, e, ci, xi, q_out + oo * nq, cube_out + oo * 12);
  }
}
#endif  // __CUDACC__

}  // namespace gik

#if defined(__CUDACC__)
namespace {

template <typename T>
int path_shortcut_api(gik_handle_t h, int64_t n_paths, int32_t n_cand, int32_t max_steps, const int64_t* offsets,
                      const T* q, const T* cube, const int32_t* pair_i, const int32_t* pair_j, const int32_t* num_steps,
                      const int32_t* n_valid, const T* q_path, double join_tol, int32_t* chosen, double* length,
                      int64_t* offsets_out, T* q_out, T* cube_out, void* stream) {
  if (n_paths < 0 || n_cand < 0 || n_cand > 32 || max_steps < 0) return GIK_E_SIZE;
  if (!(join_tol >= 0.0)) return GIK_E_PARAM;
  if (n_paths > 0 && (!offsets || !q || !cube || !chosen || !length || !offsets_out || (!q_out) != (!cube_out) ||
                      (n_cand > 0 && (!pair_i || !pair_j || !num_steps || !n_valid || (max_steps > 0 && !q_path)))))
    return GIK_E_NULL;
  if (bad_handle(h)) return GIK_E_HANDLE;
  if (n_paths == 0) return GIK_OK;
  DeviceGuard g(h->device);
  if (g.err != cudaSuccess) return (int)g.err;
  cudaStream_t st = (cudaStream_t)stream;
  const int blocks = capped_grid(h, n_paths, gik::kShortcutWarps, 16);
  if (!q_out) {
    if (int rc = launch(h, gik::gik_path_shortcut_select_kernel<T>, blocks, gik::kShortcutWarps * 32, 0, st, h->host.nq,
                        n_paths, n_cand, max_steps, offsets, q, pair_i, pair_j, num_steps, n_valid, q_path, join_tol, chosen,
                        length, offsets_out))
      return rc;
    return launch(h, gik::gik_tree_scan_kernel, 1, gik::kScanThreads, 0, st, n_paths, offsets_out);
  }
  return launch(h, gik::gik_path_shortcut_write_kernel<T>, blocks, gik::kShortcutWarps * 32, 0, st, h->host.nq, n_paths, n_cand,
                offsets, q, cube, pair_i, pair_j, num_steps, q_path, chosen, offsets_out, q_out, cube_out);
}

}  // namespace

extern "C" {
int gik_path_shortcut_f32(gik_handle_t h, int64_t n_paths, int32_t n_cand, int32_t max_steps, const int64_t* offsets,
                          const float* q, const float* cube, const int32_t* pair_i, const int32_t* pair_j,
                          const int32_t* num_steps, const int32_t* n_valid, const float* q_path, double join_tol,
                          int32_t* chosen, double* length, int64_t* offsets_out, float* q_out, float* cube_out, void* s) {
  return path_shortcut_api<float>(h, n_paths, n_cand, max_steps, offsets, q, cube, pair_i, pair_j, num_steps, n_valid,
                                  q_path, join_tol, chosen, length, offsets_out, q_out, cube_out, s);
}
int gik_path_shortcut_f64(gik_handle_t h, int64_t n_paths, int32_t n_cand, int32_t max_steps, const int64_t* offsets,
                          const double* q, const double* cube, const int32_t* pair_i, const int32_t* pair_j,
                          const int32_t* num_steps, const int32_t* n_valid, const double* q_path, double join_tol,
                          int32_t* chosen, double* length, int64_t* offsets_out, double* q_out, double* cube_out, void* s) {
  return path_shortcut_api<double>(h, n_paths, n_cand, max_steps, offsets, q, cube, pair_i, pair_j, num_steps, n_valid,
                                   q_path, join_tol, chosen, length, offsets_out, q_out, cube_out, s);
}
}  // extern "C"
#endif  // __CUDACC__
