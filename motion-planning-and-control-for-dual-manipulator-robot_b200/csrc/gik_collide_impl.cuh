// gik_collide_impl.cuh -- collision kernels + their C ABI (included at the end of gik_kernels.cu: one translation
// unit, one library).  Mapping: ONE CONFIGURATION PER WARP.  The kinematic tree is walked level by level (one joint per
// lane, warp_tree_fk), the lanes place the geometries (place_geom, gik_collide.cuh), then the collision pairs are dealt
// round-robin to the 32 lanes for the bounding-sphere test, the survivors are compacted into a per-warp list and boolean
// GJK runs on full warps of candidates, with one __any_sync per round for the early exit (warp_any_pair_hits, shared
// with the trajectory check).  The scene (geometries, pair lists) lives in global memory and is read through the
// read-only path; per-configuration traffic is q in (60 B) and one flag out.
#pragma once
#include "gik_collide.cuh"

namespace gik {

constexpr int kCollideWarps = 4;
constexpr int kMaxCand = 512;       // per-configuration candidate pairs kept for the narrow phase

// tree FK of one configuration by one warp (level by level, one joint per lane) into oMi[nq][12]; q_of(j) = q_j.
// Lane j first builds its joint's local transform jointPlacement * Rot(axis, q_j), then the joints of depth d (all
// independent) are composed with their parents' world placements of depth d - 1.
template <typename T, typename QF>
__device__ __forceinline__ void warp_tree_fk(const DevScene<T>* sc, int lane, QF q_of, T (*oMi)[12]) {
  const int nq = sc->tree.nq;
  T L[12];
  int par = -1, dep = -1;
  if (lane < nq) {
    joint_placement(sc->tree, lane, (const T*)nullptr, q_of(lane), L);
    par = sc->tree.parent[lane]; dep = sc->tree.depth[lane];
  }
  for (int d = 0; d <= sc->tree.max_depth; ++d) {
    if (dep == d) {
      if (par < 0) {
#pragma unroll
        for (int k = 0; k < 12; ++k) oMi[lane][k] = L[k];
      } else {
        se3_mul12(&oMi[par][0], L, &oMi[lane][0]);
      }
    }
    __syncwarp();
  }
}

// Does some pair (pa[k], pb[k]), k < n_pairs, intersect with its first shape inflated by `margin`?  Warp-uniform.
// oMg: the warp's geometry placements; cand: the warp's kMaxCand-entry candidate list.  The broad phase runs over all
// pairs first (bounding spheres), compacting the survivors, so that the narrow phase (GJK, a few hundred instructions,
// data dependent) runs on FULL warps of candidates instead of on the one or two lanes of each 32-pair round that happen
// to survive.
template <typename T>
__device__ __forceinline__ bool warp_any_pair_hits(const DevScene<T>* sc, const uint8_t* pa, const uint8_t* pb, int n_pairs,
                                                   const T (*oMg)[12], uint16_t* cand, T margin, int lane) {
  bool hit = false;
  int n_cand = 0;
  for (int k0 = 0; k0 < n_pairs && !hit; k0 += 32) {
    const int k = k0 + lane;
    bool pass = false;
    if (k < n_pairs) {
      const int a = pa[k], b = pb[k];
      const T dx = oMg[a][9] - oMg[b][9], dy = oMg[a][10] - oMg[b][10], dz = oMg[a][11] - oMg[b][11];
      const T reach = sc->g[a].bound + sc->g[b].bound + margin;
      pass = dx * dx + dy * dy + dz * dz <= reach * reach;
    }
    const unsigned m = __ballot_sync(0xffffffffu, pass);
    if (n_cand + __popc(m) > kMaxCand) {
      // list full (never with the reference scene): test this round's survivors in place
      if (pass) hit = gjk_intersect(make_shape(sc->g[pa[k]], oMg[pa[k]]), make_shape(sc->g[pb[k]], oMg[pb[k]]), margin);
      hit = __any_sync(0xffffffffu, hit);
    } else {
      if (pass) cand[n_cand + __popc(m & ((1u << lane) - 1u))] = (uint16_t)k;
      n_cand += __popc(m);
    }
  }
  __syncwarp();
  for (int c0 = 0; c0 < n_cand && !hit; c0 += 32) {
    if (c0 + lane < n_cand) {
      const int k = cand[c0 + lane];
      const int a = pa[k], b = pb[k];
      hit = gjk_intersect(make_shape(sc->g[a], oMg[a]), make_shape(sc->g[b], oMg[b]), margin);
    }
    hit = __any_sync(0xffffffffu, hit);
  }
  return hit;
}

template <typename T>
__global__ void __launch_bounds__(kCollideWarps * 32)
gik_collision_kernel(const DevScene<T>* __restrict__ sc, const uint8_t* __restrict__ pa, const uint8_t* __restrict__ pb,
                     int n_pairs, int64_t n, const T* __restrict__ q, const T* __restrict__ cube_pose, T margin,
                     uint8_t* __restrict__ out, int invert, const int64_t* __restrict__ sel, int64_t n_sel,
                     const int64_t* __restrict__ n_sel_dev) {
  __shared__ T s_oMi[kCollideWarps][GIK_MAX_NQ][12];
  __shared__ T s_oMg[kCollideWarps][GIK_MAX_GEOMS][12];
  __shared__ uint16_t s_cand[kCollideWarps][kMaxCand];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int ng = sc->n_geoms;
  const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  // `sel` (optional): test only the columns sel[0 .. n_sel) of the [.][n] arrays; results go to out[sel[.]]
  const int64_t count = sel ? (n_sel_dev ? *n_sel_dev : n_sel) : n;
  for (int64_t w_i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w_i < count; w_i += warps) {
    const int64_t i = sel ? __ldg(sel + w_i) : w_i;
    // q = nullptr (the cube-only test): no FK, the robot's geometries keep their local placements
    if (q) warp_tree_fk(sc, lane, [&](int j) { return __ldg(q + (int64_t)j * n + i); }, s_oMi[w]);
    for (int g = lane; g < ng; g += 32)
      place_geom(sc, g, cube_pose, n, i, q ? s_oMi[w] : nullptr, s_oMg[w][g]);
    __syncwarp();
    const bool hit = warp_any_pair_hits(sc, pa, pb, n_pairs, s_oMg[w], s_cand[w], margin, lane);
    if (lane == 0) out[i] = (uint8_t)((hit ? 1 : 0) ^ (invert ? 1 : 0));
    __syncwarp();
  }
}

// distanceToObstacle(robot, q) as a VALUE (tools.py:38-51): the smallest distance over the pairs of one list, capped at
// d_max, 0 when a pair intersects (hpp-fcl reports the negative penetration depth there; every caller in the reference
// only compares the value with a positive threshold, path.py:61-62).  One configuration per warp like the collision
// kernel; each lane takes pairs, and brackets ITS pair's distance by bisection on the margin of the boolean GJK ("A
// inflated by m intersects B") inside the running minimum of the warp -- a pair whose bounding spheres are farther apart
// than the best distance so far is skipped, a pair that does not intersect even at the best distance so far costs one
// GJK.  `rounds` bisection steps: the value is exact to d_max / 2^rounds.
template <typename T>
__global__ void __launch_bounds__(kCollideWarps * 32)
gik_distance_kernel(const DevScene<T>* __restrict__ sc, const uint8_t* __restrict__ pa, const uint8_t* __restrict__ pb,
                    int n_pairs, int64_t n, const T* __restrict__ q, const T* __restrict__ cube_pose, T d_max, int rounds,
                    T* __restrict__ out) {
  __shared__ T s_oMi[kCollideWarps][GIK_MAX_NQ][12];
  __shared__ T s_oMg[kCollideWarps][GIK_MAX_GEOMS][12];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int ng = sc->n_geoms;
  const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += warps) {
    warp_tree_fk(sc, lane, [&](int j) { return __ldg(q + (int64_t)j * n + i); }, s_oMi[w]);
    for (int g = lane; g < ng; g += 32) place_geom(sc, g, cube_pose, n, i, s_oMi[w], s_oMg[w][g]);
    __syncwarp();
    T best = d_max;                                 // running minimum, warp-uniform
    for (int k0 = 0; k0 < n_pairs && best > T(0); k0 += 32) {
      const int k = k0 + lane;
      T mine = best;
      if (k < n_pairs) {
        const int a = pa[k], b = pb[k];
        const T* Ma = &s_oMg[w][a][0];
        const T* Mb = &s_oMg[w][b][0];
        const T dx = Ma[9] - Mb[9], dy = Ma[10] - Mb[10], dz = Ma[11] - Mb[11];
        const T reach = sc->g[a].bound + sc->g[b].bound + best;
        if (dx * dx + dy * dy + dz * dz <= reach * reach) {
          const Shape<T> A = make_shape(sc->g[a], Ma), B = make_shape(sc->g[b], Mb);
          if (gjk_intersect(A, B, best)) {          // closer than the best so far: bracket it
            if (gjk_intersect(A, B, T(0))) mine = T(0);
            else {
              T lo = T(0), hi = best;
              for (int r = 0; r < rounds; ++r) {
                const T mid = T(0.5) * (lo + hi);
                if (gjk_intersect(A, B, mid)) hi = mid; else lo = mid;
              }
              mine = T(0.5) * (lo + hi);
            }
          }
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mine = min_(mine, __shfl_xor_sync(0xffffffffu, mine, o));
      best = mine;
    }
    if (lane == 0) out[i] = best;
    __syncwarp();
  }
}

// converged problems -> index list (order irrelevant) + count, everything else gets success = 0; one atomicAdd per warp
__global__ void __launch_bounds__(256) gik_compact_converged_kernel(int64_t n, const uint8_t* __restrict__ conv,
                                                                    uint8_t* __restrict__ success, int64_t* __restrict__ count,
                                                                    int64_t* __restrict__ sel) {
  const int lane = threadIdx.x & 31;
  for (int64_t i0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) & ~31ll; i0 < n; i0 += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = i0 + lane;
    const bool c = i < n && conv[i] != 0;
    const unsigned m = __ballot_sync(0xffffffffu, c);
    long long base = 0;
    if (lane == 0 && m) base = (long long)atomicAdd((unsigned long long*)count, (unsigned long long)__popc(m));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (c) sel[base + __popc(m & ((1u << lane) - 1u))] = i;
    else if (i < n) success[i] = 0;
  }
}

// pending = converged && colliding && iterations left: the problems on which the reference keeps descending
// (inverse_geometry.py:70 -- the predicate stays False while collision(q) holds).  success[] holds converged && !colliding.
__global__ void __launch_bounds__(256) gik_compact_pending_kernel(int64_t n, const uint8_t* __restrict__ conv,
                                                                  const uint8_t* __restrict__ success,
                                                                  const int32_t* __restrict__ iters, int max_iters,
                                                                  int64_t* __restrict__ count, int64_t* __restrict__ sel) {
  const int lane = threadIdx.x & 31;
  for (int64_t i0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) & ~31ll; i0 < n; i0 += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = i0 + lane;
    const bool c = i < n && conv[i] != 0 && success[i] == 0 && iters[i] < max_iters;
    const unsigned m = __ballot_sync(0xffffffffu, c);
    long long base = 0;
    if (lane == 0 && m) base = (long long)atomicAdd((unsigned long long*)count, (unsigned long long)__popc(m));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (c) sel[base + __popc(m & ((1u << lane) - 1u))] = i;
  }
}


// ---------------------------------------------------------------------------------------------------------------
// The reference's keep-descending-while-colliding tail (inverse_geometry.py:70, 97-98), ONE WARP PER PENDING PROBLEM.
//
// A pending problem converged at iteration it_c in configuration q_c and collides there.  The reference goes on
// descending -- the residual keeps shrinking, so every later iterate passes the residual test -- and re-tests
// collision(q) on every iterate until one is free (success) or the cap is reached (failure, q after max_iters updates).
// The continuation launch of the solve kernel has already produced that last configuration q_f.  Between q_c and q_f
// every point of the robot moves by a few millimetres at most, which settles almost every pair for ALL iterates at once:
//   * delta_ab = safety * (disp_a + disp_b) + floor bounds the relative displacement of geometries a, b over the tail
//     (disp_g = |p_g(q_f) - p_g(q_c)| + ||R_g(q_f) - R_g(q_c)||_F * bounding radius; the iterates lie between q_c and q_f
//     on a path that is straight to first order -- e_k = (1 - dt)^k e_c -- hence the safety factor);
//   * a pair whose shapes still intersect when both are ERODED by delta/2 collides on every iterate: the problem fails
//     with q = q_f, exactly what the reference returns, and no iterate needs testing (PERSISTENT);
//   * a pair that does not intersect even when INFLATED by delta is free on every iterate and is dropped;
//   * what is left (typically the fingers against the cube face they sit 1 mm from) is UNDECIDED: the warp then replays
//     the descent from q_c -- lanes 0 / 1 run the two hands of the pair mapping -- and tests just those pairs on every
//     iterate, stopping at the first iterate that is converged and free: the reference's decision, iterate by iterate.
// ---------------------------------------------------------------------------------------------------------------
// Two launches of the same code: STAGE 0 classifies every pending problem (persistent -> final outputs; otherwise the
// problem goes on the replay list) and compiles WITHOUT the IK replay, so that it runs at the collision kernel's
// occupancy; STAGE 1 runs over the (short) replay list, repeats the classification of its problems to rebuild their
// undecided-pair lists, and replays the descent.
template <typename T, bool WRIST, int STAGE>
__global__ void __launch_bounds__(kCollideWarps * 32, (STAGE == 0 ? 4 : 2))
gik_tail_kernel(const __grid_constant__ DevTable<T> tab, const DevScene<T>* __restrict__ sc, const uint8_t* __restrict__ pa,
                const uint8_t* __restrict__ pb, int n_pairs, int64_t n, const int64_t* __restrict__ sel,
                const int64_t* __restrict__ n_sel_dev, const T* __restrict__ pose, const T* __restrict__ q_fin,
                const T* __restrict__ resid_fin, T* q, uint8_t* success, uint8_t* conv, int32_t* iters, T* resid,
                T eps2, T dt, T lambda, int max_iters, T safety, unsigned long long* queue, unsigned long long* stats,
                int64_t* replay_count, int64_t* replay_sel) {
  __shared__ T s_oMi[kCollideWarps][GIK_MAX_NQ][12];
  __shared__ T s_oMg[kCollideWarps][GIK_MAX_GEOMS][12];
  __shared__ T s_disp[kCollideWarps][GIK_MAX_GEOMS];
  __shared__ T s_q[kCollideWarps][GIK_MAX_NQ];
  __shared__ uint16_t s_cand[kCollideWarps][kMaxCand];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int nq = sc->tree.nq, ng = sc->n_geoms;
  const int64_t count = min(n, (int64_t)*n_sel_dev);
  const T kFloor = sizeof(T) == 4 ? T(2e-5) : T(1e-9);     // round-off of the placements themselves
  const int h = lane & 1, off = 1 + 6 * h;
  const ArmConst<T>& ac = tab.arm[h];
  for (;;) {
    unsigned long long item = 0;
    if (lane == 0) item = atomicAdd(queue, 1ull);
    item = __shfl_sync(0xffffffffu, item, 0);
    if ((int64_t)item >= count) break;
    const int64_t i = sel[item];
    T cube[12];
#pragma unroll
    for (int k = 0; k < 12; ++k) cube[k] = __ldg(pose + (int64_t)k * n + i);
    // ---- displacement of every geometry between q_c and q_f
    warp_tree_fk(sc, lane, [&](int j) { return q_fin[(int64_t)j * n + i]; }, s_oMi[w]);
    T Pf[2][12];
#pragma unroll
    for (int sl = 0; sl < 2; ++sl) {
      const int g = lane + 32 * sl;
      if (g < ng) place_geom(sc, g, cube, 1, 0, s_oMi[w], Pf[sl]);
    }
    __syncwarp();
    if (lane < nq) s_q[w][lane] = q[(int64_t)lane * n + i];
    __syncwarp();
    warp_tree_fk(sc, lane, [&](int j) { return s_q[w][j]; }, s_oMi[w]);
#pragma unroll
    for (int sl = 0; sl < 2; ++sl) {
      const int g = lane + 32 * sl;
      if (g < ng) {
        T Pc[12];
        place_geom(sc, g, cube, 1, 0, s_oMi[w], Pc);
        T dR = T(0), dp = T(0);
#pragma unroll
        for (int k = 0; k < 9; ++k) { const T d = Pc[k] - Pf[sl][k]; dR += d * d; }
#pragma unroll
        for (int k = 9; k < 12; ++k) { const T d = Pc[k] - Pf[sl][k]; dp += d * d; }
        s_disp[w][g] = sqrt_(dp) + sqrt_(dR) * sc->g[g].bound;
#pragma unroll
        for (int k = 0; k < 12; ++k) s_oMg[w][g][k] = Pc[k];
      }
    }
    __syncwarp();
    // ---- broad phase with the displacement margin, candidates compacted
    int n_cand = 0;
    for (int k0 = 0; k0 < n_pairs; k0 += 32) {
      const int k = k0 + lane;
      bool pass = false;
      if (k < n_pairs) {
        const int a = pa[k], b = pb[k];
        const T* Ma = &s_oMg[w][a][0];
        const T* Mb = &s_oMg[w][b][0];
        const T dx = Ma[9] - Mb[9], dy = Ma[10] - Mb[10], dz = Ma[11] - Mb[11];
        const T reach = sc->g[a].bound + sc->g[b].bound + safety * (s_disp[w][a] + s_disp[w][b]) + kFloor;
        pass = dx * dx + dy * dy + dz * dz <= reach * reach;
      }
      const unsigned m = __ballot_sync(0xffffffffu, pass);
      if (pass && n_cand + __popc(m & ((1u << lane) - 1u)) < kMaxCand) s_cand[w][n_cand + __popc(m & ((1u << lane) - 1u))] = (uint16_t)k;
      n_cand = min(n_cand + __popc(m), kMaxCand);
    }
    __syncwarp();
    // ---- narrow phase: persistent / undecided (the undecided ones are compacted in place at the front of the list)
    bool persistent = false;
    int n_und = 0;
    for (int c0 = 0; c0 < n_cand; c0 += 32) {
      bool pers = false, und = false;
      int k = 0;
      if (c0 + lane < n_cand) {
        k = s_cand[w][c0 + lane];
        const int a = pa[k], b = pb[k];
        const T delta = safety * (s_disp[w][a] + s_disp[w][b]) + kFloor;
        pers = narrow_hits(sc->g[a], &s_oMg[w][a][0], sc->g[b], &s_oMg[w][b][0], -delta);
        if (!pers) und = narrow_hits(sc->g[a], &s_oMg[w][a][0], sc->g[b], &s_oMg[w][b][0], delta);
      }
      persistent = persistent || __any_sync(0xffffffffu, pers);
      const unsigned m = __ballot_sync(0xffffffffu, und);
      __syncwarp();
      if (und) s_cand[w][n_und + __popc(m & ((1u << lane) - 1u))] = (uint16_t)k;    // n_und <= c0: never ahead of the reads
      n_und += __popc(m);
      __syncwarp();
    }
    if (persistent) {
      // collides on every iterate: the loop runs to the cap, q after max_iters updates, success = False
      // (STAGE 1 only sees problems STAGE 0 found not persistent; the branch is kept for safety)
      if (lane < nq) q[(int64_t)lane * n + i] = q_fin[(int64_t)lane * n + i];
      if (lane == 0) {
        success[i] = 0; conv[i] = 0; iters[i] = max_iters;
        resid[i] = resid_fin[i]; resid[n + i] = resid_fin[n + i];
        if (stats) atomicAdd(stats + 0, 1ull);
      }
      __syncwarp();
      continue;
    }
    if constexpr (STAGE == 0) {
      if (lane == 0) replay_sel[atomicAdd((unsigned long long*)replay_count, 1ull)] = i;
      __syncwarp();
      continue;
    }
    if constexpr (STAGE == 1) {
    // ---- replay the descent from q_c, testing the undecided pairs on every iterate
    T qh[7], tgt[12];
    {
      qh[0] = s_q[w][tab.act_q[0]];
#pragma unroll
      for (int k = 0; k < 6; ++k) qh[1 + k] = s_q[w][tab.act_q[off + k]];
      hook_target(ac, cube, tgt);
    }
    int it = iters[i];
    unsigned long long trips = 0;
    for (;;) {
      T r = T(0), r_o = T(0), kappa = T(0), dqa[6];
      if (lane < 2) {
        T cs[kActive], sn[kActive], Sy, Sz;
#pragma unroll
        for (int k = 0; k < 7; ++k)      // (tip-aligned wrist step: the tip slot carries q6 - tip_psi, hand_wrist_phase1)
          sincos_<true>((WRIST && (kNextageTZ & kTipZ) && k == 6) ? qh[k] - ac.tip_psi : qh[k], sn[k], cs[k]);
        HandState<T> hs;
        WristState<T> wst;
        if constexpr (WRIST) hand_wrist_phase1<T, 0, kNextageTZ>(ac, cs, sn, tgt, wst, Sy, Sz, r);
        else hand_phase1<T, 0, 0, false>(ac, cs, sn, tgt, lambda, hs, Sy, Sz, r);
        const T Sy_o = __shfl_xor_sync(0x3u, Sy, 1), Sz_o = __shfl_xor_sync(0x3u, Sz, 1);
        r_o = __shfl_xor_sync(0x3u, r, 1);
        kappa = h ? chest_rate(Sy_o, Sz_o, Sy, Sz) : chest_rate(Sy, Sz, Sy_o, Sz_o);
        if constexpr (WRIST) hand_wrist_phase2(wst, kappa, dqa);
        else hand_phase2(hs, kappa, dqa);
      }
      const bool pass0 = (r < eps2) && (r_o < eps2) && (it < max_iters);
      const bool pass = __shfl_sync(0xffffffffu, (int)pass0, 0) != 0;
      bool collide = false;
      if (pass) {
        if (lane < 2) {
          if (h == 0) s_q[w][tab.act_q[0]] = qh[0];
#pragma unroll
          for (int k = 0; k < 6; ++k) s_q[w][tab.act_q[off + k]] = qh[1 + k];
        }
        __syncwarp();
        warp_tree_fk(sc, lane, [&](int j) { return s_q[w][j]; }, s_oMi[w]);
        for (int c0 = 0; c0 < n_und && !collide; c0 += 32) {
          bool hit = false;
          if (c0 + lane < n_und) {
            const int k = s_cand[w][c0 + lane];
            const int a = pa[k], b = pb[k];
            T Ma[12], Mb[12];
            place_geom(sc, a, cube, 1, 0, s_oMi[w], Ma);
            place_geom(sc, b, cube, 1, 0, s_oMi[w], Mb);
            hit = narrow_hits(sc->g[a], Ma, sc->g[b], Mb, T(0));
          }
          collide = __any_sync(0xffffffffu, hit);
        }
        __syncwarp();
      }
      const bool stop_ok = pass && !collide;
      const bool stop_cap = it >= max_iters;
      if (stop_ok || stop_cap) {
        if (lane < 2) {                      // the configuration the loop stopped at
          if (h == 0) s_q[w][tab.act_q[0]] = qh[0];
#pragma unroll
          for (int k = 0; k < 6; ++k) s_q[w][tab.act_q[off + k]] = qh[1 + k];
          resid[(int64_t)h * n + i] = sqrt_(r);
        }
        __syncwarp();
        if (lane < nq) q[(int64_t)lane * n + i] = s_q[w][lane];
        if (lane == 0) {
          success[i] = stop_ok ? 1 : 0; conv[i] = stop_ok ? 1 : 0; iters[i] = it;
          if (stats) { atomicAdd(stats + 1, 1ull); atomicAdd(stats + 2, trips); if (stop_ok) atomicAdd(stats + 3, 1ull); }
        }
        __syncwarp();
        break;
      }
      if (lane < 2) {
        qh[0] = min_(max_(tab.lo[0], qh[0] + dt * kappa), tab.hi[0]);
#pragma unroll
        for (int k = 0; k < 6; ++k) qh[1 + k] = min_(max_(tab.lo[off + k], qh[1 + k] + dt * dqa[k]), tab.hi[off + k]);
      }
      ++it; ++trips;
    }
    }
  }
}

}  // namespace gik

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
struct gik_scene_dev {
  gik::DevScene<float>* sc32 = nullptr;
  gik::DevScene<double>* sc64 = nullptr;
  uint8_t (*pairs)[2][gik::kPairListCap] = nullptr;   // gik::PairLists::pairs on the device
  int n_list[gik::kNumPairLists] = {};
};

namespace {

void free_scene(gik_scene_dev* sd) {
  if (!sd) return;
  cudaFree(sd->sc32); cudaFree(sd->sc64); cudaFree(sd->pairs);
  delete sd;
}

template <typename T> gik::DevScene<T>* scene_of(gik_scene_dev* sd);
template <> gik::DevScene<float>* scene_of<float>(gik_scene_dev* sd) { return sd->sc32; }
template <> gik::DevScene<double>* scene_of<double>(gik_scene_dev* sd) { return sd->sc64; }

// one pair list of the attached scene on the device: pair k = (a[k], b[k]), k < n
struct DevPairList { const uint8_t *a, *b; int n; };
DevPairList pair_list(const gik_scene_dev* sd, gik::PairList l) { return {sd->pairs[l][0], sd->pairs[l][1], sd->n_list[l]}; }

template <typename T>
int collide_api(gik_handle_t h, int64_t n, const T* q, const T* cube_pose, gik::PairList list, double margin, int invert,
                uint8_t* out, void* stream, const int64_t* sel = nullptr, int64_t n_sel = 0,
                const int64_t* n_sel_dev = nullptr) {
  if (bad_handle(h)) return GIK_E_HANDLE;
  if (n < 0) return GIK_E_SIZE;
  if (!(margin >= 0.0)) return GIK_E_PARAM;
  if (!h->scene) return GIK_E_NOSCENE;
  if (n == 0 || (sel && !n_sel_dev && n_sel == 0)) return GIK_OK;
  if (n_sel < 0) return GIK_E_SIZE;
  const bool cube_only = list == gik::kListCube;
  if (!out || (!cube_only && !q) || (cube_only && !cube_pose)) return GIK_E_NULL;
  DeviceGuard g(h->device);
  if (g.err != cudaSuccess) return (int)g.err;
  const int64_t work = (sel && !n_sel_dev) ? n_sel : n;     // device-side count: size the grid for the upper bound
  int64_t blocks = (work + gik::kCollideWarps - 1) / gik::kCollideWarps;
  const int64_t cap = (int64_t)h->sm_count * 16;
  if (blocks > cap) blocks = cap;
  const DevPairList pl = pair_list(h->scene, list);
  gik::gik_collision_kernel<T><<<(int)blocks, gik::kCollideWarps * 32, 0, (cudaStream_t)stream>>>(
      scene_of<T>(h->scene), pl.a, pl.b, pl.n, n, q, cube_pose, (T)margin, out, invert, sel, n_sel, n_sel_dev);
  return (int)cudaGetLastError();
}

template <typename T>
int distance_api(gik_handle_t h, int64_t n, const T* q, const T* cube_pose, gik::PairList list, double d_max, T* out,
                 void* stream) {
  if (bad_handle(h)) return GIK_E_HANDLE;
  if (n < 0) return GIK_E_SIZE;
  if (!(d_max > 0.0)) return GIK_E_PARAM;
  if (!h->scene) return GIK_E_NOSCENE;
  if (n == 0) return GIK_OK;
  if (!out || !q) return GIK_E_NULL;
  DeviceGuard g(h->device);
  if (g.err != cudaSuccess) return (int)g.err;
  int64_t blocks = (n + gik::kCollideWarps - 1) / gik::kCollideWarps;
  const int64_t cap = (int64_t)h->sm_count * 16;
  if (blocks > cap) blocks = cap;
  const DevPairList pl = pair_list(h->scene, list);
  const int rounds = sizeof(T) == 4 ? 20 : 40;       // d_max / 2^rounds: below the arithmetic's own resolution
  gik::gik_distance_kernel<T><<<(int)blocks, gik::kCollideWarps * 32, 0, (cudaStream_t)stream>>>(
      scene_of<T>(h->scene), pl.a, pl.b, pl.n, n, q, cube_pose, (T)d_max, rounds, out);
  return (int)cudaGetLastError();
}

}  // namespace

// scratch layout of gik_solve_success_* (bytes, 256-aligned blocks): two index lists with their device-side counts, the
// continuation's outputs (q_f, residuals, flags, iteration counts), the tail kernel's work queue and counters
struct SuccessScratch {
  int64_t *sel1, *sel2, *sel3; // [n + 1] each: count at [0], list from [1] (converged | pending | to replay)
  void *q_fin, *resid_fin;     // [nq][n], [2][n] of T
  uint8_t* flag_fin;           // [n]
  int32_t* iters_fin;          // [n]
  unsigned long long* queue;   // [1] + stats [4]
  size_t bytes;
};
static SuccessScratch carve_scratch(void* base, int64_t n, int nq, int esz) {
  auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
  SuccessScratch s{};
  size_t o = 0;
  char* b = (char*)base;
  s.sel1 = (int64_t*)(b + o); o += up((size_t)(n + 1) * 8);
  s.sel2 = (int64_t*)(b + o); o += up((size_t)(n + 1) * 8);
  s.sel3 = (int64_t*)(b + o); o += up((size_t)(n + 1) * 8);
  s.q_fin = b + o; o += up((size_t)nq * n * esz);
  s.resid_fin = b + o; o += up((size_t)2 * n * esz);
  s.flag_fin = (uint8_t*)(b + o); o += up((size_t)n);
  s.iters_fin = (int32_t*)(b + o); o += up((size_t)n * 4);
  s.queue = (unsigned long long*)(b + o); o += up(8 * 8);
  s.bytes = o;
  return s;
}

// K3 + the collision term in ONE stream-ordered call, no host synchronisation (inverse_geometry.py:70, 97-98):
//   1. the descent loop (stops at the first iterate with both residuals < eps);
//   2. the converged problems are compacted on the device and tested: success = converged && !collision(q);
//   3. [unless GIK_F_NO_DESCEND] the converged-but-colliding problems are the ones the reference keeps descending on:
//      a continuation launch of the solve kernel runs them to the iteration cap (q_f), and gik_tail_kernel decides each
//      one -- persistent collision (fails with q_f), or a replay that tests the undecided pairs iterate by iterate.
template <typename T>
int solve_success_api(gik_handle_t h, int64_t n, const T* q_init, const T* pose, const gik_params_t* prm, T* q_out,
                      uint8_t* success, uint8_t* conv, int32_t* iters, T* resid, void* scratch, void* stream) {
  if (bad_handle(h)) return GIK_E_HANDLE;
  if (!h->scene) return GIK_E_NOSCENE;
  if (n > 0 && (!success || !conv || !scratch || !iters || !resid)) return GIK_E_NULL;
  int rc = solve_api<T>(h, n, q_init, pose, prm, q_out, conv, iters, resid, stream);
  if (rc || n == 0) return rc;
  DeviceGuard g(h->device);
  if (g.err != cudaSuccess) return (int)g.err;
  cudaStream_t st = (cudaStream_t)stream;
  const int nq = h->host.nq;
  SuccessScratch sc = carve_scratch(scratch, n, nq, (int)sizeof(T));
  cudaError_t e = cudaMemsetAsync(sc.sel1, 0, sizeof(int64_t), st);
  if (e == cudaSuccess) e = cudaMemsetAsync(sc.sel2, 0, sizeof(int64_t), st);
  if (e == cudaSuccess) e = cudaMemsetAsync(sc.sel3, 0, sizeof(int64_t), st);
  if (e == cudaSuccess) e = cudaMemsetAsync(sc.queue, 0, 8 * 8, st);
  if (e != cudaSuccess) return (int)e;
  int64_t blocks = (n + 255) / 256;
  if (blocks > (int64_t)h->sm_count * 8) blocks = (int64_t)h->sm_count * 8;
  gik::gik_compact_converged_kernel<<<(int)blocks, 256, 0, st>>>(n, conv, success, sc.sel1, sc.sel1 + 1);
  if ((e = cudaGetLastError()) != cudaSuccess) return (int)e;
  rc = collide_api<T>(h, n, q_out, pose, gik::kListAll, 0.0, 1, success, stream, sc.sel1 + 1, 0, sc.sel1);
  if (rc || (prm->flags & GIK_F_NO_DESCEND)) return rc;
  // ---- the tail
  gik::gik_compact_pending_kernel<<<(int)blocks, 256, 0, st>>>(n, conv, success, iters, prm->max_iters, sc.sel2, sc.sel2 + 1);
  if ((e = cudaGetLastError()) != cudaSuccess) return (int)e;
  {
    SolveArgs<T> a{};
    a.q_init = q_out; a.pose = pose; a.iters = sc.iters_fin; a.resid = (T*)sc.resid_fin;
    a.q_dst[0] = (T*)sc.q_fin; a.conv_dst[0] = sc.flag_fin; a.n_dst = 1; a.out_off = 0;
    a.n = n;
    set_soa(a, n, n);
    a.sel = sc.sel2 + 1; a.n_sel = sc.sel2; a.it0 = iters;
    gik_params_t p2 = *prm;
    p2.flags &= ~GIK_F_EARLY_STOP;
    rc = launch_solve<T, MODE_BATCH>(h, a, &p2, stream, /*force=*/true);
    if (rc) return rc;
  }
  const DevPairList pl = pair_list(h->scene, gik::kListAll);
  int64_t tb = (n + gik::kCollideWarps - 1) / gik::kCollideWarps;
  const int64_t cap = (int64_t)h->sm_count * 16;
  if (tb > cap) tb = cap;
  const T safety = (T)1.5;
  const bool wrist = use_wrist<T>(h, prm);
  const T eps2 = (T)(prm->eps * prm->eps);
  // queue[0] / queue[5]: work counters of the two stages; queue[1..4]: statistics
  auto launch_tail = [&](auto kern, int64_t blocks_, const int64_t* list, unsigned long long* q_) {
    kern<<<(int)blocks_, gik::kCollideWarps * 32, 0, st>>>(
        table_of<T>(h), scene_of<T>(h->scene), pl.a, pl.b, pl.n, n, list + 1, list, pose, (const T*)sc.q_fin,
        (const T*)sc.resid_fin, q_out, success, conv, iters, resid, eps2, (T)prm->dt, (T)prm->damping, prm->max_iters, safety,
        q_, sc.queue + 1, sc.sel3, sc.sel3 + 1);
  };
  const int64_t cap2 = (int64_t)h->sm_count * 2;
  if (wrist) {
    launch_tail(gik::gik_tail_kernel<T, true, 0>, tb, sc.sel2, sc.queue);
    launch_tail(gik::gik_tail_kernel<T, true, 1>, tb < cap2 ? tb : cap2, sc.sel3, sc.queue + 5);
  } else {
    launch_tail(gik::gik_tail_kernel<T, false, 0>, tb, sc.sel2, sc.queue);
    launch_tail(gik::gik_tail_kernel<T, false, 1>, tb < cap2 ? tb : cap2, sc.sel3, sc.queue + 5);
  }
  return (int)cudaGetLastError();
}

extern "C" {

int gik_scene_attach(gik_handle_t h, const gik_scene_t* scene) {
  if (bad_handle(h)) return GIK_E_HANDLE;
  if (!scene) return GIK_E_NULL;
  int rc = gik::validate_scene(h->host, *scene);
  if (rc) return rc;
  DeviceGuard g(h->device);
  if (g.err != cudaSuccess) return (int)g.err;
  gik_scene_dev* sd = new (std::nothrow) gik_scene_dev();
  if (!sd) return (int)cudaErrorMemoryAllocation;
  gik::DevScene<float>* h32 = new (std::nothrow) gik::DevScene<float>();
  gik::DevScene<double>* h64 = new (std::nothrow) gik::DevScene<double>();
  gik::PairLists* hl = new (std::nothrow) gik::PairLists();
  cudaError_t e = (h32 && h64 && hl) ? cudaSuccess : cudaErrorMemoryAllocation;
  if (e == cudaSuccess) {
    gik::fill_dev_scene(h->host, *scene, *h32);
    gik::fill_dev_scene(h->host, *scene, *h64);
    gik::build_pair_lists(h->host, *scene, *hl);
    for (int l = 0; l < gik::kNumPairLists; ++l) sd->n_list[l] = hl->n[l];
    if ((e = cudaMalloc(&sd->sc32, sizeof(*h32))) == cudaSuccess &&
        (e = cudaMalloc(&sd->sc64, sizeof(*h64))) == cudaSuccess &&
        (e = cudaMalloc(&sd->pairs, sizeof(hl->pairs))) == cudaSuccess &&
        (e = cudaMemcpy(sd->sc32, h32, sizeof(*h32), cudaMemcpyHostToDevice)) == cudaSuccess &&
        (e = cudaMemcpy(sd->sc64, h64, sizeof(*h64), cudaMemcpyHostToDevice)) == cudaSuccess)
      e = cudaMemcpy(sd->pairs, hl->pairs, sizeof(hl->pairs), cudaMemcpyHostToDevice);
  }
  delete h32; delete h64; delete hl;
  if (e != cudaSuccess) { free_scene(sd); return (int)e; }
  cudaDeviceSynchronize();          // a previous scene may still be in use by enqueued kernels
  free_scene(h->scene);
  h->scene = sd;
  return GIK_OK;
}

int gik_collision_f32(gik_handle_t h, int64_t n, const float* q, const float* cube, uint8_t* out, void* s) { return collide_api<float>(h, n, q, cube, gik::kListAll, 0.0, 0, out, s); }
int gik_collision_f64(gik_handle_t h, int64_t n, const double* q, const double* cube, uint8_t* out, void* s) { return collide_api<double>(h, n, q, cube, gik::kListAll, 0.0, 0, out, s); }
int gik_collision_sel_f32(gik_handle_t h, int64_t n, int64_t n_sel, const int64_t* sel, const float* q, const float* cube, uint8_t* out, void* s) {
  if (!sel) return GIK_E_NULL;
  return collide_api<float>(h, n, q, cube, gik::kListAll, 0.0, 0, out, s, sel, n_sel);
}
int gik_collision_sel_f64(gik_handle_t h, int64_t n, int64_t n_sel, const int64_t* sel, const double* q, const double* cube, uint8_t* out, void* s) {
  if (!sel) return GIK_E_NULL;
  return collide_api<double>(h, n, q, cube, gik::kListAll, 0.0, 0, out, s, sel, n_sel);
}
int gik_solve_success_f32(gik_handle_t h, int64_t n, const float* q_init, const float* pose, const gik_params_t* p, float* q_out,
                          uint8_t* success, uint8_t* conv, int32_t* iters, float* resid, void* scratch, void* s) {
  return solve_success_api<float>(h, n, q_init, pose, p, q_out, success, conv, iters, resid, scratch, s);
}
int gik_solve_success_f64(gik_handle_t h, int64_t n, const double* q_init, const double* pose, const gik_params_t* p, double* q_out,
                          uint8_t* success, uint8_t* conv, int32_t* iters, double* resid, void* scratch, void* s) {
  return solve_success_api<double>(h, n, q_init, pose, p, q_out, success, conv, iters, resid, scratch, s);
}
size_t gik_solve_success_scratch_bytes(gik_handle_t h, int64_t n, int elem_size) {
  if (bad_handle(h) || n < 0 || (elem_size != 4 && elem_size != 8)) return 0;
  return carve_scratch(nullptr, n, h->host.nq, elem_size).bytes;
}
int gik_clearance_f32(gik_handle_t h, int64_t n, const float* q, const float* cube, double thr, uint8_t* out, void* s) { return collide_api<float>(h, n, q, cube, gik::kListEnv, thr, 1, out, s); }
int gik_clearance_f64(gik_handle_t h, int64_t n, const double* q, const double* cube, double thr, uint8_t* out, void* s) { return collide_api<double>(h, n, q, cube, gik::kListEnv, thr, 1, out, s); }
int gik_obstacle_distance_f32(gik_handle_t h, int64_t n, const float* q, const float* cube, double d_max, float* dist, void* s) { return distance_api<float>(h, n, q, cube, gik::kListEnv, d_max, dist, s); }
int gik_obstacle_distance_f64(gik_handle_t h, int64_t n, const double* q, const double* cube, double d_max, double* dist, void* s) { return distance_api<double>(h, n, q, cube, gik::kListEnv, d_max, dist, s); }
int gik_cube_collision_f32(gik_handle_t h, int64_t n, const float* cube, uint8_t* out, void* s) { return collide_api<float>(h, n, (const float*)nullptr, cube, gik::kListCube, 0.0, 0, out, s); }
int gik_cube_collision_f64(gik_handle_t h, int64_t n, const double* cube, uint8_t* out, void* s) { return collide_api<double>(h, n, (const double*)nullptr, cube, gik::kListCube, 0.0, 0, out, s); }

}  // extern "C"
