// gik_kernels.cu -- sm_100a kernels and the C ABI of include/gik.h.
//
// Mapping (DESIGN.md "Execution model"): ONE IK PROBLEM PER LANE (lane kernels) or per LANE PAIR (pair kernel), all
// state in registers, no shared memory and (lane kernels) no cross-lane traffic inside an iteration, so every issue
// slot of the descent loop is FP32/FP64 arithmetic.  The kernels are persistent: a lane whose problem finished
// (converged or iteration cap) stores its result and takes the next problem from a global work queue, so the bimodal
// iteration count (~740 converged vs 1000 exhausted) does not idle lanes.
// The kinematic table travels as a __grid_constant__ kernel parameter (constant bank 0): FMAs read it as
// c[0x0][...] operands, and a handle stays immutable and stream-safe.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <atomic>
#include <new>

#include "gik_table.h"

namespace gik {

constexpr int kThreads = 128;   // threads per block of the persistent solve kernels

// resident blocks per SM of the scalar lane kernel
template <typename T> struct Launch;
template <> struct Launch<float>  { static constexpr int kMinBlocks = 4; };   // 4 x 128 threads / SM -> <= 128 registers per thread
template <> struct Launch<double> { static constexpr int kMinBlocks = 3; };   // 3 x 128 threads / SM -> 168 registers per thread;
    // spills go to L1 and cost LSU issue slots, which the FP64-pipe-bound loop has to spare (measured +7 % over 2 blocks,
    // -10 % at 4 blocks)

enum { MODE_BATCH = 0, MODE_EDGES = 1 };
#define GIK_FLOPS_EXEC_F32_WRIST 945    // see gik_flops_per_iter_executed()

template <typename T>
struct SolveArgs {
  // batch mode
  const T* q_init;      // [nq][n]
  const T* pose;        // [12][n]   (edges: pose_a)
  T* q_out;             // edges: q_path [max_steps][nq][n]   (batch mode stores through q_dst / conv_dst)
  // batch-mode destinations: 1 (the caller's q_out / converged) or, for the fused all-gather, one per rank
  // (peer-mapped pointers); a result goes to column out_off + idx of arrays with out_n columns
  // (fused all-gather: [0] is THIS rank's own array, where the lanes store; [1 .. n_dst) are the peers' arrays, filled by
  // coalesced chunk pushes -- "Fused all-gather" below; marks[w] = low-water mark of compute warp w, pushed[c] = chunk c
  // of the slab has been copied to the peers)
  T* q_dst[GIK_MAX_PEERS];
  uint8_t* conv_dst[GIK_MAX_PEERS];
  int32_t n_dst;
  int64_t out_off;
  int32_t* marks;
  int32_t n_marks;
  int32_t push_blocks;         // leading blocks of the grid that push instead of solving
  int32_t top_from;            // fused launches: warps in hardware slot top_from or higher take their problems from the TOP of the
                               // slab (0: single-ended queue)
  long long* push_ctl;         // [0] F: problems [0, F) are finished, [1] every compute warp has left, [2] next chunk to push,
                               // [3] compute warps that have left; then statistics
  uint8_t* pushed;
  int32_t* warp_stats;         // measurement hook (GIK_FUSED_STATS): [2] per compute warp, or null
  // element (component c, problem i) of an array lives at ptr[c * sc + i * si]: SoA [C][n] = (n, 1), rows [n][C] = (1, C)
  int64_t q_sc, q_si, pose_sc, pose_si, out_sc, out_si, res_sc, res_si;
  // streamed input (host-resident batches): problems [0, *ready) are resident; a refill waits for the ones it takes
  const unsigned long long* ready;
  // continuation launches (the keep-descending-while-colliding tail, gik_solve_success_*): work item c of the queue is
  // column sel[c] of the arrays, *n_sel (device) items exist (n is only the upper bound the grid was sized for), and the
  // problem resumes at iteration it0[column].  All three null for an ordinary launch.
  const int64_t* sel;
  const int64_t* n_sel;
  const int32_t* it0;
  int32_t* iters;       // [n] or null (edges: iters_total)
  T* resid;             // [2][n] or null
  // edge mode
  const T* pose_b;      // [12][n]
  const int32_t* num_steps;
  int32_t* n_valid;
  int32_t max_steps;
  // common
  int64_t n;
  T eps2, dt, lambda;   // eps2 = eps^2: the predicate compares squared norms
  int32_t max_iters;
  int32_t early_stop;   // GIK_F_EARLY_STOP: give up on a problem whose squared residual fell < 10 % over 64 iterations
  int32_t lanes;        // problems per warp kept in flight (1..32); < 32 spreads a small batch over more SMs
  unsigned long long* queue;  // work queue head (zeroed on the stream before the launch): next problem to hand out
};

// Problem inputs (q_init, pose, num_steps) are read with ld.global.cg (L2 only), never with the non-coherent path:
// on the streamed host path (gik_solve_rows_*) the copy engine is still writing those staging buffers while the kernel
// runs, and ld.global.nc (__ldg) is only defined for data that is read-only during the kernel's lifetime -- a stale L1
// sector left by a warp that read the last row of one slab could otherwise serve the first row of the next slab.
// Every input is read exactly once per problem, so bypassing L1 costs nothing.
template <typename U>
__device__ __forceinline__ U ld_in(const U* p) { return __ldcg(p); }

template <typename T>
__device__ __forceinline__ void load_cube(const T* pose, int64_t sc, int64_t si, int64_t idx, T (&cube)[12]) {
#pragma unroll
  for (int c = 0; c < 12; ++c) cube[c] = ld_in(pose + (int64_t)c * sc + idx * si);
}

// the problems a refill is about to take must be resident (streamed input); no-op for device-resident batches
template <typename T>
__device__ __forceinline__ void wait_resident(const SolveArgs<T>& a, unsigned long long upto) {
  if (a.ready) {
    if (upto > (unsigned long long)a.n) upto = (unsigned long long)a.n;
    while (*(const volatile unsigned long long*)a.ready < upto) __nanosleep(200);
    __threadfence();   // acquire: the slab's rows are read only after the counter that publishes them
  }
}

// One refill of a warp: `need` = lanes (lane kernels) or even lanes of the pairs (pair kernel) without work, `rank` = this
// lane's position among them.  Returns the work item of this lane, or -1 when the queue has no more.
// Plain launches: the queue word counts the items handed out, in index order.
// Fused all-gather launches (a.top_from > 0): the word is TWO counters -- low half: items handed out from the bottom of
// the slab, high half: items handed out from the top -- and the warps in the high hardware slots (from_top) work downwards from
// the top.  Why: the SM's warp scheduler serves the co-resident warps of a sub-partition in strict slot order
// (measured with GIK_FUSED_STATS, see warp_slot(): of four co-resident warps the first finishes ~760 problems per launch,
// the others ~440 / ~180 / ~50), so a problem on a late warp lives up to 13x longer than one on an early warp and would hold the finished
// PREFIX -- all the pushers can ship -- back by a third of the launch.  With the late warps (17 % of the throughput)
// working at the other end, the prefix trails the queue by the early warps' problem duration only.  The two ends meet
// wherever they meet: no tuning, no imbalance.  A problem's arithmetic does not depend on who solves it or when.
template <typename T>
__device__ __forceinline__ int64_t queue_take(const SolveArgs<T>& a, int64_t n, unsigned need, int lane, int rank,
                                              bool from_top, bool& exhausted) {
  const int k = __popc(need), leader = __ffs(need) - 1;
  unsigned long long old = 0;
  if (lane == leader) old = atomicAdd(a.queue, from_top ? ((unsigned long long)k << 32) : (unsigned long long)k);
  old = __shfl_sync(0xffffffffu, old, leader);
  if (a.top_from == 0) {
    if (old + k >= (unsigned long long)n) exhausted = true;
    wait_resident(a, old + k);
    const int64_t cand = (int64_t)old + rank;
    return cand < n ? cand : -1;
  }
  const int64_t b = (int64_t)(old & 0xffffffffull), t = (int64_t)(old >> 32);
  if (b + t + k >= n) exhausted = true;
  const int64_t cand = from_top ? n - 1 - t - rank : b + rank;
  return (from_top ? cand >= b : cand < n - t) ? cand : -1;
}

// ---------------------------------------------------------------------------------------------------------------
// Fused all-gather (gik_solve_scatter_*): the transfer half of "solve + all-gather in one kernel".
//
// A finished problem's result is stored into this rank's OWN result arrays (q_dst[0] / conv_dst[0]) exactly as in a
// plain launch.  The leading push_blocks blocks of the grid do not solve: one warp is a lookout, the others are PUSHERS
// that copy finished chunks of kChunk consecutive problems -- nq rows of kChunk values plus kChunk flags -- into every peer's arrays with coalesced 16-byte
// stores over NVLink (loads from L2), all through the launch, so the transfer overlaps the remaining solves.  A small
// tail kernel (gik_push_rest_kernel, the whole machine) copies what is left when the last problem ends -- the chunks
// that were still in flight -- and one cross-rank barrier follows.
//
// How a pusher knows that a chunk is finished without the solving lanes paying for it: the queue hands problems out in
// index order, so "every problem below F is finished" holds for F = min(queue head, smallest index still being solved).
// Each compute warp publishes a LOW-WATER MARK -- the smallest index among its lanes' current problems, in units of
// 2^kMarkShift problems -- into marks[warp]; the lookout takes the minimum over all marks and the queue head.  (Warps
// that work from the top of the slab -- queue_take -- never hold the prefix and publish "done" at once.)  A warp
// recomputes its mark only when one of its lanes finishes (one REDUX), publishes it only when it changed (<= n >>
// kMarkShift times per launch) and one finish event LATE, before that event's own result stores: the release fence in
// front of the publication then has nothing in flight to wait for.  Stale marks are low, i.e. conservative.  [The first
// form -- every finishing lane counted its problem into a per-chunk counter with a fence + atomicAdd whose result
// decided who pushes -- cost 5.5 % of the kernel at 2 GPUs (26.17 against 24.80 ms per 2^20 problems): the fence and
// the round trip of the atomic stalled the whole warp ~440 times per launch.]
// Message passing: result stores, __threadfence, st.relaxed.gpu mark (compute warps); ld.relaxed.gpu marks,
// __threadfence, ld.global.cg results (pushers).
// ---------------------------------------------------------------------------------------------------------------
constexpr int kChunkShift = 10;
constexpr int kChunk = 1 << kChunkShift;
constexpr int kMarkShift = 13;
constexpr int kMarkDone = 0x7fffffff;

__device__ __forceinline__ int ld_relaxed(const int32_t* p) {
  int v;
  asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long ld_relaxed(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed(int32_t* p, int v) {
  asm volatile("st.relaxed.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// Hardware slot of this warp on its SM.  The warp scheduler serves the ready warps of a sub-partition in slot order --
// measured with GIK_FUSED_STATS on 2^20 problems, 16 warps per SM: slots 0-3 finish 763 problems per launch each, slots 4-7
// 441, slots 8-11 177, slots 12-15 50 -- so the slot number IS the warp's priority (see queue_take).
__device__ __forceinline__ int warp_slot() {
  unsigned w;
  asm volatile("mov.u32 %0, %%warpid;" : "=r"(w));
  return (int)w;
}

// compute-warp side -------------------------------------------------------------------------------------------------
struct MarkState { int pub = 0, pending = 0, events = 0; };
template <typename T>
__device__ __forceinline__ int mark_slot(const SolveArgs<T>& a) {          // the leading blocks hold the pushers
  return ((int)blockIdx.x - a.push_blocks) * (kThreads / 32) + ((int)threadIdx.x >> 5);
}
// a lane of this warp finished: called BEFORE the results of this event are stored
template <typename T>
__device__ __forceinline__ void mark_publish(const SolveArgs<T>& a, MarkState& ms, int lane) {
  if (ms.pending != ms.pub) {
    __threadfence();
    __syncwarp();
    if (lane == 0) st_relaxed(a.marks + mark_slot(a), ms.pending);
    ms.pub = ms.pending;
  }
}
// ... and AFTER the finished lanes were retired: the mark this warp may publish at its next event
__device__ __forceinline__ void mark_update(MarkState& ms, bool active, int64_t idx) {
  ++ms.events;
  const int m = __reduce_min_sync(0xffffffffu, active ? (int)(idx >> kMarkShift) : kMarkDone);
  if (m != kMarkDone) ms.pending = m;     // no lane active: the refill brings larger indices, or the warp leaves
}
// the warp leaves the kernel: its mark no longer holds anything back, and it is counted in push_ctl[3]
template <typename T>
__device__ __forceinline__ void mark_exit(const SolveArgs<T>& a, int lane) {
  __threadfence();
  __syncwarp();
  if (lane == 0) {
    st_relaxed(a.marks + mark_slot(a), kMarkDone);
    asm volatile("red.relaxed.gpu.global.add.u64 [%0], 1;" ::"l"(a.push_ctl + 3) : "memory");
  }
}
// a warp that takes its problems from the top of the slab (queue_take) never holds the prefix back
template <typename T>
__device__ __forceinline__ void mark_skip(const SolveArgs<T>& a, int lane) {
  if (lane == 0) st_relaxed(a.marks + mark_slot(a), kMarkDone);
}
template <typename T>
__device__ __forceinline__ void mark_stats(const SolveArgs<T>& a, const MarkState& ms, int lane, bool from_top) {
  if (a.warp_stats && lane == 0) {     // measurement hook: finish events of this warp and the end of the slab it worked from
    a.warp_stats[2 * mark_slot(a)] = ms.events;
    unsigned wid;
    asm volatile("mov.u32 %0, %%warpid;" : "=r"(wid));
    a.warp_stats[2 * mark_slot(a) + 1] = (from_top ? 1 : 0) | ((int)wid << 8);
  }
}

__device__ __forceinline__ unsigned long long now_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ int4 ld_relaxed4(const int32_t* p) {
  int4 v;
  asm volatile("ld.relaxed.gpu.global.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ long long ld_relaxed(const long long* p) {
  long long v;
  asm volatile("ld.relaxed.gpu.global.s64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed(long long* p, long long v) {
  asm volatile("st.relaxed.gpu.global.s64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// pusher side -------------------------------------------------------------------------------------------------------
// chunk ch of the slab: rows of this rank's own arrays -> the same place in every peer's arrays (one warp)
// `stop` (in-kernel pushers only): a control word that turns non-zero when the last solve has ended; the push is then
// abandoned between two batches of loads (returns false, the chunk stays unflagged and the tail kernel copies it whole)
// so that the solve kernel does not outlive its last solve by the rest of a chunk -- up to 0.1 ms with 7 destinations.
template <typename T>
__device__ __forceinline__ bool push_chunk(const SolveArgs<T>& a, int nq, int64_t n_items, int64_t ch, int lane,
                                           const long long* stop = nullptr) {
  const int64_t left = n_items - (ch << kChunkShift);
  const int cs = (int)(left < kChunk ? left : kChunk);
  const int64_t c0 = a.out_off + (ch << kChunkShift);
  constexpr int PER = 16 / (int)sizeof(T);
  bool vec = (c0 % PER) == 0 && (a.out_sc % PER) == 0 && (cs % PER) == 0;
  bool vecb = (c0 % 16) == 0 && (cs % 16) == 0;
  for (int d = 0; d < a.n_dst; ++d) {
    vec = vec && ((uintptr_t)a.q_dst[d] % 16) == 0;
    vecb = vecb && ((uintptr_t)a.conv_dst[d] % 16) == 0;
  }
  if (vec) {
    // flattened (row, 16-byte word) space, eight independent loads in flight per lane
    constexpr int U = 8;
    const int wpr = cs / PER, total = nq * wpr;
    for (int k0 = lane; k0 < total; k0 += 32 * U) {
      if (stop) {
        long long sv = 0;
        if (lane == 0) sv = ld_relaxed(stop);
        if (__shfl_sync(0xffffffffu, sv, 0) != 0) return false;
      }
      uint4 v[U];
      int64_t o[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int k = k0 + 32 * u;
        if (k < total) {
          const int r = k / wpr, w = k - r * wpr;
          o[u] = (int64_t)r * a.out_sc + c0 + (int64_t)w * PER;
          v[u] = __ldcg((const uint4*)(a.q_dst[0] + o[u]));
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (k0 + 32 * u < total)
          for (int d = 1; d < a.n_dst; ++d) *(uint4*)(a.q_dst[d] + o[u]) = v[u];
    }
  } else {
    for (int r = 0; r < nq; ++r) {
      const int64_t o = (int64_t)r * a.out_sc + c0;
      for (int k = lane; k < cs; k += 32) {
        const T v = __ldcg(a.q_dst[0] + o + k);
        for (int d = 1; d < a.n_dst; ++d) a.q_dst[d][o + k] = v;
      }
    }
  }
  if (vecb) {
    for (int k = lane; k < cs / 16; k += 32) {
      const uint4 v = __ldcg((const uint4*)(a.conv_dst[0] + c0) + k);
      for (int d = 1; d < a.n_dst; ++d) ((uint4*)(a.conv_dst[d] + c0))[k] = v;
    }
  } else {
    for (int k = lane; k < cs; k += 32) {
      const uint8_t v = __ldcg(a.conv_dst[0] + c0 + k);
      for (int d = 1; d < a.n_dst; ++d) a.conv_dst[d][c0 + k] = v;
    }
  }
  return true;
}

// The leading push_blocks blocks of a fused launch.  Warp 0 of block 0 is the LOOKOUT: it keeps reading the queue head
// and the marks (16-byte relaxed loads, eight in flight per lane: ~2.5 us per look at 2364 marks) and posts F --
// "problems [0, F) are finished" -- in push_ctl[0].  The other warps take chunks in order from push_ctl[2], wait until F
// has passed the chunk, push it and flag it.  All leave as soon as every compute warp has left (all marks kMarkDone ->
// push_ctl[1]): whatever is not pushed by then -- the ~10^5 problems that were in flight when the queue ran dry, whose
// chunks all complete in the last moments of the launch -- is the tail kernel's, which has the whole machine.
// [Measured on the way here: every pusher warp looking for itself, one dependent 4-byte load after the other: 16 us per
// look, two thirds of the pushers' time, half of the chunks pushed in-kernel.  Pushers that finish the chunks F has
// already passed before they look at the exit flag: the kernel outlives the last solve by 4 ms at 2 destinations and
// 19 ms at 8, because F sweeps the last 10 % of the slab at the very end.]
template <typename T>
__device__ __noinline__ void pusher_loop(const SolveArgs<T>& a, int nq, int64_t n) {
  const int lane = threadIdx.x & 31, warp = (int)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5);
  const int64_t n_chunks = (n + kChunk - 1) >> kChunkShift;
  unsigned long long t_a = 0, t_b = 0;    // measurement hook (GIK_FUSED_STATS): lookout: looking / sleeping; pushers: pushing / waiting
  int count = 0;                          // looks / chunks pushed
  if (warp == 0) {
    const int n4 = a.n_marks >> 2;        // (n_marks is a multiple of 4: whole blocks)
    for (;;) {
      const unsigned long long t0 = now_ns();
      unsigned long long Q = 0;
      if (lane == 0) Q = ld_relaxed(a.queue);
      Q = __shfl_sync(0xffffffffu, Q, 0);
      int m = kMarkDone, arg = -1;       // (arg: the warp holding the smallest mark, for the trace of the measurement hook)
      for (int i0 = lane; i0 < n4; i0 += 32 * 8) {
        int4 v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u)
          v[u] = (i0 + 32 * u < n4) ? ld_relaxed4(a.marks + 4 * (i0 + 32 * u)) : make_int4(kMarkDone, kMarkDone, kMarkDone, kMarkDone);
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int mu = min(min(v[u].x, v[u].y), min(v[u].z, v[u].w));
          if (mu < m) { m = mu; arg = 4 * (i0 + 32 * u) + (v[u].x == mu ? 0 : v[u].y == mu ? 1 : v[u].z == mu ? 2 : 3); }
        }
      }
      {
        const int mw = __reduce_min_sync(0xffffffffu, m);
        const unsigned who = __ballot_sync(0xffffffffu, m == mw);
        arg = __shfl_sync(0xffffffffu, arg, __ffs(who) - 1);
        m = mw;
      }
      ++count;
      long long gone = 0;
      if (lane == 0) gone = ld_relaxed(a.push_ctl + 3);
      gone = __shfl_sync(0xffffffffu, gone, 0);
      if (gone >= a.n_marks) {            // every compute warp has left
        if (lane == 0) st_relaxed(a.push_ctl + 1, 1ll);
        t_a += now_ns() - t0;
        break;
      }
      // finished prefix: below every mark and inside what the bottom end of the queue has handed out
      int64_t F = m == kMarkDone ? n : ((int64_t)m << kMarkShift);
      if (a.top_from > 0) {
        const int64_t b = (int64_t)(Q & 0xffffffffull), t = (int64_t)(Q >> 32);
        if (b < F) F = b;
        if (n - t < F) F = n - t;
      } else if ((int64_t)Q < F) {
        F = (int64_t)Q;
      }
      if (F > n) F = n;
      if (F < 0) F = 0;
      __threadfence();                    // F is posted after the marks that cover it were read
      if (lane == 0) st_relaxed(a.push_ctl, (long long)F);
      const unsigned long long t1 = now_ns();
      if (lane == 0 && (count & 255) == 1 && (count >> 8) < 60) {      // statistics: a trace of (time, F, queue head)
        long long* tr = a.push_ctl + 32 + 3 * (count >> 8);
        tr[0] = (long long)(t1 / 1000); tr[1] = (long long)F; tr[2] = ((long long)arg << 40) | (long long)(Q & 0xffffffffull);
      }
      t_a += t1 - t0;
      __nanosleep(1000);
      t_b += now_ns() - t1;
    }
  } else {
    for (;;) {
      long long c = 0;
      if (lane == 0) c = (long long)atomicAdd((unsigned long long*)(a.push_ctl + 2), 1ull);
      c = __shfl_sync(0xffffffffu, c, 0);
      if (c >= n_chunks) break;
      const int64_t end = ((int64_t)c + 1) << kChunkShift;
      const int64_t need = end < n ? end : n;
      const unsigned long long t0 = now_ns();
      bool left = false;
      for (;;) {
        long long st[2] = {0, 0};
        if (lane == 0) { st[1] = ld_relaxed(a.push_ctl + 1); st[0] = ld_relaxed(a.push_ctl); }
        const long long Fs = __shfl_sync(0xffffffffu, st[0], 0);
        left = __shfl_sync(0xffffffffu, st[1], 0) != 0;
        if (left || Fs >= need) break;
        __nanosleep(1000);
      }
      const unsigned long long t1 = now_ns();
      t_b += t1 - t0;
      if (left) break;                    // the solves are over: chunk c (not flagged) and the rest go to the tail kernel
      __threadfence();                    // results are read after the F that covers them
      const bool whole = push_chunk(a, nq, n, c, lane, a.push_ctl + 1);
      __syncwarp();
      if (!whole) break;                  // the solves ended while this chunk was on its way: the tail kernel redoes it
      if (lane == 0) a.pushed[c] = 1;
      t_a += now_ns() - t1;
      ++count;
    }
  }
  if (lane == 0 && warp < 8) {            // statistics of the first eight warps behind the control words
    long long* o = a.push_ctl + 4 + 3 * warp;
    o[0] = (long long)(t_a / 1000); o[1] = (long long)(t_b / 1000); o[2] = count;
  }
}

// after the solve kernel, stream-ordered: every chunk the pushers did not get to
template <typename T>
__global__ void __launch_bounds__(128) gik_push_rest_kernel(const __grid_constant__ SolveArgs<T> a, int nq, int tag) {
  const int lane = threadIdx.x & 31;
  const int64_t n_chunks = (a.n + kChunk - 1) >> kChunkShift;
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t c = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); c < n_chunks; c += warps)
    if (!a.pushed[c]) {
      push_chunk(a, nq, a.n, c, lane);
      if (tag && lane == 0) a.pushed[c] = (uint8_t)tag;    // (statistics of the measurement hook only)
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Per-problem code of the three solve kernels: what runs when a lane (lane pair) takes a work item, and when its problem
// or one step of its edge ends.  These rules define the results -- the start iteration, the placement of each edge step,
// when the passive joints are clamped, how n_valid counts -- so all kernels run this one copy of them.  Each kernel
// loads and stores its own ACTIVE joints, whose layout differs: load_q(idx) reads them from q_init, store_q(dst, sc, si,
// col) writes them to column col of dst (component stride sc, column stride si).  `owner` is the lane that writes the
// per-problem fields: every lane of the lane kernels, the even lane of a pair.
// ---------------------------------------------------------------------------------------------------------------
template <typename T>
struct Work {
  int64_t idx = -1;          // column of the problem (or edge) this lane works on
  bool active = false;
  int it = 0;                // descent iterations of the problem (edge: of the current step)
  T r_mark = T(3.0e38);      // early stop: squared residual sum at the last 64-iteration checkpoint
  int step = 0, nsteps = 0, it_total = 0;   // edge mode: current step (from 1), steps of the edge, iterations so far
};

// cube placement of step `step` of edge idx
template <typename T>
__device__ __forceinline__ void edge_step_cube(const SolveArgs<T>& a, int64_t idx, int step, int nsteps, T (&cube)[12]) {
  T ca[12], cb[12], xi[6];
  load_cube(a.pose, a.pose_sc, a.pose_si, idx, ca);
  load_cube(a.pose_b, a.pose_sc, a.pose_si, idx, cb);
  se3_delta(ca, cb, xi);
  edge_placement(ca, xi, step, nsteps, cube);
}

// The lane takes work item `cand`: its column, start iteration and active joints, and in `cube` the placement its hooks
// aim at (edges: that of step 1).  An edge with nothing to march ends at once with no valid step: the reference loop
// body never runs (path.py:137).
template <typename T, int MODE, typename LoadQ>
__device__ __forceinline__ void work_start(const SolveArgs<T>& a, int64_t cand, bool owner, Work<T>& w, LoadQ load_q,
                                           T (&cube)[12]) {
  w.idx = a.sel ? a.sel[cand] : cand;
  w.active = true;
  w.it = a.it0 ? a.it0[w.idx] : 0;
  w.r_mark = T(3.0e38);
  load_q(w.idx);
  if (MODE == MODE_BATCH) {
    load_cube(a.pose, a.pose_sc, a.pose_si, w.idx, cube);
    return;
  }
  w.nsteps = ld_in(a.num_steps + w.idx);
  w.step = 1;
  w.it_total = 0;
  edge_step_cube(a, w.idx, 1, w.nsteps, cube);
  if (w.nsteps < 1) {
    if (owner) {
      a.n_valid[w.idx] = 0;
      if (a.iters) a.iters[w.idx] = 0;
    }
    w.active = false;
  }
}

// passive joints of a result: q_init, clamped to their limits if an update has been applied (`moved`: the first update
// clamps the whole q, :89)
template <typename T>
__device__ __forceinline__ void store_passive(const DevTable<T>& tab, const SolveArgs<T>& a, int64_t idx, bool moved, T* dst,
                                              int64_t sc, int64_t si, int64_t col) {
  for (int p = 0; p < tab.n_passive; ++p) {
    const int j = tab.passive_q[p];
    T v = ld_in(a.q_init + (int64_t)j * a.q_sc + idx * a.q_si);
    if (moved) v = min_(max_(tab.qlo[j], v), tab.qhi[j]);
    dst[(int64_t)j * sc + col * si] = v;
  }
}

// Batch mode: the lane's problem ended (ok: converged).  Its result goes to this rank's own arrays (peers: the pushers of
// block 0) -- joints, flag, iteration count, and the residual norm of each hand this lane solved (r[k]: hand h0 + k) --
// and the lane is free.
template <typename T, int NH, typename StoreQ>
__device__ __forceinline__ void batch_finish(const DevTable<T>& tab, const SolveArgs<T>& a, Work<T>& w, bool ok, bool owner,
                                             StoreQ store_q, int h0, const T (&r)[NH]) {
  const int64_t col = a.out_off + w.idx;
  T* qo = a.q_dst[0];
  store_q(qo, a.out_sc, a.out_si, col);
  if (owner) {
    store_passive(tab, a, w.idx, w.it > 0, qo, a.out_sc, a.out_si, col);
    a.conv_dst[0][col] = ok ? 1 : 0;
    if (a.iters) a.iters[w.idx] = w.it;
  }
  if (a.resid)
#pragma unroll
    for (int k = 0; k < NH; ++k) a.resid[(int64_t)(h0 + k) * a.res_sc + w.idx * a.res_si] = sqrt_(r[k]);
  w.active = false;
}

// Edge mode: the solve of step w.step ended (ok: converged).  A converged step stores its path row, the passive joints
// clamped once any update has been applied on this edge.  Then the lane either goes on to the next step -- returns true
// with its placement in `cube` -- or the edge is finished: n_valid = the steps that converged, iters = the iterations of
// the whole edge.
template <typename T, typename StoreQ>
__device__ __forceinline__ bool edge_step_end(const DevTable<T>& tab, const SolveArgs<T>& a, Work<T>& w, bool ok, bool owner,
                                              StoreQ store_q, T (&cube)[12]) {
  w.it_total += w.it;
  if (ok) {
    T* dst = a.q_out + (int64_t)(w.step - 1) * tab.nq * a.n;
    store_q(dst, a.n, 1, w.idx);
    if (owner) store_passive(tab, a, w.idx, w.it_total > 0, dst, a.n, 1, w.idx);
  }
  if (ok && w.step < w.nsteps) {
    ++w.step;
    w.it = 0;
    w.r_mark = T(3.0e38);
    edge_step_cube(a, w.idx, w.step, w.nsteps, cube);
    return true;
  }
  if (owner) {
    a.n_valid[w.idx] = ok ? w.step : w.step - 1;
    if (a.iters) a.iters[w.idx] = w.it_total;
  }
  w.active = false;
  return false;
}

template <typename T, int MODE, uint32_t TZ, bool WRIST = false>
__global__ void __launch_bounds__(kThreads, Launch<T>::kMinBlocks)
gik_solve_kernel(const __grid_constant__ DevTable<T> tab, const __grid_constant__ SolveArgs<T> a) {
  const int lane = threadIdx.x & 31;
  const int64_t n = a.n_sel ? min(a.n, (int64_t)*a.n_sel) : a.n;          // work items of this launch
  if (MODE == MODE_BATCH && a.n_dst > 1 && (int)blockIdx.x < a.push_blocks) {   // fused all-gather: the leading blocks push, the others solve
    pusher_loop(a, tab.nq, n);
    return;
  }
  const bool from_top = MODE == MODE_BATCH && a.top_from > 0 && warp_slot() >= a.top_from;   // (see queue_take)
  if (from_top) mark_skip(a, threadIdx.x & 31);     // works outside the prefix: nothing to hold back
  const int L = a.lanes;
  const bool enabled = lane < L;

  T q[kActive], tgt[2][12];
#pragma unroll
  for (int i = 0; i < kActive; ++i) q[i] = T(0);
#pragma unroll
  for (int h = 0; h < 2; ++h)
#pragma unroll
    for (int c = 0; c < 12; ++c) tgt[h][c] = (c % 4 == 0 && c < 9) ? T(1) : T(0);
  auto load_q = [&](int64_t idx) {
#pragma unroll
    for (int i = 0; i < kActive; ++i) q[i] = ld_in(a.q_init + (int64_t)tab.act_q[i] * a.q_sc + idx * a.q_si);
  };
  auto store_q = [&](T* dst, int64_t sc, int64_t si, int64_t col) {
#pragma unroll
    for (int i = 0; i < kActive; ++i) dst[(int64_t)tab.act_q[i] * sc + col * si] = q[i];
  };
  auto set_targets = [&](const T (&cube)[12]) {
    hook_target(tab.arm[0], cube, tgt[0]);
    hook_target(tab.arm[1], cube, tgt[1]);
  };

  Work<T> w;
  bool exhausted = false;   // warp-uniform: the queue has handed out every problem
  MarkState ms;             // fused all-gather: this warp's low-water mark

  for (;;) {
    // ---------------- refill: lanes without work pull the next problems from the global queue ----------------
    // One atomicAdd per warp per refill (leader lane, count = lanes in need), so problems are handed out in index
    // order to whichever lane frees up first: the tail of the launch is bounded by ONE problem's duration instead
    // of by the slowest statically assigned lane.  The first refill of a warp takes 32 consecutive problems
    // (coalesced loads).  A problem's arithmetic does not depend on the lane it lands on: results are bit-identical.
    const unsigned need = exhausted ? 0u : __ballot_sync(0xffffffffu, enabled && !w.active);
    if (need) {
      const int64_t cand = queue_take(a, n, need, lane, __popc(need & ((1u << lane) - 1u)), from_top, exhausted);
      if (enabled && !w.active && cand >= 0) {
        T cube[12];
        work_start<T, MODE>(a, cand, true, w, load_q, cube);
        set_targets(cube);
      }
    }
    if (exhausted && !__any_sync(0xffffffffu, w.active)) break;

    // ---------------- one descent iteration for every lane ----------------
    T dq[kActive], rL, rR;
    ik_iteration<T, true, TZ, WRIST>(tab, q, tgt, a.lambda, dq, rL, rR);
    const bool ok = (rL < a.eps2) && (rR < a.eps2) && (w.it < a.max_iters);
    bool stalled = false;
    if (a.early_stop && (w.it & 63) == 63) {
      const T rs = rL + rR;
      stalled = rs > T(0.9) * w.r_mark;
      w.r_mark = rs;
    }
    const bool done = ok || (w.it >= a.max_iters) || stalled;

    const bool fused_event = MODE == MODE_BATCH && a.n_dst > 1 && __any_sync(0xffffffffu, done && w.active);
    if (fused_event && !from_top) mark_publish(a, ms, lane);
    if (!done) {
      apply_step(tab, q, dq, a.dt);
      ++w.it;
    } else if (w.active) {
      // ---------------- rare path: this lane's problem (edge step) ended ----------------
      T cube[12];
      if (MODE == MODE_BATCH) {
        const T r[2] = {rL, rR};
        batch_finish(tab, a, w, ok, true, store_q, 0, r);
      } else if (edge_step_end(tab, a, w, ok, true, store_q, cube)) {
        set_targets(cube);
      }
    }
    if (fused_event) mark_update(ms, w.active, w.idx);      // (from_top warps: statistics only)
  }
  if (MODE == MODE_BATCH && a.n_dst > 1) mark_exit(a, lane);
}


// ========================================================================================================
// fp32 lane kernel, packed: one problem per lane with the two hands carried in the halves of F2 registers, so the
// chain walks, Gram matrices, Cholesky factorisations and solves of both hands issue as FFMA2 / FMUL2 / FADD2 --
// half the issue slots of the scalar lane kernel for the same arithmetic (gik_core.cuh "F2").  Scheduling (global
// work queue, lane refill) is the scalar lane kernel's.
// Resident blocks per SM: 3 (168 registers) for the block-Cholesky step; 4 for the spherical-wrist step (128 registers,
// ~190 B of spills outside the iteration).  2^20 problems, packed log6: 42.2 M solves/s against 41.2 M at 3 blocks
// (144 registers, none) and 38.0 M at 5 (96 registers).
// ========================================================================================================
template <int MODE, uint32_t TZ, bool WRIST = false>
__global__ void __launch_bounds__(kThreads, (WRIST ? 4 : 3))
gik_solve_lane2_kernel(const __grid_constant__ DevTable<float> tab, const __grid_constant__ PackedTable pt,
                       const __grid_constant__ SolveArgs<float> a) {
  using T = float;
  const int lane = threadIdx.x & 31;
  const int64_t n = a.n_sel ? min(a.n, (int64_t)*a.n_sel) : a.n;          // work items of this launch
  if (MODE == MODE_BATCH && a.n_dst > 1 && (int)blockIdx.x < a.push_blocks) {   // fused all-gather: the leading blocks push, the others solve
    pusher_loop(a, tab.nq, n);
    return;
  }
  const bool from_top = MODE == MODE_BATCH && a.top_from > 0 && warp_slot() >= a.top_from;   // (see queue_take)
  if (from_top) mark_skip(a, threadIdx.x & 31);     // works outside the prefix: nothing to hold back
  const int L = a.lanes;
  const bool enabled = lane < L;

  T q0 = T(0);
  F2 q2[6], tgt2[12];          // (left, right) arm angles and hook targets
#pragma unroll
  for (int k = 0; k < 6; ++k) q2[k] = F2(0.0f);
#pragma unroll
  for (int c = 0; c < 12; ++c) tgt2[c] = F2((c % 4 == 0 && c < 9) ? 1.0f : 0.0f);
  auto load_q = [&](int64_t idx) {
    q0 = ld_in(a.q_init + (int64_t)tab.act_q[0] * a.q_sc + idx * a.q_si);
#pragma unroll
    for (int k = 0; k < 6; ++k)
      q2[k] = F2(ld_in(a.q_init + (int64_t)tab.act_q[1 + k] * a.q_sc + idx * a.q_si), ld_in(a.q_init + (int64_t)tab.act_q[7 + k] * a.q_sc + idx * a.q_si));
  };
  auto store_q = [&](T* dst, int64_t sc, int64_t si, int64_t col) {
    dst[(int64_t)tab.act_q[0] * sc + col * si] = q0;
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      dst[(int64_t)tab.act_q[1 + k] * sc + col * si] = q2[k].x;
      dst[(int64_t)tab.act_q[7 + k] * sc + col * si] = q2[k].y;
    }
  };
  auto set_targets = [&](const T (&cube)[12]) {
    T tl[12], tr[12];
    hook_target(tab.arm[0], cube, tl);
    hook_target(tab.arm[1], cube, tr);
#pragma unroll
    for (int c = 0; c < 12; ++c) tgt2[c] = F2(tl[c], tr[c]);
  };

  Work<T> w;
  bool exhausted = false;   // warp-uniform: the queue has handed out every problem
  MarkState ms;             // fused all-gather: this warp's low-water mark

  for (;;) {
    // ---------------- refill: lanes without work pull the next problems from the global queue ----------------
    // (as in the scalar lane kernel)
    const unsigned need = exhausted ? 0u : __ballot_sync(0xffffffffu, enabled && !w.active);
    if (need) {
      const int64_t cand = queue_take(a, n, need, lane, __popc(need & ((1u << lane) - 1u)), from_top, exhausted);
      if (enabled && !w.active && cand >= 0) {
        T cube[12];
        work_start<T, MODE>(a, cand, true, w, load_q, cube);
        set_targets(cube);
      }
    }
    if (!__any_sync(0xffffffffu, w.active)) {
      if (exhausted) break;
      continue;                                // (edges with nothing to march) back to the queue
    }

    // ---------------- one descent iteration for every lane ----------------
    // The iteration repeats in a loop of its own until an active lane finishes -- arithmetic, one vote and the back edge
    // per trip; the queue / store logic above and below runs only then (as in the pair kernel).  Measured against the
    // single-loop form on 2^20 problems: 38.30 -> 36.75 ms (27.3 -> 28.5 M solves/s).
    T rL, rR;
    bool ok, done;
    for (;;) {
      T dq0;
      F2 dq2[6];
      ik_iteration_packed<TZ, WRIST>(pt, q0, q2, tgt2, a.lambda, dq0, dq2, rL, rR);
      ok = (rL < a.eps2) && (rR < a.eps2) && (w.it < a.max_iters);
      bool stalled = false;
      if (a.early_stop && (w.it & 63) == 63) {
        const T rs = rL + rR;
        stalled = rs > T(0.9) * w.r_mark;
        w.r_mark = rs;
      }
      done = ok || (w.it >= a.max_iters) || stalled;
      if (!done) {
        q0 = min_(max_(pt.lo0, q0 + a.dt * dq0), pt.hi0);
        const F2 dt2 = F2(a.dt);
#pragma unroll
        for (int k = 0; k < 6; ++k) q2[k] = min_(max_(pt.lo[k], q2[k] + dt2 * dq2[k]), pt.hi[k]);
        ++w.it;
      }
      if (__any_sync(0xffffffffu, done && w.active)) break;
    }
    const bool fused_event = MODE == MODE_BATCH && a.n_dst > 1 && __any_sync(0xffffffffu, done && w.active);
    if (fused_event && !from_top) mark_publish(a, ms, lane);
    if (done && w.active) {
      // ---------------- rare path: this lane's problem (edge step) ended ----------------
      T cube[12];
      if (MODE == MODE_BATCH) {
        const T r[2] = {rL, rR};
        batch_finish(tab, a, w, ok, true, store_q, 0, r);
      } else if (edge_step_end(tab, a, w, ok, true, store_q, cube)) {
        set_targets(cube);
      }
    }
    if (fused_event) mark_update(ms, w.active, w.idx);      // (from_top warps: statistics only)
  }
  if (MODE == MODE_BATCH && a.n_dst > 1) mark_stats(a, ms, lane, from_top);
  if (MODE == MODE_BATCH && a.n_dst > 1) mark_exit(a, lane);
}



// ========================================================================================================
// Pair kernel: ONE PROBLEM PER LANE PAIR (even lane = left hand, odd lane = right hand).  Each lane walks its
// own hand's chain, factors its own 6x6 block and solves its two right-hand sides; the pair meets in three
// warp shuffles per iteration (the two Sherman-Morrison scalars and the residual).  Per-warp instruction count per
// iteration is about half of the lane kernel's, so this is the kernel for batches too small to give every lane of
// the machine its own problem (path.py edge projection: 4096 chains; the single-solve drop-in) -- there the cost
// is the latency of one chain-iteration, not lane occupancy -- and for every fp64 batch (half the live state per
// lane).  Same operations on the same values as the lane kernel.  Arm constants are lane dependent (hand = lane & 1):
// register-resident in the latency-bound instantiations, lane-indexed constant loads in the large-batch fp64 one
// (HOIST below).
// ========================================================================================================
// Resident blocks per SM:
//   fp32: 3 -- 165 registers: the hand's constants live in registers (HOIST below).  Measured against the 96-register
//     build with lane-indexed constant loads: config 4 40.1 -> 32.0 ms, 16 Ki problems 1.33 -> 1.02 ms, 2 Ki problems
//     0.89 -> 0.67 ms (the same code capped at 96 registers: 44.5 ms).
//   fp64: 3 -- 168 registers, 12 warps / SM.  With the constant-bank sincos / atan2 the loop is bound by its FP64-pipe
//     instruction count, not by latency: 8, 9, 10, 11, 12 warps / SM all measure 9.2-9.5 M solves/s (2^20 problems),
//     14 and 16 warps (144 / 128 registers + spills) 9.1 / 8.9 M.
//   fp64, spherical-wrist step: 4 (large batches).
//   fp64 HOIST: 1 -- launches of <= kF64HoistWarps warps per SM only: registers are free (252 used, two blocks per SM).
template <typename T, bool HOIST, bool WRIST> struct LaunchPair;
template <bool HOIST, bool WRIST> struct LaunchPair<float, HOIST, WRIST>  { static constexpr int kMinBlocks = 3; };
template <> struct LaunchPair<double, false, false> { static constexpr int kMinBlocks = 3; };
template <> struct LaunchPair<double, false, true> { static constexpr int kMinBlocks = 4; };
template <bool WRIST> struct LaunchPair<double, true, WRIST>  { static constexpr int kMinBlocks = 1; };
// warps per SM (= its two resident blocks) up to which an fp64 launch takes the register-resident instantiation:
// 12 Ki / 18 Ki problems 2.64 -> 2.47 ms against the 168-register one
constexpr int kF64HoistWarps = 8;

// HOIST: the hand's constants are selected into registers once instead of being fetched by lane-indexed constant loads
// (39 LDC + their scoreboard waits per iteration), and the tip joint's constant outer product then comes from the table
// as in the lane kernels.  fp32: always (this kernel only serves batches too small to fill the machine -- edge chains,
// single solves -- where the time is the LATENCY of one chain and registers are free).  fp64: only for launches that fit
// its two resident blocks per SM (<= 8 warps per SM); the large-batch fp64 kernel is bound by the FP64 pipe at 168 registers and keeps
// the constant loads.
template <typename T, int MODE, uint32_t TZ, bool HOIST = (sizeof(T) == 4), bool WRIST = false>
__global__ void __launch_bounds__(kThreads, (LaunchPair<T, HOIST, WRIST>::kMinBlocks))
gik_solve_pair_kernel(const __grid_constant__ DevTable<T> tab, const __grid_constant__ SolveArgs<T> a) {
  const int lane = threadIdx.x & 31;
  const int h = lane & 1;                       // hand of this lane
  const int off = 1 + 6 * h;                    // first active-joint slot of this hand's arm
  const unsigned lower_pairs = (1u << (lane & ~1)) - 1u;
  const int64_t n = a.n_sel ? min(a.n, (int64_t)*a.n_sel) : a.n;
  if (MODE == MODE_BATCH && a.n_dst > 1 && (int)blockIdx.x < a.push_blocks) {   // fused all-gather: the leading blocks push, the others solve
    pusher_loop(a, tab.nq, n);
    return;
  }
  const bool from_top = MODE == MODE_BATCH && a.top_from > 0 && warp_slot() >= a.top_from;   // (see queue_take)
  if (from_top) mark_skip(a, threadIdx.x & 31);     // works outside the prefix: nothing to hold back
  const bool enabled = (lane >> 1) < a.lanes;   // a.lanes = pairs per warp (1..16)
  ArmConst<T> acr;
  T lim_lo[7], lim_hi[7];
  if constexpr (HOIST) {
    const ArmConst<T>&L = tab.arm[0], &R = tab.arm[1];
#pragma unroll
    for (int k = 0; k < 7; ++k)
#pragma unroll
      for (int i = 0; i < 3; ++i) acr.t[k][i] = h ? R.t[k][i] : L.t[k][i];
#pragma unroll
    for (int i = 0; i < 9; ++i) acr.finv_R[i] = h ? R.finv_R[i] : L.finv_R[i];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      acr.finv_p[i] = h ? R.finv_p[i] : L.finv_p[i]; acr.tip_lin[i] = h ? R.tip_lin[i] : L.tip_lin[i];
      acr.rw[i] = h ? R.rw[i] : L.rw[i];
    }
    acr.tip_psi = h ? R.tip_psi : L.tip_psi;
#pragma unroll
    for (int i = 0; i < 21; ++i) acr.g6[i] = h ? R.g6[i] : L.g6[i];      // read by the fp32 instantiation only
    lim_lo[0] = tab.lo[0]; lim_hi[0] = tab.hi[0];
#pragma unroll
    for (int k = 0; k < 6; ++k) { lim_lo[1 + k] = h ? tab.lo[7 + k] : tab.lo[1 + k]; lim_hi[1 + k] = h ? tab.hi[7 + k] : tab.hi[1 + k]; }
  }
  const ArmConst<T>& ac = tab.arm[h];           // rare paths (hook targets at a refill / edge step) and fp64
  const ArmConst<T>& acl = HOIST ? acr : tab.arm[h];   // descent loop

  T q[7], tgt[12];                              // q[0] = chest (kept by both lanes), q[1..6] = this hand's arm
#pragma unroll
  for (int i = 0; i < 7; ++i) q[i] = T(0);
#pragma unroll
  for (int c = 0; c < 12; ++c) tgt[c] = (c % 4 == 0 && c < 9) ? T(1) : T(0);
  auto load_q = [&](int64_t idx) {
    q[0] = ld_in(a.q_init + (int64_t)tab.act_q[0] * a.q_sc + idx * a.q_si);
#pragma unroll
    for (int k = 0; k < 6; ++k) q[1 + k] = ld_in(a.q_init + (int64_t)tab.act_q[off + k] * a.q_sc + idx * a.q_si);
  };
  auto store_q = [&](T* dst, int64_t sc, int64_t si, int64_t col) {   // this hand's arm; the chest from the even lane
#pragma unroll
    for (int k = 0; k < 6; ++k) dst[(int64_t)tab.act_q[off + k] * sc + col * si] = q[1 + k];
    if (h == 0) dst[(int64_t)tab.act_q[0] * sc + col * si] = q[0];
  };

  Work<T> w;
  bool exhausted = false;
  MarkState ms;              // fused all-gather: this warp's low-water mark

  // `refill` (warp-uniform): some lane pair finished a problem in the previous trip (or the loop is starting), so the
  // queue / exit logic has to run.  GATED (the throughput-bound fp64 instantiation): while it is false -- almost every
  // trip -- the loop is the iteration, one vote and the back edge (measured +1.8 % on 2^20 fp64 problems).  The
  // latency-bound instantiations run the queue check every trip: gating it measured 6 % SLOWER on config 4 (30.0 ->
  // 31.8 ms; code layout of a 11 KB loop running from the instruction cache with one warp per sub-partition).
  // INNER (the latency-bound instantiations): the iteration repeats in a loop of its own until an active pair finishes
  // -- its trip is the arithmetic, one vote and the back edge; the queue / store logic above and below runs only then.
  // Stall samples of the single-loop form put 14 % of a lone chain's time on its four branches per trip
  // (branch_resolving + instruction fetch at the targets).  Measured against the single-loop form: config 4 29.97 ->
  // 27.12 ms, 2 Ki fp32 problems 0.64 -> 0.58 ms, 16 Ki 1.00 -> 0.93 ms, fp64 small batches unchanged.  [The same idea
  // as a FLAG in the single loop measured slower, 30.0 -> 31.8 ms.]
  constexpr bool GATED = !HOIST;
  constexpr bool INNER = HOIST;
  const T dt = a.dt, eps2 = a.eps2, lambda = a.lambda;
  const int max_iters = a.max_iters;
  bool refill = true;
  for (;;) {
    const unsigned need = ((GATED && !refill) || exhausted) ? 0u : (__ballot_sync(0xffffffffu, enabled && !w.active) & 0x55555555u);
    bool again = false;
    if (need) {
      const int64_t cand = queue_take(a, n, need, lane, __popc(need & lower_pairs), from_top, exhausted);
      if (enabled && !w.active && cand >= 0) {
        T cube[12];
        work_start<T, MODE>(a, cand, h == 0, w, load_q, cube);
        hook_target(ac, cube, tgt);
      }
      // an edge with nothing to march leaves its pair idle although the queue has more: come back next trip
      if (GATED && MODE == MODE_EDGES) again = !exhausted && __any_sync(0xffffffffu, enabled && !w.active);
    }
    if constexpr (INNER) {
      if (!__any_sync(0xffffffffu, w.active)) {
        if (exhausted) break;
        continue;                                // (edges with nothing to march) back to the queue
      }
    } else {
      if ((!GATED || refill) && exhausted && !__any_sync(0xffffffffu, w.active)) break;
    }

    // ---------------- one descent iteration: this lane's hand ----------------
    bool ok, done;
    T r;
    for (;;) {
      T cs[kActive], sn[kActive], Sy, Sz, dqa[6];
      HandState<T> hs;
      WristState<T> wst;
#pragma unroll
      for (int i = 0; i < 7; ++i)        // (tip-aligned wrist step: the tip slot carries q6 - tip_psi, hand_wrist_phase1)
        sincos_<true>((WRIST && (TZ & kTipZ) && i == 6) ? q[i] - acl.tip_psi : q[i], sn[i], cs[i]);
      // (fp64 keeps the tip products in the Gram matrix: bit-identical to the fp64 lane kernel)
      if constexpr (WRIST) hand_wrist_phase1<T, 0, TZ>(acl, cs, sn, tgt, wst, Sy, Sz, r);
      else hand_phase1<T, 0, TZ, (HOIST && sizeof(T) == 4)>(acl, cs, sn, tgt, lambda, hs, Sy, Sz, r);
      const T Sy_o = __shfl_xor_sync(0xffffffffu, Sy, 1), Sz_o = __shfl_xor_sync(0xffffffffu, Sz, 1);
      const T r_o = __shfl_xor_sync(0xffffffffu, r, 1);
      const T kappa = h ? chest_rate(Sy_o, Sz_o, Sy, Sz) : chest_rate(Sy, Sz, Sy_o, Sz_o);
      if constexpr (WRIST) hand_wrist_phase2(wst, kappa, dqa);
      else hand_phase2(hs, kappa, dqa);
      const T rL = h ? r_o : r, rR = h ? r : r_o;
      ok = (rL < eps2) && (rR < eps2) && (w.it < max_iters);
      bool stalled = false;
      if (a.early_stop && (w.it & 63) == 63) {
        const T rs = rL + rR;
        stalled = rs > T(0.9) * w.r_mark;
        w.r_mark = rs;
      }
      done = ok || (w.it >= max_iters) || stalled;
      if constexpr (GATED) refill = __any_sync(0xffffffffu, done && w.active) || again;
      if (!done) {
        if constexpr (HOIST) {
          q[0] = min_(max_(lim_lo[0], q[0] + dt * kappa), lim_hi[0]);
#pragma unroll
          for (int k = 0; k < 6; ++k) q[1 + k] = min_(max_(lim_lo[1 + k], q[1 + k] + dt * dqa[k]), lim_hi[1 + k]);
        } else {
          q[0] = min_(max_(tab.lo[0], q[0] + dt * kappa), tab.hi[0]);
#pragma unroll
          for (int k = 0; k < 6; ++k)
            q[1 + k] = min_(max_(tab.lo[off + k], q[1 + k] + dt * dqa[k]), tab.hi[off + k]);
        }
        ++w.it;
      }
      if (!INNER) break;
      if (__any_sync(0xffffffffu, done && w.active)) break;
    }
    const bool fused_event = MODE == MODE_BATCH && a.n_dst > 1 && __any_sync(0xffffffffu, done && w.active);
    if (fused_event && !from_top) mark_publish(a, ms, lane);
    if (done && w.active) {
      T cube[12];
      if (MODE == MODE_BATCH) {
        const T rh[1] = {r};
        batch_finish(tab, a, w, ok, h == 0, store_q, h, rh);
      } else if (edge_step_end(tab, a, w, ok, h == 0, store_q, cube)) {
        hook_target(ac, cube, tgt);
      }
    }
    if (fused_event) mark_update(ms, w.active, w.idx);      // (from_top warps: statistics only)
  }
  if (MODE == MODE_BATCH && a.n_dst > 1) mark_exit(a, lane);
}

// ---------------- K1 / K2: forward kinematics and LOCAL frame Jacobians (parity entries) ----------------
template <typename T>
__global__ void __launch_bounds__(128) gik_fk_kernel(const __grid_constant__ DevTable<T> tab, int64_t n,
                                                     const T* __restrict__ q, T* __restrict__ frames) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    T qa[kActive], fr[2][12];
#pragma unroll
    for (int k = 0; k < kActive; ++k) qa[k] = q[(int64_t)tab.act_q[k] * n + i];
    fk_frames<T, true>(tab, qa, fr);
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
      for (int c = 0; c < 12; ++c) frames[((int64_t)h * 12 + c) * n + i] = fr[h][c];
  }
}

template <typename T>
__global__ void __launch_bounds__(128) gik_jac_kernel(const __grid_constant__ DevTable<T> tab, int64_t n,
                                                      const T* __restrict__ q, T* __restrict__ jac) {
  const int nq = tab.nq;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    T qa[kActive], AL[6][7], AR[6][7];
#pragma unroll
    for (int k = 0; k < kActive; ++k) qa[k] = q[(int64_t)tab.act_q[k] * n + i];
    frame_jacobians<T, true>(tab, qa, AL, AR);
    for (int r = 0; r < 12 * nq; ++r) jac[(int64_t)r * n + i] = T(0);
#pragma unroll
    for (int r = 0; r < 6; ++r)
#pragma unroll
      for (int k = 0; k < 7; ++k) {
        jac[((int64_t)r * nq + tab.act_q[k == 0 ? 0 : k]) * n + i] = AL[r][k];
        jac[((int64_t)(6 + r) * nq + tab.act_q[k == 0 ? 0 : 6 + k]) * n + i] = AR[r][k];
      }
  }
}

// ---------------- K4: best-of-restarts, one warp per placement ----------------
template <typename T>
__global__ void __launch_bounds__(128) gik_best_of_kernel(int nq, int64_t n_place, int n_restart,
                                                          const T* __restrict__ q,
                                                          const uint8_t* __restrict__ conv,
                                                          const T* __restrict__ resid, T* __restrict__ q_best,
                                                          uint8_t* __restrict__ conv_best,
                                                          int32_t* __restrict__ which) {
  const int lane = threadIdx.x & 31;
  const int64_t n = n_place * n_restart;
  for (int64_t p = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; p < n_place;
       p += ((int64_t)gridDim.x * blockDim.x) >> 5) {
    // key: (not converged, max residual, restart index) -- lexicographic minimum
    int best_r = -1; int best_nc = 2; T best_m = T(0);
    for (int r = lane; r < n_restart; r += 32) {
      const int64_t i = p * n_restart + r;
      const int nc = conv[i] ? 0 : 1;
      T m = max_(resid[i], resid[n + i]);
      if (!(m == m)) m = T(INFINITY);  // NaN residual ranks last
      if (best_r < 0 || nc < best_nc || (nc == best_nc && m < best_m)) { best_r = r; best_nc = nc; best_m = m; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const int orr = __shfl_xor_sync(0xffffffffu, best_r, o);
      const int onc = __shfl_xor_sync(0xffffffffu, best_nc, o);
      const T om = __shfl_xor_sync(0xffffffffu, best_m, o);
      const bool take = orr >= 0 && (best_r < 0 || onc < best_nc ||
                                     (onc == best_nc && (om < best_m || (om == best_m && orr < best_r))));
      if (take) { best_r = orr; best_nc = onc; best_m = om; }
    }
    const int64_t src = p * n_restart + best_r;
    for (int j = lane; j < nq; j += 32) q_best[(int64_t)j * n_place + p] = q[(int64_t)j * n + src];
    if (lane == 0) {
      conv_best[p] = best_nc == 0 ? 1 : 0;
      if (which) which[p] = best_r;
    }
  }
}

// ---------------- FMA roofline microbenchmark: 8 independent register-resident chains per thread ----------
template <typename T>
__global__ void __launch_bounds__(256) gik_fma_peak_kernel(T* out, int iters, T a, T b) {
  T x0 = T(threadIdx.x) * T(1e-3), x1 = x0 + T(1), x2 = x0 + T(2), x3 = x0 + T(3);
  T x4 = x0 + T(4), x5 = x0 + T(5), x6 = x0 + T(6), x7 = x0 + T(7);
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int u = 0; u < 16; ++u) {
      x0 = x0 * a + b; x1 = x1 * a + b; x2 = x2 * a + b; x3 = x3 * a + b;
      x4 = x4 * a + b; x5 = x5 * a + b; x6 = x6 * a + b; x7 = x7 * a + b;
    }
  }
  const T s = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
  if (s == T(123456789)) out[0] = s;  // never true; keeps the chains alive
}

}  // namespace gik

// ========================================================================================================
// C ABI
// ========================================================================================================
using namespace gik;

struct gik_handle_s {
  uint32_t magic;
  int device;
  int sm_count;
  gik_table_t host;
  DevTable<float> tab32;
  PackedTable pt32;                  // (left, right)-packed constants of tab32 for the fp32 packed lane kernel
  DevTable<double> tab64;
  struct gik_scene_dev* scene;       // collision scene (gik_scene_attach), or null
  unsigned long long* queues;        // device: kQueueSlots work-queue heads, one per launch in flight
  std::atomic<uint32_t> next_queue;
};
static constexpr uint32_t kQueueSlots = 1024;   // launches that may be in flight on one handle at once
static constexpr uint32_t kMagic = 0x67696b31u;  // "gik1"
static void gik_free_scene_of(gik_handle_s* h);

namespace {

struct DeviceGuard {
  int prev = -1;
  cudaError_t err;
  explicit DeviceGuard(int dev) {
    err = cudaGetDevice(&prev);
    if (err == cudaSuccess && prev != dev) err = cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    int cur = -1;
    if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
  }
};

inline bool bad_handle(gik_handle_t h) { return h == nullptr || h->magic != kMagic; }

inline int check_params(const gik_params_t* p) {
  if (!p) return GIK_E_NULL;
  if (!(p->eps > 0.0) || !(p->dt > 0.0) || !(p->damping >= 0.0) || p->max_iters < 0 ||
      (p->flags & ~(GIK_F_LANE_KERNEL | GIK_F_PAIR_KERNEL | GIK_F_SCALAR_LANE | GIK_F_EARLY_STOP | GIK_F_CHOLESKY | GIK_F_NO_DESCEND)) != 0 ||
      (p->flags & (GIK_F_LANE_KERNEL | GIK_F_PAIR_KERNEL)) == (GIK_F_LANE_KERNEL | GIK_F_PAIR_KERNEL))
    return GIK_E_PARAM;
  return GIK_OK;
}

template <typename T> const DevTable<T>& table_of(gik_handle_t h);
template <> const DevTable<float>& table_of<float>(gik_handle_t h) { return h->tab32; }
template <> const DevTable<double>& table_of<double>(gik_handle_t h) { return h->tab64; }

// Grid for the persistent solvers: resident blocks per SM x SM count, shrunk for small batches.  `per_warp` = problems
// a warp keeps in flight (lane kernels: up to 32 lanes; pair kernel: up to 16 lane pairs).  One warp instruction costs
// the same issue slot whether 1 or 32 lanes are live, so warps are FILLED first and the batch is spread over more
// (emptier) warps only as far as it takes to give every SM sub-partition one warp: measured on 4096 edge chains,
// 7 pairs per warp (586 warps) 40.6 ms against 69.6 ms for 2 pairs per warp (2048 warps); on a 16 Ki batch 1.34 ms at
// 16 pairs per warp against 2.70 ms when spread over every resident warp slot.
template <typename Kernel>
int grid_dims(gik_handle_t h, Kernel kernel, int64_t n, int max_per_warp, int* blocks, int* per_warp, int64_t* max_warps_out,
              int reserve = 0) {   // reserve: resident block slots kept free (the pusher block of a fused launch)
  int occ = 0;
  cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, kThreads, 0);
  if (e != cudaSuccess) return (int)e;
  if (occ < 1) occ = 1;
  const int64_t warps_per_block = kThreads / 32;
  const int64_t max_blocks = (int64_t)h->sm_count * occ - reserve;
  const int64_t max_warps = max_blocks * warps_per_block;
  const int64_t target_warps = (int64_t)h->sm_count * 4;      // one warp per SM sub-partition
  int64_t Lw = (n + target_warps - 1) / target_warps;
  int L = (int)(Lw < 1 ? 1 : (Lw > max_per_warp ? max_per_warp : Lw));
  int64_t warps = (n + L - 1) / L;
  int64_t b = (warps + warps_per_block - 1) / warps_per_block;
  if (b > max_blocks) b = max_blocks;
  if (b < 1) b = 1;
  *blocks = (int)b;
  *per_warp = L;
  if (max_warps_out) *max_warps_out = max_warps;
  return GIK_OK;
}

// Which form of the step a launch runs: the spherical-wrist form (two 3x3 solves per hand) needs an undamped step and
// a table with the wrist's zero pattern (instantiated for the Nextage pattern); everything else -- damping > 0, other
// tables of the compiled topology, GIK_F_CHOLESKY -- takes the block Cholesky + Sherman-Morrison form.
template <typename T>
bool use_wrist(gik_handle_t h, const gik_params_t* prm) {
  const DevTable<T>& tab = table_of<T>(h);
  return (tab.tzero & kNextageTZ) == kNextageTZ && prm->damping == 0.0 && !(prm->flags & GIK_F_CHOLESKY);
}

// The solve kernel instantiation one launch runs.  choose_launch picks it; the grid is sized, the kernel launched and
// its name reported from this one choice.
struct SolveKernel {
  enum Family { LANE, LANE2, PAIR } family;   // scalar lane kernel, packed fp32 lane kernel, pair kernel
  bool nx;      // TZ = kNextageTZ: the table has (at least) the Nextage zero pattern, so those FMAs are skipped
  bool wrist;   // WRIST: the spherical-wrist step (implies nx)
  bool hoist;   // pair kernel, HOIST: the hand's constants in registers (fp32: always)
};

// f(kernel) for the instantiation k names
template <typename T, int MODE, typename F>
int with_kernel(const SolveKernel& k, F&& f) {
  constexpr uint32_t NX = kNextageTZ;
  if (k.family == SolveKernel::PAIR) {
    if constexpr (sizeof(T) == 8) {
      if (!k.hoist) return k.wrist ? f(gik_solve_pair_kernel<T, MODE, NX, false, true>)
                           : k.nx  ? f(gik_solve_pair_kernel<T, MODE, NX, false>) : f(gik_solve_pair_kernel<T, MODE, 0, false>);
    }
    return k.wrist ? f(gik_solve_pair_kernel<T, MODE, NX, true, true>)
         : k.nx  ? f(gik_solve_pair_kernel<T, MODE, NX, true>) : f(gik_solve_pair_kernel<T, MODE, 0, true>);
  }
  if constexpr (sizeof(T) == 4) {
    if (k.family == SolveKernel::LANE2)
      return k.wrist ? f(gik_solve_lane2_kernel<MODE, NX, true>)
           : k.nx  ? f(gik_solve_lane2_kernel<MODE, NX>) : f(gik_solve_lane2_kernel<MODE, 0>);
  }
  return k.wrist ? f(gik_solve_kernel<T, MODE, NX, true>) : k.nx ? f(gik_solve_kernel<T, MODE, NX>) : f(gik_solve_kernel<T, MODE, 0>);
}

// fp32: lane kernel when the batch can give (at least) half of the lanes of every resident warp a problem, pair kernel
// below that.  fp64: always the pair kernel -- one hand per lane halves the live state, which at 2 registers per value
// is worth more than the shared chest work (measured 7.0M vs 6.0M solves/s on 2^20 problems).
// flags can force either (GIK_F_LANE_KERNEL / GIK_F_PAIR_KERNEL) for A/B measurements, and the scalar fp32 lane kernel
// (GIK_F_SCALAR_LANE).  `reserve`: resident block slots kept free (the pusher blocks of a fused launch).
template <typename T, int MODE>
int choose_launch(gik_handle_t h, int64_t n, int flags, bool wrist, int reserve, SolveKernel* k, int* blocks, int* per_warp) {
  const bool nx = (table_of<T>(h).tzero & kNextageTZ) == kNextageTZ;
  *k = {sizeof(T) == 4 && !(flags & GIK_F_SCALAR_LANE) ? SolveKernel::LANE2 : SolveKernel::LANE, nx, wrist, false};
  int64_t max_warps = 0;
  int rc = with_kernel<T, MODE>(*k, [&](auto kern) { return grid_dims(h, kern, n, 32, blocks, per_warp, &max_warps, reserve); });
  if (rc) return rc;
  bool pair = sizeof(T) == 8 || n <= 16 * max_warps;
  if (flags & GIK_F_LANE_KERNEL) pair = false;
  if (flags & GIK_F_PAIR_KERNEL) pair = true;
  if (!pair) return GIK_OK;
  k->family = SolveKernel::PAIR;
  // fp64 pair kernel with register-resident constants: launches of at most one full warp per SM sub-partition
  k->hoist = sizeof(T) == 4 || n <= (int64_t)16 * kF64HoistWarps * h->sm_count;
  return with_kernel<T, MODE>(*k, [&](auto kern) { return grid_dims(h, kern, n, 16, blocks, per_warp, nullptr, reserve); });
}

template <typename T>
void launch_kernel(void (*kern)(DevTable<T>, SolveArgs<T>), int blocks, cudaStream_t st, gik_handle_t h, const SolveArgs<T>& a) {
  kern<<<blocks, kThreads, 0, st>>>(table_of<T>(h), a);
}
void launch_kernel(void (*kern)(DevTable<float>, PackedTable, SolveArgs<float>), int blocks, cudaStream_t st, gik_handle_t h,
                   const SolveArgs<float>& a) {
  kern<<<blocks, kThreads, 0, st>>>(h->tab32, h->pt32, a);
}

// force: a continuation launch that must run every problem to the iteration cap -- eps^2 = 0 can never be undercut
template <typename T, int MODE>
int launch_solve(gik_handle_t h, SolveArgs<T>& a, const gik_params_t* prm, void* stream, bool force = false) {
  a.eps2 = force ? T(0) : (T)(prm->eps * prm->eps);
  a.dt = (T)prm->dt;
  a.lambda = (T)prm->damping;
  a.max_iters = prm->max_iters;
  a.early_stop = (prm->flags & GIK_F_EARLY_STOP) ? 1 : 0;
  DeviceGuard g(h->device);
  if (g.err != cudaSuccess) return (int)g.err;
  int blocks = 0, lanes = 32;
  SolveKernel k;
  const int pushers = (MODE == MODE_BATCH && a.n_dst > 1) ? a.push_blocks : 0;   // fused all-gather: the leading blocks push (see "Fused all-gather")
  int rc = choose_launch<T, MODE>(h, a.n, prm->flags, use_wrist<T>(h, prm), pushers, &k, &blocks, &lanes);
  if (rc) return rc;
  if (pushers) {
    a.n_marks = blocks * (kThreads / 32);
    // the warps in the upper half of the SM's occupied warp slots -- the low-priority ones -- work from the top of the slab
    // (queue_take); needs both counters in one 64-bit word and a device-resident batch handed out by index
    const bool two_ended = a.n < (1ll << 31) && !a.ready && !a.sel;
    const int per_sm = (blocks + pushers + h->sm_count - 1) / h->sm_count;     // blocks per SM of this launch
    a.top_from = (two_ended && per_sm >= 2) ? (per_sm + 1) / 2 * (kThreads / 32) : 0;
    blocks += pushers;
  }
  a.lanes = lanes;
  a.queue = h->queues + (h->next_queue.fetch_add(1, std::memory_order_relaxed) % kQueueSlots);
  cudaError_t qe = cudaMemsetAsync(a.queue, 0, sizeof(unsigned long long), (cudaStream_t)stream);
  if (qe != cudaSuccess) return (int)qe;
  return with_kernel<T, MODE>(k, [&](auto kern) {
    launch_kernel(kern, blocks, (cudaStream_t)stream, h, a);
    return (int)cudaGetLastError();
  });
}

// The launch gik_solve_f32/f64 makes for n problems with the default parameters and these flags (GIK_F_CHOLESKY selects
// the step form, the kernel flags the kernel)
int batch_launch(gik_handle_t h, int elem_size, int64_t n, int flags, SolveKernel* k, int* blocks) {
  DeviceGuard g(h->device);
  if (g.err != cudaSuccess) return (int)g.err;
  gik_params_t dp;
  gik_default_params(&dp);
  dp.flags = flags & GIK_F_CHOLESKY;
  int lanes = 0;
  if (elem_size == 4) return choose_launch<float, MODE_BATCH>(h, n, flags, use_wrist<float>(h, &dp), 0, k, blocks, &lanes);
  return choose_launch<double, MODE_BATCH>(h, n, flags, use_wrist<double>(h, &dp), 0, k, blocks, &lanes);
}

template <typename T>
void set_soa(SolveArgs<T>& a, int64_t n_in, int64_t n_out) {
  a.q_sc = n_in; a.q_si = 1; a.pose_sc = n_in; a.pose_si = 1;
  a.out_sc = n_out; a.out_si = 1; a.res_sc = n_in; a.res_si = 1;
  a.ready = nullptr;
}

// Row-major I/O with streamed input: q_init [n][nq] and pose [n][12] are DEVICE staging buffers being filled slab by
// slab by the copy engine while the kernel runs (`ready` = device counter of resident leading problems, advanced on
// the copy stream after each slab); q_out [n][nq], converged [n], iters [n], resid [n][2] may be PINNED HOST memory
// (UVA): the kernel's stores go straight over PCIe, so no D2H copy follows the kernel.
template <typename T>
int rows_api(gik_handle_t h, int64_t n, const T* q_init, const T* pose, const gik_params_t* prm, T* q_out, uint8_t* conv,
             int32_t* iters, T* resid, const unsigned long long* ready, void* stream) {
  if (bad_handle(h)) return GIK_E_HANDLE;
  if (n < 0) return GIK_E_SIZE;
  int rc = check_params(prm);
  if (rc) return rc;
  if (n == 0) return GIK_OK;
  if (!q_init || !pose || !q_out || !conv) return GIK_E_NULL;
  SolveArgs<T> a{};
  a.q_init = q_init; a.pose = pose; a.iters = iters; a.resid = resid;
  a.q_dst[0] = q_out; a.conv_dst[0] = conv; a.n_dst = 1; a.out_off = 0;
  a.n = n;
  const int nq = h->host.nq;
  a.q_sc = 1; a.q_si = nq; a.pose_sc = 1; a.pose_si = 12;
  a.out_sc = 1; a.out_si = nq; a.res_sc = 1; a.res_si = 2;
  a.ready = ready;
  return launch_solve<T, MODE_BATCH>(h, a, prm, stream);
}

template <typename T>
int solve_api(gik_handle_t h, int64_t n, const T* q_init, const T* pose, const gik_params_t* prm, T* q_out,
              uint8_t* conv, int32_t* iters, T* resid, void* stream) {
  if (bad_handle(h)) return GIK_E_HANDLE;
  if (n < 0) return GIK_E_SIZE;
  int rc = check_params(prm);
  if (rc) return rc;
  if (n == 0) return GIK_OK;
  if (!q_init || !pose || !q_out || !conv) return GIK_E_NULL;
  SolveArgs<T> a{};
  a.q_init = q_init; a.pose = pose; a.iters = iters; a.resid = resid;
  a.q_dst[0] = q_out; a.conv_dst[0] = conv; a.n_dst = 1; a.out_off = 0;
  a.n = n;
  set_soa(a, n, n);
  return launch_solve<T, MODE_BATCH>(h, a, prm, stream);
}

template <typename T>
int scatter_api(gik_handle_t h, int64_t n, const T* q_init, const T* pose, const gik_params_t* prm, int32_t n_peers,
                T* const* q_all, uint8_t* const* conv_all, int64_t n_total, int64_t offset, int32_t* iters, T* resid,
                void* stream) {
  if (bad_handle(h)) return GIK_E_HANDLE;
  if (n < 0 || n_peers < 1 || n_peers > GIK_MAX_PEERS || offset < 0 || n_total < 0 || offset + n > n_total) return GIK_E_SIZE;
  int rc = check_params(prm);
  if (rc) return rc;
  if (n == 0) return GIK_OK;
  if (!q_init || !pose || !q_all || !conv_all) return GIK_E_NULL;
  for (int p = 0; p < n_peers; ++p)
    if (!q_all[p] || !conv_all[p]) return GIK_E_NULL;
  DeviceGuard g(h->device);
  if (g.err != cudaSuccess) return (int)g.err;
  // The lanes store into ONE array -- this rank's own, i.e. the one whose memory lives on this device -- and the chunk
  // pushes copy from it into the others.  (All on this device, as in the single-GPU test: the first one.)
  int self = 0;
  for (int p = 0; p < n_peers; ++p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, q_all[p]) == cudaSuccess && at.type == cudaMemoryTypeDevice && at.device == h->device) { self = p; break; }
  }
  (void)cudaGetLastError();
  SolveArgs<T> a{};
  a.q_init = q_init; a.pose = pose; a.iters = iters; a.resid = resid;
  a.q_dst[0] = q_all[self]; a.conv_dst[0] = conv_all[self];
  for (int p = 0, k = 1; p < n_peers; ++p)
    if (p != self) { a.q_dst[k] = q_all[p]; a.conv_dst[k] = conv_all[p]; ++k; }
  a.n_dst = n_peers; a.out_off = offset;
  a.n = n;
  set_soa(a, n, n_total);
  cudaStream_t st = (cudaStream_t)stream;
  if (n_peers == 1) return launch_solve<T, MODE_BATCH>(h, a, prm, stream);
  // scratch: marks (one per warp of the largest grid any solve kernel takes; zero = "nothing finished yet"), the pushers'
  // control words + statistics, one flag per chunk
  const int64_t n_chunks = (n + kChunk - 1) / kChunk;
  const int64_t n_marks = (int64_t)h->sm_count * 16 * (kThreads / 32);
  const size_t marks_bytes = ((size_t)n_marks * sizeof(int32_t) + 255) / 256 * 256, ctl_bytes = 2048;
  char* scratch = nullptr;
  cudaError_t e = cudaMallocAsync((void**)&scratch, marks_bytes + ctl_bytes + (size_t)n_chunks, st);
  if (e == cudaSuccess) e = cudaMemsetAsync(scratch, 0, marks_bytes + ctl_bytes + (size_t)n_chunks, st);
  if (e != cudaSuccess) return (int)e;
  a.marks = (int32_t*)scratch;
  a.push_ctl = (long long*)(scratch + marks_bytes);
  a.pushed = (uint8_t*)(scratch + marks_bytes + ctl_bytes);
  if (getenv("GIK_FUSED_STATS")) a.warp_stats = a.marks + n_marks / 2;   // (second half of the marks allocation: grids here use <= 1/4 of it)
  // pusher blocks: one (a lookout + three pushing warps) keeps pace with one or two destinations; more destinations
  // mean more stores per chunk
  a.push_blocks = n_peers <= 3 ? 1 : 2;
  const bool stats = getenv("GIK_FUSED_STATS") != nullptr;     // measurement hook (synchronises the stream)
  cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
  if (stats) {
    for (auto& x : ev) cudaEventCreate(&x);
    cudaEventRecord(ev[0], st);
  }
  rc = launch_solve<T, MODE_BATCH>(h, a, prm, stream);
  if (stats) cudaEventRecord(ev[1], st);
  if (rc == GIK_OK) {
    gik_push_rest_kernel<T><<<h->sm_count * 4, 128, 0, st>>>(a, h->host.nq, stats ? 2 : 0);
    rc = (int)cudaGetLastError();
  }
  if (stats) {
    cudaEventRecord(ev[2], st);
    uint8_t* hp = (uint8_t*)malloc((size_t)n_chunks);
    if (hp && cudaMemcpyAsync(hp, a.pushed, (size_t)n_chunks, cudaMemcpyDeviceToHost, st) == cudaSuccess &&
        cudaStreamSynchronize(st) == cudaSuccess) {
      int64_t k = 0, r = 0;
      for (int64_t c = 0; c < n_chunks; ++c) { k += hp[c] == 1; r += hp[c] == 2; }
      float t_solve = 0.f, t_rest = 0.f;
      cudaEventElapsedTime(&t_solve, ev[0], ev[1]);
      cudaEventElapsedTime(&t_rest, ev[1], ev[2]);
      fprintf(stderr, "gik fused all-gather: %lld of %lld chunks pushed inside the solve kernel (%.3f ms incl. memset), %lld by the tail kernel (%.3f ms)\n",
              (long long)k, (long long)n_chunks, t_solve, (long long)r, t_rest);
      long long pw[28];
      if (a.n_marks > 0 && cudaMemcpy(pw, a.push_ctl, sizeof(pw), cudaMemcpyDeviceToHost) == cudaSuccess)
        for (int w = 0; w < 8 && w < a.push_blocks * (kThreads / 32); ++w)
          fprintf(stderr, w == 0 ? "  lookout warp: %lld looks, looking %lld us, sleeping %lld us\n" : "  pusher warp: %lld chunks, pushing %lld us, waiting %lld us\n",
                  pw[4 + 3 * w + 2], pw[4 + 3 * w], pw[4 + 3 * w + 1]);
      if (a.warp_stats && a.n_marks > 0 && 2 * a.n_marks <= n_marks / 2) {
        int32_t* ws = (int32_t*)malloc(sizeof(int32_t) * 2 * a.n_marks);
        if (ws && cudaMemcpy(ws, a.warp_stats, sizeof(int32_t) * 2 * a.n_marks, cudaMemcpyDeviceToHost) == cudaSuccess) {
          int lo = 1 << 30, hi = 0, hist[8] = {0, 0, 0, 0, 0, 0, 0, 0};
          long long sum = 0;
          for (int w = 0; w < a.n_marks; ++w) { const int v = ws[2 * w]; lo = v < lo ? v : lo; hi = v > hi ? v : hi; sum += v; }
          for (int w = 0; w < a.n_marks; ++w) ++hist[hi > lo ? (int)((long long)(ws[2 * w] - lo) * 7 / (hi - lo)) : 0];
          fprintf(stderr, "  finish events per compute warp: min %d, mean %.1f, max %d; histogram over [min, max] in 8 bins:", lo, (double)sum / a.n_marks, hi);
          for (int b = 0; b < 8; ++b) fprintf(stderr, " %d", hist[b]);
          fprintf(stderr, "\n  by sub-partition slot (warp index in block), mean events:");
          for (int k = 0; k < kThreads / 32; ++k) {
            long long sk = 0; int nk = 0;
            for (int w = k; w < a.n_marks; w += kThreads / 32) { sk += ws[2 * w]; ++nk; }
            fprintf(stderr, " %.1f", nk ? (double)sk / nk : 0.0);
          }
          fprintf(stderr, "\n  by launch order of the block (quarters of the compute grid), mean events:");
          for (int qd = 0; qd < 4; ++qd) {
            long long sk = 0; int nk = 0;
            for (int w = a.n_marks * qd / 4; w < a.n_marks * (qd + 1) / 4; ++w) { sk += ws[2 * w]; ++nk; }
            fprintf(stderr, " %.1f", nk ? (double)sk / nk : 0.0);
          }
          {
            long long sb = 0, st2 = 0; int nb = 0, nt = 0, minb = 1 << 30;
            for (int w = 0; w < a.n_marks; ++w) {
              if (ws[2 * w + 1] & 1) { st2 += ws[2 * w]; ++nt; } else { sb += ws[2 * w]; ++nb; if (ws[2 * w] < minb) minb = ws[2 * w]; }
            }
            fprintf(stderr, "\n  warps working from the bottom: %d, mean events %.1f, min %d; from the top: %d, mean events %.1f", nb,
                    nb ? (double)sb / nb : 0.0, nb ? minb : 0, nt, nt ? (double)st2 / nt : 0.0);
          }
          fprintf(stderr, "\n  by %%warpid, mean events [warps]:");
          for (int id = 0; id < 64; ++id) {
            long long sk = 0; int nk = 0;
            for (int w = 0; w < a.n_marks; ++w) if ((ws[2 * w + 1] >> 8) == id) { sk += ws[2 * w]; ++nk; }
            if (nk) fprintf(stderr, " %d:%.0f[%d]", id, (double)sk / nk, nk);
          }
          fprintf(stderr, "\n  first 16 warps (events):");
          for (int w = 0; w < 16 && w < a.n_marks; ++w) fprintf(stderr, " %d", ws[2 * w]);
          fprintf(stderr, "\n");
        }
        free(ws);
      }
      long long tr[180];
      if (a.n_marks > 0 && getenv("GIK_FUSED_TRACE") && cudaMemcpy(tr, a.push_ctl + 32, sizeof(tr), cudaMemcpyDeviceToHost) == cudaSuccess)
        for (int k = 0; k < 60 && tr[3 * k]; ++k)
          fprintf(stderr, "  t %lld us: F %lld, queue head (bottom end) %lld, smallest mark held by compute warp %lld\n", tr[3 * k] - tr[0],
                  tr[3 * k + 1], tr[3 * k + 2] & 0xffffffffffll, tr[3 * k + 2] >> 40);
    }
    free(hp);
    for (auto& x : ev) cudaEventDestroy(x);
  }
  e = cudaFreeAsync(scratch, st);
  if (rc == GIK_OK && e != cudaSuccess) rc = (int)e;
  return rc;
}

template <typename T>
int edges_api(gik_handle_t h, int64_t n, int32_t max_steps, const T* q_start, const T* pose_a, const T* pose_b,
              const int32_t* num_steps, const gik_params_t* prm, T* q_path, int32_t* n_valid,
              int32_t* iters_total, void* stream) {
  if (bad_handle(h)) return GIK_E_HANDLE;
  if (n < 0 || max_steps < 0) return GIK_E_SIZE;
  int rc = check_params(prm);
  if (rc) return rc;
  if (n == 0) return GIK_OK;
  if (!q_start || !pose_a || !pose_b || !num_steps || !q_path || !n_valid) return GIK_E_NULL;
  SolveArgs<T> a{};
  a.q_init = q_start; a.pose = pose_a; a.pose_b = pose_b; a.num_steps = num_steps; a.q_out = q_path;
  a.n_valid = n_valid; a.iters = iters_total; a.max_steps = max_steps; a.n = n;
  set_soa(a, n, n);
  return launch_solve<T, MODE_EDGES>(h, a, prm, stream);
}

template <typename T>
int fk_api(gik_handle_t h, int64_t n, const T* q, T* frames, void* stream, bool jac) {
  if (bad_handle(h)) return GIK_E_HANDLE;
  if (n < 0) return GIK_E_SIZE;
  if (n == 0) return GIK_OK;
  if (!q || !frames) return GIK_E_NULL;
  DeviceGuard g(h->device);
  if (g.err != cudaSuccess) return (int)g.err;
  int64_t blocks = (n + 127) / 128;
  if (blocks > (int64_t)h->sm_count * 16) blocks = (int64_t)h->sm_count * 16;
  if (jac) gik_jac_kernel<T><<<(int)blocks, 128, 0, (cudaStream_t)stream>>>(table_of<T>(h), n, q, frames);
  else gik_fk_kernel<T><<<(int)blocks, 128, 0, (cudaStream_t)stream>>>(table_of<T>(h), n, q, frames);
  return (int)cudaGetLastError();
}

template <typename T>
int best_of_api(gik_handle_t h, int64_t n_place, int32_t n_restart, const T* q, const uint8_t* conv,
                const T* resid, T* q_best, uint8_t* conv_best, int32_t* which, void* stream) {
  if (bad_handle(h)) return GIK_E_HANDLE;
  if (n_place < 0 || n_restart < 1) return GIK_E_SIZE;
  if (n_place == 0) return GIK_OK;
  if (!q || !conv || !resid || !q_best || !conv_best) return GIK_E_NULL;
  DeviceGuard g(h->device);
  if (g.err != cudaSuccess) return (int)g.err;
  int64_t blocks = (n_place + 3) / 4;
  if (blocks > (int64_t)h->sm_count * 16) blocks = (int64_t)h->sm_count * 16;
  gik_best_of_kernel<T><<<(int)blocks, 128, 0, (cudaStream_t)stream>>>(h->host.nq, n_place, n_restart, q, conv,
                                                                       resid, q_best, conv_best, which);
  return (int)cudaGetLastError();
}

template <typename T>
int fma_peak(int device, int repeats, double* tflops) {
  DeviceGuard g(device);
  if (g.err != cudaSuccess) return (int)g.err;
  cudaDeviceProp prop;
  cudaError_t e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) return (int)e;
  T* out = nullptr;
  if ((e = cudaMalloc(&out, sizeof(T))) != cudaSuccess) return (int)e;
  const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  double best = 0.0;
  for (int r = 0; r < repeats + 1; ++r) {
    cudaEventRecord(e0);
    gik_fma_peak_kernel<T><<<blocks, threads>>>(out, iters, (T)0.999, (T)0.001);
    cudaEventRecord(e1);
    if ((e = cudaEventSynchronize(e1)) != cudaSuccess) break;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    const double flops = 2.0 * 8 * 16 * (double)iters * blocks * threads;
    if (r > 0 && ms > 0.f && flops / (ms * 1e-3) > best) best = flops / (ms * 1e-3);
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(out);
  if (e != cudaSuccess) return (int)e;
  *tflops = best * 1e-12;
  return GIK_OK;
}

}  // namespace

extern "C" {

void gik_default_params(gik_params_t* p) {
  if (!p) return;
  p->eps = 1e-3; p->dt = 1e-2; p->damping = 0.0; p->max_iters = 1000; p->flags = 0;
}

int gik_create(const gik_table_t* host_table, int device, gik_handle_t* out) {
  if (!host_table || !out) return GIK_E_NULL;
  *out = nullptr;
  gik_handle_s* h = new (std::nothrow) gik_handle_s();
  if (!h) return (int)cudaErrorMemoryAllocation;
  h->host = *host_table;
  int rc = build_dev_table<float>(*host_table, h->tab32);
  if (rc == GIK_OK) rc = build_dev_table<double>(*host_table, h->tab64);
  if (rc == GIK_OK) build_packed_table(h->tab32, h->pt32);
  if (rc != GIK_OK) { delete h; return rc; }
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess) { delete h; return (int)e; }
  if (device < 0 || device >= count) { delete h; return (int)cudaErrorInvalidDevice; }
  e = cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device);
  if (e != cudaSuccess) { delete h; return (int)e; }
  h->device = device;
  {
    DeviceGuard g(device);
    if (g.err == cudaSuccess) g.err = cudaMalloc(&h->queues, kQueueSlots * sizeof(unsigned long long));
    if (g.err != cudaSuccess) { delete h; return (int)g.err; }
  }
  h->next_queue.store(0);
  h->scene = nullptr;
  h->magic = kMagic;
  *out = h;
  return GIK_OK;
}

int gik_destroy(gik_handle_t h) {
  if (bad_handle(h)) return GIK_E_HANDLE;
  h->magic = 0;
  {
    DeviceGuard g(h->device);
    cudaFree(h->queues);
    gik_free_scene_of(h);
  }
  delete h;
  return GIK_OK;
}

int gik_fk_f32(gik_handle_t h, int64_t n, const float* q, float* frames, void* s) { return fk_api<float>(h, n, q, frames, s, false); }
int gik_fk_f64(gik_handle_t h, int64_t n, const double* q, double* frames, void* s) { return fk_api<double>(h, n, q, frames, s, false); }
int gik_jac_f32(gik_handle_t h, int64_t n, const float* q, float* jac, void* s) { return fk_api<float>(h, n, q, jac, s, true); }
int gik_jac_f64(gik_handle_t h, int64_t n, const double* q, double* jac, void* s) { return fk_api<double>(h, n, q, jac, s, true); }

int gik_solve_f32(gik_handle_t h, int64_t n, const float* q_init, const float* pose, const gik_params_t* p,
                  float* q_out, uint8_t* conv, int32_t* iters, float* resid, void* s) {
  return solve_api<float>(h, n, q_init, pose, p, q_out, conv, iters, resid, s);
}
int gik_solve_f64(gik_handle_t h, int64_t n, const double* q_init, const double* pose, const gik_params_t* p,
                  double* q_out, uint8_t* conv, int32_t* iters, double* resid, void* s) {
  return solve_api<double>(h, n, q_init, pose, p, q_out, conv, iters, resid, s);
}

int gik_solve_rows_f32(gik_handle_t h, int64_t n, const float* q_init, const float* pose, const gik_params_t* p, float* q_out,
                       uint8_t* conv, int32_t* iters, float* resid, const unsigned long long* ready, void* s) {
  return rows_api<float>(h, n, q_init, pose, p, q_out, conv, iters, resid, ready, s);
}
int gik_solve_rows_f64(gik_handle_t h, int64_t n, const double* q_init, const double* pose, const gik_params_t* p, double* q_out,
                       uint8_t* conv, int32_t* iters, double* resid, const unsigned long long* ready, void* s) {
  return rows_api<double>(h, n, q_init, pose, p, q_out, conv, iters, resid, ready, s);
}

int gik_solve_scatter_f32(gik_handle_t h, int64_t n, const float* q_init, const float* pose, const gik_params_t* p,
                          int32_t n_peers, float* const* q_all, uint8_t* const* conv_all, int64_t n_total, int64_t offset,
                          int32_t* iters, float* resid, void* s) {
  return scatter_api<float>(h, n, q_init, pose, p, n_peers, q_all, conv_all, n_total, offset, iters, resid, s);
}
int gik_solve_scatter_f64(gik_handle_t h, int64_t n, const double* q_init, const double* pose, const gik_params_t* p,
                          int32_t n_peers, double* const* q_all, uint8_t* const* conv_all, int64_t n_total, int64_t offset,
                          int32_t* iters, double* resid, void* s) {
  return scatter_api<double>(h, n, q_init, pose, p, n_peers, q_all, conv_all, n_total, offset, iters, resid, s);
}

int gik_best_of_f32(gik_handle_t h, int64_t n_place, int32_t n_restart, const float* q, const uint8_t* conv,
                    const float* resid, float* q_best, uint8_t* conv_best, int32_t* which, void* s) {
  return best_of_api<float>(h, n_place, n_restart, q, conv, resid, q_best, conv_best, which, s);
}
int gik_best_of_f64(gik_handle_t h, int64_t n_place, int32_t n_restart, const double* q, const uint8_t* conv,
                    const double* resid, double* q_best, uint8_t* conv_best, int32_t* which, void* s) {
  return best_of_api<double>(h, n_place, n_restart, q, conv, resid, q_best, conv_best, which, s);
}

int gik_project_edges_f32(gik_handle_t h, int64_t n_edges, int32_t max_steps, const float* q_start,
                          const float* pose_a, const float* pose_b, const int32_t* num_steps,
                          const gik_params_t* p, float* q_path, int32_t* n_valid, int32_t* iters_total, void* s) {
  return edges_api<float>(h, n_edges, max_steps, q_start, pose_a, pose_b, num_steps, p, q_path, n_valid, iters_total, s);
}
int gik_project_edges_f64(gik_handle_t h, int64_t n_edges, int32_t max_steps, const double* q_start,
                          const double* pose_a, const double* pose_b, const int32_t* num_steps,
                          const gik_params_t* p, double* q_path, int32_t* n_valid, int32_t* iters_total, void* s) {
  return edges_api<double>(h, n_edges, max_steps, q_start, pose_a, pose_b, num_steps, p, q_path, n_valid, iters_total, s);
}

// SURVEY.md 8(d) breakdown, frozen: FK 540 + pose errors 250 + LOCAL Jacobians 588 + Gram 594 + Cholesky 650 +
// triangular solves 288 + J^T z 155 + update/clamp 52.
size_t gik_flops_per_iter(void) { return 540 + 250 + 588 + 594 + 650 + 288 + 155 + 52; }

// FLOPs the kernels actually EXECUTE per descent iteration of one problem (FMA = 2, MUL / ADD = 1), from the executed
// opcode mix of the committed ncu captures (profiles/): packed instructions count both halves.
//   fp32 packed lane kernel, spherical-wrist step (profiles/r2s_solve_f32_ncu.md: 166.9 FFMA2 + 108.5 FMUL2 + 18.2 FADD2 + 2.2 FFMA + 14.1 FMUL + 5.5 FADD)
//   fp32 packed lane kernel, block-Cholesky step  (profiles/r1m_solve_f32_ncu.md: 320.8 FFMA2 + 102.6 FMUL2 + 11.1 FADD2 + 52.3 FFMA + 56.9 FMUL + 24.0 FADD)
//   fp64 pair kernel (two lanes per problem), wrist (profiles/r2p_solve_f64_ncu.md: 2 x (171.4 DFMA + 75.0 DMUL + 17.9 DADD))
//   fp64 pair kernel, block-Cholesky step          (profiles/r1i_solve_f64_ncu.md: 2 x (280.3 DFMA + 96.5 DMUL + 12.8 DADD))
size_t gik_flops_per_iter_executed(int elem_size, int wrist) {
  if (elem_size == 4) return wrist ? GIK_FLOPS_EXEC_F32_WRIST : 1696;
  if (elem_size == 8) return wrist ? 871 : 1340;
  return 0;
}

// in: q_init (nq) + pose (12); out: q (nq) + flag (1 B) + iters (4 B) + resid (2).  nq = 15.
size_t gik_bytes_per_solve(int elem_size) { return (size_t)elem_size * (15 + 12 + 15 + 2) + 1 + 4; }

int gik_measure_fma_peak(int device, int elem_size, int repeats, double* tflops) {
  if (!tflops) return GIK_E_NULL;
  if (repeats < 1) return GIK_E_SIZE;
  if (elem_size == 4) return fma_peak<float>(device, repeats, tflops);
  if (elem_size == 8) return fma_peak<double>(device, repeats, tflops);
  return GIK_E_PARAM;
}

int gik_solve_launch_dims(gik_handle_t h, int elem_size, int64_t n, int32_t* blocks, int32_t* threads) {
  if (bad_handle(h)) return GIK_E_HANDLE;
  if (!blocks || !threads) return GIK_E_NULL;
  if (n < 0) return GIK_E_SIZE;
  if (elem_size != 4 && elem_size != 8) return GIK_E_PARAM;
  SolveKernel k;
  int b = 0;
  const int rc = batch_launch(h, elem_size, n, 0, &k, &b);
  if (rc) return rc;
  *blocks = b; *threads = kThreads;
  return GIK_OK;
}

const char* gik_solve_kernel_name(gik_handle_t h, int elem_size, int64_t n, int flags) {
  if (bad_handle(h) || n < 0 || (elem_size != 4 && elem_size != 8)) return "";
  SolveKernel k;
  int b = 0;
  if (batch_launch(h, elem_size, n, flags, &k, &b)) return "";
  const bool f64 = elem_size == 8;
  switch (k.family) {
    case SolveKernel::PAIR:
      if (k.wrist) return f64 ? "gik_solve_pair_kernel<double, wrist>" : "gik_solve_pair_kernel<float, wrist>";
      return f64 ? "gik_solve_pair_kernel<double>" : "gik_solve_pair_kernel<float>";
    case SolveKernel::LANE:
      if (k.wrist) return f64 ? "gik_solve_kernel<double, wrist>" : "gik_solve_kernel<float, wrist>";
      return f64 ? "gik_solve_kernel<double>" : "gik_solve_kernel<float>";
    default:
      return k.wrist ? "gik_solve_lane2_kernel<wrist>" : "gik_solve_lane2_kernel";
  }
}

const char* gik_strerror(int code) {
  switch (code) {
    case GIK_OK: return "ok";
    case GIK_E_NULL: return "null pointer argument";
    case GIK_E_SIZE: return "invalid size";
    case GIK_E_MODEL: return "kinematic table is not a tree of 1-dof revolute joints";
    case GIK_E_TOPOLOGY: return "kinematic table does not match the compiled torso + two 6R-arm fast path";
    case GIK_E_PARAM: return "invalid solver parameter";
    case GIK_E_HANDLE: return "invalid handle";
    case GIK_E_NOSCENE: return "no collision scene attached (gik_scene_attach)";
    default: break;
  }
  if (code > 0) return cudaGetErrorString((cudaError_t)code);
  return "unknown error";
}

const char* gik_version(void) { return "gik 0.1 (sm_100a)"; }

}  // extern "C"

#include "gik_collide_impl.cuh"
#include "gik_bezier.cuh"
#include "gik_tree.cuh"
static void gik_free_scene_of(gik_handle_s* h) { free_scene(h->scene); h->scene = nullptr; }
