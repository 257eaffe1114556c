#!/usr/bin/env python
"""bench.py -- dual-arm grasp IK solves/s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dtype f32|f64] [--config 2|3|4|5]
                    [--dump-outputs DIR]

A "step" is ONE pass of the hot path over one batch of synthetic input: BASELINE config 2, 2^20 random cube
placements over the table workspace (identity rotation, path.py:47), every problem started from q0 = 0,
reference preset (eps 1e-3, dt 1e-2, max_iters 1000, undamped), fp32.  For N > 1 every rank solves its own
2^20-problem slab (weak scaling, no data-path collective) and the step ends with the all-gather of (q, converged).

Printed JSON (one line, rank 0): value = whole-job solves/s with inputs resident in HBM; e2e = the same metric
through the public API with HOST buffers (H2D + solve + D2H inside the timed region); roofline = the solve kernel
against the CUDA-core FMA peak measured in the same run; cpu_baseline = the C oracle (a port of the reference's loop;
the reference itself needs pinocchio, absent from this image) on the box's host cores.  `sub` carries short runs of
the rest of the metric: config 2 in fp64, config 3 (restarts, fp64, damped), config 4 (edge projection), the full
success predicate (collision term + the reference's keep-descending tail) and, for N > 1, config 5 (the 64 Mi-problem
strong-scaling sweep, fused scatter and NCCL gather) with a fused == all_gather check.
`--impl reference` times the CPU port alone.

`--dump-outputs DIR` writes what the timed path returned in its last timed step (rank 0's slab) as DIR/<name>.npy,
float64 arrays as float64 and everything else as float32, the problem index on the last axis.  The inputs are seeded,
so two builds run with the same arguments can be compared array for array.  Above 64 MB in all, every array keeps the
same seeded sample of problems, listed in problem_index.npy."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_PER_GPU = 1 << 20
WORKSPACE_LO = (0.20, -0.40, 0.93)      # SURVEY.md 8d config 2
WORKSPACE_HI = (0.60, 0.40, 1.40)
SAMPLER_LO = (0.33, -0.30, 1.05)        # the reference sampler's box, path.py:35-37 with config.py:36-37
SAMPLER_HI = (0.40, 0.11, 1.40)
METRIC = "dual-arm grasp IK solves/sec"
_STDOUT = sys.stdout


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dtype", default=None, choices=["f32", "f64"], help="default: f32 (f64 for --config 3)")
    ap.add_argument("--n", type=int, default=N_PER_GPU, help="problems per GPU per step")
    ap.add_argument("--cpu-sample", type=int, default=0, help="problems in the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-sub", action="store_true", help="skip the `sub` runs (fp64, configs 3 / 4 / 5, success predicate)")
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5],
                    help="BASELINE.json config: 2 (default, the metric's workload), 3 restarts fp64, 4 edge projection, 5 sharded sweep")
    ap.add_argument("--no-gather", action="store_true", help="N > 1: skip the result all-gather")
    ap.add_argument("--gather", default="fused", choices=["fused", "nccl"],
                    help="N > 1: 'fused' = the solve kernel stores results into every rank's symmetric-memory arrays over "
                         "NVLink (falls back to nccl if symmetric memory is unavailable); 'nccl' = all_gather_into_tensor")
    ap.add_argument("--box", default="workspace", choices=["workspace", "sampler"],
                    help="config 2 placement box: the table workspace (default) or the reference sampler's box (path.py:35-37)")
    ap.add_argument("--early-stop", action="store_true",
                    help="fast preset GIK_F_EARLY_STOP (NOT the reference's semantics for failed problems; never the default)")
    ap.add_argument("--kernel", default=None, choices=["lane", "pair", "lane1"], help="force a thread mapping (default: launcher's choice)")
    ap.add_argument("--step", default="auto", choices=["auto", "cholesky"],
                    help="form of the undamped step: auto = spherical-wrist 3x3 solves where the table allows it (default), "
                         "cholesky = always the general 6x6 block-Cholesky form (A/B)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step as DIR/<name>.npy; b200 arm only, since the "
                         "reference arm times a CPU port whose results the tests already compare")
    args = ap.parse_args()
    if args.dump_outputs is not None and (args.impl != "b200" or args.steps < 1):
        ap.error("--dump-outputs needs --impl b200 and --steps >= 1")
    if args.dtype is None:
        args.dtype = "f64" if args.config == 3 else "f32"
    return args


def workload_name(n, dtype):
    return (f"config2: {n} random cube placements over the table workspace x[0.20,0.60] y[-0.40,0.40] z[0.93,1.40], "
            f"identity rotation, single start q0=0, {dtype}, eps=1e-3 dt=1e-2 max_iters=1000 damping=0")


# ----------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port on the host cores (bounded sample of the same workload)
# ----------------------------------------------------------------------------------------------------------
def host_poses(n, seed):
    import numpy as np
    rng = np.random.default_rng(seed)
    P = np.zeros((n, 12))
    P[:, [0, 4, 8]] = 1.0
    P[:, 9:] = rng.uniform(WORKSPACE_LO, WORKSPACE_HI, size=(n, 3))
    return P


def cpu_solve_rate(n_sample, seed=1234, method=0):
    """Times the C oracle (oracle/grasp_ik_oracle.c, OpenMP over problems, all host threads) on n_sample problems
    of the bench workload.  method 0 = the faithful restatement (pinv through a Jacobi SVD), 1 = the same loop with
    the step solved by a 12x12 Cholesky factorisation of the normal equations (the strong CPU baseline).
    Returns (solves/s, threads, seconds)."""
    import numpy as np
    import gik_b200
    from oracle import c_oracle
    c_oracle.build()
    tc = gik_b200.nextage_table().to_c()
    threads = os.cpu_count() or 1
    P = host_poses(n_sample, seed)
    c_oracle.set_step_method(method)
    try:
        c_oracle.solve(tc, np.zeros((min(threads, n_sample), 15)), P[:min(threads, n_sample)])   # warm the threads
        t0 = time.perf_counter()
        c_oracle.solve(tc, np.zeros((n_sample, 15)), P, threads=threads)
        dt = time.perf_counter() - t0
    finally:
        c_oracle.set_step_method(0)
    return n_sample / dt, threads, dt


def numpy_solve_rate(n_sample, seed=99):
    """The numpy restatement (oracle/grasp_ik_np.py: one Python-level call per pinocchio/numpy primitive, like the
    reference's own loop) on one core -- the closest thing to the reference's Python speed this image can run."""
    import numpy as np
    from oracle import grasp_ik_np as o
    P = host_poses(n_sample, seed)
    t0 = time.perf_counter()
    for i in range(n_sample):
        o.computeqgrasppose(np.zeros(15), np.eye(3), P[i, 9:])
    return n_sample / (time.perf_counter() - t0)


def run_reference(args):
    """`--impl reference`: the reference's own CPU algorithm for the path.  The reference is Python on pinocchio
    (not installable here: no wheel, no network), so the arm times the C port of its loop (oracle/), which
    reproduces the reference's golden outputs; every step is a bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n_sample = args.cpu_sample or 16 * cores
    for _ in range(max(args.warmup, 0) and 1):
        cpu_solve_rate(min(n_sample, 2 * cores))
    t_total = 0.0
    for k in range(args.steps):
        rate, threads, dt = cpu_solve_rate(n_sample, seed=1234 + k)
        t_total += dt
    value = n_sample * args.steps / t_total
    strong, _, _ = cpu_solve_rate(64 * cores, method=1)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "solves/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(N_PER_GPU, "fp64 on CPU"),
                   "sample_per_step": n_sample},
        "cpu_baseline": {"value": value, "unit": "solves/s", "cores": threads, "kind": "port",
                         "sample": f"{n_sample} problems of the workload per step x {args.steps} steps, C oracle "
                                   f"(Jacobi-SVD pinv, -O3 -march=native, OpenMP {threads} threads)",
                         "strong": {"value": strong, "unit": "solves/s",
                                    "what": "the same C loop with the step solved by a 12x12 Cholesky of the normal "
                                            "equations instead of an SVD -- a performance-minded CPU implementation"}},
        "e2e": {"value": value, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=_STDOUT, flush=True)


# ----------------------------------------------------------------------------------------------------------
# clocks during the timed region
# ----------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.sm_max = None
        self._halt = threading.Event()
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for line in self.proc.stdout:
                f = [x.strip() for x in line.split(",")]
                if len(f) < 7:
                    continue
                try:
                    self.samples.append(float(f[0])); self.sm_max = float(f[1])
                except ValueError:
                    continue
                for nm, v in zip(names, f[3:7]):
                    if v.lower().startswith("active"):
                        self.reasons.add(nm)
                if self._halt.is_set():
                    break
        except Exception:
            pass

    def stop(self):
        self._halt.set()
        if self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass

    def summary(self):
        s = sorted(self.samples)
        med = s[len(s) // 2] if s else None
        return {"sm_mhz": med, "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons), "samples": len(s)}


# ----------------------------------------------------------------------------------------------------------
# GPU arm: workloads
# ----------------------------------------------------------------------------------------------------------
def workspace_positions(torch, n, dev, dtype, seed, box="workspace"):
    g = torch.Generator(device=dev).manual_seed(seed)
    lo = torch.tensor(WORKSPACE_LO if box == "workspace" else SAMPLER_LO, device=dev, dtype=dtype)
    hi = torch.tensor(WORKSPACE_HI if box == "workspace" else SAMPLER_HI, device=dev, dtype=dtype)
    return lo + torch.rand((n, 3), device=dev, dtype=dtype, generator=g) * (hi - lo)


def pose_rows_from(torch, pos):
    n = pos.shape[0]
    return torch.cat([torch.eye(3, device=pos.device, dtype=pos.dtype).reshape(1, 9).expand(n, 9), pos], 1).contiguous()


class Workload:
    """One BASELINE config on one rank: `launch()` enqueues the kernels of one step on the current stream and
    returns the tensors a gather would ship; `solves` = problems solved per step on this rank; `iterations()` = descent
    iterations executed by the last step (device scalar); `converged()` = fraction converged; `outputs()` = name ->
    tensor of every result the last step returned, problem index on the last axis."""
    name = ""
    solves = 0
    kernel_choice = None
    early_stop = False
    n_kernel = None          # problem count that decides the kernel mapping (edges for config 4)
    edge_mode = False


class Config2(Workload):
    def __init__(self, torch, solver, n, rank, dtype, seed_base=1000, box="workspace"):
        dev = solver.device
        self.torch, self.solver, self.solves = torch, solver, n
        self.pose_rows = pose_rows_from(torch, workspace_positions(torch, n, dev, dtype, seed_base + rank, box))
        self.pose = self.pose_rows.t().contiguous()                 # SoA [12][n]
        self.q0 = torch.zeros((15, n), device=dev, dtype=dtype)     # SoA [15][n]
        self.out = (torch.empty_like(self.q0), torch.empty(n, dtype=torch.uint8, device=dev),
                    torch.empty(n, dtype=torch.int32, device=dev), torch.empty((2, n), dtype=dtype, device=dev))
        self.name = workload_name(n, "fp32" if dtype == torch.float32 else "fp64")
        self.n_kernel = n
        if box == "sampler":
            self.name = self.name.replace("over the table workspace x[0.20,0.60] y[-0.40,0.40] z[0.93,1.40]",
                                          "over the reference sampler box x[0.33,0.40] y[-0.30,0.11] z[1.05,1.40] (path.py:35-37)")

    def launch(self):
        q, conv, _, _ = self.solver.solve_soa(self.q0, self.pose, out=self.out, kernel=self.kernel_choice,
                                              early_stop=self.early_stop)
        return q, conv

    def outputs(self):
        return dict(zip(("q", "converged", "iterations", "residual"), self.out))

    def iterations(self):
        return self.out[2].sum(dtype=self.torch.int64).double()

    def converged(self):
        return self.out[1].double().mean()


class Config3(Workload):
    """65,536 placements x 64 random-restart initial q (restart 0 = zeros), best-of, fp64 (SURVEY 8d config 3)."""
    DAMPING = 1e-6

    def __init__(self, torch, solver, n_place, restarts, rank, dtype):
        dev = solver.device
        self.torch, self.solver, self.n_place, self.R = torch, solver, n_place, restarts
        self.solves = n_place * restarts
        self.n_kernel = self.solves
        pos = workspace_positions(torch, n_place, dev, dtype, 1 + 7919 * rank)
        rows = pose_rows_from(torch, pos)
        self.pose = rows.unsqueeze(1).expand(n_place, restarts, 12).reshape(-1, 12).t().contiguous()
        lo, hi = solver.limits(dtype)
        g = torch.Generator(device=dev).manual_seed(2 + 7919 * rank)
        cand = lo + torch.rand((n_place, restarts, 15), device=dev, dtype=dtype, generator=g) * (hi - lo)
        cand[:, 0, :] = 0
        self.q0 = cand.reshape(-1, 15).t().contiguous()
        n = self.solves
        self.out = (torch.empty_like(self.q0), torch.empty(n, dtype=torch.uint8, device=dev),
                    torch.empty(n, dtype=torch.int32, device=dev), torch.empty((2, n), dtype=dtype, device=dev))
        self.best = None
        self.name = (f"config3: {n_place} workspace placements x {restarts} restarts (restart 0 = q0, others uniform in the "
                     f"joint limits), best-of, {'fp64' if dtype == torch.float64 else 'fp32'}, damping {self.DAMPING}")

    def launch(self):
        q, conv, _, resid = self.solver.solve_soa(self.q0, self.pose, out=self.out, damping=self.DAMPING, kernel=self.kernel_choice)
        self.best = self.solver.best_of_soa(q, conv, resid, self.n_place, self.R)
        return self.best[0], self.best[1]

    def outputs(self):
        return dict(zip(("q_best", "converged", "restart"), self.best))

    def iterations(self):
        return self.out[2].sum(dtype=self.torch.int64).double()

    def converged(self):
        return self.out[1].double().mean()

    def extra(self):
        return {"placements_with_a_converged_restart": float(self.best[1].double().mean()),
                "restart0_converged": float(self.out[1].reshape(self.n_place, self.R)[:, 0].double().mean())}


class Config4(Workload):
    """path.py edge projection: E edges x S interpolated placements, warm-started along each edge, march stops at the
    first non-converged step (SURVEY 8d config 4).  Step 0 starts from a converged q at cube_a."""
    edge_mode = True

    def __init__(self, torch, solver, n_edges, steps, rank, dtype):
        dev = solver.device
        self.torch, self.solver, self.E, self.S = torch, solver, n_edges, steps
        self.n_kernel = n_edges
        # endpoints a: workspace placements whose IK from q0 converges (oversample, keep the first E)
        cand = pose_rows_from(torch, workspace_positions(torch, 3 * n_edges, dev, dtype, 3 + 7919 * rank))
        q, conv = solver.solve(torch.zeros(15, device=dev, dtype=dtype), cand, dtype=dtype)
        keep = torch.nonzero(conv).flatten()[:n_edges]
        assert keep.numel() == n_edges, "not enough reachable edge starts"
        self.q_start = q[keep].t().contiguous()
        self.pose_a = cand[keep].t().contiguous()
        self.pose_b = pose_rows_from(torch, workspace_positions(torch, n_edges, dev, dtype, 4 + 7919 * rank)).t().contiguous()
        self.ns = torch.full((n_edges,), steps, dtype=torch.int32, device=dev)
        self.res = None
        self.solves = n_edges * steps          # upper bound; the executed count is reported from n_valid
        self.name = (f"config4: {n_edges} cube-pose edges x {steps} interpolated placements (SE3.Interpolate), IK "
                     f"warm-started along each edge, stop at first failure, {'fp32' if dtype == torch.float32 else 'fp64'}")

    def launch(self):
        self.res = self.solver.project_edges_soa(self.q_start, self.pose_a, self.pose_b, self.ns, self.S, kernel=self.kernel_choice)
        return self.res[0], self.res[1]

    def outputs(self):
        return dict(zip(("q_path", "n_valid", "iterations"), self.res))

    def executed(self):
        nv = self.res[1]
        return (nv + (nv < self.S).to(nv.dtype)).sum(dtype=self.torch.int64).double()   # + the failing solve

    def iterations(self):
        return self.res[2].sum(dtype=self.torch.int64).double()

    def converged(self):
        return self.res[1].double().sum() / self.executed()

    def extra(self):
        nv = self.res[1].double()
        it = self.res[2].double()
        # the launch cannot end before its LONGEST chain has been walked: iterations of one edge are strictly sequential
        return {"edges_fully_projected": float((nv == self.S).double().mean()), "mean_valid_steps": float(nv.mean()),
                "solves_executed": float(self.executed()),
                "iterations_per_edge": {"mean": float(it.mean()), "p99": float(self.torch.quantile(it, 0.99)), "max": float(it.max())}}


class SuccessPredicate(Config2):
    """Config 2 with the reference's FULL success predicate (inverse_geometry.py:70, 97-98): collision(q) on the
    converged problems and the keep-descending-while-colliding tail, all on the device (gik_solve_success_*)."""

    def __init__(self, torch, solver, n, rank, dtype):
        super().__init__(torch, solver, n, rank, dtype)
        solver._need_scene()
        self.name = "config2 + collision term and keep-descending tail on the device (gik_solve_success_*); " + self.name
        self.res = None
        self.graph, self.graph_failed = None, None

    def launch(self):
        # The call enqueues ten launches back to back; replayed from a CUDA graph they reach the GPU as ONE submission, so a
        # driver lock held by somebody else's nvidia-smi query between two of them (tens of milliseconds, measured) cannot
        # open a gap in the middle of the step.  Captured on first use; results live in the graph's static tensors.
        if self.graph is None and not self.graph_failed:
            try:
                torch = self.torch
                self.solver.solve_success_soa(self.q0, self.pose, return_stats=True)       # warm: allocator, lazy module load
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self.res = self.solver.solve_success_soa(self.q0, self.pose, return_stats=True)
                self.graph = g
            except Exception as e:                                                          # noqa: BLE001
                self.graph_failed = f"{type(e).__name__}: {e}"[:160]
                self.torch.cuda.synchronize()
        if self.graph is not None:
            self.graph.replay()
        else:
            self.res = self.solver.solve_success_soa(self.q0, self.pose, return_stats=True)
        return self.res[0], self.res[1]

    def iterations(self):
        return self.res[3].sum(dtype=self.torch.int64).double()

    def converged(self):
        return self.res[1].double().mean()       # success fraction

    def extra(self):
        st = [int(x) for x in self.res[5].tolist()]
        return {"success_fraction": float(self.res[1].double().mean()),
                "submission": "CUDA graph replay of the call's launches" if self.graph is not None else f"direct ({self.graph_failed})",
                "tail": {"persistent_collisions": st[0], "replayed_problems": st[1], "replayed_iterations": st[2],
                         "replays_that_succeeded": st[3]}}


# ----------------------------------------------------------------------------------------------------------
# GPU arm: measurement
# ----------------------------------------------------------------------------------------------------------
class Runner:
    def __init__(self, torch, dist, solver, dev, world, rank):
        self.torch, self.dist, self.solver, self.dev, self.world, self.rank = torch, dist, solver, dev, world, rank
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def time(self, step, steps, warmup):
        """W untimed + K timed calls of step(ev) bracketed by barrier + synchronize; returns (ms_total, kernel_ms), both
        the max over ranks.  step(ev) records ev[0] / ev[1] around its solve launches."""
        torch = self.torch
        for _ in range(max(warmup, 0)):
            step(None)
        self.barrier()
        kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record()
        for k in range(steps):
            step(kev[k])
        e1.record()
        self.barrier()
        t = torch.tensor([e0.elapsed_time(e1), sum(a.elapsed_time(b) for a, b in kev) / max(steps, 1)],
                         device=self.dev, dtype=torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.tolist()

    def plain_step(self, wl):
        def step(ev):
            self.flush.fill_(1)                                       # L2 flush between iterations
            if ev:
                ev[0].record()
            wl.launch()
            if ev:
                ev[1].record()
        return step

    def stats(self, wl):
        """(converged solves, iterations, solves) per step summed over ranks."""
        torch = self.torch
        solves = wl.executed() if hasattr(wl, "executed") else torch.tensor(float(wl.solves), device=self.dev, dtype=torch.float64)
        st = torch.stack([wl.converged() * solves, wl.iterations(), solves])
        if self.world > 1:
            self.dist.all_reduce(st)
        return st.tolist()


DUMP_BYTES = 64 * 1000 * 1000


def dump_outputs(out_dir, arrays, budget=DUMP_BYTES, seed=0):
    """Writes every tensor of `arrays` (problem index on the last axis) as out_dir/<name>.npy: float64 tensors as
    float64, all others as float32, and problem_index.npy (float64) with the problems kept.  When all of them would
    exceed `budget` bytes, every array keeps the same seeded sample of problems, in ascending order."""
    import numpy as np
    import torch
    n = next(iter(arrays.values())).shape[-1]
    if any(t.shape[-1] != n for t in arrays.values()):
        raise ValueError("dump_outputs: the arrays disagree on the problem count")
    per_problem = 8 + sum((8 if t.dtype == torch.float64 else 4) * (t.numel() // max(n, 1)) for t in arrays.values())
    k = min(n, (budget - 256 * (len(arrays) + 1)) // per_problem)      # 256: room for each file's .npy header
    idx = np.arange(n) if k == n else np.sort(np.random.default_rng(seed).choice(n, k, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.index_select(t.dim() - 1, torch.from_numpy(idx).to(t.device)).cpu()
        np.save(os.path.join(out_dir, name + ".npy"), (a.double() if t.dtype == torch.float64 else a.float()).numpy())
    np.save(os.path.join(out_dir, "problem_index.npy"), idx.astype(np.float64))


def roofline_of(gik_b200, solver, wl, dtype, esz, kernel_ms, iters_per_launch, solves_per_launch, peak, kernel_choice):
    """The solve kernel against the CUDA-core FMA pipe.  `frac` uses the survey's ALGORITHMIC count (3117 FLOP per
    descent iteration, frozen in SURVEY 8d for a dense-ish formulation of the step); the kernels execute far fewer
    (block structure, spherical wrist), so `frac` exceeds 1 -- `frac_executed` counts the FLOPs the kernel really
    issues (opcode mix of the committed ncu capture) and `pipe_busy_ncu` is the FMA / FP64 pipe utilisation ncu measured."""
    fpi = gik_b200.flops_per_iter()
    name = solver.kernel_name(wl.n_kernel, dtype, kernel_choice)
    damped = isinstance(wl, Config3)
    wrist = "wrist" in name and not damped
    if damped:
        name = name.replace(", wrist>", ">").replace("<wrist>", "")
    fpe = gik_b200.flops_per_iter_executed(esz, wrist)
    achieved = iters_per_launch * fpi / (kernel_ms * 1e-3) * 1e-12
    executed = iters_per_launch * fpe / (kernel_ms * 1e-3) * 1e-12
    bytes_algo = gik_b200.bytes_per_solve(esz) * solves_per_launch
    hbm_peak = None
    try:
        hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        pass
    traffic = pipe_busy = capture = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        key = ("f32" if esz == 4 else "f64") + ("_edges" if wl.edge_mode else "")
        ent = tj.get(key) if (type(wl) is Config2 and wrist) or wl.edge_mode else None
        if ent:
            traffic, pipe_busy, capture = ent.get("dram_bytes_per_launch"), ent.get("pipe_busy"), ent.get("capture")
    except Exception:
        pass
    return {
        "bound": "fp32" if esz == 4 else "fp64",
        "kernel": name + (" (edge mode)" if wl.edge_mode else ""),
        "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak if peak else None,
        "peak_source": "measured in this run: register-resident FMA chains on every SM (gik_measure_fma_peak); "
                       "MEASURED_PEAKS.json has no CUDA-core figure",
        "flops_per_iteration": fpi, "flops_per_iteration_executed": fpe,
        "achieved_executed": executed, "frac_executed": executed / peak if peak else None,
        "iterations_per_launch": iters_per_launch, "kernel_ms": kernel_ms,
        "traffic": traffic, "pipe_busy_ncu": pipe_busy, "ncu_capture": capture,
        "hbm": {"algorithmic_bytes_per_launch": bytes_algo,
                "achieved_gbs": bytes_algo / (kernel_ms * 1e-3) * 1e-9, "peak_gbs": hbm_peak,
                "frac": (bytes_algo / (kernel_ms * 1e-3) * 1e-9 / hbm_peak) if hbm_peak else None},
    }


def run_b200(args):
    import torch
    import torch.distributed as dist
    import gik_b200
    from gik_b200 import dist as gdist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product has no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    dtype = torch.float32 if args.dtype == "f32" else torch.float64
    esz = 4 if args.dtype == "f32" else 8
    solver = gik_b200.GraspIK(gik_b200.nextage_table(), dev)
    solver.force_cholesky = args.step == "cholesky"
    R = Runner(torch, dist, solver, dev, world, rank)
    peaks = {4: gik_b200.fma_peak_tflops(local, 4), 8: gik_b200.fma_peak_tflops(local, 8)}

    scaling = "weak"
    if args.config == 2:
        wl = Config2(torch, solver, args.n, rank, dtype, box=args.box)
    elif args.config == 3:
        wl = Config3(torch, solver, args.n if args.n != N_PER_GPU else 65536, 64, rank, dtype)
    elif args.config == 4:
        wl = Config4(torch, solver, args.n if args.n != N_PER_GPU else 4096, 256, rank, dtype)
    else:   # config 5: 64 Mi config-2 problems sharded over the ranks (strong scaling) + all-gather
        total = args.n if args.n != N_PER_GPU else 64 << 20
        lo_i, hi_i = gdist.shard_bounds(total, rank, world)
        wl = Config2(torch, solver, hi_i - lo_i, rank, dtype, seed_base=4000)
        wl.name = f"config5: {total} config-2 problems sharded over {world} GPU(s) + all-gather of q/converged; " + wl.name
        scaling = "strong"
    wl.kernel_choice = args.kernel
    wl.early_stop = args.early_stop
    if args.early_stop:
        wl.name += " [FAST PRESET: early stop of stalled problems -- not the reference's semantics for failed problems]"
    gather = world > 1 and not args.no_gather and args.config in (2, 5)
    if args.config == 5:
        n_total_gather, gather_off = total, lo_i
    else:
        n_total_gather, gather_off = wl.solves * world, wl.solves * rank
    fused = None
    collective = "none"
    if gather:
        collective = "all_gather_into_tensor (NCCL) of q [15][n] + converged [n] per step"
        if args.gather == "fused":
            try:
                fused = gdist.SymmetricResults(15, n_total_gather, dtype, dev)
                collective = ("fused: pusher warps of the solve kernel copy finished 1024-problem chunks of q/converged into every rank's "
                              "symmetric-memory result arrays over NVLink (coalesced 16-byte P2P stores) while the other blocks keep "
                              "solving, a tail kernel copies the chunks still in flight at the end, then one cross-rank barrier per step")
            except Exception as e:      # symmetric memory unavailable on this box: keep the NCCL gather and say so
                fused = None
                collective += f" (fused path unavailable: {type(e).__name__})"

    def make_step(w, sym, n_total, off, use_gather):
        sym_out = (w.out[2], w.out[3]) if sym is not None else None

        def step(ev):
            R.flush.fill_(1)                                       # L2 flush between iterations
            if ev:
                ev[0].record()
            if sym is not None:
                solver.solve_scatter_soa(w.q0, w.pose, sym.q_ptrs, sym.conv_ptrs, n_total, off, out=sym_out,
                                         kernel=w.kernel_choice)
            else:
                q, conv = w.launch()
            if ev:
                ev[1].record()
            if sym is not None:
                sym.barrier()
            elif use_gather:
                gdist.all_gather_results(q, conv, n_total)
        return step

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    launches0 = solver.launches
    ms_total, kernel_ms = R.time(make_step(wl, fused, n_total_gather, gather_off, gather), args.steps, args.warmup)
    launches_all = solver.launches - launches0
    launches = launches_all * args.steps // max(args.steps + max(args.warmup, 0), 1)      # launches inside the timed region
    if sampler:
        sampler.stop()
    if fused is not None:     # the local flags live in the symmetric array: bring this rank's slab back for the stats
        wl.out[1].copy_(fused.conv[gather_off:gather_off + wl.solves])
    if args.dump_outputs is not None and rank == 0:
        outs = wl.outputs()
        if fused is not None:
            outs["q"] = fused.q[:, gather_off:gather_off + wl.solves]
        dump_outputs(args.dump_outputs, outs)
    ms_per_step = ms_total / max(args.steps, 1)
    conv_solves, iters_sum, solves_all = R.stats(wl)          # per step, all ranks
    conv_frac = conv_solves / solves_all

    # ---- e2e: public batched API with HOST buffers, copies inside the timed region (default workload only)
    e2e = None
    if not args.no_e2e and args.config == 2:
        n = wl.solves
        q_host = torch.zeros((n, 15), dtype=dtype).pin_memory()
        pose_host = wl.pose_rows.cpu().pin_memory()
        q_res = torch.empty((n, 15), dtype=dtype).pin_memory()
        c_res = torch.empty((n,), dtype=torch.uint8).pin_memory()
        q_np, pose_np = q_host.numpy().copy(), pose_host.numpy().copy()          # pageable numpy arrays

        def timed_e2e(call):
            for _ in range(2):
                call()
            R.barrier()
            t0 = time.perf_counter()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(args.steps):
                call()
            a1.record()
            R.barrier()
            wall = (time.perf_counter() - t0) * 1e3
            te = torch.tensor([max(a0.elapsed_time(a1), wall)], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(te, op=dist.ReduceOp.MAX)
            return n * world * args.steps / (te.item() * 1e-3)

        # public API, HOST tensors in and out: H2D of q_init / pose, the solve and D2H of q / converged all happen inside
        # the call (one launch, inputs streamed by the copy engine, results stored to host memory by the kernel); it
        # returns when the results are in host memory
        v_out = timed_e2e(lambda: bool(gik_b200.computeqgrasppose_batch(solver, q_host, pose_host, dtype=dtype, out=(q_res, c_res))[1][0]))
        v_fresh = timed_e2e(lambda: bool(gik_b200.computeqgrasppose_batch(solver, q_host, pose_host, dtype=dtype)[1][0]))
        v_page = timed_e2e(lambda: bool(gik_b200.computeqgrasppose_batch(solver, q_np, pose_np, dtype=dtype)[1][0]))
        e2e = {"value": v_out, "unit": "solves/s",
               "h2d_bytes_per_step": int(n * (15 + 12) * esz), "d2h_bytes_per_step": int(n * (15 * esz + 1)),
               "api": "computeqgrasppose_batch(pinned host tensors, out=caller's pinned result tensors) -> host tensors",
               "variants": {"pinned_in_fresh_results_per_call": v_fresh,
                            "pageable_numpy_in_fresh_results_per_call": v_page,
                            "note": "the default API returns freshly allocated caller-owned pinned tensors; pageable inputs "
                                    "add one host memcpy into a pinned staging buffer"}}

    # ---- sub: the rest of the metric in short runs (rank-local workloads; every rank runs them, rank 0 reports)
    sub = None
    if not args.no_sub and args.config == 2 and args.box == "workspace" and not args.early_stop and args.kernel is None:
        sub = {}
        sub_sampler = ClockSampler(local) if rank == 0 else None
        if sub_sampler:
            sub_sampler.start()

        def sub_run(name, w, dt_, steps=3, warmup=1):
            ms_t, k_ms = R.time(R.plain_step(w), steps, warmup)
            cs, its, sv = R.stats(w)
            e = 4 if dt_ == torch.float32 else 8
            roof = roofline_of(gik_b200, solver, w, dt_, e, k_ms, its / world, sv / world, peaks[e], None)
            ent = {"workload": w.name, "dtype": "f32" if e == 4 else "f64", "value": sv * steps / (ms_t * 1e-3), "unit": "solves/s",
                   "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms_t / steps, "kernel_ms": k_ms,
                   "converged_fraction": cs / sv, "mean_iterations": its / sv,
                   "roofline": {k: roof[k] for k in ("kernel", "frac", "frac_executed", "achieved", "achieved_executed", "peak",
                                                     "pipe_busy_ncu", "traffic")}}
            if hasattr(w, "extra"):
                ent.update(w.extra())
                if "iterations_per_edge" in ent and ent["iterations_per_edge"]["max"] > 0:
                    # latency of one descent iteration of a lone chain, if the longest edge alone set the time
                    ent["iterations_per_edge"]["kernel_us_per_iteration_of_longest_edge"] = k_ms * 1e3 / ent["iterations_per_edge"]["max"]
            sub[name] = ent
            return ent

        f32, f64 = torch.float32, torch.float64
        sub_run("config2_fp64", Config2(torch, solver, args.n, rank, f64), f64)
        sub_run("config3_fp64_64_restarts_damped", Config3(torch, solver, 65536, 64, rank, f64), f64, steps=2)
        sub_run("config4_fp32_edges", Config4(torch, solver, 4096, 256, rank, f32), f32)
        sub_run("config4_fp64_edges", Config4(torch, solver, 4096, 256, rank, f64), f64, steps=2)
        # the sampler's nvidia-smi polling is stopped for this one: the call enqueues ten launches back to back and a
        # concurrent nvidia-smi query can hold the driver lock for tens of milliseconds between two of them (measured:
        # 89 ms per call with the 100 ms poll running against 46 ms without), which a one-launch step never sees
        if sub_sampler:
            sub_sampler.stop()
            sub_sampler.join(timeout=2.0)
        ent = sub_run("config2_fp32_success_predicate", SuccessPredicate(torch, solver, args.n, rank, f32), f32)
        ent["value_is"] = ("success-flagged solves/s: solve + collision(q) on the converged problems + the reference's "
                           "keep-descending-while-colliding tail, one stream-ordered call (gik_solve_success_f32)")
        ent["kernel_ms_is"] = "the whole call (solve, compaction, collision, continuation, tail kernels)"
        ent.pop("roofline", None)
        torch.cuda.empty_cache()
        # config 5: the 64 Mi-problem strong-scaling sweep, NCCL gather and fused scatter, with a fused == gather check
        if world > 1:
            total5 = 64 << 20
            lo5, hi5 = gdist.shard_bounds(total5, rank, world)
            w5 = Config2(torch, solver, hi5 - lo5, rank, f32, seed_base=4000)
            c5 = {"workload": f"config5: {total5} config-2 problems sharded over {world} GPUs + all-gather of q/converged; " + w5.name,
                  "scaling": "strong", "dtype": "f32", "n_gpus": world, "steps": 2, "warmup": 1}
            ms_t, k_ms = R.time(make_step(w5, None, total5, lo5, False), 2, 1)
            c5["no_gather"] = {"value": total5 * 2 / (ms_t * 1e-3), "unit": "solves/s", "ms_per_step": ms_t / 2, "kernel_ms": k_ms}
            ms_t, k_ms = R.time(make_step(w5, None, total5, lo5, True), 2, 1)
            c5["nccl_gather"] = {"value": total5 * 2 / (ms_t * 1e-3), "unit": "solves/s", "ms_per_step": ms_t / 2, "kernel_ms": k_ms}
            q_ref, c_ref = gdist.all_gather_results(w5.out[0], w5.out[1], total5)
            try:
                sym = gdist.SymmetricResults(15, total5, f32, dev)
                ms_t, k_ms = R.time(make_step(w5, sym, total5, lo5, True), 2, 1)
                c5["fused_scatter"] = {"value": total5 * 2 / (ms_t * 1e-3), "unit": "solves/s", "ms_per_step": ms_t / 2, "kernel_ms": k_ms}
                ok = torch.tensor([float(torch.equal(sym.q, q_ref) and torch.equal(sym.conv, c_ref))], device=dev)
                dist.all_reduce(ok, op=dist.ReduceOp.MIN)
                c5["gather_check"] = {"fused_equals_all_gather_on_every_rank": bool(ok.item()),
                                      "compared": "q [15][64 Mi] and converged [64 Mi], bit for bit, outside the timed region"}
                del sym
            except Exception as e:
                c5["fused_scatter"] = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
            sub["config5_strong_64Mi"] = c5
            del w5, q_ref, c_ref
            torch.cuda.empty_cache()
            # the headline's own arrays: fused scatter == NCCL gather, bit for bit
            if fused is not None:
                wl.launch()
                q_ref, c_ref = gdist.all_gather_results(wl.out[0], wl.out[1], n_total_gather)
                make_step(wl, fused, n_total_gather, gather_off, gather)(None)
                torch.cuda.synchronize()
                ok = torch.tensor([float(torch.equal(fused.q, q_ref) and torch.equal(fused.conv, c_ref))], device=dev)
                dist.all_reduce(ok, op=dist.ReduceOp.MIN)
                sub["gather_check"] = {"fused_equals_all_gather_on_every_rank": bool(ok.item()),
                                       "compared": f"headline arrays: q [15][{n_total_gather}] and converged, bit for bit, outside the timed region"}
        else:
            sub["config5_strong_64Mi"] = {"note": "needs N > 1 (the scaling runs carry it); at N = 1 it is config 2 with 64 Mi "
                                                  "problems in one launch"}
        if sub_sampler:
            sub_sampler.stop()
            sub["clocks"] = sub_sampler.summary()
            sub["clocks"]["covers"] = "the fp64 / config 3 / config 4 sub-runs (polling stopped before the success-predicate run)"

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (the solve kernel the launcher picked): CUDA-core FMA pipe, peak measured in this run
    roofline = roofline_of(gik_b200, solver, wl, dtype, esz, kernel_ms, iters_sum / world, solves_all / world, peaks[esz],
                           args.kernel)

    cpu = None
    if not args.no_cpu_baseline and world == 1 and args.config == 2:
        cores = os.cpu_count() or 1
        n_sample = args.cpu_sample or 512 * cores
        rate, threads, secs = cpu_solve_rate(n_sample)
        strong, _, s_secs = cpu_solve_rate(4096 * cores, method=1)
        np_rate = numpy_solve_rate(3)
        cpu = {"value": rate, "unit": "solves/s", "cores": threads, "kind": "port",
               "numpy_restatement_solves_per_s_1core": np_rate,
               "strong": {"value": strong, "unit": "solves/s", "cores": threads,
                          "what": f"the same C loop with the step solved by a 12x12 Cholesky of the normal equations instead of "
                                  f"an SVD ({4096 * cores} problems, {s_secs:.1f} s) -- what a performance-minded CPU "
                                  f"implementation would do; the GPU/CPU ratio against THIS figure is the honest one"},
               "sample": f"{n_sample} problems of the same workload ({secs:.1f} s), C oracle (Jacobi-SVD pinv, -O3 "
                         f"-march=native, OpenMP {threads} threads); the Python+pinocchio reference cannot be installed "
                         f"here -- its closest stand-in, the numpy restatement, is timed on 3 problems / 1 core beside it"}

    cfg = {"workload": wl.name, "problems_per_gpu_per_step": solves_all / world,
           "l2": "256 MB flush write before every step (inside the timed region)",
           "collective": collective,
           "converged_fraction": conv_frac, "mean_iterations": iters_sum / solves_all}
    if hasattr(wl, "extra"):
        cfg.update(wl.extra())
    line = {
        "metric": METRIC, "value": solves_all * args.steps / (ms_total * 1e-3), "unit": "solves/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": scaling, "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "config": cfg,
        "converged_solves_per_s": conv_solves * args.steps / (ms_total * 1e-3),
        "clocks": sampler.summary() if sampler else None,
        "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu, "sub": sub,
    }
    print(json.dumps(line), file=_STDOUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    # Exactly ONE line on stdout: libraries (NCCL prints its version banner there) are routed to stderr for the whole
    # run and the JSON line goes to the saved descriptor.
    global _STDOUT
    sys.stdout.flush()
    _STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
