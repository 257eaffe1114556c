"""The device forms of the scalar functions of csrc/gik_core.cuh, run on the device (tests/devsim/devsim.cu) and
compared with numpy longdouble: the MUFU rsqrt / rcp / sqrt (fp32, and the halves of the packed F2 type), the fp64
MUFU seed + third-order step, __sincosf and the constant-bank Cody-Waite sincos, the atan2 polynomials and log6 in
float, double and F2.  The bars are the accuracy the header and DESIGN.md state for each form.  The host build of the
header (tests/hostsim, test_device_functions_cpu.py) runs the IEEE library forms instead, so only this file measures
what the solve kernels compute."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT

CSRC = os.path.join(ROOT, "motion-planning-and-control-for-dual-manipulator-robot_b200", "csrc")
SRC = os.path.join(ROOT, "tests", "devsim", "devsim.cu")
OUT = os.path.join(ROOT, "tests", "devsim", "_build", "libdevsim.so")
LD = np.longdouble
PI = np.pi
U32, U64 = 2.0 ** -24, 2.0 ** -53


def build_devsim():
    """Compile devsim.cu with the library's own nvcc flags; rebuilt when it or gik_core.cuh is newer than the library."""
    from gik_b200 import _cabi
    deps = [SRC, os.path.join(CSRC, "gik_core.cuh")]
    if not os.path.exists(OUT) or any(os.path.getmtime(d) > os.path.getmtime(OUT) for d in deps):
        os.makedirs(os.path.dirname(OUT), exist_ok=True)
        nvcc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
        if not os.path.exists(nvcc):
            nvcc = "nvcc"
        tmp = OUT + ".tmp"
        res = subprocess.run([nvcc] + _cabi.NVCC_FLAGS + ["-I", CSRC, "-o", tmp, SRC], capture_output=True, text=True)
        assert res.returncode == 0, res.stdout + res.stderr
        os.replace(tmp, OUT)
    return OUT


class DevSim:
    """ctypes loader of libdevsim.so: numpy arrays in, numpy arrays out, through device copies."""
    OPS = {"rsqrt": 0, "rcp": 1, "sqrt": 2, "div": 3, "atan2": 4, "sincos_fast": 5, "sincos": 6}

    def __init__(self):
        self.lib = ctypes.CDLL(build_devsim())

    @staticmethod
    def _dev(a, dtype):
        import torch
        return torch.as_tensor(np.ascontiguousarray(a, dtype), device="cuda:0")

    def _run(self, fname, lead, dtype, out_shape, *args):
        import torch
        torch.cuda.synchronize()
        dev = [None if a is None else self._dev(a, dtype) for a in args]
        out = torch.zeros(out_shape, dtype=dev[0].dtype, device="cuda:0")
        ptrs = [ctypes.c_void_p(0 if d is None else d.data_ptr()) for d in dev]
        rc = getattr(self.lib, fname)(*lead, *ptrs, ctypes.c_void_p(out.data_ptr()))
        assert rc == 0, f"{fname}: CUDA error {rc}"
        return out.cpu().numpy()

    def scalar(self, op, kind, a, b=None):
        """kind: "f32", "f64" or "f2" (element i in half i % 2 of a packed value; even n)."""
        n = len(a)
        assert kind != "f2" or n % 2 == 0, "the packed forms take an even number of elements"
        dtype = np.float64 if kind == "f64" else np.float32
        shape = (2, n) if op.startswith("sincos") else (n,)
        return self._run(f"devsim_scalar_{kind}", (ctypes.c_int(self.OPS[op]), ctypes.c_int64(n)), dtype, shape, a, b)

    def log6(self, kind, R, p):
        """R [n, 9] row-major, p [n, 3] -> e [n, 6] (kind "f2": n even)"""
        n = len(R)
        assert kind != "f2" or n % 2 == 0, "the packed form takes an even number of problems"
        dtype = np.float64 if kind == "f64" else np.float32
        return self._run(f"devsim_log6_{kind}", (ctypes.c_int64(n),), dtype, (6, n), R.T, p.T).T


def test_devsim_cross_compiles():
    # nvcc cross-compiles for sm_100a without a GPU: a header change that breaks the device forms fails here first
    assert os.path.getsize(build_devsim()) > 0


@pytest.fixture(scope="module")
def dev():
    return DevSim()


def _ulp32(ref):
    return np.spacing(np.abs(ref).astype(np.float32)).astype(np.float64)


def _operands(rng, lo, hi, n):
    """log-uniform over [lo, hi], with both ends"""
    x = np.exp(rng.uniform(np.log(lo), np.log(hi), n))
    x[:2] = lo, hi
    return x


# ------------------------------------------------------------------------------------------------------ MUFU forms
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["f32", "f2"])
def test_fp32_mufu_forms_within_two_ulp(dev, kind):
    # rsqrt / rcp / sqrt .approx.ftz.f32: <= 2 ulp over the operands the kernels give them (pivots floored at
    # Num<float>::kPivotFloor = 1e-30, up to 1e12); div_ = a * rcp_(b): the reciprocal's 2 ulp + the product's rounding
    rng = np.random.default_rng(1)
    n = 1 << 20
    x = _operands(rng, 1e-30, 1e12, n).astype(np.float32)
    xl = x.astype(LD)
    worst = {}
    for op, ref in (("rsqrt", 1 / np.sqrt(xl)), ("rcp", 1 / xl), ("sqrt", np.sqrt(xl))):
        got = dev.scalar(op, kind, x)
        worst[op] = float(np.max(np.abs(got.astype(LD) - ref) / _ulp32(ref.astype(np.float64))))
        if op == "rcp":                                                          # negative operands (rcp_capped)
            gn = dev.scalar(op, kind, -x)
            worst[op] = max(worst[op], float(np.max(np.abs(gn.astype(LD) + ref) / _ulp32(ref.astype(np.float64)))))
    a = (rng.uniform(-1, 1, n) * _operands(rng, 1e-6, 1e6, n)).astype(np.float32)
    q = a.astype(LD) / xl
    ok = (np.abs(q) > 1e-37) & (np.abs(q) < 1e37)
    got = dev.scalar("div", kind, a, x)
    rel_div = float(np.max(np.abs(got.astype(LD)[ok] - q[ok]) / np.abs(q[ok])))
    print(f"{kind}: max error in ulp {worst}; div_ max relative error {rel_div:.3e} = {rel_div / 2 ** -23:.2f} * 2^-23")
    for op, w in worst.items():
        assert w <= 2.0, (op, w)
    assert rel_div <= 2.5 * 2 ** -23 * (1 + 1e-6)


@pytest.mark.gpu
def test_fp64_seed_and_step_forms(dev):
    # rcp_ / rsqrt_: MUFU seed + one third-order step, 1.1e-16 / 1.4e-16 relative (gik_core.cuh, DESIGN.md) over the
    # floors (kPivotFloor = 1e-280) to 1e12; sqrt_ is the IEEE sqrt; div_ = a * rcp_(b)
    rng = np.random.default_rng(2)
    n = 1 << 20
    x = _operands(rng, 1e-280, 1e12, n)
    xl = x.astype(LD)
    rel = {}
    for op, ref in (("rcp", 1 / xl), ("rsqrt", 1 / np.sqrt(xl)), ("sqrt", np.sqrt(xl))):
        got = dev.scalar(op, "f64", x)
        rel[op] = float(np.max(np.abs(got.astype(LD) - ref) / ref))
    gn = dev.scalar("rcp", "f64", -x)
    rel["rcp"] = max(rel["rcp"], float(np.max(np.abs(gn.astype(LD) + 1 / xl) * xl)))
    a = rng.uniform(-1, 1, n) * _operands(rng, 1e-6, 1e6, n)
    q = a.astype(LD) / xl
    ok = (np.abs(q) > 1e-300) & (np.abs(q) < 1e300)
    got = dev.scalar("div", "f64", a, x)
    rel["div"] = float(np.max(np.abs(got.astype(LD)[ok] - q[ok]) / np.abs(q[ok])))
    print(f"fp64 max relative error {rel}")
    assert rel["rcp"] <= 1.1e-16 * 1.01
    assert rel["rsqrt"] <= 1.45e-16
    assert rel["sqrt"] <= U64 * 1.0001                                          # correctly rounded
    assert rel["div"] <= 1.1e-16 * 1.01 + U64


# ------------------------------------------------------------------------------------------------------ sin / cos
def _joint_arg_range(table):
    psi = float(np.max(np.abs(np.arctan2(table.hand_R[:, 1, 0], table.hand_R[:, 0, 0]))))
    return float(np.min(table.lower)) - psi, float(np.max(table.upper)) + psi


# __sincosf: the CUDA Programming Guide documents 2^-21.41 = 3.6e-7 absolute for __sinf / __cosf on [-pi, pi]; measured
# on an NVIDIA B200 (1000 W) against the exact sin / cos of the fp32 argument: 4.0e-7 there, so the bar is the header's
# own claim (5e-7).  Beyond +-pi nothing is documented: over the joint-argument range [min lower - |tip_psi|, max upper
# + |tip_psi|] = [-5.15, 4.71] the same card measured 7.1e-7, which is the bar.  (The solve-step bound of
# test_gpu_solve_steps.py is calibrated on starts that put the arguments there.)  The accurate sincosf: 1.5 ulp.
SINCOSF_PI_ABS = 5e-7
SINCOSF_JOINT_RANGE_ABS = 7.5e-7


@pytest.mark.gpu
def test_fp32_sincos(dev, table):
    rng = np.random.default_rng(3)
    n = 1 << 20
    lo, hi = _joint_arg_range(table)
    assert lo < -PI and hi > PI
    worst = {}
    for name, x in (("pi", rng.uniform(-PI, PI, n).astype(np.float32)),
                    ("joint", rng.uniform(lo, hi, n).astype(np.float32))):
        xl = x.astype(LD)
        rs, rc = np.sin(xl), np.cos(xl)
        for op in ("sincos_fast", "sincos"):
            s, c = dev.scalar(op, "f32", x)
            err_abs = float(max(np.max(np.abs(s - rs)), np.max(np.abs(c - rc))))
            err_ulp = float(max(np.max(np.abs(s - rs) / _ulp32(rs.astype(np.float64))),
                                np.max(np.abs(c - rc) / _ulp32(rc.astype(np.float64)))))
            worst[(name, op)] = (err_abs, err_ulp)
    print("fp32 sincos (abs, ulp): " + ", ".join(f"{k}: {v[0]:.3e} / {v[1]:.1f}" for k, v in worst.items()))
    assert worst[("pi", "sincos_fast")][0] <= SINCOSF_PI_ABS
    assert worst[("joint", "sincos_fast")][0] <= SINCOSF_JOINT_RANGE_ABS
    for rng_name in ("pi", "joint"):                                        # sincosf: 2 ulp (CUDA Programming Guide)
        assert worst[(rng_name, "sincos")][1] <= 2.0


@pytest.mark.gpu
def test_fp64_sincos(dev, table):
    # the constant-bank Cody-Waite form on [-pi, pi], the joint-argument range and |x| <= 1e6, against the exact values:
    # measured 1.7e-16 absolute on an NVIDIA B200 (1000 W), the library sincos 1.3e-16
    rng = np.random.default_rng(4)
    n = 1 << 20
    lo, hi = _joint_arg_range(table)
    worst = {}
    for name, x in (("pi", rng.uniform(-PI, PI, n)), ("joint", rng.uniform(lo, hi, n)),
                    ("1e6", rng.uniform(-1e6, 1e6, n))):
        xl = x.astype(LD)
        rs, rc = np.sin(xl), np.cos(xl)
        for op in ("sincos_fast", "sincos"):
            s, c = dev.scalar(op, "f64", x)
            worst[(name, op)] = float(max(np.max(np.abs(s - rs)), np.max(np.abs(c - rc))))
    print("fp64 sincos max abs error: " + ", ".join(f"{k}: {v:.3e}" for k, v in worst.items()))
    for name in ("pi", "joint", "1e6"):
        assert worst[(name, "sincos_fast")] <= 1.8e-16, name
        assert worst[(name, "sincos")] <= 2 * 2 * U64, name


# ------------------------------------------------------------------------------------------------------ atan2_pos
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["f32", "f64", "f2"])
def test_atan2_pos(dev, kind):
    # y >= 0 (log6's |vee(R - R^T)| / 2), every ratio magnitude, both signs of x, tiny angles.  Against the exact
    # atan2 of the rounded arguments, measured on an NVIDIA B200 (1000 W): fp32 (scalar and packed) 3.0e-7 -- the
    # polynomial's 1.1e-7, the MUFU reciprocal of the ratio and the rounding of results up to pi (ulp 2.4e-7);
    # fp64 4.46e-16
    rng = np.random.default_rng(5)
    n = 1 << 20
    y = np.exp2(-60 * rng.random(n)) * rng.random(n)
    x = 2 * rng.random(n) - 1
    y[:4] = [0.0, 0.0, 1.0, 1e-30]; x[:4] = [1.0, -1.0, 0.0, 1e-30]
    dt = np.float64 if kind == "f64" else np.float32
    y, x = y.astype(dt), x.astype(dt)
    ref = np.arctan2(y.astype(LD), x.astype(LD))
    got = dev.scalar("atan2", kind, y, x).astype(LD)
    err = np.abs(got - ref)
    print(f"atan2_pos {kind}: max abs error {float(err.max()):.3e}")
    assert float(err.max()) <= (4.5e-16 if kind == "f64" else 3.2e-7)


# ------------------------------------------------------------------------------------------------------ log6
NEAR_PI_SWITCH = PI - 1e-2                      # log6_near_pi


def log6_ref(R, p, series_t2=0.0):
    """log6 of the rounded inputs in longdouble, the function the kernels evaluate: theta = atan2(|vee(R - R^T)| / 2,
    (tr R - 1) / 2), alpha / beta in their closed forms (the same cot(theta/2) branch on the sign of c), pinocchio's
    diagonal form of w from theta >= pi - 1e-2; alpha / beta from their series below theta^2 = series_t2 (the kernel's
    Num<T>::kSeriesT2).  R [n, 9], p [n, 3] -> e [n, 6], theta [n]."""
    R = R.astype(LD); p = p.astype(LD)
    v = np.stack([R[:, 7] - R[:, 5], R[:, 2] - R[:, 6], R[:, 3] - R[:, 1]], 1)
    c = np.clip((R[:, 0] + R[:, 4] + R[:, 8] - 1) / 2, -1, 1)
    s = np.sqrt((v * v).sum(1)) / 2
    th = np.arctan2(s, c)
    w = np.where((s > 0)[:, None], (th / (2 * np.where(s > 0, s, 1)))[:, None] * v, v / 2)
    front = c >= 0
    alpha = np.where(s > 0, th / 2 * np.where(front, 1 + c, s) / np.where(front, np.where(s > 0, s, 1), 1 - c), 1)
    t2 = th * th
    beta = np.where(t2 > 0, (1 - alpha) / np.where(t2 > 0, t2, 1), LD(1) / 12)
    small = t2 < 1e-6                                              # (longdouble cancellation in 1 - alpha)
    beta[small] = LD(1) / 12 + t2[small] / 720
    ser = t2 < series_t2
    z = t2[ser]
    alpha[ser] = 1 - z * (LD(1) / 12 + z * (LD(1) / 720 + z / 30240))
    beta[ser] = LD(1) / 12 + z * (LD(1) / 720 + z * (LD(1) / 30240 + z / 1209600))
    near = th >= NEAR_PI_SWITCH
    if near.any():
        cphi = -c[near]
        b2 = th[near] ** 2 / (1 + cphi)
        d = R[near][:, [0, 4, 8]]
        t = (d + cphi[:, None]) * b2[:, None]
        w[near] = np.where(v[near] > 0, 1, -1) * np.sqrt(np.maximum(t, 0))
    wp = beta * (w * p).sum(1)
    lin = alpha[:, None] * p - 0.5 * np.cross(w, p) + wp[:, None] * w
    return np.concatenate([lin, w], 1), th


def exp6_ld(xi):
    """SE3 exp of [v; w] in longdouble -> R [n, 9], p [n, 3]"""
    xi = np.asarray(xi, LD)
    v, w = xi[:, :3], xi[:, 3:]
    th = np.sqrt((w * w).sum(1))
    K = np.zeros((len(xi), 3, 3), LD)
    K[:, 0, 1], K[:, 0, 2], K[:, 1, 2] = -w[:, 2], w[:, 1], -w[:, 0]
    K[:, 1, 0], K[:, 2, 0], K[:, 2, 1] = w[:, 2], -w[:, 1], w[:, 0]
    K2 = K @ K
    ts = np.where(th > 0, th, 1)
    a = np.where(th > 1e-4, np.sin(ts) / ts, 1 - th ** 2 / 6)
    b = np.where(th > 1e-4, (1 - np.cos(ts)) / ts ** 2, 0.5 - th ** 2 / 24)
    cc = np.where(th > 1e-4, (ts - np.sin(ts)) / ts ** 3, LD(1) / 6 - th ** 2 / 120)
    I = np.eye(3, dtype=LD)[None]
    R = I + a[:, None, None] * K + b[:, None, None] * K2
    V = I + b[:, None, None] * K + cc[:, None, None] * K2
    return R.reshape(-1, 9), np.einsum("nij,nj->ni", V, v)


# theta sweep (log-spaced 1e-7 ... 3) with points on both sides of each switch: the fp32 series (theta^2 = 0.25), the
# fp64 series (theta^2 = 1e-4), the near-pi form (pi - 1e-2), and pi - 1e-4
THETA_SWITCHES = [0.5, 0.01, NEAR_PI_SWITCH]
THETAS = np.unique(np.concatenate([np.geomspace(1e-7, 3.0, 60)] + [[t * (1 - 1e-3), t * (1 + 1e-3)] for t in THETA_SWITCHES]
                                  + [[PI - 1e-4, PI - 2e-3]]))
PNORMS = np.concatenate([[0.0], np.geomspace(1e-7, 0.5, 12)])


def log6_sweep(seed, per=8):
    """(xi [n, 6], theta [n]) over THETAS x PNORMS, random axes with every component >= 0.1 in magnitude (the sign
    of a near-zero axis component is rounding noise near pi) and random directions of the translation"""
    rng = np.random.default_rng(seed)
    rows = []
    for th in THETAS:
        for pn in PNORMS:
            for _ in range(per):
                ax = rng.uniform(0.1, 1.0, 3) * rng.choice([-1.0, 1.0], 3)
                ax /= np.linalg.norm(ax)
                d = rng.standard_normal(3); d /= np.linalg.norm(d)
                rows.append(np.concatenate([pn * d, th * ax]))
    xi = np.array(rows)
    return xi, np.linalg.norm(xi[:, 3:], axis=1)


# Bars, measured on an NVIDIA B200 (1000 W): |e - e_ref| / (u (1 + |p|)), u the unit roundoff, is at most 1.0 below
# theta = 0.5 in every form -- the packed form without the series included, the accuracy DESIGN.md argues for (about
# 1e-7 (1 + |p|) in fp32) -- and 6.8 (fp32, F2) / 7.2 (fp64) from 0.5 to pi - 1e-2, where theta's own error (atan2 and
# the rounding of theta ~ 3) dominates.  Near pi (pinocchio's diagonal form) the largest absolute error is 3.9e-7 (fp32,
# F2) and 5.9e-16 (fp64).
LOG6_SMALL_K = 1.5                              # theta < 0.5
LOG6_FAR_K = {"f32": 8.0, "f2": 8.0, "f64": 8.0}
LOG6_NEAR_PI_ABS = {"f32": 6e-7, "f2": 6e-7, "f64": 1e-15}


def test_log6_reference_in_longdouble_matches_exp6():
    # the reference inverts exp6 far from pi (where it is the principal log): a check of the reference itself
    xi, th = log6_sweep(7, per=2)
    R, p = exp6_ld(xi)
    e, th_r = log6_ref(R, p)
    far = th < 3.0
    assert np.abs(e[far] - xi[far].astype(LD)).max() < 1e-15
    assert np.abs(th_r - th).max() < 1e-15


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["f32", "f2", "f64"])
def test_log6_on_device(dev, kind):
    xi, _ = log6_sweep(8)
    R, p = exp6_ld(xi)
    dt = np.float64 if kind == "f64" else np.float32
    R, p = R.astype(dt), p.astype(dt)
    e_ref, th = log6_ref(R, p)
    e_ref64 = log6_ref(R.astype(np.float64), p.astype(np.float64))[0]
    assert np.abs((e_ref64 - e_ref).astype(np.float64)).max() < 1e-12          # longdouble and fp64 references agree
    got = dev.log6(kind, R, p)
    err = np.abs(got.astype(LD) - e_ref).max(axis=1).astype(np.float64)
    pn = np.linalg.norm(p.astype(np.float64), axis=1)
    u = U64 if kind == "f64" else U32
    near = th.astype(np.float64) >= NEAR_PI_SWITCH
    k_far = err[~near] / (u * (1 + pn[~near]))
    bands = {"theta<1e-3": th < 1e-3, "1e-3..0.5": (th >= 1e-3) & (th < 0.5), "0.5..pi-1e-2": (th >= 0.5) & ~near}
    print(f"log6 {kind}: max err / (u (1 + |p|)) far from pi {k_far.max():.2f} (by band: "
          + ", ".join(f"{b} {(err[m] / (u * (1 + pn[m]))).max():.2f}" for b, m in bands.items())
          + f"); near pi max abs error {err[near].max():.3e}")
    assert k_far.max() <= LOG6_FAR_K[kind]
    small = th < 0.5
    assert (err[small] / (u * (1 + pn[small]))).max() <= LOG6_SMALL_K
    assert err[near].max() <= LOG6_NEAR_PI_ABS[kind]
