"""Scalar device functions checked without a GPU.  atan2_pos: the host build of csrc/gik_core.cuh runs the same
polynomial as the device.  fp64 sincos: device-only code (constant-bank coefficients), so its algorithm is re-executed
here in numpy from the coefficients PARSED OUT of the header -- an edited coefficient or reduction constant fails this
test before it reaches a GPU (test_gpu_device_functions.py measures the device forms themselves on the GPU)."""
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CORE = os.path.join(ROOT, "motion-planning-and-control-for-dual-manipulator-robot_b200", "csrc", "gik_core.cuh")


def test_atan2_pos_polynomials(hostsim):
    rng = np.random.default_rng(0)
    n = 200_000
    # every magnitude of the ratio, both signs of x, tiny angles (relative accuracy matters: theta / sin theta in log6)
    y = np.exp2(-60 * rng.random(n)) * rng.random(n)
    x = 2 * rng.random(n) - 1
    y[:4] = [0.0, 0.0, 1.0, 1e-300]; x[:4] = [1.0, -1.0, 0.0, 1e-300]
    ref = np.arctan2(y, x)
    got = hostsim.atan2_pos(y, x, np.float64)
    assert np.abs(got - ref).max() < 6e-16
    nz = ref > 0
    assert (np.abs(got - ref)[nz] / ref[nz]).max() < 5e-16
    got32 = hostsim.atan2_pos(y, x, np.float32).astype(np.float64)
    ref32 = np.arctan2(y.astype(np.float32).astype(np.float64), x.astype(np.float32).astype(np.float64))
    assert np.abs(got32 - ref32).max() < 4e-7


def _split(a):
    t = 134217729.0 * a          # Veltkamp split, 2^27 + 1
    hi = t - (t - a)
    return hi, a - hi


def _fma(a, b, c):
    """a * b + c with the product carried exactly (Dekker's TwoProduct + TwoSum): within an ulp of a hardware FMA,
    which is what the Cody-Waite step needs (kd * (pi/2 high) has up to 73 significant bits)."""
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64); c = np.asarray(c, np.float64)
    p = a * b
    ah, al = _split(a); bh, bl = _split(b)
    e = ((ah * bh - p) + ah * bl + al * bh) + al * bl          # p + e == a * b exactly
    s = p + c
    bb = s - p
    t = (p - (s - bb)) + (c - bb)                               # s + t == p + c exactly
    return s + (t + e)


def test_fp64_sincos_algorithm_from_header_coefficients():
    src = open(CORE).read()
    body = re.search(r"kSinCos64\[18\]\s*=\s*\{(.*?)\};", src, re.S).group(1)
    body = re.sub(r"//[^\n]*", "", body)
    K = [float(t) for t in body.replace("\n", " ").split(",") if t.strip()]
    assert len(K) == 18
    assert K[0] == 2 / np.pi and K[1] == 1.5 * 2.0 ** 52 and K[16] == -0.5 and K[17] == 1.0
    assert abs((-K[2] - K[3]) - np.pi / 2) < 1e-16 and -K[2] == np.float64(np.pi / 2)      # two-term pi/2
    for rng_max in (3.6, 100.0, 1e6):
        x = np.random.default_rng(1).uniform(-rng_max, rng_max, 200_000)
        t = _fma(x, K[0], K[1])
        kd = t - K[1]
        k = kd.astype(np.int64)
        r = _fma(kd, K[3], _fma(kd, K[2], x))
        z = r * r
        ps = _fma(K[9], z, K[8])
        for c in (K[7], K[6], K[5], K[4]):
            ps = _fma(ps, z, c)
        pc = _fma(K[15], z, K[14])
        for c in (K[13], K[12], K[11], K[10]):
            pc = _fma(pc, z, c)
        sr = _fma(r * z, ps, r)
        cr = _fma(z * z, pc, _fma(z, K[16], K[17]))
        odd = (k & 1) == 1
        s = np.where(odd, cr, sr) * np.where((k & 2) != 0, -1.0, 1.0)
        c = np.where(odd, sr, cr) * np.where(((k + 1) & 2) != 0, -1.0, 1.0)
        assert np.abs(r).max() <= np.pi / 4 + 1e-3      # (+ 2^-11 * pi/2: double rounding of the emulated FMA at the magic constant)
        assert np.abs(s - np.sin(x)).max() < 3e-16 and np.abs(c - np.cos(x)).max() < 3e-16
