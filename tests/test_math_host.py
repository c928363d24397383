"""r2ik_math.cuh on the host: accuracy and IEEE special cases of the straight-line atan2 that the
kernels use instead of the CUDA library routine.  The host build takes the exact library operation
wherever the source branches on __CUDA_ARCH__ ('/' and sqrt where the device uses a MUFU seed + Newton
steps), so these tests check the polynomials and the octant logic only; the device arithmetic itself
is compared with references in tests/test_gpu_math.py."""
import ctypes as C
import math
import os
import re
import subprocess

import numpy as np
import pytest

from parity import REPO

HS_DIR = os.path.join(REPO, "tests", "hostsim")


@pytest.fixture(scope="module")
def hs():
    subprocess.run(["make", "-C", HS_DIR], check=True, capture_output=True)
    return C.CDLL(os.path.join(HS_DIR, "_build", "libr2ik_hostsim.so"))


def run(hs, y, x):
    y = np.ascontiguousarray(y, dtype=np.float64)
    x = np.ascontiguousarray(x, dtype=np.float64)
    out = np.empty_like(y)
    ok = np.empty(len(y), np.uint8)
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    hs.hs_atan2_core(dp(y), dp(x), C.c_int64(len(y)), dp(out), ok.ctypes.data_as(C.POINTER(C.c_uint8)))
    return out, ok.astype(bool)


def test_atan2_core_accuracy_vs_mpmath(hs):
    mp = pytest.importorskip("mpmath")
    mp.mp.dps = 40
    rng = np.random.default_rng(0)
    ang = rng.uniform(-np.pi, np.pi, 20000)
    r = 10.0 ** rng.uniform(-12, 3, ang.size)
    y, x = r * np.sin(ang), r * np.cos(ang)
    # octant boundaries and tiny ratios
    y = np.concatenate([y, [1.0, 1.0, 0.41421356237309503, 0.4142135623730951, 1e-300 * 1e20, 1e-17, -1e-17]])
    x = np.concatenate([x, [1.0, -1.0, 1.0, 1.0, 1.0, 1.0, -1.0]])
    got, ok = run(hs, y, x)
    assert ok.all()
    worst = 0.0
    for yi, xi, gi in zip(y, x, got):
        want = mp.atan2(mp.mpf(float(yi)), mp.mpf(float(xi)))
        ulp = math.ulp(float(want)) if want != 0 else 5e-324
        worst = max(worst, float(abs(mp.mpf(float(gi)) - want)) / ulp)
    assert worst <= 3.0, f"atan2_core max error {worst:.2f} ulp"   # measured 2.2 (single-double pi in pi - r)
    # and against libm over a large sample
    ang = rng.uniform(-np.pi, np.pi, 1_000_000)
    y, x = np.sin(ang), np.cos(ang)
    got, ok = run(hs, y, x)
    assert ok.all()
    assert np.max(np.abs(got - np.arctan2(y, x))) < 1e-15


def test_atan2_core_special_cases(hs):
    pz, nz = 0.0, -0.0
    cases = [(pz, 1.0), (nz, 1.0), (pz, -1.0), (nz, -1.0), (1.0, pz), (1.0, nz), (-1.0, pz), (-1.0, nz),
             (pz, pz), (nz, pz), (pz, nz), (nz, nz), (3e-200, -2.0), (-3e-200, -2.0), (2.0, 3e-200), (5.0, 5.0), (-5.0, -5.0)]
    y = np.array([c[0] for c in cases])
    x = np.array([c[1] for c in cases])
    got, ok = run(hs, y, x)
    assert ok.all()
    want = np.arctan2(y, x)
    assert np.array_equal(got, want) or np.max(np.abs(got - want)) < 4e-16
    assert np.array_equal(np.signbit(got), np.signbit(want))   # signed zeros / +-pi


def test_atan2_core_ok_rejects_out_of_range(hs):
    y = np.array([5e-324, 1e-310, 1e308, np.inf, np.nan, 1.0])
    x = np.array([0.0, 1e-312, 1e308, 1.0, 1.0, np.inf])
    _, ok = run(hs, y, x)
    assert not ok.any()


def test_angle_of_unit_vs_mpmath(hs):
    """atan2 of a normalised vector without the division (used for the angles whose (cos, sin) the
    solver needs anyway): a few 1e-16 rad absolute against the true atan2 of the un-normalised input."""
    mp = pytest.importorskip("mpmath")
    mp.mp.dps = 40
    rng = np.random.default_rng(1)
    ang = rng.uniform(-np.pi, np.pi, 20000)
    r = 10.0 ** rng.uniform(-6, 2, ang.size)
    y, x = r * np.sin(ang), r * np.cos(ang)
    y = np.concatenate([y, [0.0, -0.0, 0.0, -0.0, 1.0, -1.0, 1.0, 1.0, 0.38268343236508978, 1e-9]])
    x = np.concatenate([x, [1.0, 1.0, -1.0, -1.0, 0.0, 0.0, 1.0, -1.0, 0.92387953251128674, 1.0]])
    out = np.empty_like(y)
    dp = lambda a: np.ascontiguousarray(a).ctypes.data_as(C.POINTER(C.c_double))
    y = np.ascontiguousarray(y); x = np.ascontiguousarray(x)
    hs.hs_angle_of_unit(dp(y), dp(x), C.c_int64(len(y)), dp(out))
    want = np.arctan2(y, x)
    assert np.array_equal(np.signbit(out), np.signbit(want))
    worst_abs, worst_rel = 0.0, 0.0
    assert np.max(np.abs(out - want)) < 1e-15          # incl. the signed-zero cases (+-pi, +-0)
    for yi, xi, gi in zip(y, x, out):
        if yi == 0.0:
            continue                                     # mpmath has no signed zero
        w = mp.atan2(mp.mpf(float(yi)), mp.mpf(float(xi)))
        e = float(abs(mp.mpf(float(gi)) - w))
        worst_abs = max(worst_abs, e)
        if w != 0:
            worst_rel = max(worst_rel, e / float(abs(w)))
    assert worst_abs < 1e-15, worst_abs
    assert worst_rel < 2e-15, worst_rel     # small angles keep relative accuracy (asin(u) ~ u)


def test_sincos_small_vs_mpmath(hs):
    mp = pytest.importorskip("mpmath")
    mp.mp.dps = 40
    rng = np.random.default_rng(2)
    x = np.concatenate([rng.uniform(-4, 4, 20000), rng.uniform(-40, 40, 5000), rng.uniform(-1000, 1000, 2000), [0.0, -0.0, np.pi, -np.pi, np.pi / 2, -np.pi / 2, np.pi / 4, 3 * np.pi / 4,
                                                     1e-300, 1e-9, 4.0, -4.0, 0.7417649320975901]])
    x = np.ascontiguousarray(x)
    sn = np.empty_like(x); cs = np.empty_like(x)
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    hs.hs_sincos_small(dp(x), C.c_int64(len(x)), dp(sn), dp(cs))
    worst = 0.0
    for xi, si, ci in zip(x, sn, cs):
        ws, wc = mp.sin(mp.mpf(float(xi))), mp.cos(mp.mpf(float(xi)))
        # absolute error in units of the ulp of max(|value|, 2^-54): near a zero of sin / cos the
        # two-piece reduction keeps ~1e-33 absolute accuracy, far below what any consumer resolves
        for got, want in ((si, ws), (ci, wc)):
            scale = max(abs(float(want)), 2.0 ** -54)
            worst = max(worst, float(abs(mp.mpf(float(got)) - want)) / (scale * 2.0 ** -52))
    assert worst < 2.0, worst
    assert np.max(np.abs(sn - np.sin(x))) < 3e-16 and np.max(np.abs(cs - np.cos(x))) < 3e-16


# Every call of the math routines whose domain has no validity predicate, with the reason its argument is inside the
# domain.  div_fast / rcp_fast: 2^-1022 <= |divisor| < 2^1022 (rcp.approx.ftz flushes a smaller reciprocal to zero);
# sqrt_nonneg / sqrt_rsqrt_nonneg: +-0 or a finite normal number (the root of +inf is NaN on the device).  A new call
# site fails this test until its argument has been argued into the domain here.
GUARDED_CALLS = {
    ("r2ik_math.cuh", "div_fast(num, den)"): "atan2_core: atan2_core_ok keeps den = mx or mn + mx below 2^1022",
    ("r2ik_device.cuh", "div_fast(1.0 - ux, uy * uy + uz * uz)"): "rmfv_columns: unit vector, not within isclose of +-e_x",
    ("r2ik_device.cuh", "div_fast(d_target, fabs(d) + A.proj_margin)"): "reduce_goal: d = |w - s| of a projected goal, >= margin",
    ("r2ik_device.cuh", "div_fast(A.max_arm_length, sqrt_nonneg(dg2) + A.proj_margin)"): "reach_prechecks: dg2 < inf tested",
    ("r2ik_device.cuh", "rcp_fast(2.0 * qa)"): "literal circle intersection: qa = |v|^2 of a unit direction",
    ("r2ik_device_f32.cuh", "div_fast(A64.d_min, d + A64.proj_margin)"): "FP32 front end: d < d_min, >= margin",
    ("r2ik_control.cuh", "sqrt_nonneg(cross ? s2 : 0.0)"): "interval plan: s2 = R^2 - C^2 of unit-scale coefficients",
    ("r2ik_device.cuh", "sqrt_nonneg(q12 * q12 + q22 * q22)"): "orbita3d clamp: entries of a rotation, <= 1",
    ("r2ik_device.cuh", "sqrt_nonneg(rad)"): "elbow_circle: negative rad is NaN by the select; |rad| <= 4 d^2 L1^2",
    ("r2ik_device.cuh", "sqrt_nonneg(dg2)"): "reach_prechecks: under the dg2 < inf test",
    ("r2ik_device.cuh", "sqrt_rsqrt_nonneg(dx * dx + dy * dy + dz * dz, invd)"):
        "solve_core: |w - s|^2 is finite (goal inside the reach sphere, orthonormal rotation); a wrist within ~1.5e-154 m "
        "of the shoulder gives a subnormal square and an inexact d, but then d < d_min: reduce_goal divides by "
        "|d| + proj_margin and d is recomputed from the pushed-out wrist",
    ("r2ik_device.cuh", "sqrt_nonneg(dl)"): "fast circle linking: dl >= 0 in that branch, O(1)",
    ("r2ik_device.cuh", "sqrt_nonneg(disc)"): "literal circle intersection: disc >= 0 in that branch, O(1)",
    ("r2ik_device_f32.cuh", "sqrt_rsqrt_nonneg(d2, invd64)"):
        "FP32 front end / reach map: 0 <= d2 < d_min^2; a subnormal d2 (wrist within ~1.5e-154 m of the shoulder) "
        "gives an inexact d, but such a pose is escalated (d2 <= 1e-12) and only |d| + proj_margin divides",
}


def test_call_sites_of_unguarded_routines():
    """The device calls of div_fast, rcp_fast, sqrt_nonneg and sqrt_rsqrt_nonneg are exactly the ones listed in
    GUARDED_CALLS (test_gpu_math.py measures the routines inside their domains)."""
    csrc = os.path.join(REPO, "reachy2_symbolic_ik_b200", "csrc")
    call = re.compile(r"\b(div_fast|rcp_fast|sqrt_nonneg|sqrt_rsqrt_nonneg)\(")
    found = set()
    for f in sorted(os.listdir(csrc)):
        if not f.endswith((".cuh", ".cu")):
            continue
        for line in open(os.path.join(csrc, f)):
            code = line.split("//")[0]
            if "R2IK_HD" in code:
                continue                                   # the definitions
            for m in call.finditer(code):
                depth, k = 0, m.end() - 1
                while True:                                # the call up to its closing parenthesis
                    depth += {"(": 1, ")": -1}.get(code[k], 0)
                    if depth == 0:
                        break
                    k += 1
                found.add((f, code[m.start():k + 1]))
    assert found == set(GUARDED_CALLS), (f"unlisted: {sorted(found - set(GUARDED_CALLS))}\n"
                                         f"gone: {sorted(set(GUARDED_CALLS) - found)}")
