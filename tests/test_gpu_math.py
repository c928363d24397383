"""The solver's elementary routines as the B200 runs them, against high-precision references.

tests/hostsim and test_math_host.py compile these headers for the CPU, where every `__CUDA_ARCH__` branch takes the
exact library operation ('/', sqrt, correctly rounded FP32).  Here tests/devmath/devmath.cu runs the device code -- MUFU
seeds with their Newton steps, the `.approx.ftz` FP32 instructions, the out-of-line library sincos -- built with the
flags of libr2ik.so, one kernel per routine.

Inputs: random O(1) values; every binade from 2^-1074 to 2^1023 (float32: 2^-149 to 2^127) with random mantissas, both
signs; +-0, +-inf and NaN; one ulp either side of each threshold the validity predicates test.  Wherever a routine's
stated domain or its `_ok` predicate holds, the error stays within the bound its header comment states; where a domain
has no predicate, the call sites that feed it are listed in test_math_host.py::test_call_sites_of_unguarded_routines.
"""
import ctypes as C
import hashlib
import math
import os
import subprocess

import mpmath as mp
import numpy as np
import pytest

from parity import REPO

pytestmark = pytest.mark.gpu

DM_DIR = os.path.join(REPO, "tests", "devmath")
CSRC = os.path.join(REPO, "reachy2_symbolic_ik_b200", "csrc")
TWO_PI = 2.0 * math.pi

# high words of the thresholds in the predicates: smallest normal, the sqrt seed clamp, the 1e-280 / 1e280 window of
# cs_of_atan2, and the upper bound of atan2_core_ok together with the binade above it
HI_WORDS = (0x00100000, 0x00300000, 0x05E00000, 0x7A000000, 0x7FC00000, 0x7FD00000)

# FP32 bounds.  The .approx instructions are used as they are, so their bounds are the PTX ISA's (instruction set
# reference, "rcp", "sqrt", "rsqrt": .approx.f32 accuracy over the full range).
RCP_F_ULP = 1.0                  # rcp.approx.f32: 1 ulp
SQRT_F_REL = 2.0 ** -23          # sqrt.approx.f32: relative 2^-23
RSQRT_F_REL = 2.0 ** -22.9       # rsqrt.approx.f32: relative 2^-22.9
# sincos_f, angle_of_unit_f and cs_and_angle_f feed the FP32 solve, whose decision bands (kBandLen, kBandSin, kMinH2 in
# r2ik_device_f32.cuh) are sized for "a few 1e-7" of accumulated rounding on O(1) quantities: each of these routines
# may take two float32 ulps of pi/2 .. pi of that budget.
ANGLE_F_ABS = 2.0 * float(np.spacing(np.float32(np.pi)))      # 4.8e-7 rad
SINCOS_F_ABS = 2.0 * float(np.spacing(np.float32(1.0)))       # 2.4e-7
SINCOS_F_RANGE = 64.0            # symik_pose_fast escalates |theta| > 64 (R2IK_ESC 17) before calling sincos_f


# ------------------------------------------------------------------------------------------------------------ plumbing
@pytest.fixture(scope="module")
def dm():
    """Build tests/devmath/devmath.cu with the flags of libr2ik.so (-O3, FMA contraction on: a probe built with other
    flags would test other code).  R2IK_DEVMATH_CSRC names another copy of the csrc headers to compile against (a
    patched copy, to see which test catches a change); the default is the package's own."""
    from reachy2_symbolic_ik_b200.build import NVCC_FLAGS, nvcc_path

    csrc = os.path.abspath(os.environ.get("R2IK_DEVMATH_CSRC", CSRC))
    tag = hashlib.sha1(csrc.encode()).hexdigest()[:10]
    out_dir = os.path.join(DM_DIR, "_build")
    os.makedirs(out_dir, exist_ok=True)
    lib = os.path.join(out_dir, f"libdevmath_{tag}.so")
    cmd = [nvcc_path(), *NVCC_FLAGS, "-I", csrc, "-o", lib, os.path.join(DM_DIR, "devmath.cu")]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, f"nvcc failed:\n{' '.join(cmd)}\n{res.stdout}\n{res.stderr}"
    return C.CDLL(lib)


_TORCH_DTYPES = {np.dtype(np.float64): "float64", np.dtype(np.float32): "float32", np.dtype(np.uint8): "uint8",
                 np.dtype(np.int32): "int32"}


def run(dm, name, inputs, out_dtypes):
    """dm_<name>(inputs..., outputs..., n, stream) on device copies of `inputs`; returns the outputs as numpy arrays."""
    import torch

    n = len(inputs[0])
    ins = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in inputs]
    outs = [torch.empty(n, dtype=getattr(torch, _TORCH_DTYPES[np.dtype(dt)]), device="cuda") for dt in out_dtypes]
    stream = torch.cuda.current_stream()
    fn = getattr(dm, "dm_" + name)
    err = fn(*[C.c_void_p(t.data_ptr()) for t in ins + outs], C.c_int64(n), C.c_void_p(stream.cuda_stream))
    assert err == 0, f"dm_{name}: launch failed with cudaError {err}"
    stream.synchronize()
    return [t.cpu().numpy() for t in outs]


def report(name, n, lines):
    msg = "\n  ".join([f"[device {name}] n={n}"] + lines)
    print(msg)
    return msg


def worst_line(what, err, mask, bound, unit, *args):
    """'what: worst <e> unit at (args) (bound b)' over err[mask]."""
    if not mask.any():
        return f"{what}: no inputs"
    e = np.where(mask, err, -np.inf)
    i = int(np.argmax(e))
    at = ", ".join(f"{float(a[i])!r}" for a in args)
    return f"{what}: worst {float(e[i]):.3g} {unit} at ({at}) over {int(mask.sum())} inputs (bound {bound:g})"


def from_hi(h):
    return float(np.array([h << 32], dtype=np.uint64).view(np.float64)[0])


def sweep64(rng, per=32):
    """Every binade 2^-1074 .. 2^1023 with random mantissas, both signs."""
    e = np.repeat(np.arange(-1074, 1024), per)
    v = np.ldexp(1.0 + rng.random(e.size), e)
    return np.concatenate([v, -v])


def thresholds64():
    base = [from_hi(h) for h in HI_WORDS] + [1000.0, 2.0 ** -1022, 2.0 ** 1022, 2.0 ** 1021]
    out = []
    for b in base:
        for v in (np.nextafter(b, 0.0), b, np.nextafter(b, np.inf)):
            out += [v, -v]
    return np.array(out)


SPECIALS64 = np.array([0.0, -0.0, np.inf, -np.inf, np.nan])


def sweep32(rng, per=256):
    e = np.repeat(np.arange(-149, 128), per)
    v = np.ldexp(1.0 + rng.random(e.size), e).astype(np.float32)
    v = v[np.isfinite(v)]
    return np.concatenate([v, -v])


SPECIALS32 = np.array([0.0, -0.0, np.inf, -np.inf, np.nan], np.float32)


def _order_key(a):
    i = np.asarray(a, np.float64).view(np.int64)
    return np.where(i < 0, -(i & np.int64(0x7FFFFFFFFFFFFFFF)), i)


def ulps64(got, want):
    """Distance in float64 steps between got and want (0 for +-0 vs -+0 and NaN vs NaN, inf across signs)."""
    kg, kw = _order_key(got), _order_key(want)
    with np.errstate(over="ignore"):
        d = np.abs(kg - kw).astype(np.float64)
    d[(np.sign(kg) * np.sign(kw)) < 0] = np.inf
    ng, nw = np.isnan(got), np.isnan(want)
    d[ng | nw] = np.where(ng & nw, 0.0, np.inf)[ng | nw]
    return d


def ulp_err_ld(got, want_ld):
    """|got - want| in units of the float64 ulp of want, with want given in long double."""
    w64 = want_ld.astype(np.float64)
    sp = np.spacing(np.abs(w64)).astype(np.longdouble)
    return (np.abs(got.astype(np.longdouble) - want_ld) / sp).astype(np.float64)


def mp_err(f, args, got, scale_floor=None):
    """|got - f(args)| per element, f evaluated with mpmath at 40 digits; with scale_floor, in units of
    max(|f|, scale_floor) 2^-52 instead of absolute."""
    mp.mp.dps = 40
    errs = np.empty(len(got))
    for k in range(len(got)):
        w = f(*[mp.mpf(float(a[k])) for a in args])
        scale = 1.0 if scale_floor is None else max(abs(float(w)), scale_floor) * 2.0 ** -52
        errs[k] = float(abs(mp.mpf(float(got[k])) - w)) / scale
    return errs


# ------------------------------------------------------------------------------------------------------------ FP64
def test_div_fast_and_rcp_fast(dm):
    """<= 1 ulp (against numpy's correctly rounded '/') for |b| in [2^-1022, 2^1022) and a quotient that is zero or
    normal.  Above 2^1022 the reciprocal is subnormal and rcp.approx.ftz flushes it to zero."""
    rng = np.random.default_rng(100)
    sw = sweep64(rng, 24)
    b = np.concatenate([sw, thresholds64(), SPECIALS64, rng.uniform(-4.0, 4.0, 200_000), rng.uniform(0.5, 2.0, 100_000)])
    a = np.concatenate([rng.permutation(sw), rng.uniform(-4.0, 4.0, b.size - sw.size)])
    a[-100_000:] = 1.0 + rng.uniform(-1e-3, 1e-3, 100_000)
    q, r = run(dm, "div_fast", [a, b], [np.float64])[0], run(dm, "rcp_fast", [b], [np.float64])[0]
    with np.errstate(all="ignore"):
        want_q, want_r = a / b, 1.0 / b
    ab = np.abs(b)
    b_ok = (ab >= 2.0 ** -1022) & (ab < 2.0 ** 1022)
    q_ok = b_ok & np.isfinite(a) & (((a == 0) & (want_q == 0)) | ((np.abs(want_q) >= 2.0 ** -1022) & np.isfinite(want_q)))
    eq, er = ulps64(q, want_q), ulps64(r, want_r)
    msg = report("div_fast / rcp_fast", len(b), [
        worst_line("div_fast", eq, q_ok, 1, "ulp", a, b),
        worst_line("rcp_fast", er, b_ok, 1, "ulp", b),
        worst_line("div_fast with |b| >= 2^1022 (outside the domain)", eq, np.isfinite(b) & (ab >= 2.0 ** 1022), 1, "ulp", a, b)])
    assert eq[q_ok].max() <= 1 and er[b_ok].max() <= 1, msg


def test_rsqrt_pos(dm):
    """1 / sqrt(x) for positive normal x: the MUFU seed and one cubic step, against long double."""
    rng = np.random.default_rng(101)
    x = np.concatenate([np.abs(sweep64(rng, 64)), np.abs(thresholds64()), rng.uniform(1e-3, 4.0, 500_000)])
    got = run(dm, "rsqrt_pos", [x], [np.float64])[0]
    want = 1.0 / np.sqrt(x.astype(np.longdouble))
    dom = x >= 2.0 ** -1022
    err = ulp_err_ld(got, want)
    msg = report("rsqrt_pos", len(x), [worst_line("rsqrt_pos", err, dom, RSQRT_POS_ULP, "ulp", x)])
    assert err[dom].max() <= RSQRT_POS_ULP, msg


RSQRT_POS_ULP = 1.5     # r2ik_math.cuh: "~1 ulp"


def test_sqrt_nonneg_and_sqrt_rsqrt_nonneg(dm):
    """sqrt(x) <= 1 ulp for x = +-0 or normal (numpy's sqrt is correctly rounded); the 1 / sqrt(x) of
    sqrt_rsqrt_nonneg as rsqrt_pos.  Includes [2^-1022, 2^-1020), the binades below the seed clamp."""
    rng = np.random.default_rng(102)
    x = np.concatenate([np.abs(sweep64(rng, 64)), np.abs(thresholds64()), [0.0, -0.0], rng.uniform(0.0, 4.0, 500_000),
                        np.ldexp(1.0 + rng.random(20_000), rng.integers(-1022, -1019, 20_000))])
    s1 = run(dm, "sqrt_nonneg", [x], [np.float64])[0]
    s2, inv = run(dm, "sqrt_rsqrt_nonneg", [x], [np.float64, np.float64])
    want = np.sqrt(x)
    dom = (x == 0) | ((x >= 2.0 ** -1022) & np.isfinite(x))
    e1, e2 = ulps64(s1, want), ulps64(s2, want)
    ei = ulp_err_ld(inv, 1.0 / np.sqrt(x.astype(np.longdouble)))
    pos = dom & (x > 0)
    low = dom & (x < 2.0 ** -1020) & (x > 0)
    inf_out = run(dm, "sqrt_nonneg", [np.array([np.inf])], [np.float64])[0][0]
    msg = report("sqrt_nonneg / sqrt_rsqrt_nonneg", len(x), [
        worst_line("sqrt_nonneg", e1, dom, 1, "ulp", x),
        worst_line("sqrt_nonneg on [2^-1022, 2^-1020)", e1, low, 1, "ulp", x),
        worst_line("sqrt_rsqrt_nonneg sqrt", e2, dom, 1, "ulp", x),
        worst_line("sqrt_rsqrt_nonneg inv", ei, pos, RSQRT_POS_ULP, "ulp", x),
        f"sqrt_nonneg(+inf) = {inf_out!r} (outside the domain: reach_prechecks tests dg2 for inf before the root)"])
    assert e1[dom].max() <= 1 and e2[dom].max() <= 1 and ei[pos].max() <= RSQRT_POS_ULP, msg
    assert np.array_equal(np.signbit(s1[x == 0]), np.signbit(x[x == 0])), msg


ATAN2_ULP = 3.0      # r2ik_math.cuh: polynomial 4e-18 + the single-double pi in pi - r: measured 2.2 on the host
ATAN2_NP_ULP = 4.0   # the same against np.arctan2, which is itself within 1 ulp


def _atan2_inputs(rng):
    ang = rng.uniform(-np.pi, np.pi, 600_000)
    r = 10.0 ** rng.uniform(-12, 3, ang.size)
    y, x = [r * np.sin(ang)], [r * np.cos(ang)]
    sw = sweep64(rng, 48)
    y.append(sw); x.append(rng.permutation(sw))                                    # independent magnitudes
    y.append(sw); x.append(sw * rng.uniform(0.3, 3.0, sw.size) * rng.choice([-1.0, 1.0], sw.size))   # same binade: 'big'
    th = thresholds64()
    ty, tx = np.meshgrid(np.concatenate([th, SPECIALS64, [1.0, -1.0]]), np.concatenate([th, SPECIALS64, [1.0, -1.0]]))
    y.append(ty.ravel()); x.append(tx.ravel())
    y.append(np.array([1.2 * 2.0 ** 1021])); x.append(np.array([1.5 * 2.0 ** 1021]))
    return np.concatenate(y), np.concatenate(x)


def test_atan2_core_and_its_predicate(dm):
    """Wherever atan2_core_ok(y, x) holds, atan2_core is within ATAN2_ULP of atan2 (mpmath, 40 digits, on a 20 k
    sample) and within ATAN2_NP_ULP of np.arctan2 on all ~1 M inputs, with the same sign bit; the error unit is the
    ulp of max(|atan2|, 2^-1022)."""
    rng = np.random.default_rng(103)
    y, x = _atan2_inputs(rng)
    got, ok = run(dm, "atan2_core", [y, x], [np.float64, np.uint8])
    ok = ok.astype(bool)
    want = np.arctan2(y, x)
    scale = np.maximum(np.abs(want), 2.0 ** -1022) * 2.0 ** -52
    with np.errstate(invalid="ignore"):
        err = np.where(np.isnan(want) & np.isnan(got), 0.0, np.abs(got - want) / scale)
    err[np.isnan(err)] = np.inf
    pick = rng.choice(np.nonzero(ok & (want != 0))[0], 20_000, replace=False)
    emp = mp_err(mp.atan2, [y[pick], x[pick]], got[pick], 2.0 ** -1022)
    sign_ok = np.signbit(got) == np.signbit(want)
    big = np.maximum(np.abs(y), np.abs(x))
    msg = report("atan2_core", len(y), [
        worst_line("vs mpmath", emp, np.ones(len(pick), bool), ATAN2_ULP, "ulp", y[pick], x[pick]),
        worst_line("vs np.arctan2 where atan2_core_ok", err, ok, ATAN2_NP_ULP, "ulp", y, x),
        worst_line("where not atan2_core_ok", err, ~ok & np.isfinite(err), ATAN2_NP_ULP, "ulp", y, x),
        f"atan2_core_ok: {int(ok.sum())} accepted, largest accepted max(|x|, |y|) {float(big[ok].max()):.6g}"])
    assert emp.max() <= ATAN2_ULP, msg
    assert err[ok].max() <= ATAN2_NP_ULP and sign_ok[ok].all(), msg
    # the predicate's stated domain: zero, or max(|x|, |y|) normal and < 2^1021
    dom = (big == 0) | ((big >= 2.0 ** -1020) & (big < 2.0 ** 1021))
    assert np.array_equal(ok, dom), msg


def test_cs_and_angle_fast_route(dm):
    """cs_of_atan2 normalises (x, y) with rsqrt_pos when 1e-280 < x^2 + y^2 < 1e280 (its exponent window) and
    angle_of_unit reads the angle off the unit vector: wherever the window holds, (c, s) is the unit vector to 4 ulp
    and the angle is within 1e-15 rad (2e-15 relative) of atan2(y, x) (mpmath on 20 k points, numpy on all)."""
    rng = np.random.default_rng(104)
    y, x = _atan2_inputs(rng)
    c, s, ang, deg = run(dm, "cs_and_angle", [y, x], [np.float64] * 3 + [np.uint8])
    ok = deg == 0
    want = np.arctan2(y, x)
    with np.errstate(all="ignore"):
        h = np.hypot(x.astype(np.longdouble), y.astype(np.longdouble))
        ec = np.maximum(ulp_err_ld(c, x / h), ulp_err_ld(s, y / h))
        ea = np.abs(ang - want)
    h2 = x.astype(np.longdouble) ** 2 + y.astype(np.longdouble) ** 2
    window = (h2 > 1e-280) & (h2 < 1e280)
    pick = rng.choice(np.nonzero(ok & (np.abs(want) > 1e-300))[0], 20_000, replace=False)
    emp = mp_err(mp.atan2, [y[pick], x[pick]], ang[pick])
    rel = emp / np.abs(want[pick])
    msg = report("cs_of_atan2 + angle_of_unit", len(y), [
        worst_line("(c, s) vs (x, y) / |(x, y)|", ec, ok, 4, "ulp", y, x),
        worst_line("angle vs np.arctan2", ea, ok, 1e-15, "rad", y, x),
        worst_line("angle vs mpmath, absolute", emp, np.ones(len(pick), bool), 1e-15, "rad", y[pick], x[pick]),
        worst_line("angle vs mpmath, relative", rel, np.ones(len(pick), bool), 2e-15, "", y[pick], x[pick])])
    assert ec[ok].max() <= 4 and ea[ok].max() <= 1e-15 and emp.max() <= 1e-15 and rel.max() <= 2e-15, msg
    assert (np.signbit(ang) == np.signbit(want))[ok].all(), msg
    # the window is the exponent test on the rounded x^2 + y^2: it may differ from the exact one only at its two ends
    assert not (ok & ~window & ((h2 < 1e-281) | (h2 > 1e281))).any() and not (~ok & window & (h2 > 1e-279) & (h2 < 1e279)).any(), msg


def test_angle_of_unit(dm):
    rng = np.random.default_rng(105)
    ang = rng.uniform(-np.pi, np.pi, 1_000_000)
    c, s = np.cos(ang), np.sin(ang)
    edges = np.array([0.0, np.pi / 8, np.pi / 4, 3 * np.pi / 8, np.pi / 2, np.pi, -np.pi / 8, -np.pi / 2, -np.pi])
    edges = np.concatenate([edges, np.nextafter(edges, 10), np.nextafter(edges, -10)])
    c = np.concatenate([c, np.cos(edges), [1.0, 1.0, -1.0, -1.0, 0.0, 0.0, -0.0]])
    s = np.concatenate([s, np.sin(edges), [0.0, -0.0, 0.0, -0.0, 1.0, -1.0, 1.0]])
    got = run(dm, "angle_of_unit", [c, s], [np.float64])[0]
    want = np.arctan2(s, c)
    err = np.abs(got - want)
    pick = rng.choice(np.nonzero(s != 0)[0], 20_000, replace=False)
    emp = mp_err(mp.atan2, [s[pick], c[pick]], got[pick])
    msg = report("angle_of_unit", len(c), [worst_line("vs np.arctan2", err, np.ones(len(c), bool), 1e-15, "rad", c, s),
                                           worst_line("vs mpmath", emp, np.ones(len(pick), bool), 1e-15, "rad", c[pick], s[pick])])
    assert err.max() <= 1e-15 and emp.max() <= 1e-15, msg
    assert np.array_equal(np.signbit(got), np.signbit(want)), msg


# Error unit: the ulp of max(|value|, 2^-46).  r2ik_math.cuh: "~1 ulp for |x| <= 1000", and near a zero of sin / cos
# an absolute error below 1e-30 (|k| <= 637 multiples of the 1e-33 by which HI + LO misses pi/2; 2^-46 ulp = 3.2e-30).
# The library route (|x| > 1000): 2 ulp.
SINCOS_UNITS = 2.0
SINCOS_FLOOR = 2.0 ** -46


def _sincos_err(sn, cs, x):
    with np.errstate(invalid="ignore"):
        ws, wc = np.sin(x), np.cos(x)
        es = np.abs(sn - ws) / (np.maximum(np.abs(ws), SINCOS_FLOOR) * 2.0 ** -52)
        ec = np.abs(cs - wc) / (np.maximum(np.abs(wc), SINCOS_FLOOR) * 2.0 ** -52)
    nan_ok = (np.isnan(sn) == np.isnan(ws)) & (np.isnan(cs) == np.isnan(wc))
    e = np.where(np.isnan(ws), 0.0, np.maximum(es, ec))
    return np.where(nan_ok, e, np.inf)


def test_sincos_small_and_sincos_any(dm):
    """sincos_small where sincos_small_ok (|x| <= 1000); sincos_any on both of its routes, up to 1e308, against numpy
    (glibc, full argument reduction) on ~1 M inputs and mpmath (40 digits) on 20 k."""
    rng = np.random.default_rng(106)
    sw = sweep64(rng, 48)
    x = np.concatenate([rng.uniform(-4, 4, 300_000), rng.uniform(-1000, 1000, 200_000),
                        10.0 ** rng.uniform(3, 15, 100_000) * rng.choice([-1.0, 1.0], 100_000),
                        sw, thresholds64(), SPECIALS64, np.arange(-640, 641) * (np.pi / 2)])
    sn, cs, ok = run(dm, "sincos_small", [x], [np.float64, np.float64, np.uint8])
    an, ac = run(dm, "sincos_any", [x], [np.float64, np.float64])
    ok = ok.astype(bool)
    es, ea = _sincos_err(sn, cs, x), _sincos_err(an, ac, x)
    small = np.abs(x) <= 1000.0
    pick = rng.choice(np.nonzero(np.isfinite(x) & (np.abs(x) <= 1e15))[0], 20_000, replace=False)
    emp = np.maximum(mp_err(mp.sin, [x[pick]], an[pick], SINCOS_FLOOR), mp_err(mp.cos, [x[pick]], ac[pick], SINCOS_FLOOR))
    msg = report("sincos_small / sincos_any", len(x), [
        worst_line("sincos_small where sincos_small_ok", es, ok, SINCOS_UNITS, "ulp", x),
        worst_line("sincos_any, |x| <= 1000", ea, small, SINCOS_UNITS + 1, "ulp", x),
        worst_line("sincos_any, |x| > 1000 (library route)", ea, ~small, SINCOS_UNITS + 1, "ulp", x),
        worst_line("sincos_any vs mpmath", emp, np.ones(len(pick), bool), SINCOS_UNITS, "ulp", x[pick])])
    assert np.array_equal(ok, small), msg
    assert es[ok].max() <= SINCOS_UNITS + 1 and ea.max() <= SINCOS_UNITS + 1 and emp.max() <= SINCOS_UNITS, msg


def _same_bits(got, want):
    return (got.view(np.int64) == want.view(np.int64)) | (np.isnan(got) & np.isnan(want))


def test_pymod_2pi_and_angle_diff_are_python_modulo(dm):
    """Bit-identical to Python's float `%` (and to utl:486-490 angle_diff built on it), on the fast range
    [-2 pi, 8 pi), around every multiple of pi in it, and across all binades."""
    rng = np.random.default_rng(107)
    k = np.arange(-8, 20) * np.pi
    near = np.concatenate([k + d * np.spacing(np.abs(k) + 1) for d in range(-3, 4)])
    x = np.concatenate([rng.uniform(-TWO_PI, 4 * TWO_PI, 400_000), rng.uniform(-50, 50, 100_000), near,
                        np.array([-TWO_PI, 4 * TWO_PI, 2 * TWO_PI, TWO_PI, np.nextafter(-TWO_PI, 0), np.nextafter(-TWO_PI, -10),
                                  np.nextafter(4 * TWO_PI, 0)]), sweep64(rng, 8), SPECIALS64])
    got = run(dm, "pymod_2pi", [x], [np.float64])[0]
    want = np.array([v % TWO_PI for v in x.tolist()])
    a = np.concatenate([rng.uniform(-4 * np.pi, 4 * np.pi, 300_000), x[:200_000]])
    b = np.concatenate([rng.uniform(-4 * np.pi, 4 * np.pi, 300_000), rng.permutation(x[:200_000])])
    gd = run(dm, "angle_diff", [a, b], [np.float64])[0]
    wd = np.array([((ai - bi) + math.pi) % (2 * math.pi) - math.pi for ai, bi in zip(a.tolist(), b.tolist())])
    same, samed = _same_bits(got, want), _same_bits(gd, wd)
    msg = report("pymod_2pi / angle_diff", len(x) + len(a), [
        f"pymod_2pi: {int((~same).sum())} of {len(x)} differ from Python's %" + ("" if same.all() else f", first x={x[~same][0]!r}"),
        f"angle_diff: {int((~samed).sum())} of {len(a)} differ" + ("" if samed.all() else f", first (a, b)=({a[~samed][0]!r}, {b[~samed][0]!r})")])
    assert same.all() and samed.all(), msg


def test_linspace_value_is_np_linspace(dm):
    rng = np.random.default_rng(108)
    starts = np.concatenate([rng.uniform(-2 * np.pi, 2 * np.pi, 200), [-np.pi, 0.0, 1.0, 0.0, 5e-324, -3.0]])
    stops = np.concatenate([starts[:200] + rng.uniform(-4 * np.pi, 4 * np.pi, 200), [np.pi, 1e-321, 1.0, 0.0, 1e-322, 2.5]])
    S, E, N, I, W = [], [], [], [], []
    for s0, s1 in zip(starts, stops):
        for num in (1, 2, 20, 360, 1000):
            ref = np.linspace(s0, s1, num)
            S.append(np.full(num, s0)); E.append(np.full(num, s1)); N.append(np.full(num, num, np.int32))
            I.append(np.arange(num, dtype=np.int32)); W.append(ref)
    S, E, N, I, W = map(np.concatenate, (S, E, N, I, W))
    got = run(dm, "linspace_value", [S, E, N, I], [np.float64])[0]
    same = _same_bits(got, W)
    msg = report("linspace_value", len(W), [f"{int((~same).sum())} samples differ from np.linspace" +
                                            ("" if same.all() else f", first ({S[~same][0]!r}, {E[~same][0]!r}, {N[~same][0]}, {I[~same][0]})")])
    assert same.all(), msg


# ------------------------------------------------------------------------------------------------------------ FP32
def _f32_ulps(got, want64):
    sp = np.spacing(np.abs(want64).astype(np.float32)).astype(np.float64)
    return np.abs(got.astype(np.float64) - want64) / sp


def test_fp32_rcp_sqrt_rsqrt_full_range(dm):
    """rcp_f, sqrt_f and rsqrt_f (one .approx.ftz instruction each) over every float32 binade, against float64: within
    the PTX ISA bounds wherever input and result are normal (ftz flushes subnormals)."""
    rng = np.random.default_rng(200)
    x = np.concatenate([sweep32(rng), rng.uniform(-4, 4, 300_000).astype(np.float32), SPECIALS32])
    pos = x[x > 0]
    rc = run(dm, "rcp_f", [x], [np.float32])[0]
    sq = run(dm, "sqrt_f", [pos], [np.float32])[0]
    rs = run(dm, "rsqrt_f", [pos], [np.float32])[0]
    x64, p64 = x.astype(np.float64), pos.astype(np.float64)
    tiny = float(np.finfo(np.float32).tiny)
    with np.errstate(all="ignore"):
        wr = 1.0 / x64
    dom_r = np.isfinite(x64) & (np.abs(x64) >= tiny) & (np.abs(wr) >= tiny)
    dom_s = np.isfinite(p64) & (p64 >= tiny)
    er = _f32_ulps(rc, wr)
    es = np.abs(sq - np.sqrt(p64)) / np.sqrt(p64)
    ers = np.abs(rs - 1.0 / np.sqrt(p64)) / (1.0 / np.sqrt(p64))
    msg = report("rcp_f / sqrt_f / rsqrt_f", len(x) + 2 * len(pos), [
        worst_line("rcp_f", er, dom_r, RCP_F_ULP, "ulp", x),
        worst_line("sqrt_f", es, dom_s, SQRT_F_REL, "relative", pos),
        worst_line("rsqrt_f", ers, dom_s, RSQRT_F_REL, "relative", pos)])
    assert er[dom_r].max() <= RCP_F_ULP and es[dom_s].max() <= SQRT_F_REL and ers[dom_s].max() <= RSQRT_F_REL, msg


def test_fp32_sincos_f(dm):
    rng = np.random.default_rng(201)
    x = np.concatenate([rng.uniform(-4, 4, 400_000), rng.uniform(-SINCOS_F_RANGE, SINCOS_F_RANGE, 400_000),
                        np.arange(-40, 41) * (np.pi / 2), [SINCOS_F_RANGE, -SINCOS_F_RANGE, 0.0, -0.0, 1e-30]]).astype(np.float32)
    sn, cs = run(dm, "sincos_f", [x], [np.float32, np.float32])
    x64 = x.astype(np.float64)
    e = np.maximum(np.abs(sn - np.sin(x64)), np.abs(cs - np.cos(x64)))
    msg = report("sincos_f", len(x), [worst_line(f"|x| <= {SINCOS_F_RANGE:g}", e, np.ones(len(x), bool), SINCOS_F_ABS, "abs", x)])
    assert e.max() <= SINCOS_F_ABS, msg


def test_fp32_angle_of_unit_f(dm):
    rng = np.random.default_rng(202)
    ang = np.concatenate([rng.uniform(-np.pi, np.pi, 1_000_000), np.arange(-8, 9) * (np.pi / 8)])
    c, s = np.cos(ang).astype(np.float32), np.sin(ang).astype(np.float32)
    got = run(dm, "angle_of_unit_f", [c, s], [np.float32])[0]
    e = np.abs(got - np.arctan2(s.astype(np.float64), c.astype(np.float64)))
    msg = report("angle_of_unit_f", len(c), [worst_line("unit vectors", e, np.ones(len(c), bool), ANGLE_F_ABS, "rad", c, s)])
    assert e.max() <= ANGLE_F_ABS, msg


def test_fp32_cs_and_angle_f(dm):
    """Wherever cs_and_angle_f leaves esc false the angle is within ANGLE_F_ABS of the float64 atan2 of the same float
    inputs -- in particular never on the wrong side of the +-pi cut.  Domain: x^2 + y^2 finite in float32 (the solve
    only passes coordinates inside the arm's reach sphere: a goal beyond max_arm_length returns before get_joints_f)."""
    rng = np.random.default_rng(203)
    sw = sweep32(rng, 128)
    ang = rng.uniform(-np.pi, np.pi, 400_000)
    r = 10.0 ** rng.uniform(-4, 1, ang.size)
    hmin = math.sqrt(4e-6)
    cut = rng.uniform(-3e-5, 3e-5, 50_000)
    y = np.concatenate([r * np.sin(ang), sw, hmin * np.sin(ang[:50_000]), cut, [0.0, -0.0, 1e-5, -1e-5]]).astype(np.float32)
    x = np.concatenate([r * np.cos(ang), rng.permutation(sw), hmin * np.cos(ang[:50_000]) * (1 + rng.uniform(-1e-6, 1e-6, 50_000)),
                        -np.ones(50_000), [-1.0, -1.0, -1.0, -1.0]]).astype(np.float32)
    c, s, a, esc = run(dm, "cs_and_angle_f", [y, x], [np.float32] * 3 + [np.uint8])
    y64, x64 = y.astype(np.float64), x.astype(np.float64)
    want = np.arctan2(y64, x64)
    h2 = x64 * x64 + y64 * y64
    dom = (esc == 0) & (h2 < 3.0e38)
    e = np.abs(a.astype(np.float64) - want)
    msg = report("cs_and_angle_f", len(y), [worst_line("where esc is false", e, dom, ANGLE_F_ABS, "rad", y, x),
                                            f"esc set on {int(esc.sum())} inputs"])
    assert e[dom].max() <= ANGLE_F_ABS, msg
    # what esc promises: short vectors (h^2 <= kMinH2) and the +-pi cut are always escalated
    short = h2 <= 4e-6 * (1 - 1e-6)
    cut = (x64 < 0) & (np.abs(y64) / np.sqrt(np.maximum(h2, 1e-300)) < 1e-5 * (1 - 1e-6))
    assert esc[(h2 < 3.0e38) & (short | cut)].all(), msg
