"""The device routines that are not one IEEE binary32 operation of the reference — powLikePowf and cubeLikePowf (the two powers of
Scene.cpp:175 and :196) and divExact (the three constant divisions) — compiled with the product's flags (tests/cuda/
device_math_probe.cu) and held against exact arithmetic: Python's decimal at 60 digits and fractions, rounded to binary32 in exact
rational arithmetic (never through a double).

powLikePowf targets RN(x^y) and evaluates it in binary64 with about 2^-50 relative error (rfx_device.cuh), so it may miss only where
x^y lies within 2^-26 of a float ulp of a rounding boundary, about one call in 10^7.  cubeLikePowf rounds the binary64 cube (the
square is exact, the cube rounded once) to float: it differs from RN(x^3) exactly where that double rounding lands on a float
rounding boundary.  divExact is the correctly rounded quotient for every input of its three call sites."""
import ctypes as C
import math
import os
import subprocess
from decimal import Context
from fractions import Fraction

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROBE_SRC = os.path.join(ROOT, "tests", "cuda", "device_math_probe.cu")
PROBE_SO = os.path.join(ROOT, "build", "device_math_probe.so")
DEVICE_HDRS = [os.path.join(ROOT, "reflaxman_b200", "csrc", f) for f in ("rfx_device.cuh", "rfx_types.h")]

_fp = C.POINTER(C.c_float)


def build_probe():
    """Compile the probe with the product's nvcc flags into build/ (git-ignored) unless it is newer than its sources."""
    from reflaxman_b200 import build as B
    deps = [PROBE_SRC, os.path.abspath(B.__file__)] + DEVICE_HDRS
    if os.path.exists(PROBE_SO) and all(os.path.getmtime(d) <= os.path.getmtime(PROBE_SO) for d in deps):
        return PROBE_SO
    os.makedirs(os.path.dirname(PROBE_SO), exist_ok=True)
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    tmp = PROBE_SO + ".%d.tmp" % os.getpid()
    subprocess.run([nvcc, *B.NVCC_FLAGS, "-o", tmp, PROBE_SRC], check=True)
    os.replace(tmp, PROBE_SO)
    return PROBE_SO


def test_probe_compiles():
    """The probe builds for sm_100a (nvcc cross-compiles without a GPU) and exports its three entry points."""
    so = build_probe()
    out = subprocess.run(["nm", "-D", "--defined-only", so], check=True, capture_output=True, text=True).stdout
    for sym in ("probe_pow", "probe_cube", "probe_div"):
        assert " " + sym + "\n" in out, sym


@pytest.fixture(scope="module")
def probe():
    L = C.CDLL(build_probe())
    L.probe_pow.argtypes = [C.c_int, _fp, _fp, _fp]
    L.probe_cube.argtypes = [C.c_int, _fp, _fp]
    L.probe_div.argtypes = [C.c_int, C.c_int, _fp, _fp]
    return L


def _call(fn, *arrays, extra=()):
    ins = [np.ascontiguousarray(a, np.float32) for a in arrays]
    out = np.zeros(len(ins[0]), np.float32)
    rc = fn(len(out), *extra, *[a.ctypes.data_as(_fp) for a in ins], out.ctypes.data_as(_fp))
    assert rc == 0, "probe failed (%d)" % rc
    return out


# ---------------------------------------------------------------------------------------------------------------- exact rounding
def rn32(F):
    """Round a positive Fraction to binary32, ties to even, denormals included.  Returns (float32 value, distance of F from the
    nearest rounding boundary in units of the float ulp at F, True when F lies exactly on a boundary)."""
    n, d = F.numerator, F.denominator
    e = n.bit_length() - d.bit_length()
    if (n << max(0, -e)) < (d << max(0, e)):
        e -= 1                                    # 2^e <= F < 2^(e+1)
    qe = max(e - 23, -149)                        # exponent of the ulp
    num, den = (n, d << qe) if qe >= 0 else (n << -qe, d)
    k, rem = divmod(num, den)
    c = 2 * rem - den                             # sign of (fraction - 1/2)
    if c > 0 or (c == 0 and k & 1):
        k += 1
    return np.float32(math.ldexp(k, qe)), Fraction(abs(c), 2 * den), c == 0


def rn32_dyadic(N, E):
    """rn32 of the positive dyadic N * 2^E, in integer arithmetic: (float32 value, True when N * 2^E lies exactly on a boundary)."""
    qe = max(N.bit_length() - 1 + E - 23, -149)
    shift = qe - E
    if shift <= 0:
        return np.float32(math.ldexp(N, E)), False
    k, rem, half = N >> shift, N & ((1 << shift) - 1), 1 << (shift - 1)
    if rem > half or (rem == half and k & 1):
        k += 1
    return np.float32(math.ldexp(k, qe)), rem == half


def on_f32_boundary(v):
    """Elementwise: the binary64 values v > 0 that lie exactly on a binary32 rounding boundary (halfway between adjacent floats)."""
    v = np.asarray(v, np.float64)
    e = np.frexp(v)[1] - 1                            # 2^e <= v < 2^(e+1)
    r = np.ldexp(v, -np.maximum(e - 23, -149))        # v in units of the float ulp at v (exact: a power-of-two scaling)
    return (v > 0) & (r - np.floor(r) == 0.5)


def _ulps_apart(a, b):
    return abs(int(np.float32(a).view(np.int32)) - int(np.float32(b).view(np.int32)))


# ---------------------------------------------------------------------------------------------------------------- powLikePowf
POW_BAND = Fraction(1, 1 << 26)    # in ulps: what a ~2^-50 relative error can move across


def _pow_inputs():
    """~200k (x, y) pairs: the three modes of tools/pow_check.cu, y = 1 across every exponent, powers of two with integer exponents
    (exact results, denormals, 2^-150), results straddling 2^-126 and 2^-149, and x = 2^-63."""
    rng = np.random.default_rng(20261020)
    xs, ys = [], []

    def add(x, y):
        xs.append(np.asarray(x, np.float32).ravel()); ys.append(np.asarray(y, np.float32).ravel())

    n = 66000
    u = rng.random(n, np.float32)
    add(np.float32(1) - u, np.float32(1) + np.float32(120) * rng.random(n, np.float32))                           # (0, 1] x [1, 121)
    k = rng.integers(0, 20, n)
    add(np.float32(1) - np.ldexp(rng.random(n, np.float32), -k).astype(np.float32), np.float32(1) + np.float32(4096) * rng.random(n, np.float32))
    k = rng.integers(0, 63, n)
    add(np.ldexp(np.float32(0.5) + np.float32(0.5) * rng.random(n, np.float32), -k).astype(np.float32),
        np.float32(1) + np.float32(8) * rng.random(n, np.float32))                                                # log-uniform x, y in [1, 9)
    xs[0][xs[0] == 0] = 1.0; xs[1][xs[1] == 0] = 1.0
    # y = 1 for x across all exponents down to 2^-63 (and a few mantissas each)
    xe = np.array([np.ldexp(np.float32(m), -e) for e in range(0, 64) for m in (1.0, 0.75, 0.999999, 0.5000001, 0.6180339)], np.float32)
    add(xe, np.ones_like(xe))
    # x = 2^-k, integer y: exact results, into the denormals, 2^-149, 2^-150 (a tie that rounds to 0) and below
    px, py = [], []
    for k in range(1, 64):
        for y in range(1, 160):
            if k * y <= 160:
                px.append(2.0 ** -k); py.append(float(y))
    add(px, py)
    # results straddling 2^-126 and 2^-149: y = t / log2(1/x) for t around 126 and 149
    x = (np.float32(1) - rng.random(4000, np.float32) * np.float32(0.999)).astype(np.float32)
    t = np.where(rng.random(4000) < 0.5, 126.0, 149.0) + rng.uniform(-1.5, 1.5, 4000)
    y = (t / -np.log2(x.astype(np.float64))).astype(np.float32)
    ok = (y >= 1) & np.isfinite(y)
    add(x[ok], y[ok])
    # x = 2^-63 (the smallest argument Scene.cpp:175 passes) with every kind of y
    add(np.full(200, 2.0 ** -63, np.float32), np.float32(1) + np.float32(3) * rng.random(200, np.float32))
    return np.concatenate(xs), np.concatenate(ys)


def _pow_exact(x, y, ctx=Context(prec=60)):
    """x^y as a Fraction: exact for integer y (x is dyadic), else exp(y ln x) in 60-digit decimal.  Second item: exact or not."""
    if y == int(y) and y <= 200:
        return Fraction(float(x)) ** int(y), True
    from decimal import Decimal
    return Fraction(ctx.exp(ctx.multiply(Decimal(float(y)), ctx.ln(Decimal(float(x)))))), False


@pytest.mark.gpu
def test_pow_like_powf_is_correctly_rounded_outside_the_band(probe):
    x, y = _pow_inputs()
    assert len(x) > 190000
    got = _call(probe.probe_pow, x, y)
    misses = []
    for i in range(len(x)):
        F, exact = _pow_exact(x[i], y[i])
        want, dist, tie = rn32(F)
        if got[i].view(np.uint32) == want.view(np.uint32):
            continue
        # a miss: allowed only next to a rounding boundary, never by more than one ulp, and never on an exact result
        assert _ulps_apart(got[i], want) == 1, (float(x[i]), float(y[i]), float(got[i]), float(want))
        assert not exact, ("exact result missed", float(x[i]), float(y[i]), float(got[i]), float(want))
        assert dist < POW_BAND, ("miss away from a rounding boundary", float(x[i]), float(y[i]), float(got[i]), float(want), float(dist))
        misses.append((float(x[i]), float(y[i]), float(dist)))
    print("powLikePowf: %d inputs, %d within %g ulp of a boundary and missed: %s" % (len(x), len(misses), float(POW_BAND), misses))
    assert len(misses) <= 3, misses          # DESIGN.md: about one call in 10^7


@pytest.mark.gpu
def test_pow_like_powf_special_cases(probe):
    """x = 1 with any finite y or +inf gives 1; x < 1 with y = +inf gives 0; 2^-150 (a tie) rounds to 0, 2^-149 and 2^-140 are exact;
    y = 1 returns x itself at the extremes of the range."""
    inf = np.float32(np.inf)
    cases = [(1.0, 1.0, 1.0), (1.0, 5.0, 1.0), (1.0, 4096.5, 1.0), (1.0, inf, 1.0), (0.5, inf, 0.0), (0.99999994, inf, 0.0),
             (2.0 ** -63, inf, 0.0), (0.5, 150.0, 0.0), (0.5, 149.0, 2.0 ** -149), (0.5, 140.0, 2.0 ** -140), (2.0 ** -10, 15.0, 0.0),
             (0.25, 0.5, 0.5), (2.0 ** -63, 1.0, 2.0 ** -63), (0.99999994, 1.0, 0.99999994), (0.5, 151.0, 0.0)]
    x, y, want = (np.array(c, np.float32) for c in zip(*cases))
    got = _call(probe.probe_pow, x, y)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), list(zip(x, y, got, want))


# ---------------------------------------------------------------------------------------------------------------- cubeLikePowf
def _binade(lo_exp, hi_exp):
    """every float in [2^lo_exp, 2^hi_exp)"""
    a, b = np.float32(2.0 ** lo_exp).view(np.uint32), np.float32(2.0 ** hi_exp).view(np.uint32)
    return np.arange(a, b, dtype=np.uint32).view(np.float32)


@pytest.mark.gpu
def test_cube_like_powf_is_the_correctly_rounded_cube(probe):
    """The device cube is (float)((d * d) * d): the square is exact, the cube is rounded to binary64 once, then to float.  That
    differs from RN(x^3) exactly where the binary64 cube lies on a float rounding boundary while x^3 does not (double rounding).
    Exhaustively over [1/2, 1) (every other binade of normal results is that one scaled by a power of 8, which leaves the boundary
    test unchanged) and over [2^-51, 2^-41) (cubes in the float denormals and across 2^-126, 2^-149 and 2^-150): the device equals
    the binary64 model bit for bit, and the model lands on a boundary only where the exact cube does, so the device cube is RN(x^3)
    on all of [0, 1]: there is no double-rounding case.
    The 10^6 random inputs and the edges are also rounded exactly in integer arithmetic."""
    for lo, hi in [(-1, 0)] + [(e, e + 1) for e in range(-51, -41)]:
        x = _binade(lo, hi)
        got = _call(probe.probe_cube, x)
        d = x.astype(np.float64)
        dbl = (d * d) * d
        assert np.array_equal(got.view(np.uint32), dbl.astype(np.float32).view(np.uint32)), (lo, hi)
        # a binary64 cube on a boundary is harmless only when it is the exact cube (then both roundings see the same tie)
        for i in np.nonzero(on_f32_boundary(dbl))[0]:
            M, E = int(np.frexp(d[i])[0] * (1 << 24)), int(np.frexp(d[i])[1]) - 24
            assert Fraction(M ** 3) * Fraction(2) ** (3 * E) == Fraction(float(dbl[i])), ("double rounding", float(x[i]))
    rng = np.random.default_rng(31337)
    edges = [0.0, 1.0, 2.0 ** -149, 2.0 ** -126, 2.0 ** -127, 2.0 ** -50, 2.0 ** -42]
    edges += list(np.arange(1, 4097) * 2.0 ** -149)                         # denormal x
    edges += list(1.0 - np.arange(1, 4097) * 2.0 ** -24)                    # just below 1
    x = np.concatenate([np.array(edges, np.float32), rng.random(1_000_000, np.float32)])
    got = _call(probe.probe_cube, x)
    m, ex = np.frexp(x.astype(np.float64))
    for i in range(len(x)):
        M, E = int(m[i] * (1 << 24)), int(ex[i]) - 24   # x = M * 2^E exactly
        want = rn32_dyadic(M ** 3, 3 * E)[0] if M else np.float32(0)
        assert got[i].view(np.uint32) == want.view(np.uint32), (float(x[i]), float(got[i]), float(want))


# ---------------------------------------------------------------------------------------------------------------- divExact
@pytest.mark.gpu
@pytest.mark.parametrize("which,D,hi", [(0, Fraction(32767, 2), 32768), (1, Fraction(32767), 32768), (2, Fraction(255), 256)],
                         ids=["16383.5", "32767", "255"])
def test_div_exact_is_the_correctly_rounded_quotient_on_every_input(probe, which, D, hi):
    """Every input of each call site (the 15-bit draws, the 8-bit texel channels), through the compiled device code and the
    constants the kernels use."""
    r = np.arange(hi, dtype=np.float32)
    got = _call(probe.probe_div, r, extra=(which,))
    want = np.array([rn32(Fraction(k) / D)[0] if k else np.float32(0) for k in range(hi)], np.float32)
    bad = np.nonzero(got.view(np.uint32) != want.view(np.uint32))[0]
    assert len(bad) == 0, [(int(k), float(got[k]), float(want[k])) for k in bad[:8]]
