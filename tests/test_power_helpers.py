"""The literal-power helpers of csrc/inflx_device.cuh against the correctly rounded power, over the
whole double range: every instance the generator can emit (inflx_powi<3..64>, inflx_powi_neg<2..64>,
inflx_powh<1..63>, inflx_powh_neg<0..63>), under the exact policy (slow path, pre-passes, point
kernels) and the speculative one as the grid kernel runs it (its value, or the exact policy's where
it flags the point).  Host build (tests/native/pow_check.cpp, seeds are IEEE values); the GPU twin
with the hardware seeds is tests/test_gpu_power_helpers.py.

Reference: libquadmath's powq rounded to double; where the quad value lies within 2^-40 ulp of a
rounding boundary the rounding is decided exactly (rational arithmetic for x^N, squares compared
for x^(N+1/2))."""
import ctypes
import math
import os
import subprocess
from fractions import Fraction

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NATIVE = os.path.join(ROOT, "tests", "native")
HEADER = os.path.join(ROOT, "inflatox_b200", "csrc", "inflx_device.cuh")
_DP = ctypes.POINTER(ctypes.c_double)

KINDS = {0: "inflx_powi", 1: "inflx_powi_neg", 2: "inflx_powh", 3: "inflx_powh_neg"}
N_RANGE = {0: range(3, 65), 1: range(2, 65), 2: range(1, 64), 3: range(0, 64)}
BAND = (2.0**-969, 2.0**969)  # results in here: the double-double chains' own range
NEAR = 2.0**-40  # quad value this close (in ulps) to a rounding boundary: decided exactly
# the chains' double-double value is within ~2^-100 (relative) of the power, i.e. ~2^-47 ulp: they may
# round the wrong way only for a power this close to a rounding boundary (e.g. x = 1 - 2^-53,
# x^(3/2) = 1 - 1.5 2^-53 + 0.375 2^-106, which lies 2^-54.4 ulp above a midpoint)
HARD = 2.0**-40


def exponent(kind: int, n: int) -> float:
    return float((n, -n, n + 0.5, -(n + 0.5))[kind])


# ---------------------------------------------------------------------------------------------
# arguments
# ---------------------------------------------------------------------------------------------
def _base_arguments(n_random: int = 5, seed: int = 11) -> np.ndarray:
    """Every binade from 2^-1074 to 2^1023, both signs: mantissas 1, 1 + ulp, all ones and
    `n_random` random ones (subnormal binades: the same patterns below their leading bit);
    +-0, +-inf, NaN."""
    rng = np.random.default_rng(seed)
    frac = (1 << 52) - 1
    bits = []
    for e in range(1, 2047):  # normal binades
        m = [0, 1, frac] + [int(v) for v in rng.integers(2, frac, n_random)]
        bits += [(e << 52) | v for v in m]
    for j in range(52):  # subnormal binades [2^(j-1074), 2^(j-1073))
        top = 1 << j
        m = {top, top | 1, (top << 1) - 1} | {top | int(v) for v in rng.integers(0, top, n_random)} if j else {1}
        bits += sorted(m)
    pos = np.array(bits, dtype=np.uint64)
    x = np.concatenate([pos, pos | np.uint64(1 << 63)]).view(np.float64)
    special = np.array([0.0, -0.0, np.inf, -np.inf, np.nan])
    return np.concatenate([special, x])


_BASE = None


def arguments(kind: int, n: int) -> np.ndarray:
    """The base set plus a few ulps around each band edge of x^M, M = |exponent|: the overflow
    threshold DBL_MAX^(1/M), 2^(-1022/M), 2^(-1074/M), 2^(-1075/M), 2^(+-969/M), and for the
    negative powers the x where x^-M becomes subnormal or rounds to zero, 2^(1022/M),
    2^(1074/M), 2^(1075/M)."""
    global _BASE
    if _BASE is None:
        _BASE = _base_arguments()
    m = abs(exponent(kind, n))
    edges = []
    for e in (1024, -1022, -1074, -1075, 969, -969, 1022, 1074, 1075):
        t = e / m
        if not -1074 < t < 1024:
            continue
        v = math.ldexp(2.0 ** (t - math.floor(t)), math.floor(t))
        for k in range(-6, 7):
            w = v
            for _ in range(abs(k)):
                w = math.nextafter(w, math.inf if k > 0 else 0.0)
            edges += [w, -w]
    # and 4096 random operands spread over the operand band and a little beyond it
    rng = np.random.default_rng(1000 * kind + n)
    lo, hi = operand_band(kind, n)
    e = rng.uniform(math.log2(lo) - 2, math.log2(hi) + 2, 4096)
    inner = np.exp2(e) * rng.uniform(1, 2, e.size) * np.where(rng.random(e.size) < 0.25, -1.0, 1.0)
    return np.ascontiguousarray(np.concatenate([_BASE, np.array(edges), inner]))


# ---------------------------------------------------------------------------------------------
# reference
# ---------------------------------------------------------------------------------------------
def build_host_checker(workdir) -> ctypes.CDLL:
    so = os.path.join(str(workdir), "pow_check.so")
    subprocess.run(
        ["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-fopenmp", "-shared", "-fPIC",
         f"-I{NATIVE}", f'-DINFLX_DEVICE_HEADER="{HEADER}"', os.path.join(NATIVE, "pow_check.cpp"),
         "-o", so, "-lquadmath"],
        check=True,
    )  # fmt: skip
    lib = ctypes.CDLL(so)
    lib.pow_eval.argtypes = [ctypes.c_int, ctypes.c_int, _DP, ctypes.c_long, _DP, _DP,
                             ctypes.POINTER(ctypes.c_ubyte)]  # fmt: skip
    lib.pow_ref.argtypes = [ctypes.c_double, _DP, ctypes.c_long, _DP, _DP, _DP]
    return lib


def _exact_round(kind: int, n: int, x: float, r: float) -> float:
    """The correctly rounded power of x, given r = a rounding of it that is at most one step off."""
    neg = kind in (1, 3)
    if kind in (0, 1):
        p, v = 1, Fraction(x) ** n
    else:  # compare squares: v^2 = x^(2n+1)
        p, v = 2, Fraction(x) ** (2 * n + 1)
    if neg:
        v = 1 / v
    sign = -1.0 if v < 0 else 1.0
    v = abs(v)
    top = Fraction(2) ** 1024  # stands for +inf: the first value past DBL_MAX

    def frac(d):
        return Fraction(d) if d < math.inf else top

    def step(d, up):
        if d == math.inf:
            return d if up else 1.7976931348623157e308
        return math.nextafter(d, math.inf if up else 0.0)

    def odd(d):
        return d < math.inf and int(np.float64(d).view(np.uint64)) & 1

    best = abs(r)
    for _ in range(2):  # r is at most one step off
        below, above = step(best, False), step(best, True)
        m_dn, m_up = (frac(best) + frac(below)) / 2, (frac(best) + frac(above)) / 2
        if best > 0 and v < m_dn**p:
            best = below
        elif v > m_up**p:
            best = above
        else:
            if best > 0 and v == m_dn**p and odd(best):  # ties to even
                best = below
            elif v == m_up**p and odd(best):
                best = above
            break
    return sign * best


def reference(lib, kind: int, n: int, x: np.ndarray):
    """(correctly rounded power, distance of the quad value from a rounding boundary in ulps,
    glibc pow)"""
    m = x.size
    ref, dist, libm = np.empty(m), np.empty(m), np.empty(m)
    lib.pow_ref(exponent(kind, n), x.ctypes.data_as(_DP), m, ref.ctypes.data_as(_DP),
                dist.ctypes.data_as(_DP), libm.ctypes.data_as(_DP))  # fmt: skip
    for i in np.flatnonzero(dist < NEAR):
        xi = float(x[i])
        if math.isfinite(xi) and xi != 0.0 and not (kind >= 2 and xi < 0):
            ref[i] = _exact_round(kind, n, xi, float(ref[i]))
    return ref, dist, libm


# ---------------------------------------------------------------------------------------------
# the contract
# ---------------------------------------------------------------------------------------------
def operand_band(kind: int, n: int):
    """[2^lo, 2^hi) of |x| on which the chains run: x^M in [2^-969, 2^969] for M = |exponent|, and
    x >= 2^-969 for the half powers (inflx_pow_band)"""
    m2 = int(2 * abs(exponent(kind, n)))
    klo = -(1938 // m2)
    if m2 & 1:
        klo = max(klo, -969)
    khi = min(1938 // m2, 1017)
    return 2.0**klo, 2.0**khi


def classify(v: np.ndarray) -> np.ndarray:
    """0 NaN, +-1 inf, +-2 zero, +-3 subnormal, +-4 normal (sign of the value)"""
    a = np.abs(v)
    c = np.where(np.isnan(v), 0, np.where(np.isinf(v), 1, np.where(a == 0, 2, np.where(a < 2.0**-1022, 3, 4))))
    return np.where(np.signbit(v) & ~np.isnan(v), -c, c)


def same_bits(a, b):
    return (a.view(np.uint64) == b.view(np.uint64)) | (np.isnan(a) & np.isnan(b))


def ulps(a, b):
    """distance in ulps of two values of the same class and sign (0 where both are NaN)"""
    ia, ib = np.abs(a).view(np.int64), np.abs(b).view(np.int64)
    d = np.abs(ia - ib)
    return np.where(np.isnan(a) & np.isnan(b), 0, d)


def check_instance(kind, n, x, exact, spec, flag, cr, dist, hard=HARD):
    """Assert the contract for one instance; return (arguments outside the band, results that
    differ from the correctly rounded one).

    Every result is the correctly rounded power, except where the exact power lies within `hard`
    ulps of a rounding boundary: there the double-double value (~2^-100 relative) may round to the
    neighbour, 1 ulp off."""
    name = f"{KINDS[kind]}<{n}>"
    run = np.where(flag != 0, exact, spec)  # the grid kernel: speculative value unless flagged
    ccr = classify(cr)
    for pol, got in (("exact", exact), ("speculative", run)):
        bad = np.flatnonzero(classify(got) != ccr)
        assert bad.size == 0, (name, pol, "class", x[bad[:4]], got[bad[:4]], cr[bad[:4]])
    free = flag == 0
    bad = np.flatnonzero(free & ~same_bits(spec, exact))
    assert bad.size == 0, (name, "unflagged speculative != exact", x[bad[:4]], spec[bad[:4]], exact[bad[:4]])
    # the fast path is taken on the whole operand band (negative operands of a half power included:
    # their NaN is legitimate and costs no recomputation)
    lo, hi = operand_band(kind, n)
    a = np.abs(x)
    bad = np.flatnonzero((a >= lo) & (a < hi) & ~free)
    assert bad.size == 0, (name, "flagged inside the operand band", x[bad[:4]])
    a = np.abs(cr)
    inband = (a >= BAND[0]) & (a <= BAND[1])
    n_off = 0
    for pol, got in (("exact", exact), ("speculative", run)):
        off = ~same_bits(got, cr)
        bad = np.flatnonzero(off & ~((ulps(got, cr) <= 1) & (dist < hard)))
        assert bad.size == 0, (name, pol, "not correctly rounded", x[bad[:4]], got[bad[:4]], cr[bad[:4]],
                               dist[bad[:4]])  # fmt: skip
        n_off = max(n_off, int(off.sum()))
    return int((~inband).sum()), n_off


@pytest.fixture(scope="module")
def host(tmp_path_factory):
    return build_host_checker(tmp_path_factory.mktemp("pow"))


def eval_host(lib, kind, n, x):
    m = x.size
    exact, spec, flag = np.empty(m), np.empty(m), np.zeros(m, dtype=np.uint8)
    lib.pow_eval(kind, n, x.ctypes.data_as(_DP), m, exact.ctypes.data_as(_DP), spec.ctypes.data_as(_DP),
                 flag.ctypes.data_as(ctypes.POINTER(ctypes.c_ubyte)))  # fmt: skip
    return exact, spec, flag


@pytest.mark.parametrize("kind", sorted(KINDS))
def test_power_helper_is_correctly_rounded_over_the_double_range(host, kind):
    """Every instance, every binade, the band edges and the special values: result class and
    sign of the correctly rounded power, the speculative value equal to the exact one wherever it
    does not flag, no flag inside the operand band, and every result bit-identical to the correctly
    rounded one - inside the chains' band and, through the scaled forms, outside it (overflow,
    subnormal and zero results) - unless the power lies within 2^-40 ulp of a rounding boundary."""
    outside = off = libm_diff = total = 0
    for n in N_RANGE[kind]:
        x = arguments(kind, n)
        cr, dist, libm = reference(host, kind, n, x)
        exact, spec, flag = eval_host(host, kind, n, x)
        o, f = check_instance(kind, n, x, exact, spec, flag, cr, dist)
        outside, off, total = outside + o, off + f, total + x.size
        libm_diff += int((~same_bits(libm, cr)).sum())
    print(f"{KINDS[kind]}: {len(N_RANGE[kind])} instances, {total} arguments, {outside} results outside "
          f"[2^-969, 2^969], {off} within 2^-40 ulp of a rounding boundary and 1 ulp off; glibc pow "
          f"differs from the correctly rounded power on {libm_diff}")
    assert off <= total * 1e-3


def test_reference_decides_midpoints_exactly(host):
    """3^34 is a double midpoint (54 significant bits): ties to even; and a few exact powers."""
    for kind, n, xi, want in ((0, 34, 3.0, float(3**34 - 1)), (0, 3, 0.75, 0.421875),
                              (1, 4, 2.0**-300, math.inf), (1, 3, 2.0**300, 2.0**-900),
                              (3, 1, 4.0, 0.125), (2, 3, 4.0, 128.0)):  # fmt: skip
        cr, _, _ = reference(host, kind, n, np.array([xi]))
        assert cr[0] == want, (kind, n, xi, cr[0], want)
        exact, spec, flag = eval_host(host, kind, n, np.array([xi]))
        assert exact[0] == want and (flag[0] or spec[0] == want)
    assert _exact_round(0, 34, 3.0, float(3**34 + 1)) == float(3**34 - 1)


def test_issue_examples_no_longer_nan_or_zero(host):
    """Overflow gives +-inf, an underflowing reciprocal the correctly rounded subnormal."""
    cases = [
        (0, 3, float.fromhex("0x1.b399103b55abfp+341"), math.inf),
        (0, 3, -float.fromhex("0x1.b399103b55abfp+341"), -math.inf),
        (2, 3, float.fromhex("0x1.b399103b55abfp+341"), math.inf),
        (1, 3, 2.0**350, 2.0**-1050),
        (1, 2, 2.0**520, 2.0**-1040),
        (3, 1, float.fromhex("0x1.cc721bacf9358p+682"), None),
    ]
    for kind, n, xi, want in cases:
        x = np.array([xi])
        cr, _, _ = reference(host, kind, n, x)
        exact, spec, flag = eval_host(host, kind, n, x)
        run = exact if flag[0] else spec
        if want is not None:
            assert cr[0] == want
        assert cr[0] != 0 and not np.isnan(cr[0])
        assert exact[0] == cr[0] and run[0] == cr[0], (kind, n, xi, exact[0], run[0], cr[0])
