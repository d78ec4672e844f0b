"""The step kernel's math and layout primitives on the device, against exact references.

roadsurf_eval_primitive runs exp, log, the stability correction and the three division forms exactly as the
step kernel does (same definitions, constant-bank coefficients, global or shared-memory tables, fallbacks,
build flags).  The references:
  - glibc's exp / log through ctypes: the libm the oracle links, which rs_libm.h mirrors bit for bit on its
    fast path;
  - Decimal exp / ln at 60 digits, as an error in ulps;
  - the host's IEEE a / b, and for the cases outside the exact domain of the division forms a host model of
    the same fused operations in exact rational arithmetic.
Bit patterns are compared (parity.bit_mismatch): zeros must have the same sign, any two NaNs are equal.

The transpose and fill kernels are compared with NumPy, guard values around the written region included.
"""
import ctypes as C
import ctypes.util
import math
from decimal import Decimal, localcontext
from fractions import Fraction

import numpy as np
import pytest

from parity import bit_mismatch, same_bits
from roadsurf_b200 import lib

DIGITS = 60
# maximum errors documented for the algorithms (glibc sysdeps/ieee754/dbl-64/e_exp.c / e_log.c, FMA code path)
# and for CUDA's double-precision exp / log (CUDA Math API, "Mathematical Functions Appendix")
GLIBC_EXP_ULP, GLIBC_LOG_ULP, CUDA_ULP = 0.511, 0.519, 1.0
DBL_MIN = 2.2250738585072014e-308
LN2 = math.log(2.0)

_libm = C.CDLL(ctypes.util.find_library("m"))
for _f in ("exp", "log"):
    getattr(_libm, _f).restype = C.c_double
    getattr(_libm, _f).argtypes = [C.c_double]


def glibc(name, x):
    f = getattr(_libm, name)
    return np.array([f(float(v)) for v in x])


# ---- exact references ------------------------------------------------------------------------------------

def exp_ref(x):
    with localcontext() as ctx:
        ctx.prec = DIGITS
        return Decimal(float(x)).exp()


def log_ref(x):
    with localcontext() as ctx:
        ctx.prec = DIGITS
        return Decimal(float(x)).ln()


def ulp_of(ref):
    """Spacing of the doubles at the real number `ref` (below a power of two: the smaller spacing)."""
    f = abs(float(ref))
    u = math.ulp(f)
    if f > DBL_MIN and math.frexp(f)[0] == 0.5 and Decimal(f) > abs(ref):
        u /= 2
    return u


def ulp_error(y, ref):
    """|y - ref| in ulps of ref (y a finite double, ref a Decimal)."""
    with localcontext() as ctx:
        ctx.prec = DIGITS
        return float(abs(Decimal(float(y)) - ref) / Decimal(ulp_of(ref)))


def fma(x, y, z):
    """Correctly rounded x * y + z for finite operands, with IEEE's sign of an exact zero."""
    s = Fraction(x) * Fraction(y) + Fraction(z)
    if s == 0:
        return -0.0 if (math.copysign(1, x) * math.copysign(1, y) < 0 and math.copysign(1, z) < 0) else 0.0
    return float(s)


def div_const_model(a, c, rc):
    """The kernel's div_const (and fdiv, whose frcp(c) equals RN(1 / c) on its domain), operation by operation."""
    q = a * rc
    return fma(fma(-q, c, a), rc, q)


def f64(bits):
    return np.asarray(bits, dtype=np.uint64).view(np.float64)


def neighbours(x):
    return [math.nextafter(x, -math.inf), x, math.nextafter(x, math.inf)]


def exp_fast_path(x):
    """The arguments rs_libm.h's exp evaluates itself (|x| < 512; |x| < 2^-54 is 1 + x)."""
    return np.abs(x) < 512.0


def log_fast_path(x):
    """The arguments rs_libm.h's log evaluates itself (positive, normal, finite)."""
    return (x >= DBL_MIN) & (x < math.inf)


# ---- CPU: the references themselves ------------------------------------------------------------------------

def test_decimal_references_and_ulp_error_on_hand_computed_values():
    e = "2.71828182845904523536028747135266249775724709369995957496697"
    ln2 = "0.693147180559945309417232121458176568075500134360255254120680"
    assert str(exp_ref(1.0))[:55] == e[:55]
    assert str(log_ref(2.0))[:55] == ln2[:55]
    assert exp_ref(0.0) == 1 and log_ref(1.0) == 0
    assert ulp_error(1.0, Decimal(1)) == 0.0
    assert ulp_error(1.0 + 2.0 ** -52, Decimal(1)) == 1.0
    with localcontext() as ctx:
        ctx.prec = 400   # the references below are exact
        assert ulp_error(1.0, Decimal(1) - Decimal(2) ** -54) == 0.5      # below 1 the spacing is 2^-53
        assert ulp_error(2.0 ** -1074, Decimal(0)) == 1.0                  # subnormal spacing
        assert ulp_error(2.0 ** -1022, Decimal(2) ** -1022 - Decimal(2) ** -1075) == 0.5
    # glibc itself, at a few arguments, within its documented bound
    for x in (1.0, -1.0, 0.5, 100.0, -700.0, 1e-10):
        assert ulp_error(_libm.exp(x), exp_ref(x)) <= GLIBC_EXP_ULP
    for x in (2.0, 0.5, 1e-300, 1e300, 1.0 + 2.0 ** -30):
        assert ulp_error(_libm.log(x), log_ref(x)) <= GLIBC_LOG_ULP


def test_division_model_reproduces_the_known_sign_and_subnormal_cases():
    assert fma(2.0, 3.0, 1.0) == 7.0 and fma(0.1, 10.0, -1.0) == 5.551115123125783e-17
    assert math.copysign(1, fma(-0.0, 3.0, -0.0)) < 0 and math.copysign(1, fma(0.0, 3.0, -0.0)) > 0
    assert math.copysign(1, div_const_model(-0.0, 3.0, 1 / 3.0)) > 0          # IEEE: -0.0
    assert math.copysign(1, div_const_model(0.0, -3.0, 1 / -3.0)) < 0         # as IEEE
    assert div_const_model(1.0, 3.0, 1 / 3.0) == 1.0 / 3.0
    # a subnormal quotient the form rounds differently from IEEE division
    bad = [(a, c) for a, c in _subnormal_quotients(2000) if div_const_model(a, c, 1.0 / c) != a / c]
    assert bad


# ---- CPU: argument checks (no device work happens before them) ---------------------------------------------

def test_argument_checks_of_the_primitive_and_layout_entries():
    h = lib.load()
    fake = C.c_void_p(0x1000)  # never dereferenced: every call below is rejected or a no-op
    bad, ok = -2, 0             # RS_ERR_BAD_ARGUMENT, RS_OK
    ev = h.roadsurf_eval_primitive
    assert ev(-1, fake, fake, fake, 1, None) == bad
    assert ev(lib.PRIM_N, fake, fake, fake, 1, None) == bad
    assert ev(lib.PRIM_EXP, fake, None, fake, -1, None) == bad
    assert ev(lib.PRIM_EXP, None, None, fake, 1, None) == bad
    assert ev(lib.PRIM_EXP, fake, None, None, 1, None) == bad
    for fn in (lib.PRIM_FRCP, lib.PRIM_FDIV, lib.PRIM_DIV_CONST):
        assert ev(fn, fake, None, fake, 1, None) == bad
    assert b"bad arguments" in h.roadsurf_last_error()
    for fn in range(lib.PRIM_N):
        assert ev(fn, fake, fake, fake, 0, None) == ok
    to, frm = h.roadsurf_transpose_to_soa, h.roadsurf_transpose_from_soa
    # to_soa(src, src_ld, npoints, n, dst, ld) / from_soa(src, ld, npoints, n, dst, dst_ld)
    assert to(None, 4, 32, 4, fake, 32, None) == bad and to(fake, 4, 32, 4, None, 32, None) == bad
    assert to(fake, 4, -1, 4, fake, 32, None) == bad and to(fake, 4, 32, -1, fake, 32, None) == bad
    assert to(fake, 4, 33, 4, fake, 32, None) == bad and to(fake, 3, 32, 4, fake, 32, None) == bad
    assert frm(None, 32, 32, 4, fake, 4, None) == bad and frm(fake, 32, 32, 4, None, 4, None) == bad
    assert frm(fake, 32, -1, 4, fake, 4, None) == bad and frm(fake, 32, 32, -1, fake, 4, None) == bad
    assert frm(fake, 31, 32, 4, fake, 4, None) == bad and frm(fake, 32, 32, 4, fake, 3, None) == bad
    assert to(fake, 4, 0, 4, fake, 32, None) == ok and to(fake, 4, 32, 0, fake, 32, None) == ok
    assert frm(fake, 32, 0, 4, fake, 4, None) == ok and frm(fake, 32, 32, 0, fake, 4, None) == ok
    assert h.roadsurf_fill(None, 4, 1.0, None) == bad and h.roadsurf_fill(fake, -1, 1.0, None) == bad
    assert h.roadsurf_fill(fake, 0, 1.0, None) == ok


# ---- argument sets -------------------------------------------------------------------------------------------

F4 = lambda v: float(np.float32(v))  # noqa: E731  Fortran REAL(4) literals, as the kernel's F4()


def magnus_args():
    """fdiv(a * T, T + b) of CalcLE for surface / air temperatures in [-100, 100] (both coefficient sets)."""
    T = np.concatenate([np.linspace(-100.0, 100.0, 20001), [0.0, -0.0, 1e-300, -1e-300, 2.0 ** -1074]])
    a = np.where(T < 0, F4(21.875), F4(17.269))
    b = np.where(T < 0, F4(265.5), F4(237.3))
    return (a * T) / (T + b)


def pexp_args():
    """PExp = 22 - 2.7 Tair - 0.2 Rhz over the input-check ranges Tair in [-90, 100], Rhz in [-0.1, 120]."""
    tair, rhz = np.meshgrid(np.linspace(-90.0, 100.0, 381), np.concatenate([np.linspace(-0.1, 120.0, 121), [F4(-0.1)]]))
    return ((22.0 - F4(2.7) * tair) - F4(0.20) * rhz).ravel()


def decay_args():
    """The coupling and relaxation decays: -(DT i - DT end) / c for c = 4 h (the default couplingEffectReduction
    and the relaxation constant), time steps of 30 s to 1 h."""
    out = []
    for dt in (30.0, 60.0, 300.0, 3600.0):
        i = np.arange(0, int(10 * 86400 / dt) + 1, dtype=np.float64)   # up to 10 days past the window end
        out.append(-((dt * (i + 120)) - (dt * 120)) / (4.0 * 3600.0))
    return np.concatenate(out)


def exp_args(rng):
    sets = {}
    # every table index (k mod 128 of k = round(x * 128 / ln 2)) at the centre and both ends of its reduction
    # interval, over a spread of exponents
    k = np.concatenate([np.arange(128) + 128 * m for m in (-738, -500, -200, -40, -7, -1, 0, 1, 3, 20, 150, 600, 738)])
    c = k * (LN2 / 128)
    h = 0.4999 * LN2 / 128
    x = np.concatenate([c, c - h, c + h])
    sets["table"] = x[np.abs(x) < 512]
    sets["boundaries"] = np.array([s * v for v in (2.0 ** -54, 512.0) for s in (1, -1) for v in neighbours(v)])
    sets["special"] = np.array([0.0, -0.0, 2.0 ** -1074, -2.0 ** -1074, 2.0 ** -1030, -DBL_MIN, math.inf, -math.inf,
                                math.nan, 708.0, -708.0, 709.78, -709.78, 709.782712893384, 709.7827128933841,
                                745.13, -745.13, -745.1332191019411, -745.1332191019412, 710.0, -746.0, 1e300,
                                -1e300])
    sets["magnus"] = magnus_args()
    sets["pexp"] = pexp_args()
    sets["decay"] = decay_args()
    sets["random"] = np.exp2(rng.uniform(-60, 10, 1_000_000)) * rng.choice([-1.0, 1.0], 1_000_000)
    return sets


def psih_stab():
    s = -np.concatenate([[0.0, 1e6, 2.0 ** -1074], np.logspace(-12, 6, 20001), np.linspace(0, 50, 5001)])
    return np.concatenate([s, [-0.0]])


def log_args(rng):
    sets = {}
    # every table interval i = ((bits(x) - bits(0x1.6p-1)) >> 45) & 127: its first, middle and last argument,
    # at exponents from the subnormal boundary to the overflow boundary
    base = np.uint64(0x3FE6000000000000)
    xs = []
    for e in (-1000, -600, -100, -10, -1, 0, 1, 10, 100, 600, 1000):
        for i in range(128):
            for off in (0, 1 << 44, (1 << 45) - 1):
                bits = int(base) + (i << 45) + off + (e << 52)
                if 0 < bits < 0x7FF0000000000000:
                    xs.append(bits)
    sets["table"] = f64(xs)
    sets["boundaries"] = np.array(neighbours(1.0 - 2.0 ** -4) + neighbours(1.0 + float.fromhex("0x1.09p-4"))
                                  + neighbours(1.0) + neighbours(DBL_MIN) + neighbours(1.7976931348623157e308)[:2])
    sets["special"] = np.array([0.0, -0.0, 2.0 ** -1074, 1e-310, 2.0 ** -1023, math.nextafter(DBL_MIN, 0), -1.0,
                                -1e-300, -2.0 ** -1074, -math.inf, math.inf, math.nan, -math.nan])
    s = psih_stab()
    sets["psih"] = (1.0 + np.sqrt(1.0 - 16.0 * s)) / 2.0
    ex = rng.integers(1, 2047, 1_000_000, dtype=np.uint64)
    mant = rng.integers(0, 1 << 52, 1_000_000, dtype=np.uint64)
    sets["random"] = f64((ex << np.uint64(52)) | mant)
    return sets


def _subnormal_quotients(n, seed=5):
    r = np.random.default_rng(seed)
    out = []
    while len(out) < n:
        c = math.ldexp(1.0 + r.random(), int(r.integers(1, 60))) * (1 if r.random() < 0.5 else -1)
        a = math.ldexp(1.0 + r.random(), int(r.integers(-1074, -1021)))
        if a / c != 0 and abs(a / c) < DBL_MIN:
            out.append((a, c))
    return out


# ---- GPU: exp / log ----------------------------------------------------------------------------------------------

def _device(fn, a, b=None):
    import torch
    ta = torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()
    tb = None if b is None else torch.from_numpy(np.ascontiguousarray(b, dtype=np.float64)).cuda()
    return lib.eval_primitive(fn, ta, tb).cpu().numpy()


def _check_libm(name, fn, sets, fast_path, ref, glibc_ulp, special):
    x = np.concatenate(list(sets.values()))
    y = _device(fn, x)
    g = glibc(name, x)
    fast = fast_path(x)
    bad = bit_mismatch(y[fast], g[fast])
    assert not bad.any(), (name, fn, x[fast][bad][:8], y[fast][bad][:8], g[fast][bad][:8])
    # accuracy against the exact value: every structured argument, a sample of the random ones
    sample = np.concatenate([v if len(v) < 10_000 else v[::4] for k, v in sets.items() if k != "random"]
                            + [sets["random"][::500]])
    ys = _device(fn, sample)
    for xv, yv in zip(sample, ys):
        if fast_path(np.array([xv]))[0]:
            assert ulp_error(yv, ref(xv)) <= glibc_ulp, (name, xv, yv)
    # outside the fast path: the device library; special values exact, finite values within its 1 ulp
    slow = ~fast
    for xv, yv in zip(x[slow], y[slow]):
        want = special(xv)
        if want is not None:
            assert same_bits(np.array([yv]), np.array([want])), (name, xv, yv, want)
        else:
            r = ref(xv)   # next to the overflow threshold inf is as good as the largest double
            assert ((np.isinf(yv) and yv > 0 and r > Decimal(1.7976931348623157e308)) or
                    (np.isfinite(yv) and ulp_error(yv, r) <= CUDA_ULP)), (name, xv, yv)
    differ = int(bit_mismatch(y[slow], g[slow]).sum())
    print(f"{name} fn={fn}: {fast.sum()} fast-path arguments bit-equal to glibc; outside the fast path "
          f"{differ} of {slow.sum()} results differ from glibc")
    return y


def _exp_special(x):
    if math.isnan(x):
        return math.nan
    # overflow to inf / underflow to +0, except next to the thresholds (checked to 1 ulp there)
    if x > 710.0 or (x > 709.0 and exp_ref(x) > Decimal(1.7976931348623157e308) * (1 + Decimal(2) ** -40)):
        return math.inf
    if x < -746.0 or (x < -745.0 and exp_ref(x) < Decimal(2) ** -1075 * (1 - Decimal(2) ** -40)):
        return 0.0
    return None


def _log_special(x):
    if math.isnan(x) or x < 0:
        return math.nan
    if x == 0:
        return -math.inf
    if x == math.inf:
        return math.inf
    return None


EXP_FNS = [lib.PRIM_EXP, lib.PRIM_EXP_SMEM, lib.PRIM_EXP_FLAT, lib.PRIM_EXP_FLAT_SMEM]
LOG_FNS = [lib.PRIM_LOG, lib.PRIM_LOG_SMEM]


@pytest.mark.gpu
@pytest.mark.parametrize("fn", EXP_FNS, ids=["exp", "exp_smem", "exp_flat", "exp_flat_smem"])
def test_device_exp_equals_glibc_on_its_fast_path_and_cuda_exp_outside(rslib, exact, fn):
    sets = exp_args(np.random.default_rng(101))
    assert sets["pexp"].min() > -273 and sets["pexp"].max() < 266
    for k in ("magnus", "pexp", "decay", "table"):
        assert exp_fast_path(sets[k]).all(), k      # the model's call sites never leave the fast path
    _check_libm("exp", fn, sets, exp_fast_path, exp_ref, GLIBC_EXP_ULP, _exp_special)


@pytest.mark.gpu
@pytest.mark.parametrize("fn", LOG_FNS, ids=["log", "log_smem"])
def test_device_log_equals_glibc_on_its_fast_path_and_cuda_log_outside(rslib, exact, fn):
    sets = log_args(np.random.default_rng(102))
    assert log_fast_path(sets["psih"]).all() and log_fast_path(sets["table"]).all()
    _check_libm("log", fn, sets, log_fast_path, log_ref, GLIBC_LOG_ULP, _log_special)


@pytest.mark.gpu
@pytest.mark.parametrize("fn", [lib.PRIM_PSIH_UNSTABLE, lib.PRIM_PSIH_UNSTABLE_SMEM], ids=["psih", "psih_smem"])
def test_stability_correction_equals_the_host_expression_bitwise(rslib, exact, fn):
    s = psih_stab()
    y = _device(fn, s)
    want = np.array([-2.0 * math.log((1.0 + math.sqrt(1.0 - 16.0 * v)) / 2.0) for v in s])
    bad = bit_mismatch(y, want)
    assert not bad.any(), (s[bad][:8], y[bad][:8], want[bad][:8])


# ---- GPU: divisions ------------------------------------------------------------------------------------------------

DIV_FNS = [lib.PRIM_FDIV, lib.PRIM_DIV_CONST]

# Operand ranges of the divisions of model_step, from the input checks (Tair, Tdew in [-90, 100], VZ clamped to
# [0.4, 100], Rhz in [-0.1, 120], SW <= 4000, LW <= 1000, prec <= 500) and the model's constants; each range is
# sampled log-uniformly in magnitude with both signs where the numerator can take both.
CALL_SITES = {
    "WatSnowRat = SrfExtmms / RDummy": ((1e-6, 10.0), (1e-3, 100.0)),
    "PRain = 1 / (1 + exp(PExp))": ((1.0, 1.0), (1.0, 1e116)),
    "capDZ = 1 / (DyC VSH)": ((1.0, 1.0), (1e2, 1e9)),
    "AirDens = 1e5 / (287.05 TaK)": ((1e5, 1e5), (5e4, 1.1e5)),
    "UStar = kv / (logUstar + PSIM)": ((0.16, 40.0), (1e-3, 1e3)),
    "BLC = ck UStar / (logCond + PSIH)": ((1e-6, 1e6), (1e-3, 1e3)),
    "Stab = sfac BLC dT / (den0 UStar^3)": ((1e-12, 1e9), (1e-6, 1e12)),
    "Magnus = a T / (T + b)": ((1e-15, 2200.0), (165.0, 370.0)),
    "RAero = (...)(...) / (VK^2 VZ)": ((1e-6, 1e6), (0.064, 16.0)),
    "LE = ... / (PsychC RAero)": ((1e-9, 1e7), (1e-4, 3.0)),
    "Evap = LE / (L WatDen)": ((1e-9, 1e7), (3e8, 3e9)),
    "div_const by run constants (DT, 3600, 1000, ...)": ((1e-12, 1e9), (0.5, 14400.0)),
}
DOMAIN_LO, DOMAIN_HI = 2.0 ** -960, 2.0 ** 960   # |a| and |a / b|, with |b| in [2^-500, 2^500]


def _all_ones_mantissa(b):
    return (np.asarray(b, dtype=np.float64).view(np.uint64) & np.uint64(0xFFFFFFFFFFFFF)) == np.uint64(0xFFFFFFFFFFFFF)


def _log_uniform(rng, lo, hi, n, signed=True):
    v = np.exp(rng.uniform(math.log(lo), math.log(hi), n)) if hi > lo else np.full(n, lo)
    return v * (rng.choice([-1.0, 1.0], n) if signed else 1.0)


def _division_operands(rng):
    """(a, b) pairs inside the exact domain: a = +0, or a finite with |a| and |a / b| in [2^-960, 2^960], and
    |b| in [2^-500, 2^500]."""
    A, B = [], []
    # divisors: powers of two and all-ones mantissas across the range, a few constants, random
    special_b = [math.ldexp(m, e) for e in range(-500, 500, 3) for m in (1.0, 2.0 - 2.0 ** -52, 1.5, 1.0 + 2.0 ** -52)]
    special_b += [3.0, 10.0, 1000.0, 3364.0, 3600.0, 14400.0, 287.05, F4(287.05) * 273.15]
    for b in special_b:
        for s in (1.0, -1.0):
            bb = s * b
            # quotients at 1 - ulp, 1, 1 + ulp and their neighbours in the numerator
            for a in neighbours(bb) + [0.0, 1.0, -1.0, 2.0 * bb, bb * 3.0]:
                A.append(a)
                B.append(bb)
    n = 400_000
    b = np.exp2(rng.uniform(-500, 500, n)) * rng.choice([-1.0, 1.0], n)
    q = np.exp2(rng.uniform(-450, 450, n)) * rng.choice([-1.0, 1.0], n)
    A.extend(q * b)
    B.extend(b)
    for (alo, ahi), (blo, bhi) in CALL_SITES.values():
        A.extend(_log_uniform(rng, alo, ahi, 20_000))
        B.extend(_log_uniform(rng, blo, bhi, 20_000, signed=False))
    A, B = np.array(A), np.array(B)
    q = A / B
    keep = ((A == 0) & ~np.signbit(A)) | ((np.abs(A) >= DOMAIN_LO) & (np.abs(A) <= DOMAIN_HI) &
                                          (np.abs(q) >= DOMAIN_LO) & (np.abs(q) <= DOMAIN_HI))
    assert keep.mean() > 0.95
    return A[keep], B[keep]


def test_call_site_ranges_lie_inside_the_exact_division_domain():
    for name, ((alo, ahi), (blo, bhi)) in CALL_SITES.items():
        assert 2.0 ** -500 <= blo and bhi <= 2.0 ** 500, name
        assert DOMAIN_LO <= alo and ahi <= DOMAIN_HI, name
        assert DOMAIN_LO <= alo / bhi and ahi / blo <= DOMAIN_HI, name


@pytest.mark.gpu
def test_reciprocal_is_ieee_exact_over_its_documented_range(rslib):
    rng = np.random.default_rng(201)
    b = np.concatenate([[math.ldexp(m, e) for e in range(-500, 500) for m in (1.0, 2.0 - 2.0 ** -52, 1.5)],
                        np.exp2(rng.uniform(-500, 500, 1_000_000)), [2.0 ** 500, math.nextafter(2.0 ** -500, 1)]])
    b = np.concatenate([b, -b])
    y = _device(lib.PRIM_FRCP, np.zeros_like(b), b)
    bad = bit_mismatch(y, 1.0 / b)
    ones = _all_ones_mantissa(b)
    assert not (bad & ~ones).any(), (b[bad & ~ones][:8], y[bad & ~ones][:8])
    # b = (2 - 2^-52) 2^k: 1/b lies just above a rounding tie; the Newton steps can land on the tie itself and
    # round it to even, one ulp toward zero
    r = 1.0 / b[ones]
    assert (~bit_mismatch(y[ones], r) | ~bit_mismatch(y[ones], np.nextafter(r, 0.0))).all(), (b[ones][:4], y[ones][:4])
    print(f"frcp: {int(bad.sum())} of {int(ones.sum())} all-ones divisors one ulp toward zero, all others exact")


@pytest.mark.gpu
@pytest.mark.parametrize("fn", DIV_FNS, ids=["fdiv", "div_const"])
def test_division_forms_are_ieee_exact_on_their_domain(rslib, fn):
    a, b = _division_operands(np.random.default_rng(202))
    y = _device(fn, a, b)
    bad = bit_mismatch(y, a / b)
    # fdiv takes frcp's reciprocal: for all-ones divisors it is one ulp low and some quotients are, too
    allowed = _all_ones_mantissa(b) if fn == lib.PRIM_FDIV else np.zeros_like(bad)
    assert not (bad & ~allowed).any(), (a[bad & ~allowed][:8], b[bad & ~allowed][:8], y[bad & ~allowed][:8])
    q = a[bad] / b[bad]
    assert (np.abs(y[bad] - q) <= np.spacing(np.abs(q))).all()
    print(f"fn={fn}: {int(bad.sum())} of {int(allowed.sum())} quotients by all-ones divisors one ulp off")


# Outside the domain, as the forms behave (IEEE's answer in the comment).  The reciprocal's rcp.approx.ftz seed
# is infinite for a zero divisor and zero for an infinite one; the Newton steps then produce NaN.
OUT_OF_DOMAIN = [
    # (fn, a, b, result)
    (lib.PRIM_FRCP, 0.0, 0.0, math.nan),            # inf
    (lib.PRIM_FRCP, 0.0, -0.0, math.nan),           # -inf
    (lib.PRIM_FRCP, 0.0, math.inf, math.nan),       # 0
    (lib.PRIM_FRCP, 0.0, -math.inf, math.nan),      # -0
    (lib.PRIM_FRCP, 0.0, math.nan, math.nan),
    (lib.PRIM_FDIV, 1.0, 0.0, math.nan),            # inf
    (lib.PRIM_FDIV, -1.0, 0.0, math.nan),           # -inf
    (lib.PRIM_FDIV, 1.0, math.inf, math.nan),       # 0
    (lib.PRIM_FDIV, math.inf, 2.0, math.nan),       # inf
    (lib.PRIM_FDIV, -0.0, 3.0, 0.0),                # -0
    (lib.PRIM_FDIV, -0.0, -3.0, 0.0),               # 0
    (lib.PRIM_FDIV, 0.0, -3.0, -0.0),               # -0
    (lib.PRIM_DIV_CONST, 1.0, 0.0, math.nan),       # inf
    (lib.PRIM_DIV_CONST, 0.0, 0.0, math.nan),       # nan
    (lib.PRIM_DIV_CONST, 1.0, math.inf, math.nan),  # 0
    (lib.PRIM_DIV_CONST, math.inf, 2.0, math.nan),  # inf
    (lib.PRIM_DIV_CONST, -0.0, 3.0, 0.0),           # -0
    (lib.PRIM_DIV_CONST, -0.0, -3.0, 0.0),          # 0
    (lib.PRIM_DIV_CONST, 0.0, -3.0, -0.0),          # -0
]


@pytest.mark.gpu
def test_division_forms_outside_their_domain_behave_as_pinned(rslib):
    for fn in (lib.PRIM_FRCP, lib.PRIM_FDIV, lib.PRIM_DIV_CONST):
        rows = [r for r in OUT_OF_DOMAIN if r[0] == fn]
        y = _device(fn, [r[1] for r in rows], [r[2] for r in rows])
        want = np.array([r[3] for r in rows])
        bad = bit_mismatch(y, want)
        assert not bad.any(), [(rows[i], y[i]) for i in np.nonzero(bad)[0]]
    # subnormal quotients: the forms follow their operation sequence, which rounds some of them differently
    pairs = _subnormal_quotients(3000)
    a = np.array([p[0] for p in pairs])
    b = np.array([p[1] for p in pairs])
    want = np.array([div_const_model(x, c, 1.0 / c) for x, c in pairs])
    for fn in DIV_FNS:
        y = _device(fn, a, b)
        bad = bit_mismatch(y, want)
        assert not bad.any(), (fn, a[bad][:4], b[bad][:4], y[bad][:4], want[bad][:4])
        print(f"fn={fn}: {int(bit_mismatch(y, a / b).sum())} of {len(a)} subnormal quotients differ from IEEE")


# ---- GPU: layout kernels ------------------------------------------------------------------------------------------

GUARD = -12345.678


def _payload(rng, shape):
    v = rng.standard_normal(shape)
    flat = v.reshape(-1)
    flat[::7] = -0.0
    flat[3::11] = f64(np.uint64(0x7FF4000000000123))   # NaN payloads are copied, not re-encoded
    flat[5::13] = f64(np.uint64(0xFFF8000000000001))
    flat[1::17] = 2.0 ** -1074
    return v


def _transpose_both_ways(h, npoints, n, src_ld, ld, rng):
    import torch
    src = np.full((npoints, src_ld), GUARD)
    src[:, :n] = _payload(rng, (npoints, n))
    dst = np.full((n, ld), GUARD)
    ts, td = torch.from_numpy(src).cuda(), torch.from_numpy(dst).cuda()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert h.roadsurf_transpose_to_soa(ts.data_ptr(), src_ld, npoints, n, td.data_ptr(), ld, st) == 0, \
        h.roadsurf_last_error()
    want = dst.copy()
    want[:, :npoints] = src[:, :n].T
    got = td.cpu().numpy()
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64))    # payloads and guards, bit for bit
    back = torch.full((npoints, src_ld), GUARD, dtype=torch.float64, device="cuda")
    assert h.roadsurf_transpose_from_soa(td.data_ptr(), ld, npoints, n, back.data_ptr(), src_ld, st) == 0, \
        h.roadsurf_last_error()
    got = back.cpu().numpy()
    assert np.array_equal(got.view(np.uint64), src.view(np.uint64))


@pytest.mark.gpu
def test_transposes_copy_bit_exactly_and_touch_nothing_else(rslib):
    h = rslib.load()
    rng = np.random.default_rng(301)
    for npoints in (1, 31, 32, 33, 1000):
        for n in (1, 31, 33, 8881):
            if npoints * n > 2_000_000:
                continue
            _transpose_both_ways(h, npoints, n, n, npoints, rng)
    _transpose_both_ways(h, 33, 31, 40, 64, rng)        # row stride > n, plane stride > npoints
    _transpose_both_ways(h, 1000, 33, 33, 1003, rng)
    _transpose_both_ways(h, 1000, 8881, 8881, 1024, rng)


@pytest.mark.gpu
def test_transposes_of_more_points_than_one_grid_column(rslib):
    """More than 65535 * 32 points: the point tiles no longer fit one launch's grid.y."""
    _transpose_both_ways(rslib.load(), 2_097_153, 2, 2, 2_097_153, np.random.default_rng(302))


@pytest.mark.gpu
def test_empty_transposes_and_fill_are_no_ops(rslib):
    import torch
    h = rslib.load()
    t = torch.full((64,), GUARD, dtype=torch.float64, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = t.data_ptr()
    assert h.roadsurf_transpose_to_soa(p, 2, 0, 2, p, 32, st) == 0
    assert h.roadsurf_transpose_to_soa(p, 2, 32, 0, p, 32, st) == 0
    assert h.roadsurf_transpose_from_soa(p, 32, 0, 2, p, 2, st) == 0
    assert h.roadsurf_transpose_from_soa(p, 32, 32, 0, p, 2, st) == 0
    assert h.roadsurf_fill(p, 0, 1.0, st) == 0
    torch.cuda.synchronize()
    assert (t.cpu().numpy() == GUARD).all()


@pytest.mark.gpu
def test_fill_writes_exactly_its_range(rslib):
    import torch
    h = rslib.load()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    full_pass = 148 * 16 * 256
    for n, start in ((1, 0), (1, 3), (1000, 1), (full_pass, 0), (full_pass + 1, 0), (full_pass + 1, 5)):
        buf = torch.full((n + start + 9,), GUARD, dtype=torch.float64, device="cuda")
        value = -0.0 if n == 1000 else -9999.0
        assert h.roadsurf_fill(buf.data_ptr() + 8 * start, n, value, st) == 0, h.roadsurf_last_error()
        want = np.full(n + start + 9, GUARD)
        want[start:start + n] = value
        assert same_bits(buf.cpu().numpy(), want), (n, start)
