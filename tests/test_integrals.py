"""The host half of the exact integrals (mpas_b200.h, MpasIntegral): mpasb200_integral_value rounds the sum the limbs
represent exactly once, and mpasb200_integral_merge is exact and order-independent.  Accumulators are built here from the
documented representation, sum = sum_j limb[j] * 2^(32 j - 1088); no GPU is needed."""
import ctypes as C
import math
import struct
from fractions import Fraction

import numpy as np
import pytest

from mpas_regent_b200 import _abi, dynamics, parallel

NL, BIAS = _abi.INTEGRAL_LIMBS, _abi.INTEGRAL_BIAS
MASK = (1 << 32) - 1


def acc_of(N, limbs=None, **counts):
    """the canonical accumulator of the integer N (the sum in units of 2^-1088), or raw limbs as given"""
    a = _abi.MpasIntegral()
    if limbs is None:
        limbs = []
        for _ in range(NL - 1):
            limbs.append(N & MASK)
            N >>= 32
        limbs.append(N)
    a.limb[:] = [int(x) for x in limbs]
    for k, v in counts.items():
        setattr(a, k, v)
    return a


def exact(a):
    return sum(int(a.limb[j]) << (32 * j) for j in range(NL))


def value(a):
    return dynamics.load_library().mpasb200_integral_value(C.byref(a))


def ref(N):
    """float(Fraction) is correctly rounded (ties to even); it raises where the rounded value is out of range"""
    try:
        return float(Fraction(N, 1 << BIAS))
    except OverflowError:
        return math.inf if N > 0 else -math.inf


def same_bits(x, y):
    return struct.pack("<d", x) == struct.pack("<d", y)


def check(N):
    got, want = value(acc_of(N)), ref(N)
    assert same_bits(got, want), (N, got, want)


def units(x: float) -> int:
    """a double as an exact integer multiple of 2^-1088"""
    n, d = x.as_integer_ratio()
    return n * ((1 << BIAS) // d)


def test_ties_round_to_even():
    one = 1 << BIAS
    for base in (1 << 53, 3 << 60, (1 << 53) * 7):
        for m in (base + 1, base + 3, base + 5):               # odd multiples of half an ulp above 2^53-sized integers
            for sign in (1, -1):
                check(sign * m * one)
                check(sign * (m * one + 1))                    # just above the tie
                check(sign * (m * one - 1))                    # just below it
    assert value(acc_of(((1 << 53) + 1) * one)) == 2.0 ** 53
    assert value(acc_of(((1 << 53) + 3) * one)) == 2.0 ** 53 + 4


def test_subnormal_results():
    tiny = 1 << (BIAS - 1074)                                  # 2^-1074 in units
    for n in (1, 2, 3, tiny // 2, tiny // 2 + 1, tiny, 3 * tiny // 2, 5 * tiny // 2, 12345 * tiny + 7, (1 << 52) * tiny - 1,
              (1 << 52) * tiny, ((1 << 52) - 1) * tiny + tiny // 2):
        for sign in (1, -1):
            check(sign * n)
    assert same_bits(value(acc_of(-3)), -0.0)                  # a negative sum below half of 2^-1074 rounds to -0
    assert value(acc_of(tiny // 2 + 1)) == 5e-324 and value(acc_of(tiny // 2)) == 0.0


def test_sums_that_cancel_to_zero():
    rng = np.random.default_rng(0)
    xs = [float(x) for x in rng.standard_normal(200) * 10.0 ** rng.integers(-300, 300, 200)]
    acc = _abi.MpasIntegral()
    lib = dynamics.load_library()
    for x in xs + [-x for x in reversed(xs)]:
        assert lib.mpasb200_integral_merge(C.byref(acc), C.byref(acc_of(units(x)))) == 0
    assert list(acc.limb) == [0] * NL
    assert same_bits(value(acc), 0.0)
    assert same_bits(value(acc_of(0)), 0.0)
    assert same_bits(value(acc_of(0, limbs=[1 << 32, -1] + [0] * (NL - 2))), 0.0)      # non-canonical zero


def test_overflow_to_infinity():
    big = 1 << (1024 + BIAS)                                   # 2^1024 in units
    half_ulp = 1 << (970 + BIAS)
    for n in (big, big - half_ulp, big - half_ulp - 1, big - 2 * half_ulp, 5 * big, (1 << (NL * 32 - 2)) - 1):
        for sign in (1, -1):
            check(sign * n)
    assert value(acc_of(big - half_ulp)) == math.inf           # the tie with the largest double goes to even = 2^1024
    assert value(acc_of(big - half_ulp - 1)) == np.finfo(np.float64).max
    assert value(acc_of(-big)) == -math.inf


def test_nan_and_inf_rules():
    n = units(1.5)
    assert math.isnan(value(acc_of(n, n_nan=1)))
    assert math.isnan(value(acc_of(n, n_pinf=2, n_ninf=1)))
    assert math.isnan(value(acc_of(n, n_nan=1, n_pinf=1)))
    assert value(acc_of(n, n_pinf=3)) == math.inf
    assert value(acc_of(-n, n_ninf=1)) == -math.inf
    assert value(acc_of(n, count=10)) == 1.5


def test_random_sums_and_raw_limbs():
    """random doubles of every magnitude, subnormals included, and accumulators with arbitrary (non-canonical) limbs"""
    rng = np.random.default_rng(1)
    for _ in range(40):
        xs = rng.standard_normal(300) * 10.0 ** rng.integers(-320, 308, 300)
        xs[rng.random(300) < 0.1] = rng.integers(-1000, 1000, 1).astype(float) * 5e-324
        check(sum(units(float(x)) for x in xs if np.isfinite(x)))
    for _ in range(200):
        limbs = [int(x) for x in rng.integers(-(1 << 62), 1 << 62, NL)]
        limbs[rng.integers(0, NL)] = int(rng.integers(-(1 << 63), (1 << 63) - 1))
        a = acc_of(0, limbs=limbs)
        top = int(rng.integers(0, NL))
        for j in range(top + 1, NL):                           # a random size, from subnormal to overflow
            a.limb[j] = 0
        got, want = value(a), ref(exact(a))
        assert same_bits(got, want), (limbs, got, want)


def test_merge_is_exact_and_order_independent():
    rng = np.random.default_rng(2)
    xs = rng.standard_normal(400) * 10.0 ** rng.integers(-300, 300, 400)
    parts = [{"limbs": np.array(acc_of(units(float(x))).limb[:], dtype=np.int64), "count": 1, "n_nan": int(i % 7 == 0),
              "n_pinf": 0, "n_ninf": 0} for i, x in enumerate(xs)]
    want = sum(units(float(x)) for x in xs)
    outs = []
    for _ in range(6):                                          # random splits into partitions, merged in random orders
        perm = rng.permutation(len(parts))
        cuts = sorted(rng.choice(np.arange(1, len(parts)), size=int(rng.integers(1, 20)), replace=False))
        groups = [dynamics.merge_integrals([parts[i] for i in g]) for g in np.split(perm, cuts)]
        rng.shuffle(groups)
        outs.append(parallel.merge_integrals(groups))
    for o in outs:
        assert np.array_equal(o["limbs"], outs[0]["limbs"])
        assert exact(dynamics.as_integral(o)) == want
        assert np.array_equal(o["limbs"], np.array(acc_of(want).limb[:], dtype=np.int64))     # canonical form
        assert o["count"] == len(xs) and o["n_nan"] == sum(p["n_nan"] for p in parts)
        assert math.isnan(o["value"])
    unflagged = parallel.merge_integrals([dict(p, n_nan=0) for p in parts])
    assert same_bits(unflagged["value"], ref(want)) and unflagged["bits"] == f"{struct.unpack('<Q', struct.pack('<d', ref(want)))[0]:016x}"


def test_merge_refuses_a_sum_out_of_range():
    lib = dynamics.load_library()
    a = acc_of(0, limbs=[0] * (NL - 1) + [(1 << 63) - 1])
    assert lib.mpasb200_integral_merge(C.byref(a), C.byref(acc_of(0, limbs=[0] * (NL - 1) + [1]))) == _abi.E_INVAL
    assert lib.mpasb200_integral_merge(None, C.byref(a)) == _abi.E_INVAL
    with pytest.raises(dynamics.MpasB200Error):
        dynamics.merge_integrals([{"limbs": np.array(a.limb[:]), "count": 0, "n_nan": 0, "n_pinf": 0, "n_ninf": 0}] * 2)
