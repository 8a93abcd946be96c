"""Two steps of the INT8 digit GEMM (hk_gemm_i8.cu) in the form the kernels compute them, restated in Python and
checked against ``hk_digits_reference``:

- ``split_q_digits``: the 8 phase digits with rint done by adding and subtracting 1.5 2^52 and the digit read from the
  low word of the sum (no conversions), must be byte for byte ``split_digits(q, 8)``;
- the epilogue's two-part combination ``t = (hi + lo 2^-35) 2^-28`` of the ten int32 class sums (``ref.combine``) must
  be the correctly rounded class sum up to 31 K steps of 32 rows, stay within ``error_bound``'s combination term above,
  and equal the kernel's fma with its single rounding done exactly;
- the reference's own shortcuts must be exact: float64 matrix products for the integer class sums, and ``fma_int`` (the
  once-rounded fma of the phase arguments) on the cases where a double rounding would show.
"""
import math
from fractions import Fraction

import numpy as np
import pytest

import hk_digits_reference as ref


def split_q_digits(q: float) -> list:
    """hk_gemm_i8.cu ``split_q_digits``: rint(t) as (t + 1.5 2^52) - 1.5 2^52, the digit from the low word of the sum."""
    magic = np.float64(1.5 * 2.0**52)
    t = np.float64(q) * 64.0
    d = []
    for _ in range(ref.Q_DIGITS):
        s = t + magic
        lo = int(np.array(s).view(np.uint64)) & 0xFFFFFFFF
        d.append(lo - (1 << 32) if lo >= 1 << 31 else lo)
        t = (t - (s - magic)) * 128.0
    return d


def _check_split(qs):
    want = ref.split_digits(np.asarray(qs, dtype=np.float64), ref.Q_DIGITS)
    for i, q in enumerate(qs):
        got = split_q_digits(float(q))
        assert got == [int(v) for v in want[:, i]], f"q = {q!r}: {got} != {want[:, i].tolist()}"
        assert all(-64 <= v <= 64 for v in got)


def test_split_special_values():
    _check_split([0.0, -0.0, 1.0, -1.0, 0.5, -0.5, 2.0**-55, -(2.0**-55), 2.0**-56, 3 * 2.0**-57, 2.0**-1074, 1 - 2.0**-53])


@pytest.mark.parametrize("level", range(8))
def test_split_exact_ties_at_every_level(level):
    """q 2^(6 + 7 level) an exact half-integer, and the doubles either side of it, where rint's tie rule decides."""
    rng = np.random.default_rng(level)
    qs = []
    for _ in range(200):
        m = int(rng.integers(-(2 ** (6 + 7 * level)), 2 ** (6 + 7 * level)))
        q = (m + 0.5) * 2.0 ** -(6 + 7 * level)
        if abs(q) <= 1:
            qs += [q, np.nextafter(q, 2.0), np.nextafter(q, -2.0)]
    # q 2^6 = 1.5 -+ 2^-51: rounding q 2^55 first would make these exact ties
    qs += [(3 * 2.0**48 - 0.25) * 2.0**-55, -(3 * 2.0**48 - 0.25) * 2.0**-55, (3 * 2.0**48 + 0.25) * 2.0**-55]
    _check_split(qs)


def test_split_random_sample():
    rng = np.random.default_rng(1)
    x = rng.uniform(-2 * np.pi, 2 * np.pi, 100_000)
    qs = np.concatenate([np.cos(x), np.sin(x), rng.uniform(-1, 1, 50_000), np.ldexp(rng.uniform(-1, 1, 20_000), -rng.integers(0, 80, 20_000))])
    _check_split(qs)


def combine_two_part(acc: np.ndarray) -> np.ndarray:
    """``ref.combine`` with unit scaling (``s_j 2^-12 = 1``)."""
    return ref.combine(acc, np.full(acc.shape[1], 2.0**12))


def fma_with_fractions(acc: np.ndarray) -> np.ndarray:
    """The epilogue as the kernel writes it: hi and lo in int64, converted to double (rounded to nearest), then
    fma(lo, 2^-35, hi) 2^-28 with the fma's single rounding done exactly with Fractions."""
    hi = sum(acc[c].astype(object) * 2 ** (7 * (4 - c)) for c in range(5))
    lo = sum(acc[c].astype(object) * 2 ** (7 * (9 - c)) for c in range(5, 10))
    assert all(abs(v) < 2**63 for v in np.concatenate([hi.ravel(), lo.ravel()]))
    out = np.empty(acc.shape[1:])
    for idx in np.ndindex(out.shape):
        h, l = float(hi[idx]), float(lo[idx])  # int64 -> double conversions, rounded to nearest
        out[idx] = float(Fraction(l) * Fraction(1, 2**35) + Fraction(h)) * 2.0**-28
    return out


def exact_class_sum(acc: np.ndarray, idx) -> Fraction:
    return sum((Fraction(int(acc[c][idx]), 2 ** (7 * c)) for c in range(ref.CLASSES)), Fraction(0))


def _adversarial_acc(ksteps, rng, n=64):
    """Class sums of K steps at their largest: |s_c| up to n_c 64^2 32 K (n_c digit pairs of class c)."""
    n_c = np.array([min(c + 1, ref.Q_DIGITS, ref.W_DIGITS, ref.Q_DIGITS + ref.W_DIGITS - 1 - c) for c in range(ref.CLASSES)])
    top = n_c * 64 * 64 * 32 * ksteps
    acc = np.stack([rng.integers(-top[c], top[c] + 1, n) for c in range(ref.CLASSES)])
    acc[:, 0] = top  # all at the top
    acc[:, 1] = -top
    acc[:, 2] = 0
    acc[:, 3] = 0
    acc[0, 3] = 1
    acc[9, 3] = -1
    return acc


@pytest.mark.parametrize("ksteps", [1, 2, 16, 31])
def test_two_part_combination_is_correctly_rounded(ksteps):
    acc = _adversarial_acc(ksteps, np.random.default_rng(ksteps))
    got = combine_two_part(acc)
    for i in range(acc.shape[1]):
        want = float(exact_class_sum(acc, i))  # Fraction -> float rounds to nearest, ties to even
        assert got[i] == want, f"K steps {ksteps}, column {i}: {got[i]!r} != {want!r}"


@pytest.mark.parametrize("ksteps", [32, 63, 500, 2047])
def test_two_part_combination_within_bound_above_31_steps(ksteps):
    """Above 31 K steps hi and lo may round when converted: three roundings, well inside the ten of error_bound."""
    acc = _adversarial_acc(ksteps, np.random.default_rng(ksteps))
    got = combine_two_part(acc)
    u = 2.0**-53
    for i in range(acc.shape[1]):
        exact = exact_class_sum(acc, i)
        mag = sum(abs(int(acc[c][i])) * 2.0 ** (-7 * c) for c in range(ref.CLASSES))
        assert abs(Fraction(got[i]) - exact) <= Fraction(10 * u * mag * (1 + 16 * u)), f"K steps {ksteps}, column {i}"


def test_two_part_combination_exact_zero_and_power_of_two_scaling():
    acc = np.zeros((ref.CLASSES, 3), dtype=np.int64)
    acc[:, 1] = np.arange(1, 11) * 12345
    acc[:, 2] = -acc[:, 1]
    t = combine_two_part(acc)
    assert t[0] == 0.0 and math.copysign(1.0, t[0]) == 1.0
    for e in (-600, -64, 64, 600):
        s = np.ldexp(1.0, e - 12)
        assert np.array_equal(np.ldexp(t * s, -e), t * np.ldexp(1.0, -12))


@pytest.mark.parametrize("ksteps", [1, 31, 32, 2047])
def test_numpy_combination_is_the_kernels_fma(ksteps):
    acc = _adversarial_acc(ksteps, np.random.default_rng(100 + ksteps), n=200)
    assert np.array_equal(combine_two_part(acc), fma_with_fractions(acc))


def _class_sums_int64(qd, wd):
    acc = np.zeros((ref.CLASSES, qd.shape[1], wd.shape[2]), dtype=np.int64)
    for a in range(ref.Q_DIGITS):
        for b in range(ref.W_DIGITS):
            if a + b < ref.CLASSES:
                acc[a + b] += qd[a] @ wd[b]
    return acc


@pytest.mark.parametrize("K", [32, 1000, 65504])
def test_float64_class_sums_are_exact(K):
    """Digits at +-64 on every row (the largest sums), alternating signs and random digits: the float64 products of
    ``class_sums`` must equal int64 products, up to the kernel's 65 504 rows (2047 K steps)."""
    rng = np.random.default_rng(K)
    n_k, NN = 3, 5
    qd = rng.integers(-64, 65, (ref.Q_DIGITS, n_k, K))
    wd = rng.integers(-64, 65, (ref.W_DIGITS, K, NN))
    qd[:, 0] = 64
    wd[:, :, 0] = 64
    wd[:, :, 1] = -64
    qd[:, 1] = np.where(np.arange(K) % 2, 64, -64)
    wd[:, :, 2] = np.where(np.arange(K) % 2, -64, 64)[None, :]
    got = ref.class_sums(qd, wd)
    want = _class_sums_int64(qd, wd)
    assert np.array_equal(got, want)
    assert got[4, 0, 0] == 5 * 64 * 64 * K  # five digit pairs of class 4, all at the top


def test_fma_int_is_rounded_once():
    """``fma_int(a, n, c)`` against the exactly rounded Fraction value: random arguments, and sums placed exactly one
    longdouble ulp from a double midpoint, where rounding twice would go the wrong way."""
    rng = np.random.default_rng(5)
    a = np.concatenate([rng.uniform(-2, 2, 3000), rng.uniform(-1e3, 1e3, 3000), np.ldexp(rng.uniform(-1, 1, 2000), -rng.integers(0, 60, 2000))])
    n = rng.integers(-40, 41, len(a))
    c = np.concatenate([rng.uniform(-50, 50, 4000), rng.uniform(-5e4, 5e4, 4000)])
    # a n = c' + 2^-53 (1 +- 2^-11): c' + a n is a double midpoint plus or minus a tail below the longdouble grid of c'
    m = 2000
    cc = rng.uniform(1, 2, m)
    tail = np.ldexp(1.0, -53) * (1 + np.where(rng.random(m) < 0.5, 1, -1) * 2.0**-12)
    a2, n2, c2 = tail, np.ones(m, dtype=np.int64), cc
    a = np.concatenate([a, a2, -a2])
    n = np.concatenate([n, n2, n2])
    c = np.concatenate([c, c2, -c2])
    got = ref.fma_int(a, n, c)
    for i in range(len(a)):
        want = float(Fraction(float(a[i])) * int(n[i]) + Fraction(float(c[i])))
        assert got[i] == want, f"fma({a[i]!r}, {n[i]}, {c[i]!r}) = {want!r}, got {got[i]!r}"
