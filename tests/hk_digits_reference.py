"""Python restatement of the INT8 digit GEMM of the H(k) build (tbmodels_b200/csrc/hk_gemm_i8.cu).

``Hp[k, j] = sum_r Q[k, r] W[r, j]`` with |Q| <= 1 (the [cos | sin] phase rows) and W the Hermitian-split weights:

- ``q = sum_{a=0..7} q_a 2^(-6-7a)``, ``q_a`` in [-64, 64], rounded at 2^-55;
- ``W_rj / s_j = sum_{b=0..8} w_b 2^(-6-7b)``, rounded at 2^-62, ``s_j`` the power of two with
  ``2^-1 s_j <= max_r |W_rj| < s_j`` (0 for an all-zero column, whose digits are all 0);
- class ``c = a + b`` has weight ``2^(-12-7c)``; the class sums ``s_c``, c <= 9, are exact integers (int32 on the GPU);
- the epilogue combines them exactly into ``hi = sum_{c<=4} s_c 2^(7(4-c))`` and ``lo = sum_{c>=5} s_c 2^(7(9-c))``
  (int64), converts each to double (exact up to 31 K steps of 32 rows), forms ``fma(lo, 2^-35, hi)`` (one rounding) and
  scales by ``2^-28`` and ``s_j 2^-12`` (both exact).

The phase rows are those of the kernel too (:func:`phase_rows`): ``x = fma(k_{D-1}, R_{D-1}, ... fma(k_0, R_0, 0.0))``
with every fma rounded once, then ``sincospi_lean(2 x)`` of ``tbk_math.cuh``, run on the host through
``tbk_host_sincospi``.  Every operation is an exact integer operation or a correctly rounded double operation, so
:func:`hamilton_int8` gives the kernel's bits for a model and a set of k-points (convention 2).  Neither the order of the
stored R nor the power-of-two normalisation of the model on the device changes a bit: integer sums do not depend on
order, and scaling by 2^e commutes with every step.  ``error_bound`` is the a-priori bound of the scheme per element.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

Q_DIGITS = 8
W_DIGITS = 9
CLASSES = 10


def split_digits(x: np.ndarray, n_digits: int) -> np.ndarray:
    """Balanced digits ``d[a]`` in [-64, 64] of ``x`` (|x| <= 1) with ``x ~ sum_a d[a] 2^(-6-7a)``: shape
    ``(n_digits,) + x.shape``, int64.  Every step but the last ``rint`` is exact."""
    t = np.asarray(x, dtype=np.float64) * 64.0
    out = np.empty((n_digits,) + t.shape, dtype=np.int64)
    for a in range(n_digits):
        r = np.rint(t)
        out[a] = r.astype(np.int64)
        t = (t - r) * 128.0
    return out


def column_exponents(W: np.ndarray) -> np.ndarray:
    """``e_j`` with ``s_j = 2^e_j``, ``2^(e_j - 1) <= max_r |W_rj| < 2^e_j`` (0 for all-zero columns)."""
    _, e = np.frexp(np.abs(W).max(axis=0) if W.shape[0] else np.zeros(W.shape[1]))
    return e.astype(np.int64)


def w_digits(W: np.ndarray):
    """(digits ``[9, K, NN]``, scales ``s_j``): all-zero columns get zero digits and ``s_j = 0``."""
    e = column_exponents(W)
    nz = np.abs(W).max(axis=0) > 0 if W.shape[0] else np.zeros(W.shape[1], dtype=bool)
    d = split_digits(np.ldexp(W, -e[None, :]), W_DIGITS)
    d[:, :, ~nz] = 0
    s = np.where(nz, np.ldexp(1.0, e), 0.0)
    return d, s


def q_digits(Q: np.ndarray) -> np.ndarray:
    """Digits ``[8, n_k, K]`` of the phase rows (|Q| <= 1)."""
    return split_digits(Q, Q_DIGITS)


def class_sums(qd: np.ndarray, wd: np.ndarray) -> np.ndarray:
    """Exact ``acc[c, k, j] = sum_{a + b = c} sum_r q_a[k, r] w_b[r, j]`` for c = 0 .. 9 (int64).

    The products run as float64 matrix products: digits are at most 64 in magnitude and K below 2^16 rows, so every
    partial sum of every product is an integer below 2^28 and the result is exact in any summation order."""
    K = qd.shape[2]
    assert K < 2**16, "more rows than the int32 class sums of the kernel allow"
    n_k, NN = qd.shape[1], wd.shape[2]
    qf = qd.reshape(Q_DIGITS * n_k, K).astype(np.float64)
    acc = np.zeros((CLASSES, n_k, NN), dtype=np.int64)
    for b in range(W_DIGITS):
        prod = (qf @ wd[b].astype(np.float64)).reshape(Q_DIGITS, n_k, NN)
        for a in range(min(Q_DIGITS, CLASSES - b)):
            acc[a + b] += prod[a].astype(np.int64)
    return acc


def combine(acc: np.ndarray, s: np.ndarray) -> np.ndarray:
    """The epilogue: ``hi`` and ``lo`` in int64, ``t = fma(double(lo), 2^-35, double(hi)) 2^-28``, times ``s_j 2^-12``.

    ``double(lo) 2^-35`` is exact (a power-of-two scaling far from the subnormals), so ``double(lo) 2^-35 +
    double(hi)`` rounds once, exactly as the fma does; the two scalings are exact."""
    hi = np.zeros(acc.shape[1:], dtype=np.int64)
    lo = np.zeros(acc.shape[1:], dtype=np.int64)
    for c in range(5):
        hi += acc[c] << (7 * (4 - c))
        lo += acc[c + 5] << (7 * (4 - c))
    t = (lo.astype(np.float64) * 2.0**-35 + hi.astype(np.float64)) * 2.0**-28
    return t * np.ldexp(s, -12)  # s_j along the last axis


def digit_gemm(Q: np.ndarray, W: np.ndarray) -> np.ndarray:
    """``Q [n_k, K] @ W [K, NN]`` as the INT8 kernel computes it."""
    wd, s = w_digits(W)
    return combine(class_sums(q_digits(Q), wd), s)


def error_bound(Q: np.ndarray, W: np.ndarray) -> np.ndarray:
    """Per-element bound ``[n_k, NN]`` on ``|digit_gemm(Q, W) - Q @ W|`` (exact product):

    - dropped classes c >= 10: per row at most sum_c n_c 2^(-7c) <= 11 2^-70 of s_j (n_c pairs of 64 x 64 digits);
    - W rounding: 2^-63 s_j per row (|q| <= 1);
    - Q rounding: 2^-56 |W_rj| per row;
    - the combination: at most three roundings (hi, lo, the fma; only the fma up to 31 K steps), bounded here by the ten
      of a Horner chain, 10 u sum_c |acc_c| 2^(-12-7c) s_j.
    """
    K = W.shape[0]
    wd, s = w_digits(W)
    acc = class_sums(q_digits(Q), wd)
    mag = np.zeros(acc.shape[1:])
    for c in range(CLASSES):
        mag += np.abs(acc[c]).astype(np.float64) * 2.0 ** (-12 - 7 * c)
    u = 2.0**-53
    dropped_and_w = K * s * (11 * 2.0**-70 + 2.0**-63)
    return dropped_and_w[None, :] + 2.0**-56 * np.abs(W).sum(axis=0)[None, :] + 10 * u * mag * s[None, :] * (1 + 16 * u)


def digits_fraction(d) -> "Fraction":
    """Exact value ``sum_a d[a] 2^(-6-7a)`` of one digit vector."""
    from fractions import Fraction

    return sum((Fraction(int(v), 2 ** (6 + 7 * a)) for a, v in enumerate(d)), Fraction(0))


# ------------------------------------------------------------------------------------ the kernel's inputs, restated
def fma_int(a: np.ndarray, n: np.ndarray, c: np.ndarray) -> np.ndarray:
    """``fma(a, n, c)`` rounded once, for float64 ``a``, ``c`` and integers ``|n| < 2^11`` (broadcast).

    ``a n`` has at most 64 significant bits, so it is exact in the 80-bit ``np.longdouble``; the sum ``s = a n + c`` is
    rounded there, and its exact error ``e`` follows from TwoSum.  Converting ``s`` to double is then the correctly
    rounded result except when ``s`` lies exactly halfway between two doubles and ``e != 0``: the exact sum is off the
    midpoint, on the side of ``e``."""
    LD = np.longdouble
    if np.finfo(LD).nmant < 63:
        raise RuntimeError("fma_int needs an 80-bit np.longdouble")
    n = np.asarray(n)
    assert np.all(np.abs(n) < 2**11)
    p = np.asarray(a, dtype=np.float64).astype(LD) * n.astype(LD)
    cl = np.asarray(c, dtype=np.float64).astype(LD)
    s = p + cl
    bb = s - p
    err = (p - (s - bb)) + (cl - bb)
    d = s.astype(np.float64)
    off = s - d.astype(LD)  # exact: s and d are within half an ulp of d
    other = np.nextafter(d, np.where(off > 0, np.inf, -np.inf))
    tie = (off != 0) & (err != 0) & (other.astype(LD) - s == off)
    fix = tie & ((err > 0) == (off > 0))
    return np.where(fix, other, d)


def phase_args(k: np.ndarray, R: np.ndarray) -> np.ndarray:
    """``2 x`` ``[n_k, n_R]`` with ``x = fma(k_{D-1}, R_{D-1}, ... fma(k_0, R_0, 0.0))``: the argument of
    ``sincospi_lean`` in hk_phase_kernel and hk_qdigits_kernel."""
    k = np.asarray(k, dtype=np.float64)
    R = np.asarray(R, dtype=np.int64)
    x = np.zeros((k.shape[0], R.shape[0]))
    for d in range(R.shape[1]):
        x = fma_int(k[:, d : d + 1], R[None, :, d], x)
    return 2.0 * x


def sincospi(t: np.ndarray):
    """(sin, cos) of ``pi t`` by ``sincospi_lean`` (tbk_math.cuh, compiled for the host), elementwise."""
    from tbmodels_b200 import _capi

    f = _capi.load().tbk_host_sincospi
    t = np.asarray(t, dtype=np.float64)
    tu, inv = np.unique(t.ravel(), return_inverse=True)
    sv, cv = np.empty(len(tu)), np.empty(len(tu))
    s, c = C.c_double(), C.c_double()
    ps, pc = C.byref(s), C.byref(c)
    for i, v in enumerate(tu.tolist()):
        f(v, ps, pc)
        sv[i] = s.value
        cv[i] = c.value
    return sv[inv].reshape(t.shape), cv[inv].reshape(t.shape)


def phase_rows(k: np.ndarray, R: np.ndarray) -> np.ndarray:
    """The kernel's phase rows ``[n_k, 2 n_R]``: cos and sin of ``2 pi k.R`` interleaved, the row order of W."""
    sn, cs = sincospi(phase_args(k, R))
    Q = np.empty((sn.shape[0], 2 * sn.shape[1]))
    Q[:, 0::2] = cs
    Q[:, 1::2] = sn
    return Q


def packed_weights(p) -> np.ndarray:
    """The Hermitian-split weights ``[2 n_R, N^2]`` of a packed model (``tbk_host_pack_weights``, the host pack of
    tbk_api.cu): rows ``2 r`` = hp(T_r + T_r^H) and ``2 r + 1`` = hp(i (T_r - T_r^H))."""
    from tbmodels_b200 import _capi

    dp = C.POINTER(C.c_double)
    hop = np.ascontiguousarray(p.hop, dtype=np.complex128)
    W = np.zeros((2 * p.n_R, p.size * p.size))
    rc = _capi.load().tbk_host_pack_weights(p.size, p.n_R, hop.view(np.float64).ctypes.data_as(dp), W.ctypes.data_as(dp))
    assert rc == 0
    return W


def unpack_hermitian(hp: np.ndarray, N: int) -> np.ndarray:
    """Packed ``[n_k, N^2]`` -> complex ``[n_k, N, N]`` as expand.cu writes convention 2: the lower triangle as stored,
    a zero imaginary diagonal, the upper triangle the conjugate of the lower one."""
    nre = N * (N + 1) // 2
    i, j = np.tril_indices(N)
    diag = i == j
    re = hp[:, i * (i + 1) // 2 + j]
    im = hp[:, np.where(diag, 0, nre + i * (i - 1) // 2 + j)]
    im[:, diag] = 0.0
    H = np.empty((hp.shape[0], N, N), dtype=np.complex128)
    H.real[:, j, i] = re
    H.imag[:, j, i] = -im
    H.real[:, i, j] = re
    H.imag[:, i, j] = im  # last, so that the diagonal keeps +0
    return H


def hamilton_int8(p, k: np.ndarray, W: np.ndarray | None = None) -> np.ndarray:
    """H(k) ``[n_k, N, N]`` (convention 2) of the packed model ``p`` with the bits of the INT8 build.  ``W`` overrides
    the weights (default: :func:`packed_weights` of ``p``)."""
    k = np.asarray(k, dtype=np.float64).reshape(-1, p.dim)
    Wp = packed_weights(p) if W is None else W
    return unpack_hermitian(digit_gemm(phase_rows(k, p.R), Wp), p.size)
