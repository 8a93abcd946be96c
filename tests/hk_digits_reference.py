"""Python restatement of the INT8 digit GEMM of the H(k) build (tbmodels_b200/csrc/hk_gemm_i8.cu).

``Hp[k, j] = sum_r Q[k, r] W[r, j]`` with |Q| <= 1 (the [cos | sin] phase rows) and W the Hermitian-split weights:

- ``q = sum_{a=0..7} q_a 2^(-6-7a)``, ``q_a`` in [-64, 64], rounded at 2^-55;
- ``W_rj / s_j = sum_{b=0..8} w_b 2^(-6-7b)``, rounded at 2^-62, ``s_j`` the power of two with
  ``2^-1 s_j <= max_r |W_rj| < s_j`` (0 for an all-zero column, whose digits are all 0);
- class ``c = a + b`` has weight ``2^(-12-7c)``; the classes ``c <= 9`` are summed exactly (int32 on the GPU, int64
  here), combined in double from c = 9 down to 0 by ``t = t 2^-7 + acc_c`` (one rounding per step), and scaled by
  ``s_j 2^-12`` (exact).

Every operation is an exact integer or a correctly rounded double operation, so this restatement gives the kernel's
bits for the same Q and W.  ``error_bound`` is the a-priori bound of the scheme per element.
"""
from __future__ import annotations

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
    """Exact ``acc[c, k, j] = sum_{a + b = c} sum_r q_a[k, r] w_b[r, j]`` for c = 0 .. 9 (int64)."""
    acc = np.zeros((CLASSES, qd.shape[1], wd.shape[2]), dtype=np.int64)
    for a in range(Q_DIGITS):
        for b in range(W_DIGITS):
            if a + b < CLASSES:
                acc[a + b] += qd[a] @ wd[b]
    return acc


def combine(acc: np.ndarray, s: np.ndarray) -> np.ndarray:
    """The epilogue: Horner steps from class 9 down to 0 in double, then the exact scaling by ``s_j 2^-12``."""
    t = acc[CLASSES - 1].astype(np.float64)
    for c in range(CLASSES - 2, -1, -1):
        t = t * 2.0**-7 + acc[c].astype(np.float64)  # t 2^-7 is exact: one rounding per step, as fma on the GPU
    return t * np.ldexp(s, -12)[None, :]


def digit_gemm(Q: np.ndarray, W: np.ndarray) -> np.ndarray:
    """``Q [n_k, K] @ W [K, NN]`` as the INT8 kernel computes it."""
    wd, s = w_digits(W)
    return combine(class_sums(q_digits(Q), wd), s)


def error_bound(Q: np.ndarray, W: np.ndarray) -> np.ndarray:
    """Per-element bound ``[n_k, NN]`` on ``|digit_gemm(Q, W) - Q @ W|`` (exact product):

    - dropped classes c >= 10: per row at most sum_c n_c 2^(-7c) <= 11 2^-70 of s_j (n_c pairs of 64 x 64 digits);
    - W rounding: 2^-63 s_j per row (|q| <= 1);
    - Q rounding: 2^-56 |W_rj| per row;
    - the ten Horner roundings: 10 u sum_c |acc_c| 2^(-12-7c) s_j.
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
