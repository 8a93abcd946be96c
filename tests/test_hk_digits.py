"""The INT8 digit scheme of the H(k) build (tests/hk_digits_reference.py) on the CPU: the digit split is exact to its
rounding, the class-sum result stays within the scheme's bound on random and adversarial columns, and the H(k) it
builds (``hamilton_int8``: the kernel's phases, weights and epilogue) is within the longdouble budget of
``test_gpu_accuracy.py``."""
from fractions import Fraction

import numpy as np
import pytest

import hk_digits_reference as hd
from oracle import exact_spectra as xs
from oracle import workloads as wl
from oracle.accuracy import C_H, check_h


def _edge_values():
    rng = np.random.default_rng(1)
    special = [0.0, 1.0, -1.0, 0.5, -0.5, 2.0**-55, -(2.0**-56), 2.0**-56 * 3, 1 - 2.0**-53, -(1 - 2.0**-53), 2.0**-1074,
               1 / 128, 63.5 / 64, 64.5 / 128 / 64, np.nextafter(1 / 128, 0), 5e-324, 2.0**-300]
    return np.concatenate([special, rng.uniform(-1, 1, 300), rng.uniform(-1, 1, 100) * 2.0 ** rng.integers(-80, 0, 100)])


@pytest.mark.parametrize("n_digits, last", [(hd.Q_DIGITS, 55), (hd.W_DIGITS, 62)])
def test_digit_split_is_exact_to_its_rounding(n_digits, last):
    x = _edge_values()
    d = hd.split_digits(x, n_digits)
    assert d.min() >= -64 and d.max() <= 64
    for i, v in enumerate(x):
        err = abs(hd.digits_fraction(d[:, i]) - Fraction(float(v)))
        assert err <= Fraction(1, 2 ** (last + 1)), f"x = {v!r}: digits off by {float(err):.3e}"
    # values on the digit grid are represented exactly
    grid = np.array([Fraction(int(m), 2**last) for m in (1, -3, 2**40 + 7, -(2**50) - 11)], dtype=object)
    dg = hd.split_digits(grid.astype(np.float64), n_digits)
    for i, v in enumerate(grid):
        assert hd.digits_fraction(dg[:, i]) == v


def _exact_product(Q, W):
    """Q @ W with exact rational sums, rounded once to double."""
    out = np.empty((Q.shape[0], W.shape[1]))
    for k in range(Q.shape[0]):
        for j in range(W.shape[1]):
            out[k, j] = float(sum((Fraction(float(q)) * Fraction(float(w)) for q, w in zip(Q[k], W[:, j])), Fraction(0)))
    return out


def _adversarial_columns(K, rng):
    cols = [
        rng.standard_normal(K),                                   # random
        np.where(np.arange(K) == 3, 1.0, 1e-9 * rng.standard_normal(K)),  # one dominant R
        rng.standard_normal(K) * 10.0 ** rng.integers(-12, 3, K),  # mixed magnitudes
        np.zeros(K),                                              # all zero
        np.where(rng.random(K) < 0.5, 0.0, rng.standard_normal(K)),  # half zeros
        np.full(K, 2.0**-1000) * rng.standard_normal(K),         # tiny scale, far from overflow of the digits
        np.full(K, 2.0**-1022) * rng.integers(-3, 4, K),          # subnormal-adjacent scale
        np.full(K, 1.0 - 2.0**-53),                               # s_j = 1 exactly at the top of the binade
        np.full(K, 0.5),                                          # a power of two: s_j = 2 max
        rng.standard_normal(K) * 2.0**900,                        # large scale
    ]
    return np.stack(cols, axis=1)


@pytest.mark.parametrize("K", [16, 64, 512])
def test_class_sums_within_bound(K):
    rng = np.random.default_rng(K)
    W = _adversarial_columns(K, rng)
    Q = np.concatenate([np.cos(rng.uniform(0, 7, (6, K))), np.ones((1, K)), -np.ones((1, K)), np.zeros((1, K)),
                        np.where(rng.random((1, K)) < 0.5, 1.0, -1.0)])
    got = hd.digit_gemm(Q, W)
    exact = _exact_product(Q, W)
    bound = hd.error_bound(Q, W)
    err = np.abs(got - exact)
    assert np.all(err <= bound + 0.5 * np.abs(np.spacing(exact))), f"worst err / bound {float((err / np.maximum(bound, 1e-300)).max()):.3f}"
    assert np.all(got[:, 3] == 0) and not np.signbit(got[:, 3]).any(), "an all-zero column must give +0"
    # with |q| <= 1 the bound is a few eps of sum_r |W_rj| (and of s_j K 2^-63 when one R dominates)
    S = np.abs(W).sum(axis=0)
    assert np.all(bound <= 12 * 2.0**-53 * S[None, :] + K * 2.0**-62 * np.abs(W).max(axis=0)[None, :] * 2)


def _packed_weights(p):
    """Hermitian-split weights [2 n_R, N^2] in the packed layout of tbk_math.cuh (host_pack_weights restated)."""
    N = p.size
    nre = N * (N + 1) // 2
    W = np.zeros((2 * p.n_R, N * N))
    for r in range(p.n_R):
        T = p.hop[r]
        for q, M in ((2 * r, T + T.conj().T), (2 * r + 1, 1j * (T - T.conj().T))):
            for i in range(N):
                for j in range(i + 1):
                    W[q, i * (i + 1) // 2 + j] = M[i, j].real
                    if j < i:
                        W[q, nre + i * (i - 1) // 2 + j] = M[i, j].imag
    return W


def _unpack(hp, N):
    nre = N * (N + 1) // 2
    H = np.zeros((hp.shape[0], N, N), dtype=np.complex128)
    for i in range(N):
        for j in range(i + 1):
            v = hp[:, i * (i + 1) // 2 + j] + (1j * hp[:, nre + i * (i - 1) // 2 + j] if j < i else 0)
            H[:, i, j] = v
            H[:, j, i] = np.conj(v)
    return H


@pytest.mark.parametrize("model", ["n9", "n36"])
def test_host_pack_and_unpack_restated(model):
    """``hd.packed_weights`` (the library's host pack) equals its Python restatement bit for bit, and
    ``hd.unpack_hermitian`` mirrors as the restatement does, with a +0 imaginary diagonal."""
    p = wl.synthetic(9, 30, seed=11) if model == "n9" else wl.synthetic(36, 60, seed=12)
    W = hd.packed_weights(p)
    assert np.array_equal(W, _packed_weights(p))
    hp = np.random.default_rng(2).standard_normal((3, p.size * p.size))
    H = hd.unpack_hermitian(hp, p.size)
    assert np.array_equal(H, _unpack(hp, p.size))
    d = np.diagonal(H, axis1=1, axis2=2)
    assert np.all(d.imag == 0) and not np.signbit(d.imag).any()


@pytest.mark.skipif(not xs.longdouble_is_extended(), reason="the exact references need an 80-bit np.longdouble")
@pytest.mark.parametrize("kscale", [2.0, 1e3])
@pytest.mark.parametrize("model", ["n9", "n36"])
def test_digit_hamilton_against_longdouble(model, kscale):
    """``hamilton_int8`` (the kernel's phases, digits and epilogue) within the longdouble budget of the GPU tests."""
    from oracle import tb_oracle as orc

    p = wl.synthetic(9, 30, seed=11) if model == "n9" else wl.synthetic(36, 60, seed=12)
    k = np.random.default_rng(4).uniform(-kscale, kscale, (5, p.dim))
    H = hd.hamilton_int8(p, k)
    want = orc.hamilton_longdouble(p.R, p.hop, p.pos, k, 2)
    check_h(H, want, xs.hamilton_scale(p, k, 2), f"digit GEMM {model} |k|<={kscale:g}", c=C_H)
