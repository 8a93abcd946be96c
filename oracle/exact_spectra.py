"""TEST INFRASTRUCTURE ONLY -- models whose spectra and Hamiltonians are known beyond float64 accuracy.

A float64 reference (LAPACK ``eigvalsh``, the numpy Fourier sum of ``tb_oracle.hamilton``) is itself off by several
ulps, and by ~1000 ulps for H(k) at |k| ~ 1e3, so it cannot judge a kernel at rounding level.  The constructions here
give references that are accurate to ``np.longdouble`` (64-bit mantissa on x86) rounding, cheap at N = 808:

* **Folded supercells** (:func:`folded_spectrum`): the ``supercell(size)`` of a base model with N_b <= 2 orbitals, at
  supercell momentum K, has exactly the eigenvalues of the base model at the momenta ``(K + o) / size`` for every cell
  offset o (Bloch's theorem on the folded zone).  For N_b <= 2 these are closed forms, evaluated in longdouble.
* **Designed spectra** (:func:`designed_model`): ``H = Q diag(lam) Q^H`` built in longdouble with Q a product of
  Householder reflectors and a diagonal phase, rounded to a Hermitian float64 matrix and stored as the R = 0 hopping
  ``0.5 H`` (the packing adds the Hermitian conjugate exactly).  ``delta = ||H_f64 - H_ld||_2`` bounds, by Weyl's
  theorem, how far the eigenvalues of the stored matrix can be from ``lam``.
* **k.p expansions** (:func:`kdotp_coefficients_longdouble`, :func:`kdotp_hamilton_longdouble`): the Taylor terms of
  ``construct_kdotp`` and the k.p Hamiltonian with extended-precision phases, powers and sums.

``tests/test_exact_spectra.py`` pins these down on the CPU (against scipy and mpmath); ``tests/test_gpu_accuracy.py``
holds the kernels to them.  The product package never imports this module.
"""
from __future__ import annotations

import itertools
import math

import numpy as np

from tbmodels_b200._pack import PackedModel, pack_arrays

from . import tb_oracle
from . import workloads as wl

LD = np.longdouble
CLD = np.clongdouble
PI_LD = LD("3.14159265358979323846264338327950288")


def longdouble_is_extended() -> bool:
    """True where ``np.longdouble`` carries at least the 64-bit mantissa of x87 extended precision."""
    return np.finfo(np.longdouble).nmant >= 63


# ----------------------------------------------------------------------------------------------- base models (N_b <= 2)
def band1(dim: int = 3, n_half: int = 13, seed: int = 1, real: bool = False) -> PackedModel:
    """One orbital, real on-site energy, complex hoppings on the ``n_half`` shortest half-set lattice vectors (the first
    shells of the lattice, so ``|R_d| <= 1`` for n_half <= 13 in 3-D) with amplitudes decaying like ``0.7^|R|^2``.
    ``real=True``: real hoppings, so e(k) = e(-k) and folded spectra at Gamma and the zone boundary are degenerate."""
    rng = np.random.default_rng(seed)
    Rs = wl.shortest_half_vectors(n_half, dim)
    R = np.concatenate([np.zeros((1, dim), np.int32), Rs])
    amp = 0.7 ** (Rs * Rs).sum(axis=1)
    hop = np.empty((n_half + 1, 1, 1), dtype=complex)
    hop[0, 0, 0] = 0.5 * rng.normal()
    hop[1:, 0, 0] = amp * (rng.normal(size=n_half) + 1j * rng.normal(size=n_half))
    if real:
        hop = hop.real.astype(complex)
    return pack_arrays(R, hop, np.zeros((1, dim)))


def band2(dim: int = 2, n_half: int = 6, seed: int = 2, m: float = 0.3) -> PackedModel:
    """Haldane-like two-band model: staggered on-site energies +-m, and on every stored lattice vector a general complex
    2 x 2 hopping (complex first- and second-neighbour terms on both sublattices), so H(k) is genuinely complex.  The
    orbitals sit at distinct positions, so convention 1 differs from convention 2."""
    rng = np.random.default_rng(seed)
    Rs = wl.shortest_half_vectors(n_half, dim)
    R = np.concatenate([np.zeros((1, dim), np.int32), Rs])
    hop = np.zeros((n_half + 1, 2, 2), dtype=complex)
    t01 = 0.8 * (rng.normal() + 1j * rng.normal())
    hop[0] = 0.5 * np.array([[m, t01], [np.conj(t01), -m]])
    amp = 0.6 ** (Rs * Rs).sum(axis=1)
    hop[1:] = amp[:, None, None] * (rng.normal(size=(n_half, 2, 2)) + 1j * rng.normal(size=(n_half, 2, 2)))
    pos = np.zeros((2, dim))
    pos[1] = rng.random(dim)
    return pack_arrays(R, hop, pos)


def base_eigenvalues(base: PackedModel, k) -> np.ndarray:
    """Ascending eigenvalues ``[n_k, N_b]`` (longdouble) of a base model with N_b <= 2 at the momenta ``k`` (any float
    or longdouble array ``[n_k, dim]``), from the longdouble Fourier sum and the closed forms."""
    if base.size > 2:
        raise ValueError("closed forms exist for one or two orbitals only")
    H = tb_oracle.hamilton_longdouble(base.R, base.hop, base.pos, np.asarray(k), 2)
    if base.size == 1:
        return H[:, :, 0].real.copy()
    a, d, b = H[:, 0, 0].real, H[:, 1, 1].real, H[:, 1, 0]
    mean = (a + d) / 2
    rad = np.sqrt(((a - d) / 2) ** 2 + b.real * b.real + b.imag * b.imag)
    return np.stack([mean - rad, mean + rad], axis=1)


def cell_offsets(size) -> np.ndarray:
    """Every cell offset o of a ``size`` supercell, ``[prod(size), dim]``."""
    return np.array(list(itertools.product(*[range(int(s)) for s in size])), dtype=np.int64).reshape(-1, len(size))


def folded_spectrum(base: PackedModel, size, K) -> np.ndarray:
    """Exact ascending eigenvalues ``[n_k, N_b * prod(size)]`` (longdouble) of ``supercell(size)`` at the supercell
    momenta ``K`` ``[n_k, dim]`` (float64, as handed to the kernels): the base spectra at ``(K + o) / size``."""
    K = np.asarray(K, dtype=np.float64).reshape(-1, base.dim)
    size_l = np.asarray(size, dtype=LD)
    offs = cell_offsets(size).astype(LD)
    kb = (K.astype(LD)[:, None, :] + offs[None, :, :]) / size_l  # [n_k, vol, dim]
    ev = base_eigenvalues(base, kb.reshape(-1, base.dim))
    return np.sort(ev.reshape(K.shape[0], -1), axis=1)


# ------------------------------------------------------------------------------------------------------ designed spectra
SPECTRA = ("uniform", "clusters", "multiple", "graded", "outlier", "offset")


def spectrum(kind: str, n: int, rng) -> np.ndarray:
    """Eigenvalues of one designed family, ascending float64 (exactly representable, so ``lam`` is exact)."""
    if kind == "uniform":
        lam = rng.uniform(-1.0, 1.0, n)
    elif kind == "clusters":  # four clusters of width 1e-9 rho
        centres = np.array([-0.9, -0.3, 0.4, 1.0])
        lam = centres[np.arange(n) % 4] + rng.uniform(-0.5e-9, 0.5e-9, n)
    elif kind == "multiple":  # integers, each (about) n / 4 times
        lam = np.array([-2.0, -1.0, 1.0, 3.0])[np.arange(n) % 4]
    elif kind == "graded":  # +-10^(-12 i / n)
        lam = rng.choice([-1.0, 1.0], n) * 10.0 ** (-12.0 * np.arange(n) / n)
    elif kind == "outlier":
        lam = rng.uniform(-1.0, 1.0, n)
        lam[0] = 1e6
    elif kind == "offset":
        lam = 1e4 + rng.uniform(-1.0, 1.0, n)
    else:
        raise ValueError(f"unknown spectrum {kind!r}")
    return np.sort(lam)


def random_unitary_similarity(lam, rng, n_reflectors: int | None = None):
    """``(Q diag(lam) Q^H, Q)`` in clongdouble, Q = (random diagonal phases) x (product of random Householder reflectors).

    Each reflector ``P = I - 2 v v^H / (v^H v)`` is unitary to longdouble rounding; it is applied as two rank-1 updates,
    so the cost is O(m N^2).  Default m: N reflectors up to N = 128 (a Haar-like basis), 32 above.  Column j of Q is the
    eigenvector of ``lam[j]``."""
    n = len(lam)
    m = n_reflectors if n_reflectors is not None else (n if n <= 128 else 32)
    A = np.diag(np.asarray(lam, dtype=LD)).astype(CLD)
    Q = np.eye(n, dtype=CLD)
    for _ in range(m):
        v = (rng.normal(size=n) + 1j * rng.normal(size=n)).astype(CLD)
        tau = LD(2) / (v.real * v.real + v.imag * v.imag).sum()
        A = A - np.outer(v, tau * (v.conj() @ A))  # P A
        A = A - np.outer(A @ v, tau * v.conj())  # (P A) P^H, P Hermitian
        Q = Q - np.outer(v, tau * (v.conj() @ Q))  # P Q
    ph = rng.uniform(0.0, 2.0, n).astype(LD) * PI_LD
    d = np.cos(ph) + 1j * np.sin(ph)
    A = d[:, None] * A * d.conj()[None, :]
    return (A + A.conj().T) / 2, d[:, None] * Q


def round_hermitian(A_ld) -> np.ndarray:
    """Exactly Hermitian complex128 rounding of a Hermitian clongdouble matrix (lower triangle rounded, mirrored)."""
    low = np.tril(A_ld.astype(np.complex128), -1)
    return low + low.conj().T + np.diag(A_ld.diagonal().real.astype(np.float64)).astype(complex)


def designed_model(kind: str, n: int, seed: int = 0, dim: int = 3, n_reflectors: int | None = None,
                   return_vectors: bool = False):
    """R = 0-only model with the designed spectrum ``kind`` -> ``(packed, lam, delta)`` (``+ (Q,)`` with
    ``return_vectors``: the exact eigenvectors, rounded to complex128).

    ``lam`` (float64, ascending) is the exact spectrum of the longdouble matrix; ``delta`` bounds ``||H_f64 - H_ld||_2``
    (the spectral norm, which Weyl's theorem needs; it is <= the Frobenius norm), so every eigenvalue of the stored
    float64 matrix lies within ``delta`` of ``lam``.  H(k) of the model is the same matrix at every k."""
    rng = np.random.default_rng([seed, n, SPECTRA.index(kind)])
    lam = spectrum(kind, n, rng)
    A, Q = random_unitary_similarity(lam, rng, n_reflectors)
    H = round_hermitian(A)
    err = (H.astype(CLD) - A).astype(np.complex128)  # tiny entries: converting them to float64 costs nothing
    delta = float(np.linalg.norm(err, 2)) * (1 + 1e-6) if n > 1 else float(np.abs(err).max())
    packed = pack_arrays(np.zeros((1, dim), np.int32), (0.5 * H)[None], np.zeros((n, dim)))
    if return_vectors:
        return packed, lam, delta, Q.astype(np.complex128)
    return packed, lam, delta


# ------------------------------------------------------------------------------------- extended-precision Hamiltonians
def _phases_ld(k, vecs):
    """``exp(2 pi i k.v)`` ``[n_k, n_v]`` in clongdouble with the argument reduced exactly, and ``max |k.v|``."""
    x = np.asarray(k, dtype=LD) @ np.asarray(vecs, dtype=LD).T
    xr = x - np.rint(x)
    return np.cos(2 * PI_LD * xr) + 1j * np.sin(2 * PI_LD * xr), (float(np.abs(x).max()) if x.size else 0.0)


def phase_budget(k, vecs) -> np.ndarray:
    """``1 + 2 pi sum_d |k_d v_d|`` ``[n_k, n_v]``: the phase ``exp(2 pi i k.v)`` of a kernel that forms ``k.v`` in double
    is off by at most a few eps times this (the dot product rounds relative to ``sum_d |k_d v_d|``, not to ``|k.v|``)."""
    return 1 + 2 * np.pi * (np.abs(np.asarray(k, dtype=np.float64))[:, None, :] * np.abs(np.asarray(vecs, dtype=np.float64))[None]).sum(-1)


def hamilton_scale(packed: PackedModel, k, convention: int = 2) -> np.ndarray:
    """Per k-point and element ``sum_R (|T_R,ij| + |T_R,ji|) (1 + 2 pi sum_d |k_d R_d|)``: what one rounding of every
    term of the Fourier sum, and the unavoidable rounding of that term's k.R in double, can move H_ij by.  Convention 1
    adds ``S_ij 2 pi sum_d |k_d| (|pos_i,d| + |pos_j,d|)`` for the orbital-position phases, ``S_ij = sum_R (|T_R,ij| +
    |T_R,ji|)``.  ``[n_k, N, N]`` float64."""
    hop = np.abs(np.asarray(packed.hop))
    A = hop + hop.transpose(0, 2, 1)  # [n_R, N, N]
    k = np.asarray(k, dtype=np.float64).reshape(-1, packed.dim)
    if not packed.n_R:
        return np.zeros((len(k), packed.size, packed.size))
    scale = np.einsum("kr,rij->kij", phase_budget(k, packed.R), A)
    if convention == 1:
        p = np.abs(k) @ np.abs(np.asarray(packed.pos, dtype=np.float64)).T  # [n_k, N]
        scale = scale + A.sum(axis=0)[None] * 2 * np.pi * (p[:, :, None] + p[:, None, :])
    return scale


def kdotp_coefficients_longdouble(packed: PackedModel, k, order: int):
    """Taylor coefficients of ``construct_kdotp(k, order)`` with longdouble phases, powers and sums:
    ``C_p = (2 pi i)^|p| / p! sum_R [R^p e^{2 pi i k.R} T_R + (-R)^p e^{-2 pi i k.R} T_R^H]``.
    Returns ``(powers [n_terms, dim], coeff clongdouble [n_terms, N, N], scale float64 [n_terms, N, N])``; ``scale`` is
    the matching sum of magnitudes (the float64 rounding budget of every term)."""
    R = np.asarray(packed.R, dtype=np.int64)
    T = np.asarray(packed.hop).astype(CLD)
    k = np.asarray(k, dtype=np.float64).reshape(packed.dim)
    ph, _ = _phases_ld(k[None], R)
    ph = ph[0]
    budget = phase_budget(k[None], R)[0]  # [n_R]
    powers = [p for p in itertools.product(range(order + 1), repeat=packed.dim) if sum(p) <= order]
    n = packed.size
    coeff = np.zeros((len(powers), n, n), dtype=CLD)
    scale = np.zeros((len(powers), n, n))
    absT = np.abs(np.asarray(packed.hop))
    for q, p in enumerate(powers):
        mono = np.prod(R.astype(LD) ** np.array(p), axis=1)  # R^p, exact for these small integers
        sign = LD(-1) ** sum(p)
        fac = (2j * PI_LD) ** sum(p) / LD(math.prod(math.factorial(x) for x in p))
        acc = np.einsum("r,rij->ij", mono * ph, T) + sign * np.einsum("r,rji->ij", mono * ph.conj(), T.conj())
        coeff[q] = fac * acc
        mag = np.abs(mono.astype(np.float64)) * budget
        scale[q] = float(abs(fac)) * np.einsum("r,rij->ij", mag, absT + absT.transpose(0, 2, 1))
    return np.array(powers, dtype=np.int32).reshape(len(powers), packed.dim), coeff, scale


def kdotp_hamilton_longdouble(powers, coeff, k):
    """``H(k) = sum_q prod_d k_d^{p_qd} C_q`` in clongdouble for float64 ``k`` ``[n_k, dim]`` and complex128 ``coeff``;
    also returns the float64 rounding budget ``sum_q |prod k^p| |C_q|`` ``[n_k, N, N]``."""
    k = np.asarray(k, dtype=LD)
    mono = np.prod(k[:, None, :] ** np.asarray(powers)[None, :, :].astype(LD), axis=2)  # [n_k, n_terms]
    H = np.einsum("kq,qij->kij", mono, np.asarray(coeff).astype(CLD))
    scale = np.einsum("kq,qij->kij", np.abs(mono.astype(np.float64)), np.abs(np.asarray(coeff)))
    return H, scale
