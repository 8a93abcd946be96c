"""TEST INFRASTRUCTURE ONLY -- references for the Berry curvature of every band (``Evaluator.berry_curvature``).

* :func:`berry_curvature`: numpy / scipy on the packed arrays, the semantics of the device path (singletons: the
  sum over states; clusters of ascending eigenvalues with gaps ``<= degen_tol * rho``: the eigenvalues of the Hermitian
  non-Abelian curvature F).  ``dH/dk`` comes from :func:`velocity_reference.dhamilton`, its closed form.
* :func:`base_curvature` / :func:`folded_curvature`: exact (longdouble) curvature of base models with N_b <= 2 orbitals
  (two bands: ``+- d.(d_a d x d_b d) / (2 |d|^3)``, lower band first, with ``H = d_0 + d.sigma`` of the convention's
  H(k); the sign is the one the plaquette phases of tests/test_berry_curvature_oracle.py pin) and of their
  folded supercells (the base values at ``(K + o) / size`` divided by ``size_a size_b``).
* :func:`curvature_budget`: ``S_a >= ||X_a||_2`` for either convention.

The product package never imports this module.
"""
from __future__ import annotations

import numpy as np
import scipy.linalg as la

from oracle import exact_spectra as xs
from oracle import tb_oracle

import velocity_reference as vr

LD = xs.LD
PI_LD = xs.PI_LD


def pairs(dim: int):
    """The direction pairs a < b in the order of the curvature's last axis."""
    return [(a, b) for a in range(dim) for b in range(a + 1, dim)]


def x_matrices(R, hop, pos, k, convention):
    """``X_a`` ``[n_k, dim, N, N]``: ``dH/dk_a`` (convention 2) or ``dH/dk_a + 2 pi i [H, T_a]`` (convention 1), both
    in the orbital basis of the convention-2 H(k)."""
    pos = np.asarray(pos, dtype=np.float64)
    k = np.asarray(k, dtype=np.float64).reshape(-1, pos.shape[1])
    X = vr.dhamilton(R, hop, k)
    if convention == 1:
        H = tb_oracle.hamilton(R, hop, pos, k)
        for a in range(pos.shape[1]):
            X[:, a] += 2j * np.pi * (pos[None, :, a] - pos[:, None, a])[None] * H
    return X


def berry_curvature(R, hop, pos, k, convention=2, degen_tol=1e-8):
    """``(w [n_k, N], curv [n_k, N, P])`` with ``la.eigh`` of the convention-2 H(k) and ``eigvalsh`` of the F blocks."""
    pos = np.asarray(pos, dtype=np.float64)
    k = np.asarray(k, dtype=np.float64).reshape(-1, pos.shape[1])
    H = tb_oracle.hamilton(R, hop, pos, k)
    X = x_matrices(R, hop, pos, k, convention)
    n_k, dim, n = k.shape[0], k.shape[1], H.shape[1]
    prs = pairs(dim)
    w = np.empty((n_k, n))
    curv = np.zeros((n_k, n, len(prs)))
    for i in range(n_k):
        w[i], V = la.eigh(H[i])
        M = np.einsum("ji,ajk,kl->ail", V.conj(), X[i], V)
        for s, t in vr.clusters(w[i], degen_tol):
            out = np.r_[0:s, t:n]
            d = w[i][s:t, None] - w[i][None, out]  # [m, n - m]
            den = d[:, None, :] * d[None, :, :]  # (E_n - E_l)(E_m - E_l)
            for p, (a, b) in enumerate(prs):
                if t - s == 1:
                    z = M[a][s, out] * M[b][out, s]
                    curv[i, s, p] = -2 * np.sum(z.imag / (d[0] * d[0]))
                    continue
                za = M[a][s:t, out][:, None, :] * M[b][out, s:t].T[None, :, :]
                zb = M[b][s:t, out][:, None, :] * M[a][out, s:t].T[None, :, :]
                F = 1j * np.sum((za - zb) / den, axis=2)
                curv[i, s:t, p] = la.eigvalsh((F + F.conj().T) / 2)
    return w, curv


def _h_dh_longdouble(base, k, convention):
    """``H [n_k, N, N]`` and ``dH/dk_a [n_k, dim, N, N]`` (clongdouble) of the convention's H(k)."""
    R = np.asarray(base.R, dtype=np.int64)
    T = np.asarray(base.hop).astype(xs.CLD)
    ph, _ = xs._phases_ld(k, R)  # [n_k, n_R] e^{2 pi i k.R}
    H = tb_oracle.hamilton_longdouble(base.R, base.hop, base.pos, k, 2)
    dH = np.empty((k.shape[0], base.dim) + H.shape[1:], dtype=xs.CLD)
    for a in range(base.dim):
        wgt = 2 * PI_LD * R[:, a].astype(LD)
        S = np.einsum("kr,rij->kij", 1j * wgt[None, :] * ph, T)
        dH[:, a] = S + S.conj().transpose(0, 2, 1)
    if convention == 1:
        pos = np.asarray(base.pos, dtype=LD)
        x = np.asarray(k).astype(LD) @ pos.T
        x = x - np.rint(x)
        pe = np.cos(2 * PI_LD * x) + 1j * np.sin(2 * PI_LD * x)  # [n_k, N]
        rot = pe.conj()[:, :, None] * pe[:, None, :]
        H = rot * H
        for a in range(base.dim):
            dH[:, a] = rot * dH[:, a] + 2j * PI_LD * (pos[None, :, a] - pos[:, None, a])[None] * H
    return H, dH


def base_curvature(base, k, convention) -> np.ndarray:
    """Exact curvature ``[n_k, N_b, P]`` (longdouble) of a base model with N_b <= 2, lower band first: zero for one
    orbital, ``+- d.(d_a d x d_b d) / (2 |d|^3)`` for two (``H = d_0 + d.sigma``, d = (Re H_10, Im H_10, (H_00 - H_11) / 2)
    of the convention's H(k))."""
    if base.size > 2:
        raise ValueError("closed forms exist for one or two orbitals only")
    k = np.asarray(k).reshape(-1, base.dim)
    prs = pairs(base.dim)
    out = np.zeros((k.shape[0], base.size, len(prs)), dtype=LD)
    if base.size == 1:
        return out
    H, dH = _h_dh_longdouble(base, k, convention)

    def dvec(A):
        return np.stack([A[..., 1, 0].real, A[..., 1, 0].imag, (A[..., 0, 0].real - A[..., 1, 1].real) / 2], axis=-1)

    d = dvec(H)
    norm3 = np.sqrt((d * d).sum(axis=-1)) ** 3
    for p, (a, b) in enumerate(prs):
        trip = (d * np.cross(dvec(dH[:, a]), dvec(dH[:, b]))).sum(axis=-1)
        out[:, 0, p] = trip / (2 * norm3)
        out[:, 1, p] = -trip / (2 * norm3)
    return out


def folded_curvature(base, size, K, convention, degen_tol=1e-8):
    """Exact ``(w [n_k, N], curv [n_k, N, P])`` (longdouble) of ``supercell(size)`` at the supercell momenta ``K``: the base
    curvature at ``(K + o) / size`` divided by ``size_a size_b``, ordered like the folded spectrum and sorted per pair
    inside every cluster of that spectrum (``degen_tol``)."""
    K = np.asarray(K, dtype=np.float64).reshape(-1, base.dim)
    size_l = np.asarray(size, dtype=LD)
    offs = xs.cell_offsets(size).astype(LD)
    kb = ((K.astype(LD)[:, None, :] + offs[None, :, :]) / size_l).reshape(-1, base.dim)
    ev = xs.base_eigenvalues(base, kb).reshape(K.shape[0], -1)
    div = np.array([size_l[a] * size_l[b] for a, b in pairs(base.dim)], dtype=LD)
    cb = (base_curvature(base, kb, convention) / div).reshape(K.shape[0], -1, len(div))
    order = np.argsort(ev, axis=1, kind="stable")
    w = np.take_along_axis(ev, order, axis=1)
    c = np.take_along_axis(cb, order[:, :, None], axis=1)
    for i in range(K.shape[0]):
        for s, t in vr.clusters(w[i].astype(np.float64), degen_tol):
            c[i, s:t] = np.sort(c[i, s:t], axis=0)
    return w, c


def curvature_budget(packed, convention) -> np.ndarray:
    """``S_a`` ``[dim]`` >= ``||X_a||_2``: :func:`velocity_budget` for convention 2; for convention 1
    ``2 pi max_i sum_j sum_R (|R_a + pos_j,a - pos_i,a| |T_R,ij| + |R_a + pos_i,a - pos_j,a| |T_R,ji|)``."""
    if convention == 2:
        return vr.velocity_budget(packed)
    if not packed.n_R:
        return np.zeros(packed.dim)
    A = np.abs(np.asarray(packed.hop))  # [n_R, N, N]
    R = np.asarray(packed.R, dtype=np.float64)
    pos = np.asarray(packed.pos, dtype=np.float64)
    out = np.empty(packed.dim)
    for a in range(packed.dim):
        dp = pos[None, :, a] - pos[:, None, a]  # [i, j] = pos_j - pos_i
        w1 = np.abs(R[:, a, None, None] + dp[None])  # |R_a + pos_j - pos_i|
        w2 = np.abs(R[:, a, None, None] - dp[None])  # |R_a + pos_i - pos_j|
        rows = (w1 * A + w2 * A.transpose(0, 2, 1)).sum(axis=(0, 2))
        out[a] = 2 * np.pi * rows.max()
    return out
