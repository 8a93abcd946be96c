"""TEST INFRASTRUCTURE ONLY -- references for the band velocities dE_n/dk_d (``Evaluator.band_velocity``).

* :func:`band_velocity`: numpy / scipy on the packed arrays, the same semantics as the device path (clusters of
  ascending eigenvalues with gaps ``<= degen_tol * rho`` get the eigenvalues of their projected blocks).  ``dH/dk_d`` is
  built from its closed form ``2 pi i sum_R R_d (e^{2 pi i k.R} T_R - e^{-2 pi i k.R} T_R^H)``, not from
  ``construct_kdotp``, so the two cross-check.
* :func:`base_velocities` / :func:`folded_velocities`: exact (longdouble) velocities of folded supercells of base models
  with N_b <= 2 orbitals.  ``d_K H`` of a folded supercell is block-diagonal in the base momentum, so every projected
  block of a cluster is diagonal and its eigenvalues are the base velocities, whatever the cluster threshold merges:
  the reference is exact for every cluster.
* :func:`velocity_budget`: ``S_d = 2 pi max_i sum_j sum_R |R_d| (|T_R,ij| + |T_R,ji|)``, a bound on ``||dH/dk_d||_2``.

The product package never imports this module.
"""
from __future__ import annotations

import numpy as np
import scipy.linalg as la

from oracle import exact_spectra as xs
from oracle import tb_oracle

LD = xs.LD
PI_LD = xs.PI_LD


def dhamilton(R, hop, k) -> np.ndarray:
    """``dH/dk_d`` of the convention-2 H(k), ``[n_k, dim, N, N]`` complex128."""
    R = np.asarray(R)
    hop = np.asarray(hop)
    k = np.asarray(k, dtype=np.float64).reshape(-1, R.shape[1] if R.ndim == 2 and R.size else 1)
    n = hop.shape[1]
    out = np.zeros((k.shape[0], k.shape[1], n, n), dtype=complex)
    for r_vec, mat in zip(R, hop):
        ph = np.exp(2j * np.pi * (k @ r_vec))  # [n_k]
        term = ph[:, None, None] * mat[None]
        term = term - term.conj().transpose(0, 2, 1)
        out += 2j * np.pi * r_vec[None, :, None, None] * term[:, None]
    return out


def clusters(w, degen_tol):
    """``[(start, stop)]`` of the maximal runs of ascending ``w`` whose consecutive gaps are ``<= degen_tol * rho``."""
    w = np.asarray(w)
    thr = degen_tol * float(np.abs(w).max()) if w.size else 0.0
    cuts = np.flatnonzero(~(np.diff(w) <= thr)) + 1
    bounds = np.concatenate([[0], cuts, [len(w)]])
    return list(zip(bounds[:-1].tolist(), bounds[1:].tolist()))


def cluster_gaps(w, degen_tol):
    """``[N]``: for every index, the gap from its cluster to the nearest other cluster (inf if there is none)."""
    g = np.full(len(w), np.inf)
    for a, b in clusters(w, degen_tol):
        left = w[a] - w[a - 1] if a > 0 else np.inf
        right = w[b] - w[b - 1] if b < len(w) else np.inf
        g[a:b] = min(left, right)
    return g


def band_velocity(R, hop, pos, k, degen_tol=1e-8):
    """``(w [n_k, N], v [n_k, N, dim])`` with ``la.eigh`` and ``eigvalsh`` of the projected blocks of every cluster."""
    k = np.asarray(k, dtype=np.float64).reshape(-1, np.asarray(pos).shape[1])
    H = tb_oracle.hamilton(R, hop, pos, k)
    dH = dhamilton(R, hop, k)
    n_k, dim, n = k.shape[0], k.shape[1], H.shape[1]
    w = np.empty((n_k, n))
    v = np.empty((n_k, n, dim))
    for i in range(n_k):
        w[i], V = la.eigh(H[i])
        for a, b in clusters(w[i], degen_tol):
            Vc = V[:, a:b]
            for d in range(dim):
                blk = Vc.conj().T @ dH[i, d] @ Vc
                v[i, a:b, d] = la.eigvalsh((blk + blk.conj().T) / 2)
    return w, v


def velocity_budget(packed) -> np.ndarray:
    """``S_d`` ``[dim]``: ``2 pi max_i sum_j sum_R |R_d| (|T_R,ij| + |T_R,ji|)`` >= ``||dH/dk_d||_2``."""
    if not packed.n_R:
        return np.zeros(packed.dim)
    A = np.abs(np.asarray(packed.hop))
    A = A + A.transpose(0, 2, 1)  # [n_R, N, N]
    rows = A.sum(axis=2)  # [n_R, N]
    return np.array([2 * np.pi * (np.abs(packed.R[:, d])[:, None] * rows).sum(axis=0).max() for d in range(packed.dim)])


def base_velocities(base, k) -> np.ndarray:
    """Exact ``dE/dk`` ``[n_k, N_b, dim]`` (longdouble) of a base model with N_b <= 2, in the order of
    :func:`oracle.exact_spectra.base_eigenvalues` (lower band first): for N_b = 1 ``dH_00``, for N_b = 2
    ``d mean -+ d rad`` with ``d rad = [((a - d)/2)(da - dd)/2 + Re(conj(b) db)] / rad``."""
    if base.size > 2:
        raise ValueError("closed forms exist for one or two orbitals only")
    k = np.asarray(k).reshape(-1, base.dim)
    R = np.asarray(base.R, dtype=np.int64)
    T = np.asarray(base.hop).astype(xs.CLD)
    ph, _ = xs._phases_ld(k, R)  # [n_k, n_R] e^{2 pi i k.R}
    H = tb_oracle.hamilton_longdouble(base.R, base.hop, base.pos, k, 2)
    out = np.empty((k.shape[0], base.size, base.dim), dtype=LD)
    for d in range(base.dim):
        wgt = 2 * PI_LD * R[:, d].astype(LD)  # dH = sum_R 2 pi i R_d (e T - conj(e) T^H)
        S = np.einsum("kr,rij->kij", 1j * wgt[None, :] * ph, T)
        dH = S + S.conj().transpose(0, 2, 1)
        if base.size == 1:
            out[:, 0, d] = dH[:, 0, 0].real
            continue
        a, dd, b = H[:, 0, 0].real, H[:, 1, 1].real, H[:, 1, 0]
        da, ddd, db = dH[:, 0, 0].real, dH[:, 1, 1].real, dH[:, 1, 0]
        rad = np.sqrt(((a - dd) / 2) ** 2 + b.real * b.real + b.imag * b.imag)
        drad = (((a - dd) / 2) * (da - ddd) / 2 + (b.real * db.real + b.imag * db.imag)) / rad
        out[:, 0, d] = (da + ddd) / 2 - drad
        out[:, 1, d] = (da + ddd) / 2 + drad
    return out


def folded_velocities(base, size, K, degen_tol=1e-8):
    """Exact ``(w [n_k, N], v [n_k, N, dim])`` (longdouble) of ``supercell(size)`` at the supercell momenta ``K``: the base
    velocities at ``(K + o) / size`` divided by ``size_d``, ordered like the folded spectrum and sorted per direction
    inside every cluster of that spectrum (``degen_tol``)."""
    K = np.asarray(K, dtype=np.float64).reshape(-1, base.dim)
    size_l = np.asarray(size, dtype=LD)
    offs = xs.cell_offsets(size).astype(LD)
    kb = ((K.astype(LD)[:, None, :] + offs[None, :, :]) / size_l).reshape(-1, base.dim)
    ev = xs.base_eigenvalues(base, kb).reshape(K.shape[0], -1)
    vb = (base_velocities(base, kb) / size_l).reshape(K.shape[0], -1, base.dim)
    order = np.argsort(ev, axis=1, kind="stable")
    w = np.take_along_axis(ev, order, axis=1)
    v = np.take_along_axis(vb, order[:, :, None], axis=1)
    for i in range(K.shape[0]):
        for a, b in clusters(w[i].astype(np.float64), degen_tol):
            v[i, a:b] = np.sort(v[i, a:b], axis=0)
    return w, v
