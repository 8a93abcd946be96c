"""TEST INFRASTRUCTURE ONLY -- exact references with large, non-trivial degenerate clusters ("orbit sums").

Take base models b with N_b <= 2 orbitals (``oracle.exact_spectra.band2``) and a group G of signed permutation matrices
P.  For every P add a copy of b whose hopping ``T_R`` sits at the lattice vector ``P R`` and whose orbitals sit at
``P pos``: copy g has ``H_g(k) = h(P^T k)`` in both conventions, with no arithmetic on the hoppings.  Hence, from the
longdouble closed forms of the base model (:func:`oracle.exact_spectra.base_eigenvalues`,
:func:`velocity_reference.base_velocities`, :func:`curvature_reference.base_curvature`), for every band of the sum

* ``E = E_b(P^T k)``, ``v = P v_b(P^T k)``, ``Omega^{ab} = sum_{cd} P_ac P_bd Omega_b^{cd}(P^T k)`` (either convention).

At a k fixed by a subgroup of G the copies are exactly degenerate, with different (permuted) velocities and curvatures.
Copies do not couple, so the exact projected velocity block and the exact non-Abelian curvature F of a cluster are
diagonal in the copy basis: the cluster's answer is the sorted list of its members' values.  The orbitals of the copies
are interleaved by a seeded permutation, so that a solver's eigenvectors inside a cluster mix the copies and the
cluster's blocks are far from diagonal (the GPU tests assert that they are).

Optional exact on-site shifts delta_g per copy (added to the copy's own R = 0 hopping, so the references use the very
same stored numbers) split a cluster into levels a chosen distance apart, which tests where ``degen_tol`` cuts.

Folded supercells of an orbit sum (``supercell(size)`` at supercell momentum K) are the orbit sum at the base momenta
``(K + o) / size``: :func:`orbit_exact` accepts ``size``.  There X_a of convention 1 and dH/dk are block-diagonal in the
base momentum, so velocities and convention-1 curvatures are exact member by member; convention-2 X is not (see
tests/test_gpu_berry_curvature.py), so only the traces of its clusters are exact.

The product package never imports this module.
"""
from __future__ import annotations

import itertools
from dataclasses import dataclass

import numpy as np

from oracle import exact_spectra as xs
from tbmodels_b200 import pack_arrays
from tbmodels_b200._pack import PackedModel

import curvature_reference as cr
import velocity_reference as vr

LD = xs.LD


def signed_permutations(dim: int, perms: bool = True, signs: bool = True) -> np.ndarray:
    """``[|G|, dim, dim]`` int64: all permutation matrices (``perms``), times all sign flips (``signs``); both False
    gives the trivial group.  The identity comes first."""
    ps = list(itertools.permutations(range(dim))) if perms else [tuple(range(dim))]
    ss = list(itertools.product((1, -1), repeat=dim)) if signs else [(1,) * dim]
    out = []
    for p in ps:
        for s in ss:
            P = np.zeros((dim, dim), dtype=np.int64)
            P[np.arange(dim), p] = s
            out.append(P)
    return np.stack(out)


@dataclass
class Orbit:
    """An orbit sum: ``packed`` the model, ``copies`` its (base model with its shift applied, P) pairs in block order,
    ``perm`` the orbital interleaving (block orbital i is model orbital ``perm[i]``)."""

    packed: PackedModel
    copies: list
    perm: np.ndarray


def shifted(base: PackedModel, delta: float) -> PackedModel:
    """``base`` with ``delta`` added to every on-site energy: ``delta / 2`` on the diagonal of its R = 0 hopping (H(k)
    adds ``T_0 + T_0^H``); exact in H for dyadic ``delta``, and the references use the stored result either way."""
    if not delta:
        return base
    r0 = np.flatnonzero(~np.asarray(base.R).any(axis=1))
    if len(r0) != 1:
        raise ValueError("the base model needs exactly one R = 0 hopping")
    hop = np.array(base.hop, copy=True)
    hop[r0[0]] += (delta / 2) * np.eye(base.size)
    return pack_arrays(base.R, hop, base.pos)


def orbit_sum(bases, G, perm_seed: int = 0, shifts=None) -> Orbit:
    """The direct sum of the G-orbits of ``bases`` (copy ``i |G| + g`` is base i moved by ``G[g]``), with ``shifts``
    (``[len(bases) |G|]`` on-site shifts, or None) and the orbitals interleaved by a permutation of seed ``perm_seed``
    (None: blocks left contiguous).  Lattice vectors R and -R are merged onto the half set as ``workloads.supercell``
    merges them: ``T`` at ``P R`` becomes ``T^H`` at ``-P R`` when the first non-zero component of ``P R`` is negative."""
    G = np.asarray(G, dtype=np.int64)
    dim = G.shape[1]
    copies = []
    for i, b in enumerate(bases):
        for g, P in enumerate(G):
            copies.append((shifted(b, 0.0 if shifts is None else float(shifts[i * len(G) + g])), P))
    n = sum(b.size for b, _ in copies)
    raw: dict = {}
    pos = np.empty((n, dim))
    off = 0
    for b, P in copies:
        sl = slice(off, off + b.size)
        pos[sl] = np.asarray(b.pos) @ P.T
        for R, T in zip(np.asarray(b.R, dtype=np.int64), np.asarray(b.hop)):
            Rp = P @ R
            nz = Rp[Rp != 0]
            if nz.size and nz[0] < 0:
                Rp, T = -Rp, T.conj().T
            key = tuple(int(x) for x in Rp)
            if key not in raw:
                raw[key] = np.zeros((n, n), dtype=complex)
            raw[key][sl, sl] += T  # blocks of different copies are disjoint: exact
        off += b.size
    perm = np.arange(n) if perm_seed is None else np.random.default_rng(perm_seed).permutation(n)
    inv = np.argsort(perm)
    keys = sorted(raw, key=lambda r: (any(r), r))  # R = 0 first
    hop = np.stack([raw[key][np.ix_(inv, inv)] for key in keys])
    return Orbit(pack_arrays(np.array(keys, dtype=np.int32), hop, pos[inv]), copies, perm)


def _full_curvature(c, dim):
    """``[..., P]`` pair values -> ``[..., dim, dim]`` antisymmetric tensors."""
    W = np.zeros(c.shape[:-1] + (dim, dim), dtype=c.dtype)
    for p, (a, b) in enumerate(cr.pairs(dim)):
        W[..., a, b] = c[..., p]
        W[..., b, a] = -c[..., p]
    return W


def orbit_values(orbit: Orbit, kb, convention: int = 2):
    """Unsorted exact ``(E [n_k, N], v [n_k, N, dim], Omega [n_k, N, P])`` (longdouble) at the base momenta ``kb``
    ``[n_k, dim]`` (float64 or longdouble), bands in copy order (two per copy: lower, upper)."""
    kb = np.asarray(kb).reshape(-1, orbit.packed.dim)
    dim = kb.shape[1]
    E, V, C = [], [], []
    for b, P in orbit.copies:
        q = kb.astype(LD) @ P.astype(LD)  # P^T k, exact
        PL = P.astype(LD)
        E.append(xs.base_eigenvalues(b, q))
        V.append(vr.base_velocities(b, q) @ PL.T)  # v_a = sum_c P_ac v_b,c
        W = _full_curvature(cr.base_curvature(b, q, convention), dim)
        W = np.einsum("ac,knce,be->knab", PL, W, PL)  # Omega^{ab} = sum P_ac P_be Omega_b^{ce}
        C.append(np.stack([W[..., a, b] for a, b in cr.pairs(dim)], axis=-1))
    return np.concatenate(E, axis=1), np.concatenate(V, axis=1), np.concatenate(C, axis=1)


def orbit_exact(orbit: Orbit, k, convention: int = 2, degen_tol: float = 1e-8, size=None):
    """Exact ``(w [n_k, N], v [n_k, N, dim], Omega [n_k, N, P])`` (longdouble) in the model's band order (ascending
    energies), with the members of every cluster of that spectrum (``degen_tol``) sorted per component, the semantics of
    ``band_velocity`` / ``berry_curvature``.  ``size``: ``k`` are momenta K of ``supercell(size)``, whose bands are those
    of the base momenta ``(K + o) / size``, with ``v_a / size_a`` and ``Omega^{ab} / (size_a size_b)``."""
    dim = orbit.packed.dim
    k = np.asarray(k, dtype=np.float64).reshape(-1, dim)
    if size is None:
        E, v, c = orbit_values(orbit, k, convention)
    else:
        size_l = np.asarray(size, dtype=LD)
        offs = xs.cell_offsets(size).astype(LD)
        kb = ((k.astype(LD)[:, None, :] + offs[None, :, :]) / size_l).reshape(-1, dim)
        E, v, c = orbit_values(orbit, kb, convention)
        div = np.array([size_l[a] * size_l[b] for a, b in cr.pairs(dim)], dtype=LD)
        E = E.reshape(k.shape[0], -1)
        v = (v / size_l).reshape(k.shape[0], -1, dim)
        c = (c / div).reshape(k.shape[0], -1, len(div))
    order = np.argsort(E, axis=1, kind="stable")
    w = np.take_along_axis(E, order, axis=1)
    v = np.take_along_axis(v, order[:, :, None], axis=1)
    c = np.take_along_axis(c, order[:, :, None], axis=1)
    for i in range(k.shape[0]):
        for s, t in vr.clusters(w[i].astype(np.float64), degen_tol):
            v[i, s:t] = np.sort(v[i, s:t], axis=0)
            c[i, s:t] = np.sort(c[i, s:t], axis=0)
    return w, v, c


def cluster_sizes(w, degen_tol: float = 1e-8) -> set:
    """The set of cluster sizes of an ascending spectrum."""
    return {t - s for s, t in vr.clusters(np.asarray(w, dtype=np.float64), degen_tol)}
