"""The orbit-sum references (tests/symmetric_reference.py) pinned on the CPU: exact velocities and curvatures against the
numpy oracles in both conventions at symmetric and generic momenta, the cluster sizes of the designed points, the sum
rule, exact shifts and the folded composition against the oracle on the explicit supercell."""
import numpy as np
import pytest

from oracle import exact_spectra as xs
from oracle import workloads as wl
from oracle.accuracy import EPS

import curvature_reference as cr
import symmetric_reference as sr
import velocity_reference as vr

pytestmark = pytest.mark.skipif(not xs.longdouble_is_extended(), reason="the exact references need an 80-bit np.longdouble")

C_REF = 4.0  # numpy oracle vs exact: units of sqrt(N) eps S (1 + rho / g) (velocities), times S / g^2 more (curvature)
KAPPA = 0.137
GENERIC2 = [0.31, -0.42]
GENERIC3 = [0.31, -0.42, 0.11]


def _b2():
    return xs.band2(2, 6, seed=2)


def _b3(seed=4):
    return xs.band2(3, 13, seed=seed)


# name -> (orbit, [(k, cluster sizes at degen_tol 1e-8)])
DESIGNED = {
    "2d-flips": (lambda: sr.orbit_sum([_b2()], sr.signed_permutations(2, perms=False), 1),
                 [([0, 0], {4}), ([0.5, 0.5], {4}), ([0, 0.5], {4}), (GENERIC2, {1})]),
    "2d-signed-perms": (lambda: sr.orbit_sum([_b2()], sr.signed_permutations(2), 2),
                        [([KAPPA, KAPPA], {2}), ([0.5, 0.5], {8}), (GENERIC2, {1})]),
    "3d-perms": (lambda: sr.orbit_sum([_b3()], sr.signed_permutations(3, signs=False), 3),
                 [([KAPPA] * 3, {6}), (GENERIC3, {1})]),
    "3d-signed-perms": (lambda: sr.orbit_sum([_b3()], sr.signed_permutations(3), 4),
                        [([0.5] * 3, {48}), ([0, 0.5, 0], {16}), ([KAPPA] * 3, {6}), (GENERIC3, {1})]),
}


def _ratios(p, w, v, c, ow, ov, oc, convention, traces=False):
    """Worst ``|oracle - exact|`` in units of ``sqrt(N) eps S_d (1 + rho / g)`` and ``sqrt(N) eps S_a S_b (1 + rho / g) /
    g^2``; ``traces``: curvature clusters compared by their sums."""
    w64 = np.asarray(w, dtype=np.float64)
    rho = float(np.abs(w64).max())
    g = np.array([vr.cluster_gaps(row, 1e-8) for row in w64])[:, :, None]
    unit = np.sqrt(p.size) * EPS
    rv = float((np.abs(ov - v).astype(np.float64) / (unit * vr.velocity_budget(p) * (1 + rho / g))).max())
    S = cr.curvature_budget(p, convention)
    sab = np.array([S[a] * S[b] for a, b in cr.pairs(p.dim)])
    err = np.abs(oc - c).astype(np.float64)
    if traces:
        for i, row in enumerate(w64):
            for s, t in vr.clusters(row, 1e-8):
                err[i, s:t] = np.abs(oc[i, s:t].sum(axis=0) - c[i, s:t].sum(axis=0)).astype(np.float64)
    rc = float((err / (unit * sab * (1 + rho / g) / (g * g))).max())
    assert float(np.abs(ow - w).max()) <= 64 * unit * rho
    return rv, rc


@pytest.mark.parametrize("convention", (1, 2))
@pytest.mark.parametrize("name", list(DESIGNED))
def test_orbit_exact_against_oracles(name, convention):
    """Every band, clusters member by member (the exact blocks are diagonal in the copy basis), and the designed sizes."""
    build, pts = DESIGNED[name]
    orbit = build()
    p = orbit.packed
    k = np.array([q for q, _ in pts], dtype=np.float64)
    w, v, c = sr.orbit_exact(orbit, k, convention)
    for row, (q, sizes) in zip(w, pts):
        assert sr.cluster_sizes(row) == sizes, f"{name} at {q}: cluster sizes {sr.cluster_sizes(row)} != {sizes}"
    ow, ov = vr.band_velocity(p.R, p.hop, p.pos, k)
    _, oc = cr.berry_curvature(p.R, p.hop, p.pos, k, convention)
    rv, rc = _ratios(p, w, v, c, ow, ov, oc, convention)
    print(f"[orbit] {name} N={p.size} conv {convention}: vel {rv:.3g}, curv {rc:.3g} x sqrt(N) eps units")
    assert rv <= C_REF and rc <= C_REF
    assert float(np.abs(c.sum(axis=1)).max()) <= 1e-15 * float(np.abs(c).max()), "sum over bands not zero"
    assert float(np.abs(c).max()) > 1 and float(np.abs(v).max()) > 1


def test_several_bases():
    """Two bases: their orbits' clusters stay apart, and the union is still exact."""
    orbit = sr.orbit_sum([_b3(4), _b3(5)], sr.signed_permutations(3, signs=False), 6)
    p = orbit.packed
    k = np.array([[KAPPA] * 3, GENERIC3])
    w, v, c = sr.orbit_exact(orbit, k, 1)
    assert sr.cluster_sizes(w[0]) == {6} and sr.cluster_sizes(w[1]) == {1}
    ow, ov = vr.band_velocity(p.R, p.hop, p.pos, k)
    _, oc = cr.berry_curvature(p.R, p.hop, p.pos, k, 1)
    rv, rc = _ratios(p, w, v, c, ow, ov, oc, 1)
    print(f"[orbit] two bases N={p.size}: vel {rv:.3g}, curv {rc:.3g}")
    assert rv <= C_REF and rc <= C_REF


def test_interleaving_only_relabels():
    """The interleaving permutes orbitals and nothing else: H(k) of the contiguous and the interleaved sum agree exactly
    after the permutation, and R / -R are merged onto the half set."""
    from oracle import tb_oracle as orc

    G = sr.signed_permutations(3)
    a = sr.orbit_sum([_b3()], G, None).packed
    b = sr.orbit_sum([_b3()], G, 4)
    assert a.n_R == b.packed.n_R == _b3().n_R  # the shells of the base are closed under G
    for R in np.asarray(b.packed.R):
        nz = R[R != 0]
        assert not nz.size or nz[0] > 0
    k = np.array([GENERIC3])
    Ha = orc.hamilton(a.R, a.hop, a.pos, k)[0]
    Hb = orc.hamilton(b.packed.R, b.packed.hop, b.packed.pos, k)[0]
    assert np.array_equal(Hb[np.ix_(b.perm, b.perm)], Ha)


def test_shifts():
    """Dyadic on-site shifts: levels of a cluster exactly delta apart in the exact spectrum, the oracle agrees, and the
    cut falls where ``degen_tol rho`` says."""
    G = sr.signed_permutations(3, signs=False)
    base = _b3()
    k = np.array([[KAPPA] * 3])
    rho0 = float(np.abs(sr.orbit_exact(sr.orbit_sum([base], G, 3), k)[0]).max())
    delta = 2.0 ** (np.floor(np.log2(rho0)) - 10)
    for offset in (0.0, -64.0):
        orbit = sr.orbit_sum([base], G, 3, shifts=offset + delta * np.arange(len(G)))
        p = orbit.packed
        w, _, _ = sr.orbit_exact(orbit, k, degen_tol=0.0)
        rho = float(np.abs(w).max())
        if offset:
            assert float(-w[0, 0]) == rho, "rho must come from a negative eigenvalue"
        d = np.diff(w[0].astype(np.float64))
        assert np.sum(np.abs(d - delta) <= 1e-12 * rho) == 2 * (len(G) - 1)
        assert sr.cluster_sizes(w[0], delta / (2 * rho)) == {1}
        assert sr.cluster_sizes(w[0], 2 * delta / rho) == {len(G)}
        for tol in (delta / (2 * rho), 2 * delta / rho):
            w, v, c = sr.orbit_exact(orbit, k, 1, degen_tol=tol)
            ow, ov = vr.band_velocity(p.R, p.hop, p.pos, k, degen_tol=tol)
            _, oc = cr.berry_curvature(p.R, p.hop, p.pos, k, 1, degen_tol=tol)
            assert np.abs(ov - v).max() <= 1e-10 * vr.velocity_budget(p).max() * rho / delta
            assert np.abs(oc - c).max() <= 1e-10 * cr.curvature_budget(p, 1).max() ** 2 * rho / delta**3


@pytest.mark.parametrize("convention", (1, 2))
def test_folded_composition(convention):
    """``orbit_exact(size=...)`` against the oracle on ``workloads.supercell`` of the orbit sum: every member of velocities
    and convention-1 curvature, cluster traces of convention-2 curvature; K on the diagonal clusters folds and orbits."""
    orbit = sr.orbit_sum([_b3()], sr.signed_permutations(3, signs=False), 3)
    size = (2, 2, 2)
    sup = wl.supercell(orbit.packed, size)
    K = np.array([[KAPPA] * 3, GENERIC3])
    w, v, c = sr.orbit_exact(orbit, K, convention, size=size)
    assert sr.cluster_sizes(w[0]) == {6} and sr.cluster_sizes(w[1]) == {1}
    ow, ov = vr.band_velocity(sup.R, sup.hop, sup.pos, K)
    _, oc = cr.berry_curvature(sup.R, sup.hop, sup.pos, K, convention)
    rv, rc = _ratios(sup, w, v, c, ow, ov, oc, convention, traces=convention == 2)
    print(f"[orbit] folded {size} N={sup.size} conv {convention}: vel {rv:.3g}, curv {rc:.3g}")
    assert rv <= C_REF and rc <= C_REF
    # the composition itself: the unfolded values at the base momenta (K + o) / size, divided by size_a size_b
    kb = (K[:1, None, :].astype(sr.LD) + xs.cell_offsets(size)[None].astype(sr.LD)) / sr.LD(2)
    ew, _, ec = sr.orbit_values(orbit, kb.reshape(-1, 3), convention)
    assert np.array_equal(np.sort(ew.ravel()), w[0])
    assert np.array_equal(np.sort(ec.reshape(-1, 3) / 4, axis=0), np.sort(c[0], axis=0))
