"""Band velocities and Berry curvature inside degenerate clusters of 2 to 48 bands (band_velocity.cu, berry_curvature.cu,
jacobi_eig.cuh) against the exact orbit-sum references of tests/symmetric_reference.py, on every kernel path.

A cluster's answer is the eigenvalues of an m x m Hermitian block (the projected velocity block, or the non-Abelian
curvature F), found by cyclic complex Jacobi.  Orbit sums have exact clusters of up to 48 bands whose exact blocks are
diagonal in the copy basis, with distinct diagonal entries, and whose interleaved orbitals make a solver's blocks far from
diagonal (asserted for every case): so a Jacobi that stops early, drops the phase of a rotation, or a block with missing
entries gives wrong members.

* velocities to ``C_VEL sqrt(N) eps S_d (1 + rho / g_n)``, curvatures to ``C_CURV sqrt(N) eps S_a S_b (1 + rho / g_n) /
  g_n^2`` (the bounds of tests/test_gpu_velocity.py and tests/test_gpu_berry_curvature.py), g_n the exact gap from n's
  cluster to the next cluster at the ``degen_tol`` in use; folded cases compare convention-2 clusters by their traces;
* host and device entry points, host-packed models and ``Evaluator.from_supercell``; clusters and singletons in one call;
* where ``degen_tol`` cuts: exact on-site shifts a known distance apart are split or merged, also when rho = max |E| comes
  from a negative eigenvalue; ``degen_tol = 0`` at generic k; ``degen_tol = 4`` (one cluster of N bands);
* 2^+-600 scaled models bit-equal.

Every check prints its worst ratio (``pytest -s``).
"""
import numpy as np
import pytest

from oracle import exact_spectra as xs
from oracle import workloads as wl
from oracle.accuracy import EPS, check_eig

import curvature_reference as cr
import symmetric_reference as sr
import velocity_reference as vr

pytestmark = [
    pytest.mark.gpu,
    pytest.mark.skipif(not xs.longdouble_is_extended(), reason="the exact references need an 80-bit np.longdouble"),
]

C_VEL = 4.0  # units of sqrt(N) eps S_d (1 + rho / g_n), as tests/test_gpu_velocity.py
C_CURV = 4.0  # units of sqrt(N) eps S_a S_b (1 + rho / g_n) / g_n^2, as tests/test_gpu_berry_curvature.py
MIN_MIXING = 0.05  # max |off-diagonal| / eigenvalue spread of V_c^H dH_0 V_c, in at least one cluster of m >= 3
KAPPA = 0.137
CONVENTIONS = (1, 2)


@pytest.fixture(scope="module")
def tbk():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import tbmodels_b200

    return tbmodels_b200


def _b2():
    return xs.band2(2, 6, seed=2)


def _b3(seed=4):
    return xs.band2(3, 13, seed=seed)


def _perms3():
    return sr.orbit_sum([_b3()], sr.signed_permutations(3, signs=False), 3)


def _signed3(n_bases=1):
    return sr.orbit_sum([_b3(4 + i) for i in range(n_bases)], sr.signed_permutations(3), 4 + n_bases)


# name -> (orbit, supercell size or None, points, their cluster sizes at degen_tol 1e-8).  Paths: N = 8 fused H(k) + eigh
# and FMA products; N = 12 GEMM H(k), shared-memory eigh, DMMA products; N >= 16 global-scratch eigh; N >= 224 two-stage
# tridiagonalisation.
CASES = {
    "2d-flips-N8": (lambda: sr.orbit_sum([_b2()], sr.signed_permutations(2, perms=False), 1), None,
                    [[0, 0], [0.5, 0.5], [0, 0.5]], {4}),
    "2d-signed-perms-N16": (lambda: sr.orbit_sum([_b2()], sr.signed_permutations(2), 2), None,
                            [[KAPPA, KAPPA], [0.5, 0.5], [0, 0], [0, 0.5]], {2, 8, 4}),
    "3d-perms-N12": (_perms3, None, [[KAPPA] * 3], {6}),
    "3d-signed-perms-N96": (_signed3, None, [[0.5] * 3, [0, 0.5, 0], [KAPPA] * 3, [0.31, -0.42, 0.11]], {48, 16, 6, 1}),
    "4x3d-signed-perms-N384": (lambda: _signed3(4), None, [[0.5] * 3], {48}),
    "8x3d-signed-perms-N768": (lambda: _signed3(8), None, [[0.5] * 3], {48}),
    "3d-perms-2x2x2-N96": (_perms3, (2, 2, 2), [[KAPPA] * 3], {6}),
    "3d-perms-4x4x4-N768": (_perms3, (4, 4, 4), [[KAPPA] * 3], {6}),
}
WORST: dict = {}


def _note(key, ratio):
    WORST[key] = max(WORST.get(key, 0.0), ratio)


def _case(name):
    """``(orbit, size, explicit packed model, k)``; k: the designed points (their cluster sizes asserted) followed by two
    generic points."""
    build, size, pts, sizes = CASES[name]
    orbit = build()
    dim = orbit.packed.dim
    k = np.concatenate([np.array(pts, dtype=np.float64), np.random.default_rng(len(name)).uniform(-1, 1, (2, dim))])
    w = sr.orbit_exact(orbit, k, size=size)[0]
    got = set().union(*(sr.cluster_sizes(row) for row in w[: len(pts)]))
    assert got == sizes, f"{name}: cluster sizes {got} != {sizes}"
    packed = orbit.packed if size is None else wl.supercell(orbit.packed, size)
    return orbit, size, packed, k


def _evaluators(tbk, orbit, size, packed):
    """Host-packed and device-packed (``from_supercell``; size 1 for plain orbit sums) evaluators of the same model."""
    return [("host-packed", tbk.Evaluator(packed)),
            ("from_supercell", tbk.Evaluator.from_supercell(orbit.packed, size or (1,) * orbit.packed.dim))]


def _gaps(w_exact, degen_tol):
    return np.array([vr.cluster_gaps(row, degen_tol) for row in np.asarray(w_exact, dtype=np.float64)])


def check_vel(got, want, w_exact, S, what, degen_tol=1e-8, c=C_VEL):
    """``|got - want| <= c sqrt(N) eps S_d (1 + rho / g_n)``, g_n from the clusters at ``degen_tol``."""
    got = np.asarray(got, dtype=np.float64)
    assert got.shape == want.shape, f"{what}: shape {got.shape} != {want.shape}"
    assert np.all(np.isfinite(got)), f"{what}: velocities not finite"
    w64 = np.asarray(w_exact, dtype=np.float64)
    rho = float(np.abs(w64).max())
    g = _gaps(w64, degen_tol)[:, :, None]
    bound = np.sqrt(w64.shape[-1]) * EPS * np.maximum(S, 1e-300)[None, None, :] * (1 + rho / g)
    ratio = float((np.abs(got.astype(np.longdouble) - want).astype(np.float64) / bound).max())
    print(f"[clusters] {what}: vel err {ratio:.3g} x sqrt(N) eps S_d (1 + rho / g)")
    _note("velocity", ratio)
    assert ratio <= c, f"{what}: velocity error {ratio:.2f} > {c:g} units of sqrt(N) eps S_d (1 + rho / g)"
    return ratio


def check_curv(got, want, w_exact, S, dim, what, degen_tol=1e-8, traces=False, c=C_CURV):
    """``|got - want| <= c sqrt(N) eps S_a S_b (1 + rho / g_n) / g_n^2``; ``traces``: clusters compared by their sums."""
    got = np.asarray(got, dtype=np.float64)
    assert got.shape == want.shape, f"{what}: shape {got.shape} != {want.shape}"
    assert np.all(np.isfinite(got)), f"{what}: curvature not finite"
    w64 = np.asarray(w_exact, dtype=np.float64)
    rho = float(np.abs(w64).max())
    g = _gaps(w64, degen_tol)[:, :, None]
    sab = np.array([S[a] * S[b] for a, b in cr.pairs(dim)])
    bound = np.sqrt(w64.shape[-1]) * EPS * sab[None, None, :] * (1 + rho / g) / (g * g)
    err = np.abs(got.astype(np.longdouble) - want).astype(np.float64)
    if traces:
        for i, row in enumerate(w64):
            for s, t in vr.clusters(row, degen_tol):
                err[i, s:t] = np.abs(got[i, s:t].astype(np.longdouble).sum(axis=0) - want[i, s:t].sum(axis=0))
    ratio = float((err / bound).max())
    print(f"[clusters] {what}: curv err {ratio:.3g} x sqrt(N) eps S_a S_b (1 + rho / g) / g^2")
    _note("curvature", ratio)
    assert ratio <= c, f"{what}: curvature error {ratio:.2f} > {c:g} units"
    return ratio


def _dh(packed, k, d):
    """``dH/dk_d`` ``[N, N]`` at one momentum (the closed form of velocity_reference.dhamilton, one direction)."""
    out = np.zeros((packed.size, packed.size), dtype=complex)
    for R, T in zip(np.asarray(packed.R), np.asarray(packed.hop)):
        if R[d]:
            term = np.exp(2j * np.pi * float(np.dot(k, R))) * T
            out += 2j * np.pi * R[d] * (term - term.conj().T)
    return out


# ------------------------------------------------------------------------------------------------------- non-vacuity
@pytest.mark.parametrize("name", list(CASES))
def test_clusters_are_mixed(tbk, name):
    """The blocks the kernels diagonalise are far from diagonal: with the eigenvectors of ``Evaluator.eigh`` (the same
    eigh launch as band_velocity / berry_curvature, whose w those entry points reproduce bit for bit),
    ``max |offdiag(V_c^H dH_0 V_c)| / spread`` >= MIN_MIXING in some cluster of m >= 3.  Otherwise the other tests of this
    file would say nothing about Jacobi."""
    orbit, size, packed, k = _case(name)
    for label, ev in _evaluators(tbk, orbit, size, packed):
        w, V = ev.eigh(k)
        wv, _ = ev.band_velocity(k)
        ev.close()
        assert np.array_equal(w, wv), f"{name} {label}: eigh's w differs from band_velocity's"
        best = 0.0
        for i in range(k.shape[0]):
            dH = None
            for s, t in vr.clusters(w[i], 1e-8):
                if t - s < 3:
                    continue
                dH = _dh(packed, k[i], 0) if dH is None else dH
                B = V[i][:, s:t].conj().T @ dH @ V[i][:, s:t]
                e = np.linalg.eigvalsh((B + B.conj().T) / 2)
                off = float(np.abs(B - np.diag(np.diag(B))).max())
                best = max(best, off / float(e[-1] - e[0]))
        print(f"[clusters] {name} {label}: mixing max |offdiag| / spread = {best:.3g}")
        _note(f"mixing {name} {label}", best)
        assert best >= MIN_MIXING, f"{name} {label}: eigh's cluster vectors are (nearly) localised on copies ({best:.3g})"


# ----------------------------------------------------------------------------------------------------- every member
@pytest.mark.parametrize("name", list(CASES))
def test_velocities(tbk, name):
    import torch

    orbit, size, packed, k = _case(name)
    want_w, want_v, _ = sr.orbit_exact(orbit, k, size=size)
    S = vr.velocity_budget(packed)
    for label, ev in _evaluators(tbk, orbit, size, packed):
        w, v = ev.band_velocity(k)
        wd, vd = ev.band_velocity_device(torch.from_numpy(k).cuda())
        ev.check()
        ev.close()
        assert np.array_equal(wd.cpu().numpy(), w) and np.array_equal(vd.cpu().numpy(), v), "host != device entry point"
        check_eig(w, want_w, f"{name} {label}")
        check_vel(v, want_v, want_w, S, f"{name} {label}")


@pytest.mark.parametrize("convention", CONVENTIONS)
@pytest.mark.parametrize("name", list(CASES))
def test_curvature(tbk, name, convention):
    import torch

    orbit, size, packed, k = _case(name)
    want_w, _, want_c = sr.orbit_exact(orbit, k, convention, size=size)
    S = cr.curvature_budget(packed, convention)
    traces = size is not None and convention == 2
    for label, ev in _evaluators(tbk, orbit, size, packed):
        w, c = ev.berry_curvature(k, convention=convention)
        wd, cd = ev.berry_curvature_device(torch.from_numpy(k).cuda(), convention=convention)
        ev.check()
        ev.close()
        assert np.array_equal(wd.cpu().numpy(), w) and np.array_equal(cd.cpu().numpy(), c), "host != device entry point"
        check_eig(w, want_w, f"{name} {label}")
        check_curv(c, want_c, want_w, S, packed.dim, f"{name} {label} conv {convention}", traces=traces)


# ------------------------------------------------------------------------------------------------------------ degen_tol
# a 6-fold (N = 12) and a 48-fold (N = 96) point; copy g shifted by offset + g delta, delta = 2^-10 rho to within a factor
# of two (much smaller spacings would drown the curvature's ordering in its g^-2 bound)
SHIFTED = {"3d-perms-N12": (lambda: _b3(), sr.signed_permutations(3, signs=False), [KAPPA] * 3),
           "3d-signed-perms-N96": (lambda: _b3(), sr.signed_permutations(3), [0.5] * 3)}


@pytest.mark.parametrize("offset", [16.0, -64.0])
@pytest.mark.parametrize("name", list(SHIFTED))
def test_degen_tol_cut(tbk, name, offset):
    """``degen_tol = delta / (2 rho)`` splits the shifted cluster (the exact values in energy order), ``2 delta / rho``
    merges it (the sorted exact values).  The whole model is shifted up by 16 (rho = max |E| is the largest eigenvalue) or
    down by 64 (rho is |E_0|, the spectrum negative)."""
    base_fn, G, pt = SHIFTED[name]
    k = np.array([pt])
    orbit = sr.orbit_sum([base_fn()], G, 3, shifts=np.full(len(G), offset))
    rho = float(np.abs(sr.orbit_exact(orbit, k)[0]).max())
    delta = 2.0 ** (np.floor(np.log2(rho)) - 10)
    orbit = sr.orbit_sum([base_fn()], G, 3, shifts=offset + delta * np.arange(len(G)))
    p = orbit.packed
    w_ex = sr.orbit_exact(orbit, k, degen_tol=0.0)[0]
    rho = float(np.abs(w_ex).max())
    assert (float(w_ex.min()) > 0) if offset > 0 else (float(w_ex.max()) < 0)
    ev = tbk.Evaluator(p)
    for tol, sizes in ((delta / (2 * rho), {1}), (2 * delta / rho, {len(G)})):
        w_ex, v_ex, _ = sr.orbit_exact(orbit, k, degen_tol=tol)
        assert sr.cluster_sizes(w_ex[0], tol) == sizes
        w, v = ev.band_velocity(k, degen_tol=tol)
        check_eig(w, w_ex, f"{name} offset {offset}")
        check_vel(v, v_ex, w_ex, vr.velocity_budget(p), f"shifted {name} offset {offset} degen_tol {tol:.3g}", degen_tol=tol)
        for convention in CONVENTIONS:
            _, _, c_ex = sr.orbit_exact(orbit, k, convention, degen_tol=tol)
            _, c = ev.berry_curvature(k, convention=convention, degen_tol=tol)
            check_curv(c, c_ex, w_ex, cr.curvature_budget(p, convention), 3,
                       f"shifted {name} offset {offset} conv {convention} degen_tol {tol:.3g}", degen_tol=tol)
    ev.close()


@pytest.mark.parametrize("name", ["2d-flips-N8", "3d-signed-perms-N96"])
def test_degen_tol_zero_generic(tbk, name):
    """At generic k every band is a singleton: ``degen_tol = 0`` gives the default's bits."""
    orbit = CASES[name][0]()
    p = orbit.packed
    k = np.random.default_rng(11).uniform(-1, 1, (5, p.dim))
    w_ex = sr.orbit_exact(orbit, k)[0]
    assert all(sr.cluster_sizes(row) == {1} for row in w_ex)
    ev = tbk.Evaluator(p)
    w, v = ev.band_velocity(k)
    w0, v0 = ev.band_velocity(k, degen_tol=0.0)
    assert np.array_equal(w0, w) and np.array_equal(v0, v)
    for convention in CONVENTIONS:
        _, c = ev.berry_curvature(k, convention=convention)
        _, c0 = ev.berry_curvature(k, convention=convention, degen_tol=0.0)
        assert np.array_equal(c0, c), f"{name} conv {convention}: degen_tol 0 differs from the default at generic k"
    ev.close()


@pytest.mark.parametrize("name", ["2d-flips-N8", "3d-perms-N12", "2d-signed-perms-N16", "3d-signed-perms-N96"])
def test_degen_tol_whole_spectrum(tbk, name):
    """``degen_tol = 4``: one cluster of all N bands.  Velocities are the eigenvalues of dH/dk_d itself (V^H dH_d V is
    similar to it), to ``C_VEL sqrt(N) eps S_d``; the curvature is exactly zero (F has no states outside).  N <= 96: the
    N x N Jacobi runs on one thread (N = 384 took 6 minutes on an NVIDIA B200)."""
    orbit, size, packed, k = _case(name)
    ev = tbk.Evaluator(packed)
    w, v = ev.band_velocity(k, degen_tol=4.0)
    S = vr.velocity_budget(packed)
    want = np.stack([np.stack([np.linalg.eigvalsh(_dh(packed, q, d)) for d in range(packed.dim)], axis=-1) for q in k])
    ratio = float((np.abs(v - want) / (np.sqrt(packed.size) * EPS * S)).max())
    print(f"[clusters] {name} degen_tol 4: vel err {ratio:.3g} x sqrt(N) eps S_d")
    _note("velocity, one cluster", ratio)
    assert ratio <= C_VEL
    for convention in CONVENTIONS:
        wc, c = ev.berry_curvature(k, convention=convention, degen_tol=4.0)
        assert np.array_equal(wc, w) and not c.any(), f"{name} conv {convention}: curvature of one cluster is not zero"
    ev.close()


# ----------------------------------------------------------------------------------------------------------------- scale
@pytest.mark.parametrize("e", [-600, 600])
def test_scaled_48_fold_bitwise(tbk, e):
    """H -> 2^e H at a 48-fold point: velocities exactly 2^e times, curvature bit-equal."""
    orbit, _, packed, k = _case("3d-signed-perms-N96")
    ev = tbk.Evaluator(packed)
    evs = tbk.Evaluator(xs.scaled(packed, e))
    w, v = ev.band_velocity(k)
    ws, vs = evs.band_velocity(k)
    assert np.array_equal(ws, np.ldexp(w, e)) and np.array_equal(vs, np.ldexp(v, e)), f"2^{e}: velocities not scaled exactly"
    for convention in CONVENTIONS:
        _, c = ev.berry_curvature(k, convention=convention)
        _, cs = evs.berry_curvature(k, convention=convention)
        assert np.array_equal(cs, c), f"2^{e} conv {convention}: curvature differs from the unscaled one"
    ev.close()
    evs.close()


def test_worst_ratios():
    """Prints the worst ratio of every check of this module (run last, ``pytest -s``)."""
    for key, val in sorted(WORST.items()):
        print(f"[clusters] worst {key}: {val:.3g}")
