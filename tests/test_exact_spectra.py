"""The exact-spectrum references of ``oracle/exact_spectra.py``, pinned on the CPU.

``tests/test_gpu_accuracy.py`` holds the kernels to these references at a few ulps, so the references themselves must be
right to much better than that: the folding identity and the closed forms against LAPACK on the supercell Hamiltonian and
against 40-digit mpmath, the designed spectra against LAPACK and their rounding bound delta.
"""
import numpy as np
import pytest
import scipy.linalg as la

from oracle import exact_spectra as xs
from oracle import tb_oracle as orc
from oracle import workloads as wl

EPS = np.finfo(np.float64).eps

pytestmark = pytest.mark.skipif(
    not xs.longdouble_is_extended(),
    reason=f"np.longdouble has a {np.finfo(np.longdouble).nmant}-bit mantissa here; the exact references need >= 63 bits",
)

FOLD_CASES = [
    ("band1-3d", lambda: xs.band1(3), (2, 2, 1)),
    ("band1-3d", lambda: xs.band1(3), (3, 3, 1)),
    ("band1-3d", lambda: xs.band1(3), (4, 4, 2)),
    ("band1-3d-long", lambda: xs.band1(3, n_half=40, seed=3), (3, 2, 2)),
    ("band2-2d", lambda: xs.band2(2, 4), (4, 4)),
    ("band2-2d-long", lambda: xs.band2(2, 8, seed=5), (3, 2)),
    ("band2-3d", lambda: xs.band2(3, 13, seed=4), (2, 2, 2)),
    ("band1-1d", lambda: xs.band1(1, 3, seed=6), (7,)),
]


def _kpoints(dim, seed=0):
    """Gamma, the zone boundary (highly degenerate folded spectra) and random points, incl. |K| > 1."""
    rng = np.random.default_rng(seed)
    return np.concatenate([np.zeros((1, dim)), np.full((1, dim), 0.5), rng.uniform(-1, 1, (3, dim)), rng.uniform(-40, 40, (1, dim))])


@pytest.mark.parametrize("name,make,size", FOLD_CASES, ids=[f"{c[0]}-{'x'.join(map(str, c[2]))}" for c in FOLD_CASES])
def test_folded_spectrum_matches_lapack_on_the_supercell(name, make, size):
    """The folded spectrum is the spectrum of wl.supercell(...)'s H(K): LAPACK agrees within 32 sqrt(N) eps rho."""
    base = make()
    sup = wl.supercell(base, size)
    K = _kpoints(base.dim)
    want = xs.folded_spectrum(base, size, K)
    assert want.shape == (len(K), sup.size) and want.dtype == np.longdouble
    H = orc.hamilton(sup.R, sup.hop, sup.pos, K, 2)
    got = np.array([la.eigvalsh(h) for h in H])
    rho = float(np.abs(want).max())
    err = float(np.abs(got - want.astype(np.float64)).max())
    assert err <= 32 * np.sqrt(sup.size) * EPS * rho, f"{name} {size}: {err / (EPS * rho):.1f} eps rho"


MPMATH_CASES = [c for c in FOLD_CASES if c[1]().size * int(np.prod(c[2])) <= 16]


@pytest.mark.parametrize("name,make,size", MPMATH_CASES, ids=[f"{c[0]}-{'x'.join(map(str, c[2]))}" for c in MPMATH_CASES])
def test_folded_spectrum_matches_mpmath(name, make, size):
    """N <= 16: the supercell H(K) and its eigenvalues in 40-digit arithmetic (the float64 hoppings are exact there) agree
    with the folding identity evaluated in 40 digits to 1e-25, and the longdouble closed forms with both to ~ 1e-18."""
    mpmath = pytest.importorskip("mpmath")
    base = make()
    sup = wl.supercell(base, size)
    K = _kpoints(base.dim, seed=1)[[0, 1, 2, 5]]
    with mpmath.workdps(40):
        two_pi_i = 2j * mpmath.pi

        def h_mp(packed, k):
            n = packed.size
            H = mpmath.matrix(n, n)
            for R, T in zip(packed.R, packed.hop):
                x = sum((kd if isinstance(kd, mpmath.mpf) else mpmath.mpf(float(kd))) * int(rd) for kd, rd in zip(k, R))
                ph = mpmath.exp(two_pi_i * x)
                for i in range(n):
                    for j in range(n):
                        if T[i, j] != 0:
                            H[i, j] += ph * mpmath.mpc(T[i, j].real, T[i, j].imag)
            return H + H.transpose_conj()

        ld = xs.folded_spectrum(base, size, K)
        for ik, Kp in enumerate(K):
            w_sup = sorted(mpmath.eighe(h_mp(sup, Kp), eigvals_only=True))
            w_fold = []
            for o in xs.cell_offsets(size):
                kb = [(mpmath.mpf(float(Kp[d])) + int(o[d])) / int(size[d]) for d in range(base.dim)]
                Hb = h_mp(base, kb)
                if base.size == 1:
                    w_fold.append(mpmath.re(Hb[0, 0]))
                else:
                    mean, half = (Hb[0, 0] + Hb[1, 1]) / 2, (Hb[0, 0] - Hb[1, 1]) / 2
                    rad = mpmath.sqrt(mpmath.re(half) ** 2 + abs(Hb[1, 0]) ** 2)
                    w_fold += [mpmath.re(mean) - rad, mpmath.re(mean) + rad]
            w_fold.sort()
            rho = max(abs(x) for x in w_fold)
            assert max(abs(a - b) for a, b in zip(w_sup, w_fold)) <= 1e-25 * rho, f"K={Kp}: folding identity"
            err_ld = max(abs(mpmath.mpf(float(a)) + mpmath.mpf(float(a - np.longdouble(float(a)))) - b)
                         for a, b in zip(ld[ik], w_fold))
            assert err_ld <= 64 * float(np.finfo(np.longdouble).eps) * float(rho), f"K={Kp}: longdouble closed form"


def test_folded_supercell_sizes_reach_the_large_classes():
    """The (8, 101, 1) supercell (N = 808) is cheap: the reference of 3 momenta takes one vectorised longdouble sum.
    With real hoppings (time-reversal symmetric) the Gamma spectrum is degenerate: e(o / size) = e(-o / size), so every
    level but those of the mirror-symmetric offsets is double."""
    K = _kpoints(3)[:3]
    w = xs.folded_spectrum(xs.band1(3), (8, 101, 1), K)
    assert w.shape == (3, 808) and np.all(np.diff(w.astype(np.float64), axis=1) >= 0)
    w = xs.folded_spectrum(xs.band1(3, real=True), (8, 101, 1), K)
    vals = np.round(w[0].astype(np.float64), 12)
    assert len(np.unique(vals)) <= 808 // 2 + 2


@pytest.mark.parametrize("kind", xs.SPECTRA)
@pytest.mark.parametrize("n", [1, 3, 12, 33, 130, 260])
def test_designed_spectrum_is_exact(kind, n):
    """H_f64 is exactly Hermitian, its rounding bound delta is <= 2 eps rho, and LAPACK finds lam within 32 sqrt(N) eps rho
    + delta (in practice within ~ sqrt(N) eps rho)."""
    p, lam, delta, Q = xs.designed_model(kind, n, seed=7, return_vectors=True)
    H = 2 * p.hop[0]
    # Q holds the exact eigenvectors: unitary, and H Q = Q diag(lam) up to the float64 roundings of H and Q
    assert np.abs(Q.conj().T @ Q - np.eye(n)).max() <= 4 * n * EPS
    assert np.abs(H @ Q - Q * lam).max() <= 4 * n * EPS * float(np.abs(lam).max())
    assert p.n_R == 1 and not p.R.any()
    assert np.array_equal(H, H.conj().T)
    assert np.array_equal(lam, np.sort(lam)) and lam.shape == (n,)
    rho = float(np.abs(lam).max())
    assert delta <= 2 * EPS * rho, f"delta = {delta / (EPS * rho):.2f} eps rho"
    w = la.eigvalsh(H)
    assert np.abs(w - lam).max() <= 32 * np.sqrt(n) * EPS * rho + delta
    # the model's H(k) is that matrix at every k (R = 0 only), through the reference's own sum
    k = np.random.default_rng(n).uniform(-3, 3, (2, 3))
    assert np.array_equal(orc.hamilton(p.R, p.hop, p.pos, k, 2), np.stack([H, H]))


def test_designed_spectrum_families_have_their_structure():
    rng = np.random.default_rng(0)
    c = xs.spectrum("clusters", 64, rng)
    assert np.ptp(c[:16]) <= 1e-9 and np.diff(c).max() > 0.5
    m = xs.spectrum("multiple", 64, rng)
    assert sorted(np.unique(m, return_counts=True)[1]) == [16] * 4
    g = xs.spectrum("graded", 64, rng)
    assert np.abs(g).min() < 1e-11 and np.abs(g).max() == 1.0
    assert xs.spectrum("outlier", 64, rng).max() == 1e6
    assert np.all(np.abs(xs.spectrum("offset", 64, rng) - 1e4) <= 1)


def test_hamilton_longdouble_beats_the_float64_sum_at_large_k():
    """At |k| ~ 1e3 the float64 Fourier sum is off by ~ 1e3 eps (the phase argument k.R loses its low digits before the
    exponential); longdouble keeps 11 more bits, so it still judges a kernel at rounding level there."""
    p = wl.synthetic(4, 30, seed=5)
    k = np.random.default_rng(1).uniform(-1e3, 1e3, (20, 3))
    ld = orc.hamilton_longdouble(p.R, p.hop, p.pos, k, 2)
    f64 = orc.hamilton(p.R, p.hop, p.pos, k, 2)
    scale = xs.hamilton_scale(p, k)
    assert (np.abs(f64 - ld) / scale).max() <= 2 * EPS  # the budget covers the float64 sum ...
    assert np.abs(f64 - ld).max() > 50 * EPS * (np.abs(p.hop).sum(axis=0) * 2).max()  # ... which is far from exact


@pytest.mark.parametrize("name", ["band2", "syn3"])
def test_kdotp_longdouble_references_match_the_oracle(name):
    """The longdouble construct_kdotp coefficients and k.p Hamiltonian agree with the float64 restatements of the
    reference within their own rounding budgets."""
    p = xs.band2(2, 4) if name == "band2" else wl.synthetic(3, 9, seed=11)
    k0 = np.random.default_rng(3).uniform(-0.7, 0.7, p.dim)
    powers, coeff, scale = xs.kdotp_coefficients_longdouble(p, k0, 3)
    want = orc.construct_kdotp(p.R, p.hop, p.pos, k0, 3)
    assert [tuple(x) for x in powers] == list(want)
    for q, key in enumerate(want):
        assert np.all(np.abs(want[key] - coeff[q]) <= 8 * EPS * scale[q] + 1e-300), key
    c64 = coeff.astype(np.complex128)
    tc = {tuple(int(x) for x in pw): c64[q] for q, pw in enumerate(powers)}
    k = np.random.default_rng(4).uniform(-2, 2, (9, p.dim))
    H, hs = xs.kdotp_hamilton_longdouble(powers, c64, k)
    assert np.all(np.abs(orc.kdotp_hamilton(tc, k) - H) <= 8 * EPS * hs + 1e-300)
