"""TEST INFRASTRUCTURE ONLY -- the rounding-level checks shared by ``tests/test_gpu_accuracy.py`` and
``tests/test_gpu_scale.py``.

* eigenvalues: ``max |lam_gpu - lam_exact| <= C_EIG sqrt(N) eps rho + delta`` (``delta`` the rounding of the stored
  matrix, see :func:`oracle.exact_spectra.designed_model`);
* H(k) and k.p coefficients elementwise within ``C_H eps`` times the budget of :func:`oracle.exact_spectra.hamilton_scale`
  or the k.p budgets.

Every check prints its worst ratio (``pytest -s``), so the margin of every path can be read off a run.
"""
import numpy as np

EPS = np.finfo(np.float64).eps
C_EIG = 16.0  # eigenvalues, residuals, orthogonality: units of sqrt(N) eps rho (sqrt(N) eps)
C_H = 4.0  # H(k) and k.p coefficients: units of the per-element budget (xs.hamilton_scale)


def check_eig(got, want, what, delta=0.0):
    """``got`` ``[n_k, N]`` against the exact ``want`` (longdouble or float64) at ``C_EIG sqrt(N) eps rho + delta``."""
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want)
    assert got.shape == want.shape, f"{what}: shape {got.shape} != {want.shape}"
    assert np.all(np.isfinite(got)), f"{what}: {int((~np.isfinite(got)).sum())} eigenvalues are not finite"
    n = want.shape[-1]
    rho = float(np.abs(want).max())
    err = float(np.abs(got.astype(np.longdouble) - want).max())
    unit = np.sqrt(n) * EPS * rho
    ratio = max(err - delta, 0.0) / unit
    print(f"[accuracy] {what}: eig err {err / (EPS * rho):.2f} eps rho = {ratio:.2f} sqrt(N) eps rho (+ delta "
          f"{delta / (EPS * rho):.2f} eps rho)")
    assert np.all(np.diff(got, axis=-1) >= 0), f"{what}: eigenvalues not ascending"
    assert err <= C_EIG * unit + delta, (f"{what}: max|d lambda| = {err / (EPS * rho):.1f} eps rho = {ratio:.1f} sqrt(N) eps rho "
                                         f"> {C_EIG:g} sqrt(N) eps rho + delta")
    return ratio


def check_h(got, want_ld, scale, what, c=C_H):
    """Elementwise ``|got - want| <= c eps scale`` (``scale`` from :func:`xs.hamilton_scale` or the k.p budgets)."""
    got = np.asarray(got)
    assert got.shape == want_ld.shape, f"{what}: shape {got.shape} != {want_ld.shape}"
    assert np.all(np.isfinite(got)), f"{what}: {int((~np.isfinite(got)).sum())} elements are not finite"
    err = np.abs(got.astype(np.clongdouble) - want_ld).astype(np.float64)
    ratio = float((err / (EPS * np.maximum(scale, 1e-300))).max())
    print(f"[accuracy] {what}: H err {ratio:.2f} eps budget")
    assert ratio <= c, f"{what}: max |dH_ij| / (eps budget_ij) = {ratio:.2f} > {c:g}"
    return ratio


def kset(dim, n_random=3, seed=0, scale=1.0):
    """Gamma, the zone boundary (degenerate folded spectra with real hoppings) and random points: an odd batch."""
    rng = np.random.default_rng(seed)
    return np.concatenate([np.zeros((1, dim)), np.full((1, dim), 0.5), rng.uniform(-scale, scale, (n_random, dim))])
