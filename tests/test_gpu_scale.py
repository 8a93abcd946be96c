"""Every kernel path on models scaled by powers of two, 2^-960 .. 2^960.

Multiplying every hopping by 2^e multiplies the exact spectra, H(k) and the k.p coefficients by 2^e (``xs.scaled``), so
the rounding-level bounds of ``tests/test_gpu_accuracy.py`` apply unchanged at every scale.  The kernels square matrix
entries (Householder norms, QL rotations, the Sturm sequence's e^2, the 2 x 2 closed form), which overflow beyond about
2^+-510 unless the model is normalised; the handle does that (``tbk_api.cu``, ``normalise_exponent``).  LAPACK rescales
the same way, so the reference holds at every scale (the CPU tests below).

Exponents: +-520 lie past the squares' overflow and underflow; at -470 a 2^-26 rho splitting squared (~1e-299) falls
below any absolute cut-off near 1e-290 in the 2 x 2 closed form, +470 is its mirror; +-960 is the farthest binade where the designed entries, the
graded family's 1e-12 rho eigenvalues and the H budget all stay normal and N rho cannot overflow.

The bitwise tests hold the kernels to exact power-of-two equivariance: eigenvalues(2^e T) == 2^e eigenvalues(T), and the
same for H(k) and eigenvectors, at even e, where every operation (``rsqrt.approx`` included) is exactly equivariant.
"""
import functools

import numpy as np
import pytest
import scipy.linalg

from oracle import exact_spectra as xs
from oracle import workloads as wl
from oracle.accuracy import C_EIG, EPS, check_eig, check_h, kset

pytestmark = pytest.mark.skipif(not xs.longdouble_is_extended(), reason="the exact references need an 80-bit np.longdouble")

E = (-960, -700, -520, -470, -300, -64, 0, 64, 300, 470, 520, 700, 960)
E_ROUTES = (-700, -520, 520, 960)
E_BITWISE = (-700, -300, -64, 64, 300, 700)  # +-700: the normalisation itself must keep the bits


def ldexp(x, e):
    return np.ldexp(np.asarray(x), e)


@functools.lru_cache(maxsize=None)
def designed(kind, n, seed):
    return xs.designed_model(kind, n, seed=seed)


# -------------------------------------------------------------------------------------------------- CPU: the references
@pytest.mark.parametrize("e", E)
def test_lapack_holds_at_every_scale(e):
    """scipy eigvalsh (LAPACK zheevr, which rescales) on the scaled designed spectra stays within 32 sqrt(N) eps rho:
    the accuracy asked of the kernels is the reference's own at every scale."""
    worst = 0.0
    for i, n in enumerate((2, 12, 64)):
        kind = xs.SPECTRA[(i + n) % len(xs.SPECTRA)]
        p, lam, delta = designed(kind, n, 7)
        H = 2 * xs.scaled(p, e).hop[0]
        with np.errstate(all="raise"):
            got = scipy.linalg.eigvalsh(H)
            want = ldexp(lam, e)
            rho = float(np.abs(want).max())
            ratio = (float(np.abs(got - want).max()) - float(ldexp(delta, e))) / (np.sqrt(n) * EPS * rho)
        worst = max(worst, ratio)
        assert ratio <= 32, f"eigvalsh N={n} {kind} 2^{e}: {ratio:.2f} sqrt(N) eps rho"
    print(f"[scale] eigvalsh 2^{e}: worst {worst:.2f} sqrt(N) eps rho")


@pytest.mark.parametrize("e", E)
def test_folded_spectrum_scales_exactly(e):
    for base, size in ((xs.band1(3), (3, 2, 1)), (xs.band2(2, 4), (2, 3))):
        K = kset(base.dim, seed=1)
        with np.errstate(all="raise"):
            want = ldexp(xs.folded_spectrum(base, size, K), e)
            got = xs.folded_spectrum(xs.scaled(base, e), size, K)
        assert got.dtype == want.dtype and np.array_equal(got, want)


# ------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def tbk():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import tbmodels_b200

    return tbmodels_b200


def _ref(fn, *args):
    with np.errstate(all="raise"):
        return fn(*args)


# folded supercells, one per size class: basis kernel (N = 1, 2), fused small kernel (3 .. 8), staged and register
# kernels, QL / bisection boundary (128 / 129), two-stage reduction (200, 512)
FOLDED = [("b1", (1, 1, 1)), ("b2", (1, 1)), ("b1", (5, 1, 1)), ("b1r", (2, 2, 2)), ("b1", (3, 2, 2)),
          ("b1", (11, 3, 1)), ("b1r", (4, 4, 4)), ("b1r", (8, 4, 4)), ("b1", (43, 3, 1)), ("b1", (5, 5, 8)),
          ("b1", (8, 8, 8))]
BASES = {
    "b1": lambda: xs.band1(3),
    "b1r": lambda: xs.band1(3, real=True, seed=4),
    "b2": lambda: xs.band2(2, 4),
}


@pytest.mark.gpu
@pytest.mark.parametrize("e", E)
@pytest.mark.parametrize("case", FOLDED, ids=[f"{c[0]}-{'x'.join(map(str, c[1]))}" for c in FOLDED])
def test_folded_supercell_scaled(tbk, case, e):
    import torch

    name, size = case
    base = xs.scaled(BASES[name](), e)
    n = base.size * int(np.prod(size))
    K = kset(base.dim, n_random=9 if n <= 8 else (3 if n <= 300 else 1), seed=n)
    want = _ref(xs.folded_spectrum, base, size, K)
    what = f"2^{e} N={n} {name}"
    dev = tbk.Evaluator.from_supercell(base, size)
    check_eig(dev.eigenval_array(K), want, f"{what} device-packed")
    got = dev.eigenval_device(torch.from_numpy(K).cuda())
    dev.check()
    check_eig(got.cpu().numpy(), want, f"{what} device-packed eigenval_device")
    dev.close()
    host = tbk.Evaluator(wl.supercell(base, size))
    check_eig(host.eigenval_array(K), want, f"{what} host-packed")
    host.close()


def _routes():
    from test_gpu_accuracy import ROUTES

    return ROUTES


@pytest.mark.gpu
@pytest.mark.parametrize("e", E_ROUTES)
@pytest.mark.parametrize("env,n", [pytest.param(env, sizes[-1], id=rid) for rid, env, sizes in _routes()])
def test_forced_solver_routes_scaled(tbk, monkeypatch, env, n, e):
    """Every tuning-hook route of test_gpu_accuracy.ROUTES at its largest size, one designed spectrum."""
    for key, val in env.items():
        monkeypatch.setenv(key, val)
    kind = xs.SPECTRA[n % len(xs.SPECTRA)]
    p, lam, delta = designed(kind, n, 11)
    k = np.random.default_rng(n).uniform(-1, 1, (3, 3))
    ev = tbk.Evaluator(xs.scaled(p, e))
    route = ",".join(f"{k[4:]}={v}" for k, v in env.items())
    check_eig(ev.eigenval_array(k), np.tile(ldexp(lam, e), (3, 1)), f"2^{e} {route} N={n} {kind}", ldexp(delta, e))
    ev.close()


@pytest.mark.gpu
@pytest.mark.parametrize("e", E)
@pytest.mark.parametrize("n", (3, 33, 130, 260))
def test_eigh_scaled(tbk, n, e):
    """eigh on a scaled designed spectrum: eigenvalues, residual, V^H V - I and cluster projectors (computed on the
    unscaled problem: 2^-e w is exact) at the bounds of test_gpu_accuracy."""
    from test_gpu_accuracy import _clusters

    kind = xs.SPECTRA[n % len(xs.SPECTRA)]
    p, lam, delta, Q = xs.designed_model(kind, n, seed=5, return_vectors=True)
    H = 2 * p.hop[0]
    k = np.random.default_rng(n).uniform(-1, 1, (3, 3))
    ev = tbk.Evaluator(xs.scaled(p, e))
    w, v = ev.eigh(k)
    ev.close()
    what = f"2^{e} eigh N={n} {kind}"
    assert np.all(np.isfinite(w)) and np.all(np.isfinite(v)), f"{what}: non-finite output"
    check_eig(w, np.tile(ldexp(lam, e), (3, 1)), what, ldexp(delta, e))
    w = ldexp(w, -e)
    rho = float(np.abs(lam).max())
    unit = np.sqrt(n) * EPS
    resid = float(np.linalg.norm(H[None] @ v - v * w[:, None, :], axis=1).max())
    gram = float(np.abs(v.conj().transpose(0, 2, 1) @ v - np.eye(n)).max())
    worst = 0.0
    for a, b, gap in _clusters(lam, rho):
        if np.isfinite(gap):
            P_exact = Q[:, a:b] @ Q[:, a:b].conj().T
            for i in range(3):
                P = v[i][:, a:b] @ v[i][:, a:b].conj().T
                worst = max(worst, float(np.abs(P - P_exact).max()) * gap / (unit * rho))
    print(f"[accuracy] {what}: residual {resid / (unit * rho):.2f}, V^H V - I {gram / unit:.2f}, projectors {worst:.2f}")
    assert resid <= C_EIG * unit * rho, f"{what}: residual {resid / (unit * rho):.1f} sqrt(N) eps rho"
    assert gram <= C_EIG * unit, f"{what}: |V^H V - I| = {gram / unit:.1f} sqrt(N) eps"
    assert worst <= C_EIG, f"{what}: spectral projector off by {worst:.1f} sqrt(N) eps rho / gap"


@pytest.mark.gpu
@pytest.mark.parametrize("e", E)
@pytest.mark.parametrize("factor", ["factorised", "explicit"])
def test_mesh_scaled(tbk, monkeypatch, factor, e):
    if factor == "explicit":
        monkeypatch.setenv("TBK_NO_MESH_FACTOR", "1")
    base, size, dims = xs.scaled(BASES["b1"](), e), (3, 3, 4), (2, 3, 8)
    want = _ref(xs.folded_spectrum, base, size, wl.kgrid_points(dims))
    ev = tbk.Evaluator(wl.supercell(base, size))
    assert ev.mesh_factorised(dims) == (factor == "factorised")
    check_eig(ev.eigenval_mesh(dims), want, f"2^{e} mesh N={ev.size} {factor}")
    ev.close()


@pytest.mark.gpu
@pytest.mark.parametrize("e", E)
def test_kdotp_scaled(tbk, e):
    """KdotpModel.eigenval on a designed constant term plus a zero linear term (exact spectrum at every k), k.p H of an
    order-3 expansion against the longdouble sum, and kdotp_coefficients, all with coefficients scaled by 2^e."""
    p, lam, delta = designed("clusters", 12, 9)
    H0 = 2 * p.hop[0]
    tc = xs.scaled_kdotp({(0, 0, 0): H0, (1, 0, 0): np.zeros_like(H0)}, e)
    k = np.random.default_rng(1).uniform(-1, 1, (5, 3))
    check_eig(tbk.KdotpModel(tc).eigenval(k), np.tile(ldexp(lam, e), (5, 1)), f"2^{e} kdotp eigenval N=12", ldexp(delta, e))

    base = xs.scaled(xs.band2(2, 4), e)
    k0 = np.random.default_rng(5).uniform(-0.5, 0.5, 2)
    powers, coeff, _ = _ref(xs.kdotp_coefficients_longdouble, base, k0, 3)
    c64 = coeff.astype(np.complex128)
    kk = np.random.default_rng(6).uniform(-2, 2, (17, 2))
    H, hs = _ref(xs.kdotp_hamilton_longdouble, powers, c64, kk)
    tc = {tuple(int(x) for x in pw): c64[q] for q, pw in enumerate(powers)}
    check_h(tbk.KdotpModel(tc).hamilton(kk), H, hs, f"2^{e} kdotp hamilton")

    ev = tbk.Evaluator(base)
    got_p, got = ev.kdotp_coefficients(k0, 3)
    ev.close()
    _, want, scale = _ref(xs.kdotp_coefficients_longdouble, base, k0, 3)
    assert np.array_equal(got_p, powers)
    check_h(got, want, scale, f"2^{e} kdotp coefficients")


def _hk_models():
    from test_gpu_accuracy import _hk_models as models

    return models()


@pytest.mark.gpu
@pytest.mark.parametrize("e", E)
def test_hamilton_scaled(tbk, monkeypatch, e):
    """H(k) of every model of test_gpu_accuracy._hk_models and the device-packed supercell (block-sparse and dense
    GEMM), both conventions, against the scaled longdouble H at the scaled budget."""
    from oracle import tb_oracle as orc

    for mid, p0 in _hk_models():
        p = xs.scaled(p0, e)
        k = np.random.default_rng(len(mid)).uniform(-2, 2, (9, p.dim))
        ev = tbk.Evaluator(p)
        for conv in (1, 2):
            want = _ref(orc.hamilton_longdouble, p.R, p.hop, p.pos, k, conv)
            check_h(ev.hamilton(k, convention=conv), want, xs.hamilton_scale(p, k, conv), f"2^{e} H {mid} conv{conv}")
        ev.close()
    base = xs.scaled(BASES["b2"](), e)
    sup = wl.supercell(base, (4, 3))
    k = np.random.default_rng(3).uniform(-2, 2, (9, 2))
    want = _ref(orc.hamilton_longdouble, sup.R, sup.hop, sup.pos, k, 2)
    for dense in (False, True):
        if dense:
            monkeypatch.setenv("TBK_GEMM_DENSE", "1")
        ev = tbk.Evaluator.from_supercell(base, (4, 3))
        check_h(ev.hamilton(k), want, xs.hamilton_scale(sup, k, 2), f"2^{e} H supercell {'dense' if dense else 'sparse'}")
        ev.close()


@pytest.mark.gpu
@pytest.mark.parametrize("e", (0, -470, 470))
@pytest.mark.parametrize("env", [{}, {"TBK_NO_BASIS": "1"}, {"TBK_FORCE_GEMM": "1"}], ids=["basis", "no-basis", "gemm"])
def test_two_level_probe(tbk, monkeypatch, env, e):
    """Levels (1, 1 + 2^-26) 2^e: at 2^-470 the squared splitting (~1e-299) lies far below the float64 range's middle;
    the 2 x 2 closed form must still resolve it."""
    for key, val in env.items():
        monkeypatch.setenv(key, val)
    lam = np.array([1.0, 1.0 + 2.0 ** -26])
    p, lam, delta = xs.model_with_spectrum(lam, np.random.default_rng(26), dim=2)
    k = kset(2, n_random=5, seed=2)
    ev = tbk.Evaluator(xs.scaled(p, e))
    if not env:
        assert ev.path == "fused-product"
    check_eig(ev.eigenval_array(k), np.tile(ldexp(lam, e), (len(k), 1)), f"2^{e} two-level {ev.path}", ldexp(delta, e))
    ev.close()


# ---------------------------------------------------------------------------------------- bitwise power-of-two shifts
def _bitwise_models():
    from conftest import load_golden, packed_from

    return {
        "silicon": packed_from(load_golden("silicon.npz")),
        "haldane": wl.haldane(),
        "synthetic36-gemm": wl.synthetic(36, 30, seed=12),
    }


def _same(got, ref, e, what):
    """got == 2^e ref bit for bit wherever 2^e ref is normal (H(k): tiny elements may round to subnormals)."""
    want = ldexp(ref, e) if not np.iscomplexobj(ref) else xs.scale_complex(ref, e)
    normal = lambda a: np.abs(a) >= np.finfo(np.float64).tiny  # noqa: E731
    parts = [(got, want)] if not np.iscomplexobj(ref) else [(got.real, want.real), (got.imag, want.imag)]
    for g, w in parts:
        mask = normal(w)
        bad = int((g[mask] != w[mask]).sum())
        assert bad == 0, f"{what}: {bad} of {int(mask.sum())} normal outputs differ from 2^{e} x the unscaled run"


@pytest.mark.gpu
@pytest.mark.parametrize("e", E_BITWISE)
@pytest.mark.parametrize("mid", ["silicon", "haldane", "synthetic36-gemm"])
def test_bitwise_equivariance(tbk, mid, e):
    p = _bitwise_models()[mid]
    k = np.random.default_rng(7).uniform(-1, 1, (33, p.dim))
    runs = []
    for s in (0, e):
        ev = tbk.Evaluator(xs.scaled(p, s))
        w, v = ev.eigh(k)
        runs.append((ev.eigenval_array(k), ev.hamilton(k), ev.hamilton(k, convention=1), w, v))
        ev.close()
    (e0, h0, h10, w0, v0), (e1, h1, h11, w1, v1) = runs
    _same(e1, e0, e, f"{mid} eigenval")
    _same(h1, h0, e, f"{mid} H conv2")
    _same(h11, h10, e, f"{mid} H conv1")
    _same(w1, w0, e, f"{mid} eigh eigenvalues")
    _same(v1, v0, 0, f"{mid} eigh eigenvectors")


@pytest.mark.gpu
@pytest.mark.parametrize("e", E_BITWISE)
def test_bitwise_equivariance_supercell_and_mesh(tbk, e):
    """Device-packed N = 512 supercell (two-stage reduction, bisection) and the factorised mesh path."""
    base = BASES["b1"]()
    K = kset(3, n_random=1, seed=4)
    out = []
    for s in (0, e):
        ev = tbk.Evaluator.from_supercell(xs.scaled(base, s), (8, 8, 8))
        sup = ev.eigenval_array(K)
        ev.close()
        ev = tbk.Evaluator(wl.synthetic(36, 30, seed=12) if s == 0 else xs.scaled(wl.synthetic(36, 30, seed=12), s))
        assert ev.mesh_factorised((2, 3, 16))
        out.append((sup, ev.eigenval_mesh((2, 3, 16))))
        ev.close()
    _same(out[1][0], out[0][0], e, "supercell N=512 device-packed")
    _same(out[1][1], out[0][1], e, "mesh synthetic36 factorised")
