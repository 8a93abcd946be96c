"""Rounding-level accuracy of every kernel path against references that are better than float64.

The parity tests hold the kernels to the north-star bounds (1e-10 rho for eigenvalues), about 25 000 times what LAPACK
loses: a kernel that drops four digits passes them.  Here the references are exact spectra and longdouble Hamiltonians
(``oracle/exact_spectra.py``, pinned on the CPU by ``tests/test_exact_spectra.py``), and the bounds are a few ulps:

* eigenvalues: ``max |lam_gpu - lam_exact| <= C_EIG sqrt(N) eps rho + delta``, delta the rounding of the stored matrix
  (designed spectra; for folded supercells the rounding of the summed supercell hoppings, ~ eps rho, sits inside the
  constant);
* eigenvectors: residual ``max_j ||H v_j - w_j v_j|| <= C_EIG sqrt(N) eps rho``, ``max |V^H V - I| <= C_EIG sqrt(N) eps``,
  and inside a cluster of eigenvalues the spectral projector within ``C_EIG sqrt(N) eps rho / gap`` of the exact one;
* H(k) elementwise: ``|dH_ij| <= C_H eps sum_R (|T_R,ij| + |T_R,ji|) (1 + 2 pi sum_d |k_d R_d|)`` -- one rounding per
  term of the Fourier sum, and the rounding of that term's k.R in double that no kernel forming it can avoid.

LAPACK sits near 1.1 sqrt(N) eps rho on these spectra.  Every check prints its worst ratio (``pytest -s``) in units of
``sqrt(N) eps rho`` (eigenvalues) or of the H budget, so the margin of every path can be read off a run.
"""
import numpy as np
import pytest

from oracle import exact_spectra as xs
from oracle.accuracy import C_EIG, EPS, check_eig, check_h, kset
from oracle import workloads as wl

pytestmark = [
    pytest.mark.gpu,
    pytest.mark.skipif(not xs.longdouble_is_extended(), reason="the exact references need an 80-bit np.longdouble"),
]


@pytest.fixture(scope="module")
def tbk():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import tbmodels_b200

    return tbmodels_b200


# ------------------------------------------------------------------------- folded supercells through the default dispatch
# (base, size): N = N_b prod(size) covers every size class of the default dispatch -- trigonometric-product kernel (N <= 2:
# size 1 of a base model with |R_d| <= 1, k-dependent spectrum), fused small kernel (N <= 8), staged
# shared-memory kernels, register kernel (21 .. 40), staged -> register hand-over, QL / bisection boundary (128 / 129),
# two-stage reduction (128 .. 808), the last size 808
FOLDED = [
    ("b1", (3, 1, 1)), ("b1", (2, 2, 1)), ("b1", (5, 1, 1)), ("b1", (3, 2, 1)), ("b1", (7, 1, 1)), ("b1", (2, 2, 2)),
    ("b1", (3, 3, 1)), ("b1", (3, 2, 2)), ("b1", (4, 4, 2)), ("b1", (11, 3, 1)), ("b1r", (3, 3, 4)), ("b1", (4, 4, 4)),
    ("b1", (41, 2, 1)), ("b1", (83, 1, 1)), ("b1r", (5, 5, 5)), ("b1", (8, 4, 4)), ("b1", (43, 3, 1)), ("b1", (5, 5, 8)),
    ("b1r", (8, 8, 4)), ("b1", (7, 7, 7)), ("b1", (8, 8, 8)), ("b1", (10, 10, 6)), ("b1", (9, 9, 9)), ("b1", (8, 101, 1)),
    ("b1", (1, 1, 1)), ("b2", (1, 1)), ("b2-3d", (1, 1, 1)), ("b2", (2, 2)), ("b2", (4, 4)), ("b2", (6, 6)), ("b2", (8, 8)), ("b2-3d", (2, 2, 2)), ("b2-3d", (3, 3, 2)),
    ("b2-3d", (4, 4, 4)),
] + [("b1-600", (3, 3, 1)), ("b2-1500", (2, 2, 2)), ("b1-3000", (3, 3, 4)), ("b2-3000", (3, 3, 2)), ("b1-4000", (4, 4, 4))]
# the last five: long-range bases whose supercells have 138 .. 309 stored R, so their explicit-k H(k) runs on the INT8
# digit GEMM by default (>= 81 stored R; tests/test_gpu_hk_int8_exact.py checks that it does)
BASES = {
    "b1": lambda: xs.band1(3),
    "b1r": lambda: xs.band1(3, real=True, seed=4),
    "b2": lambda: xs.band2(2, 4),
    "b2-3d": lambda: xs.band2(3, 13, seed=4),
    "b1-600": lambda: xs.band1(3, 600),
    "b2-1500": lambda: xs.band2(3, 1500),
    "b1-3000": lambda: xs.band1(3, 3000),
    "b2-3000": lambda: xs.band2(3, 3000),
    "b1-4000": lambda: xs.band1(3, 4000),
}
INT8_FOLDED = FOLDED[-5:]


def _fold_id(case):
    base, size = case
    return f"{base}-{'x'.join(map(str, size))}"


@pytest.mark.parametrize("case", FOLDED, ids=[_fold_id(c) for c in FOLDED])
def test_folded_supercell_default_dispatch(tbk, case):
    """Host-packed (Evaluator(wl.supercell(...))) and device-packed (Evaluator.from_supercell, block-sparse GEMM)
    supercells, explicit k through the host and the device-buffer entry points, against the folded spectrum."""
    import torch

    name, size = case
    base = BASES[name]()
    n = base.size * int(np.prod(size))
    K = kset(base.dim, n_random=33 if n <= 8 else (3 if n <= 300 else 1), seed=n)
    want = xs.folded_spectrum(base, size, K)
    dev = tbk.Evaluator.from_supercell(base, size)
    check_eig(dev.eigenval_array(K), want, f"N={n} {name} device-packed")
    got = dev.eigenval_device(torch.from_numpy(K).cuda())
    dev.check()
    check_eig(got.cpu().numpy(), want, f"N={n} {name} device-packed eigenval_device")
    dev.close()
    host = tbk.Evaluator(wl.supercell(base, size))
    check_eig(host.eigenval_array(K), want, f"N={n} {name} host-packed")
    host.close()


# the last mesh dimension holds at least two points per class of stored R (last components -1, 0, 1): factorisable.
# The long-range cases run explicit k-points only (TBK_NO_MESH_FACTOR=1), where run_eigenval builds H(k) on INT8.
MESH = [("b1", (3, 3, 4), (2, 3, 8)), ("b1", (5, 5, 5), (1, 2, 7)), ("b2-3d", (4, 4, 4), (1, 1, 8)), ("b2", (4, 4), (3, 8))]
MESH_INT8 = [("b1-600", (3, 3, 1), (2, 3, 5)), ("b2-3000", (3, 3, 2), (2, 2, 3))]


def _mesh_cases():
    for c in MESH:
        for factor in ("factorised", "explicit"):
            yield pytest.param(c, factor, id=f"{c[0]}-{'x'.join(map(str, c[1]))}-{factor}")
    for c in MESH_INT8:
        yield pytest.param(c, "explicit", id=f"{c[0]}-{'x'.join(map(str, c[1]))}-explicit")


@pytest.mark.parametrize("case,factor", list(_mesh_cases()))
def test_folded_supercell_mesh(tbk, monkeypatch, case, factor):
    """eigenval_mesh on a folded supercell: the factorised line sums and (TBK_NO_MESH_FACTOR=1) device-generated
    explicit k-points (host-packed supercell, and the device-packed one as well); the mesh contains Gamma and, for even
    sizes, the zone boundary."""
    name, size, dims = case
    if factor == "explicit":
        monkeypatch.setenv("TBK_NO_MESH_FACTOR", "1")
    base = BASES[name]()
    want = xs.folded_spectrum(base, size, wl.kgrid_points(dims))
    ev = tbk.Evaluator(wl.supercell(base, size))
    assert ev.mesh_factorised(dims) == (factor == "factorised")
    check_eig(ev.eigenval_mesh(dims), want, f"mesh N={ev.size} {name} {dims} {factor}")
    ev.close()
    if factor == "explicit":
        ev = tbk.Evaluator.from_supercell(base, size)
        check_eig(ev.eigenval_mesh(dims), want, f"mesh N={ev.size} {name} {dims} device-packed")
        ev.close()


# ------------------------------------------------------------------------------------------- forced solver routes
# (route id, environment, sizes): every solver route the tuning hooks reach.  Each size runs one designed spectrum
# (the families rotate with the size) in an odd batch, and a folded supercell of the same size where one exists.
ROUTES = [
    ("force-gemm", {"TBK_FORCE_GEMM": "1"}, (1, 2, 3, 5, 8)),
    ("no-basis", {"TBK_NO_BASIS": "1"}, (1, 2, 4, 7)),
    ("tridiag-g1", {"TBK_TRIDIAG_G": "1"}, (9, 33, 64)),
    ("tridiag-g32", {"TBK_TRIDIAG_G": "32"}, (9, 33, 64)),
    ("tridiag-g64", {"TBK_TRIDIAG_G": "64"}, (12, 36, 100)),
    ("stages-0", {"TBK_TRIDIAG_STAGES": "0"}, (25, 49, 97)),
    ("stages-50", {"TBK_TRIDIAG_STAGES": "50"}, (25, 64, 119)),
    ("stages-80", {"TBK_TRIDIAG_STAGES": "80"}, (36, 97, 119)),
    ("reg-stop0", {"TBK_TRIDIAG_REG_STOP": "0"}, (21, 33, 40)),
    ("reg-stop2", {"TBK_TRIDIAG_REG_STOP": "2"}, (24, 36, 64)),
    ("reg-stop9-mid21", {"TBK_TRIDIAG_REG_STOP": "9", "TBK_TRIDIAG_REG_MID": "21"}, (25, 32, 40)),
    ("reg-stop12-mid24", {"TBK_TRIDIAG_REG_STOP": "12", "TBK_TRIDIAG_REG_MID": "24"}, (29, 33, 64)),
    ("panel-t128-lpr16", {"TBK_TRIDIAG_PANEL_MIN": "2", "TBK_PANEL_T": "128", "TBK_PANEL_LPR": "16"}, (17, 65, 129)),
    ("panel-t128-lpr32", {"TBK_TRIDIAG_PANEL_MIN": "2", "TBK_PANEL_T": "128", "TBK_PANEL_LPR": "32"}, (9, 40, 200)),
    ("panel-t256-lpr16", {"TBK_TRIDIAG_PANEL_MIN": "2", "TBK_PANEL_T": "256", "TBK_PANEL_LPR": "16"}, (31, 100, 256)),
    ("panel-t256-lpr32", {"TBK_TRIDIAG_PANEL_MIN": "2", "TBK_PANEL_T": "256", "TBK_PANEL_LPR": "32"}, (16, 63, 129)),
    ("panel-t512-lpr16", {"TBK_TRIDIAG_PANEL_MIN": "2", "TBK_PANEL_T": "512", "TBK_PANEL_LPR": "16"}, (33, 255, 300)),
    ("panel-t512-lpr32", {"TBK_TRIDIAG_PANEL_MIN": "2", "TBK_PANEL_T": "512", "TBK_PANEL_LPR": "32"}, (24, 129, 200)),
    ("twostage-12", {"TBK_TRIDIAG_TWOSTAGE": "12"}, (12, 13, 33, 65, 100)),
    ("twostage-0", {"TBK_TRIDIAG_TWOSTAGE": "0"}, (128, 200, 343, 600)),
    ("band-t128", {"TBK_TRIDIAG_TWOSTAGE": "12", "TBK_BAND_T": "128"}, (17, 129)),
    ("band-t256", {"TBK_TRIDIAG_TWOSTAGE": "12", "TBK_BAND_T": "256"}, (40, 200)),
    ("band-t257", {"TBK_TRIDIAG_TWOSTAGE": "12", "TBK_BAND_T": "257"}, (47, 256)),
    ("band-t512", {"TBK_TRIDIAG_TWOSTAGE": "12", "TBK_BAND_T": "512"}, (64, 256)),
    ("band-chase1", {"TBK_BAND_CHASE": "1"}, (128, 131, 230)),
    ("band-chase4", {"TBK_BAND_CHASE": "4"}, (128, 200, 343)),
    ("nopanel", {"TBK_TRIDIAG_NOPANEL": "1"}, (121, 165, 300, 620)),
    ("bisect-small", {"TBK_QL_BISECT_MIN": "9"}, (9, 12, 33, 64, 128)),
    ("ql-large", {"TBK_QL_BISECT_MIN": "100000"}, (129, 200, 512, 808)),
    ("ql-global", {"TBK_QL_GLOBAL_MIN": "9"}, (9, 36, 128, 200)),
]

# folded supercells for some of the route sizes (1-band 3-D unless noted): size -> (base, supercell)
FOLDED_AT = {
    1: ("b1", (1, 1, 1)), 2: ("b2", (1, 1)), 3: ("b1", (3, 1, 1)), 4: ("b1", (2, 2, 1)), 5: ("b1", (5, 1, 1)),
    7: ("b1", (7, 1, 1)), 8: ("b1r", (2, 2, 2)), 9: ("b1r", (3, 3, 1)), 12: ("b1", (3, 2, 2)), 16: ("b2-3d", (2, 2, 2)),
    24: ("b1", (4, 3, 2)), 25: ("b1", (5, 5, 1)), 32: ("b2", (4, 4)), 33: ("b1", (11, 3, 1)), 36: ("b1r", (3, 3, 4)),
    40: ("b1", (5, 4, 2)), 49: ("b1", (7, 7, 1)), 64: ("b1r", (4, 4, 4)), 65: ("b1", (13, 5, 1)), 97: ("b1", (97, 1, 1)),
    100: ("b1", (5, 5, 4)), 119: ("b1", (17, 7, 1)), 121: ("b1", (11, 11, 1)), 128: ("b1r", (8, 4, 4)),
    129: ("b1", (43, 3, 1)), 131: ("b1", (131, 1, 1)), 165: ("b1", (11, 5, 3)), 200: ("b1", (5, 5, 8)),
    230: ("b2", (23, 5)), 255: ("b1", (17, 5, 3)), 256: ("b1r", (8, 8, 4)), 300: ("b1", (10, 10, 3)),
    343: ("b1r", (7, 7, 7)), 512: ("b1", (8, 8, 8)), 600: ("b1", (10, 10, 6)), 620: ("b1", (31, 5, 4)),
    808: ("b1", (8, 101, 1)),
}


def _route_sizes():
    for rid, env, sizes in ROUTES:
        yield pytest.param(env, sizes, id=rid)


@pytest.mark.parametrize("env,sizes", list(_route_sizes()))
def test_forced_solver_routes(tbk, monkeypatch, env, sizes):
    for key, val in env.items():
        monkeypatch.setenv(key, val)
    route = ",".join(f"{k[4:]}={v}" for k, v in env.items())
    for i, n in enumerate(sizes):
        kind = xs.SPECTRA[(i + n) % len(xs.SPECTRA)]
        p, lam, delta = xs.designed_model(kind, n, seed=11)
        nk = 3 if n > 300 else 5
        k = np.random.default_rng(n).uniform(-1, 1, (nk, 3))
        ev = tbk.Evaluator(p)
        check_eig(ev.eigenval_array(k), np.tile(lam, (nk, 1)), f"{route} N={n} {kind}", delta)
        ev.close()
        if n in FOLDED_AT:
            name, size = FOLDED_AT[n]
            base = BASES[name]()
            K = kset(base.dim, n_random=3 if n <= 300 else 1, seed=n)
            ev = tbk.Evaluator(wl.supercell(base, size)) if n <= 300 else tbk.Evaluator.from_supercell(base, size)
            check_eig(ev.eigenval_array(K), xs.folded_spectrum(base, size, K), f"{route} N={n} folded {name}")
            ev.close()


@pytest.mark.parametrize("kind", xs.SPECTRA)
def test_default_dispatch_designed_spectra(tbk, kind):
    """Every designed family through the default dispatch at the size classes (batch of 3: an odd batch)."""
    for n in (1, 2, 3, 6, 8, 9, 16, 21, 33, 40, 41, 64, 82, 127, 128, 129, 260, 600):
        p, lam, delta = xs.designed_model(kind, n, seed=3)
        k = np.random.default_rng(n).uniform(-1, 1, (3, 3))
        ev = tbk.Evaluator(p)
        check_eig(ev.eigenval_array(k), np.tile(lam, (3, 1)), f"default N={n} {kind}", delta)
        ev.close()


# ---------------------------------------------------------------------------------------------------------------- eigh
EIGH_SIZES = (1, 3, 12, 13, 31, 32, 33, 36, 64, 82, 83, 130, 260)


def _clusters(lam, rho):
    """Index ranges of the groups of lam separated by more than 1e-6 rho, and each group's gap to the rest."""
    cuts = np.flatnonzero(np.diff(lam) > 1e-6 * rho) + 1
    bounds = np.concatenate([[0], cuts, [len(lam)]])
    out = []
    for a, b in zip(bounds[:-1], bounds[1:]):
        left = lam[a] - lam[a - 1] if a > 0 else np.inf
        right = lam[b] - lam[b - 1] if b < len(lam) else np.inf
        out.append((a, b, min(left, right)))
    return out


@pytest.mark.parametrize("kind", xs.SPECTRA)
@pytest.mark.parametrize("n", EIGH_SIZES)
def test_eigh_designed_spectra(tbk, n, kind):
    """Eigenvalues against lam, residual and orthogonality at rounding level, and the spectral projector of every
    cluster (a multiple eigenvalue, a 1e-9 rho cluster, or a single level) against the exact eigenvectors."""
    p, lam, delta, Q = xs.designed_model(kind, n, seed=5, return_vectors=True)
    H = 2 * p.hop[0]
    k = np.random.default_rng(n).uniform(-1, 1, (3, 3))
    ev = tbk.Evaluator(p)
    w, v = ev.eigh(k)
    ev.close()
    what = f"eigh N={n} {kind}"
    check_eig(w, np.tile(lam, (3, 1)), what, delta)
    rho = float(np.abs(lam).max())
    unit = np.sqrt(n) * EPS
    resid = float(np.linalg.norm(H[None] @ v - v * w[:, None, :], axis=1).max())
    gram = float(np.abs(v.conj().transpose(0, 2, 1) @ v - np.eye(n)).max())
    print(f"[accuracy] {what}: residual {resid / (unit * rho):.2f}, V^H V - I {gram / unit:.2f} (sqrt(N) eps [rho])")
    assert resid <= C_EIG * unit * rho, f"{what}: residual {resid / (unit * rho):.1f} sqrt(N) eps rho"
    assert gram <= C_EIG * unit, f"{what}: |V^H V - I| = {gram / unit:.1f} sqrt(N) eps"
    worst = 0.0
    for a, b, gap in _clusters(lam, rho):
        if not np.isfinite(gap):
            continue
        P_exact = Q[:, a:b] @ Q[:, a:b].conj().T
        for i in range(3):
            P = v[i][:, a:b] @ v[i][:, a:b].conj().T
            worst = max(worst, float(np.abs(P - P_exact).max()) * gap / (unit * rho))
    print(f"[accuracy] {what}: cluster projectors {worst:.2f} sqrt(N) eps rho / gap")
    assert worst <= C_EIG, f"{what}: spectral projector off by {worst:.1f} sqrt(N) eps rho / gap"


EIGH_FOLDED = [("b1", (3, 3, 4)), ("b2-3d", (2, 2, 2))] + INT8_FOLDED


@pytest.mark.parametrize("case", EIGH_FOLDED, ids=[_fold_id(c) for c in EIGH_FOLDED])
def test_eigh_folded_supercells(tbk, case):
    """eigh of folded supercells, host- and device-packed (the last five through the INT8 H(k) build, the first two
    through DMMA): eigenvalues against the folded spectrum, the residual against the longdouble H(k), and V^H V - I,
    all at C_EIG sqrt(N) eps (rho)."""
    from oracle import tb_oracle as orc

    name, size = case
    base = BASES[name]()
    sup = wl.supercell(base, size)
    n = sup.size
    K = kset(base.dim, n_random=3, seed=n)
    want = xs.folded_spectrum(base, size, K)
    H = orc.hamilton_longdouble(sup.R, sup.hop, sup.pos, K, 2)
    rho = float(np.abs(want).max())
    unit = np.sqrt(n) * EPS
    for what, ev in (("device-packed", tbk.Evaluator.from_supercell(base, size)), ("host-packed", tbk.Evaluator(sup))):
        w, v = ev.eigh(K)
        ev.close()
        label = f"eigh N={n} {name} {what}"
        check_eig(w, want, label)
        vl = v.astype(np.clongdouble)
        resid = float(np.abs(np.sqrt((np.abs(H @ vl - vl * w.astype(np.longdouble)[:, None, :]) ** 2).sum(axis=1))).max())
        gram = float(np.abs(v.conj().transpose(0, 2, 1) @ v - np.eye(n)).max())
        print(f"[accuracy] {label}: residual {resid / (unit * rho):.2f}, V^H V - I {gram / unit:.2f} (sqrt(N) eps [rho])")
        assert resid <= C_EIG * unit * rho, f"{label}: residual {resid / (unit * rho):.1f} sqrt(N) eps rho"
        assert gram <= C_EIG * unit, f"{label}: |V^H V - I| = {gram / unit:.1f} sqrt(N) eps"


# ------------------------------------------------------------------------------------------------ H(k), elementwise
def _hk_models():
    """(id, packed): every H(k) build path.  N <= 2 nearest-cell models run the trigonometric-product (basis) kernel,
    N 3..8 the fused small kernel (nearest-cell product phases or general R), larger N the DMMA GEMM."""
    return [
        ("basis-n1-d1", xs.band1(1, 1, seed=1)), ("basis-n1-d2", xs.band1(2, 4, seed=2)), ("basis-n1-d3", xs.band1(3, 13)),
        ("basis-n2-d1", xs.band2(1, 1, seed=3)), ("basis-n2-d2", xs.band2(2, 4)), ("basis-n2-d3", xs.band2(3, 13, seed=4)),
        ("small-n2-longR", xs.band2(2, 12, seed=5)), ("small-n3-usez", wl.synthetic(3, 13, seed=6)),
        ("small-n5-usez", wl.synthetic(5, 13, seed=7)), ("small-n8-usez", wl.synthetic(8, 13, seed=8)),
        ("small-n4-longR", wl.synthetic(4, 60, seed=9)), ("small-n7-longR", wl.synthetic(7, 40, seed=10)),
        ("gemm-n9", wl.synthetic(9, 30, seed=11)), ("gemm-n36", wl.synthetic(36, 60, seed=12)),
        ("gemm-n64-2d", wl.synthetic(64, 20, seed=13, dim=2)),
    ]


HK_IDS = [m[0] for m in _hk_models()]


@pytest.mark.parametrize("kscale", [2.0, 1e3])
@pytest.mark.parametrize("convention", [1, 2])
@pytest.mark.parametrize("mid", HK_IDS)
def test_hamilton_against_longdouble(tbk, mid, convention, kscale):
    from oracle import tb_oracle as orc

    p = dict(_hk_models())[mid]
    k = np.random.default_rng(len(mid)).uniform(-kscale, kscale, (33, p.dim))
    ev = tbk.Evaluator(p)
    got = ev.hamilton(k, convention=convention)
    ev.close()
    want = orc.hamilton_longdouble(p.R, p.hop, p.pos, k, convention)
    check_h(got, want, xs.hamilton_scale(p, k, convention), f"H {mid} conv{convention} |k|<={kscale:g}")


@pytest.mark.parametrize("kscale", [2.0, 1e3])
@pytest.mark.parametrize("dense", [False, True], ids=["block-sparse", "dense"])
@pytest.mark.parametrize("case", [("b1", (3, 3, 4)), ("b2", (4, 3)), ("syn", (2, 2, 2))], ids=["b1-3x3x4", "b2-4x3", "syn5-2x2x2"])
def test_supercell_hamilton_against_longdouble(tbk, monkeypatch, case, dense, kscale):
    """Device-packed supercells, block-sparse and dense GEMM (TBK_GEMM_DENSE), both conventions."""
    from oracle import tb_oracle as orc

    if dense:
        monkeypatch.setenv("TBK_GEMM_DENSE", "1")
    name, size = case
    base = wl.synthetic(5, 9, seed=21) if name == "syn" else BASES[name]()
    sup = wl.supercell(base, size)
    k = np.random.default_rng(3).uniform(-kscale, kscale, (9, base.dim))
    ev = tbk.Evaluator.from_supercell(base, size)
    for conv in (1, 2):
        want = orc.hamilton_longdouble(sup.R, sup.hop, sup.pos, k, conv)
        check_h(ev.hamilton(k, convention=conv), want, xs.hamilton_scale(sup, k, conv),
                f"H supercell {name} {size} {'dense' if dense else 'sparse'} conv{conv} |k|<={kscale:g}")
    ev.close()


KDOTP_MODELS = {"band2-2d": lambda: xs.band2(2, 4), "syn3": lambda: wl.synthetic(3, 9, seed=11),
                "syn12-2d": lambda: wl.synthetic(12, 12, seed=12, dim=2)}


@pytest.mark.parametrize("kscale", [2.0, 1e3])
@pytest.mark.parametrize("name", list(KDOTP_MODELS))
def test_kdotp_coefficients_against_longdouble(tbk, name, kscale):
    """construct_kdotp's Taylor coefficients (kdotp_construct.cu) against the longdouble expansion, at expansion points
    with |k0| <= 2 and |k0| ~ 1e3."""
    p = KDOTP_MODELS[name]()
    ev = tbk.Evaluator(p)
    for i, k0 in enumerate(np.random.default_rng(5).uniform(-kscale, kscale, (2, p.dim))):
        powers, coeff = ev.kdotp_coefficients(k0, 3)
        want_p, want, scale = xs.kdotp_coefficients_longdouble(p, k0, 3)
        assert np.array_equal(powers, want_p)
        check_h(coeff, want, scale, f"kdotp coefficients {name} |k0|<={kscale:g} #{i}")
    ev.close()


@pytest.mark.parametrize("kscale", [2.0, 1e3])
@pytest.mark.parametrize("name", list(KDOTP_MODELS))
def test_kdotp_hamilton_against_longdouble(tbk, name, kscale):
    """The k.p Hamiltonian (monomial GEMM) of an order-3 expansion against the longdouble sum of its terms, at |k| <= 2
    and |k| ~ 1e3 (monomials up to 1e9: the budget sum_q |prod k^p| |C_q| scales with them)."""
    p = KDOTP_MODELS[name]()
    k0 = np.random.default_rng(5).uniform(-0.5, 0.5, p.dim)
    powers, coeff, _ = xs.kdotp_coefficients_longdouble(p, k0, 3)
    c64 = coeff.astype(np.complex128)
    tc = {tuple(int(x) for x in pw): c64[q] for q, pw in enumerate(powers)}
    k = np.random.default_rng(6).uniform(-kscale, kscale, (17, p.dim))
    H, hs = xs.kdotp_hamilton_longdouble(powers, c64, k)
    check_h(tbk.KdotpModel(tc).hamilton(k), H, hs, f"kdotp hamilton {name} |k|<={kscale:g}")
