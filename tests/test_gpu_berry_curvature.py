"""Berry curvature of every band on the GPU (``Evaluator.berry_curvature``, berry_curvature.cu) on every kernel path.

Curvatures are held to ``C_CURV sqrt(N) eps S_a S_b (1 + rho / g_n) / g_n^2``: S_a >= ||X_a||_2 the budget of the
convention (tests/curvature_reference.py), g_n the exact gap from n's cluster to the next cluster (``S_a S_b / g_n^2``
bounds |Omega_n|).
* every dispatch class against the exact curvature of folded supercells: every member in convention 1, singletons and
  cluster traces in convention 2 (there X is not block-diagonal in the base momentum, so F of a cross-block cluster is
  not diagonal);
* the numpy oracle on the golden models, to ``1e-10 S_a S_b (1 + rho / g_n) / g_n^2``;
* consistency (w bit-equal to eigh's, host / device and chunk sizes bit-equal, the sum rule, Omega(-k) = -Omega(k) for
  real hoppings), the Haldane Chern numbers, degenerate models (H (x) I_2, H = 0, N = 1), power-of-two scaled models
  (bit-equal), argument errors.

Every check prints its worst ratio (``pytest -s``).
"""
import numpy as np
import pytest

from conftest import EIG_TOL, load_golden, packed_from
from oracle import exact_spectra as xs
from oracle import workloads as wl
from oracle.accuracy import EPS, check_eig, kset
from tbmodels_b200 import pack_arrays

import curvature_reference as cr
import velocity_reference as vr
from test_gpu_velocity import BASES, FOLDED, SCALE_MODELS, _fold_id, _golden_models

pytestmark = [
    pytest.mark.gpu,
    pytest.mark.skipif(not xs.longdouble_is_extended(), reason="the exact references need an 80-bit np.longdouble"),
]

C_CURV = 4.0  # units of sqrt(N) eps S_a S_b (1 + rho / g_n) / g_n^2; measured worst 0.30 (sum rule), 0.14 (folded), NVIDIA B200
CONVENTIONS = (1, 2)


@pytest.fixture(scope="module")
def tbk():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import tbmodels_b200

    return tbmodels_b200


def _bound(w_exact, S, dim, unit):
    """``[n_k, N, P]`` ``unit S_a S_b (1 + rho / g_n) / g_n^2``."""
    w64 = np.asarray(w_exact, dtype=np.float64)
    rho = float(np.abs(w64).max())
    g = np.array([vr.cluster_gaps(row, 1e-8) for row in w64])[:, :, None]
    sab = np.array([S[a] * S[b] for a, b in cr.pairs(dim)])
    return unit * np.maximum(sab, 1e-300)[None, None, :] * (1 + rho / g) / (g * g)


def check_curv(got, want, w_exact, S, dim, what, c=C_CURV, unit=None, traces=False):
    """``|got - want| <= c unit S_a S_b (1 + rho / g_n) / g_n^2``; ``unit`` defaults to ``sqrt(N) eps``.  ``traces``:
    clusters are compared by the sums of their members."""
    got = np.asarray(got, dtype=np.float64)
    assert got.shape == want.shape, f"{what}: shape {got.shape} != {want.shape}"
    assert np.all(np.isfinite(got)), f"{what}: curvature not finite"
    n = got.shape[1]
    label = "sqrt(N) eps" if unit is None else f"{unit:g}"
    bound = _bound(w_exact, S, dim, np.sqrt(n) * EPS if unit is None else unit)
    err = np.abs(got.astype(np.longdouble) - want).astype(np.float64)
    if traces:
        for i, row in enumerate(np.asarray(w_exact, dtype=np.float64)):
            for s, t in vr.clusters(row, 1e-8):
                if t - s > 1:
                    err[i, s:t] = np.abs(got[i, s:t].astype(np.longdouble).sum(axis=0) - want[i, s:t].sum(axis=0))
    # N = 1 has no other band (g = inf, bound 0): the curvature must then be exactly zero
    rel = np.where(err == 0, 0.0, np.divide(err, bound, out=np.full_like(err, np.inf), where=bound > 0))
    ratio = float(rel.max()) if err.size else 0.0
    print(f"[curvature] {what}: curv err {ratio:.3g} x {label} S_a S_b (1 + rho / g) / g^2")
    assert ratio <= c, f"{what}: curvature error {ratio:.2f} > {c:g} units"
    return ratio


# ------------------------------------------------------------------------- folded supercells through the default dispatch
@pytest.mark.parametrize("convention", CONVENTIONS)
@pytest.mark.parametrize("case", FOLDED, ids=[_fold_id(c) for c in FOLDED])
def test_folded_supercell_curvature(tbk, case, convention):
    """Device-packed (host and device entry points) and host-packed supercells against the exact curvature."""
    import torch

    name, size = case
    base = BASES[name]()
    sup = wl.supercell(base, size)
    n = sup.size
    K = kset(base.dim, n_random=9 if n <= 8 else (3 if n <= 300 else 1), seed=n)
    want_w, want_c = cr.folded_curvature(base, size, K, convention)
    S = cr.curvature_budget(sup, convention)
    tr = convention == 2
    dev = tbk.Evaluator.from_supercell(base, size)
    w, c = dev.berry_curvature(K, convention=convention)
    check_eig(w, want_w, f"N={n} {name} device-packed")
    check_curv(c, want_c, want_w, S, base.dim, f"N={n} {name} conv {convention} device-packed", traces=tr)
    wd, cd = dev.berry_curvature_device(torch.from_numpy(K).cuda(), convention=convention)
    dev.check()
    assert np.array_equal(wd.cpu().numpy(), w) and np.array_equal(cd.cpu().numpy(), c), "host and device entry points differ"
    dev.close()
    host = tbk.Evaluator(sup)
    w, c = host.berry_curvature(K, convention=convention)
    host.close()
    check_eig(w, want_w, f"N={n} {name} host-packed")
    check_curv(c, want_c, want_w, S, base.dim, f"N={n} {name} conv {convention} host-packed", traces=tr)


# ------------------------------------------------------------------------------------------------- oracle parity (goldens)
GOLDEN = [m[0] for m in _golden_models()]


@pytest.mark.parametrize("convention", CONVENTIONS)
@pytest.mark.parametrize("name", GOLDEN)
def test_oracle_parity(tbk, name, convention):
    p, k = dict(_golden_models())[name]
    ow, oc = cr.berry_curvature(p.R, p.hop, p.pos, k, convention)
    ev = tbk.Evaluator(p)
    w, c = ev.berry_curvature(k, convention=convention)
    ev.close()
    rho = float(np.abs(ow).max())
    assert np.abs(w - ow).max() <= EIG_TOL * rho, f"{name}: eigenvalues beyond the north-star bound"
    check_curv(c, oc, ow, cr.curvature_budget(p, convention), p.dim, f"oracle {name} conv {convention}", c=1.0, unit=1e-10)


# ------------------------------------------------------------------------------------------------------------ consistency
CONSISTENCY = {
    "haldane-basis": lambda: packed_from(load_golden("haldane.npz")),
    "syn5-small": lambda: wl.synthetic(5, 13, seed=7),
    "syn12-gemm": lambda: wl.synthetic(12, 20, seed=8),
    "syn36-gemm": lambda: wl.synthetic(36, 60, seed=12),
    "syn90-gemm": lambda: wl.synthetic(90, 20, seed=13),
}


@pytest.mark.parametrize("convention", CONVENTIONS)
@pytest.mark.parametrize("name", list(CONSISTENCY))
def test_consistency(tbk, monkeypatch, name, convention):
    """w bit-equal to eigh's; host and device entry points bit-equal; a 1 MB workspace (many chunks) bit-equal to the
    default; sum over bands zero within the budget."""
    import torch

    p = CONSISTENCY[name]()
    k = np.random.default_rng(3).uniform(-1, 1, (37, p.dim))
    ev = tbk.Evaluator(p)
    w, c = ev.berry_curvature(k, convention=convention)
    we, _ = ev.eigh(k)
    assert np.array_equal(w, we), f"{name}: w differs from eigh's"
    wd, cd = ev.berry_curvature_device(torch.from_numpy(k).cuda(), convention=convention)
    ev.check()
    ev.close()
    assert np.array_equal(wd.cpu().numpy(), w) and np.array_equal(cd.cpu().numpy(), c), f"{name}: host != device"
    bound = _bound(w, cr.curvature_budget(p, convention), p.dim, np.sqrt(p.size) * EPS).max(axis=1)  # [n_k, P]
    ratio = float((np.abs(c.sum(axis=1)) / bound).max())
    print(f"[curvature] {name} conv {convention}: sum over bands {ratio:.3g} x sqrt(N) eps S_a S_b (1 + rho / g) / g^2")
    assert ratio <= C_CURV
    monkeypatch.setenv("TBK_WORKSPACE_MB", "1")
    small = tbk.Evaluator(p)
    w1, c1 = small.berry_curvature(k, convention=convention)
    small.close()
    assert np.array_equal(w1, w) and np.array_equal(c1, c), f"{name}: results depend on the chunk size"


def _real_part(p):
    """The model with the imaginary parts of its hoppings dropped (the silicon golden model has some, up to 4e-4)."""
    return pack_arrays(p.R, np.asarray(p.hop).real.astype(complex), p.pos)


TIME_REVERSAL = {
    "silicon-real": lambda: _real_part(packed_from(load_golden("silicon.npz"))),
    "b1r-3x3x4": lambda: wl.supercell(xs.band1(3, real=True, seed=4), (3, 3, 4)),
    "b1r-5x5x5": lambda: wl.supercell(xs.band1(3, real=True, seed=4), (5, 5, 5)),
}


@pytest.mark.parametrize("convention", CONVENTIONS)
@pytest.mark.parametrize("name", list(TIME_REVERSAL))
def test_time_reversal(tbk, name, convention):
    """Real hoppings: Omega(-k) = -Omega(k); inside a cluster the ascending list is negated and reversed."""
    p = TIME_REVERSAL[name]()
    k = np.random.default_rng(6).uniform(-1, 1, (5, p.dim))
    ev = tbk.Evaluator(p)
    w, c = ev.berry_curvature(k, convention=convention)
    wm, cm = ev.berry_curvature(-k, convention=convention)
    ev.close()
    rho = float(np.abs(w).max())
    assert np.abs(wm - w).max() <= EIG_TOL * rho
    flipped = -cm
    for i in range(k.shape[0]):
        for s, t in vr.clusters(w[i], 1e-8):
            flipped[i, s:t] = flipped[i, s:t][::-1]
    check_curv(c, flipped.astype(np.longdouble), w, cr.curvature_budget(p, convention), p.dim,
               f"time reversal {name} conv {convention}")


@pytest.mark.parametrize("convention", CONVENTIONS)
def test_haldane_chern_numbers(tbk, convention):
    """128^2 mid-point mesh on the device: lower band C = -1, upper +1."""
    import torch

    p = packed_from(load_golden("haldane.npz"))
    g = (np.arange(128) + 0.5) / 128
    k = np.stack(np.meshgrid(g, g, indexing="ij"), axis=-1).reshape(-1, 2)
    ev = tbk.Evaluator(p)
    _, c = ev.berry_curvature_device(torch.from_numpy(k).cuda(), convention=convention)
    ev.check()
    ev.close()
    chern = c[:, :, 0].sum(dim=0).cpu().numpy() / k.shape[0] / (2 * np.pi)
    print(f"[curvature] Haldane conv {convention}: Chern numbers {chern}")
    np.testing.assert_allclose(chern, [-1.0, 1.0], atol=1e-10)


# ---------------------------------------------------------------------------------------------------- degenerate models
def _doubled(p):
    hop = np.stack([np.kron(h, np.eye(2)) for h in p.hop])
    return pack_arrays(p.R, hop, np.repeat(p.pos, 2, axis=0))


@pytest.mark.parametrize("convention", CONVENTIONS)
@pytest.mark.parametrize("n", [8, 36, 128])
def test_doubled_model(tbk, n, convention):
    """H (x) I_2: every eigenvalue exactly doubly degenerate; the curvatures come in equal pairs, those of H."""
    base = wl.synthetic(n // 2, 13, seed=n)
    p = _doubled(base)
    k = np.random.default_rng(n).uniform(-1, 1, (5, 3))
    ev = tbk.Evaluator(p)
    w, c = ev.berry_curvature(k, convention=convention)
    ev.close()
    bw, bc = cr.berry_curvature(base.R, base.hop, base.pos, k, convention)
    S = cr.curvature_budget(base, convention)
    rho = float(np.abs(bw).max())
    assert np.abs(w[:, 0::2] - bw).max() <= EIG_TOL * rho and np.abs(w[:, 1::2] - bw).max() <= EIG_TOL * rho
    for half in (0, 1):
        check_curv(c[:, half::2], bc, bw, S, 3, f"H x I2 N={n} conv {convention} member {half}", c=1.0, unit=1e-10)


@pytest.mark.parametrize("n", [1, 4, 40])
def test_zero_model(tbk, n):
    """H = 0: one cluster of size N, all curvatures zero."""
    p = pack_arrays(np.array([[0, 0, 0], [1, 0, 0]], np.int32), np.zeros((2, n, n), complex), np.zeros((n, 3)))
    ev = tbk.Evaluator(p)
    for convention in CONVENTIONS:
        w, c = ev.berry_curvature(np.random.default_rng(0).random((5, 3)), convention=convention)
        assert w.shape == (5, n) and c.shape == (5, n, 3)
        assert not w.any() and not c.any()
    ev.close()


def test_one_band_model(tbk):
    ev = tbk.Evaluator(xs.band1(2))
    for convention in CONVENTIONS:
        _, c = ev.berry_curvature(np.random.default_rng(1).random((7, 2)), convention=convention)
        assert c.shape == (7, 1, 1) and not c.any()
    ev.close()


# ----------------------------------------------------------------------------------------------------------------- scale
@pytest.mark.parametrize("e", [-600, -64, 64, 600])
@pytest.mark.parametrize("name", list(SCALE_MODELS))
def test_scaled_models_bitwise(tbk, name, e):
    """Omega is invariant under H -> 2^e H: bit-equal to the unscaled run; w exactly 2^e times."""
    p = SCALE_MODELS[name]()
    k = kset(p.dim, n_random=5, seed=2)
    for convention in CONVENTIONS:
        ev = tbk.Evaluator(p)
        w, c = ev.berry_curvature(k, convention=convention)
        ev.close()
        ev = tbk.Evaluator(xs.scaled(p, e))
        ws, cs = ev.berry_curvature(k, convention=convention)
        ev.close()
        assert np.array_equal(ws, np.ldexp(w, e)), f"{name} 2^{e}: eigenvalues are not 2^e times the unscaled ones"
        assert np.array_equal(cs, c), f"{name} 2^{e} conv {convention}: curvature differs from the unscaled one"


# ---------------------------------------------------------------------------------------------------------------- errors
def test_errors(tbk):
    import torch

    kp = tbk.Evaluator.from_kdotp(np.array([[0, 0], [1, 0]], dtype=np.int32), np.stack([np.eye(2), np.diag([1.0, -1.0])]).astype(complex))
    with pytest.raises(tbk.TbkError):
        kp.berry_curvature([0.1, 0.2])
    kp.close()
    line = tbk.Evaluator(pack_arrays(np.array([[0], [1]], np.int32), np.ones((2, 2, 2), complex), np.zeros((2, 1))))
    with pytest.raises(tbk.TbkError):
        line.berry_curvature([0.1])
    line.close()
    ev = tbk.Evaluator(wl.synthetic(4, 6, seed=1))
    kd = torch.zeros((3, 3), dtype=torch.float64, device="cuda")
    for bad in (0, 3):
        with pytest.raises(ValueError):
            ev.berry_curvature([0.1, 0.2, 0.3], convention=bad)
        with pytest.raises(ValueError):
            ev.berry_curvature_device(kd, convention=bad)
    for bad in (-1e-8, float("nan")):
        with pytest.raises(ValueError):
            ev.berry_curvature([0.1, 0.2, 0.3], degen_tol=bad)
        with pytest.raises(ValueError):
            ev.berry_curvature_device(kd, degen_tol=bad)
    with pytest.raises(ValueError):
        ev.berry_curvature_device(kd, out_w=torch.empty((3, 5), dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        ev.berry_curvature_device(kd, out_c=torch.empty((3, 4, 2), dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        ev.berry_curvature_device(kd, out_c=torch.empty((3, 4, 3), dtype=torch.float32, device="cuda"))
    with pytest.raises(ValueError):
        ev.berry_curvature_device(kd, out_c=torch.empty((3, 3, 4), dtype=torch.float64, device="cuda").transpose(1, 2))
    w, c = ev.berry_curvature(np.zeros((0, 3)))
    assert w.shape == (0, 4) and c.shape == (0, 4, 3)
    w, c = ev.berry_curvature_device(torch.zeros((0, 3), dtype=torch.float64, device="cuda"))
    assert tuple(w.shape) == (0, 4) and tuple(c.shape) == (0, 4, 3)
    w, c = ev.berry_curvature([0.1, 0.2, 0.3])
    assert w.shape == (4,) and c.shape == (4, 3)
    ev.close()
