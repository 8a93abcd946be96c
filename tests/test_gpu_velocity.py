"""Band velocities dE_n/dk_d on the GPU (``Evaluator.band_velocity``, band_velocity.cu) on every kernel path.

* every dispatch class against the exact velocities of folded supercells (tests/velocity_reference.py):
  eigenvalues to ``C_EIG sqrt(N) eps rho``, velocities to ``C_VEL sqrt(N) eps S_d (1 + rho / g_n)``, S_d the velocity
  budget (a bound on ||dH/dk_d||), g_n the exact gap from n's cluster to the next cluster;
* the numpy oracle on the golden models, to ``1e-10 S_d (1 + rho / g_n)``;
* consistency (w bit-equal to eigh's, host / device and chunk sizes bit-equal, finite differences of eigenval),
  degenerate models (H (x) I_2, H = 0), power-of-two scaled models (bit-equal), argument errors.

Every check prints its worst ratio (``pytest -s``).
"""
import numpy as np
import pytest

from conftest import EIG_TOL, load_golden, packed_from
from oracle import exact_spectra as xs
from oracle import workloads as wl
from oracle.accuracy import C_EIG, EPS, check_eig, kset
from tbmodels_b200 import pack_arrays

import velocity_reference as vr

pytestmark = [
    pytest.mark.gpu,
    pytest.mark.skipif(not xs.longdouble_is_extended(), reason="the exact references need an 80-bit np.longdouble"),
]

C_VEL = 4.0  # velocities: units of sqrt(N) eps S_d (1 + rho / g_n); the worst path measured 0.39 (NVIDIA B200)


@pytest.fixture(scope="module")
def tbk():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import tbmodels_b200

    return tbmodels_b200


def check_vel(got, want, w_exact, S, what, c=C_VEL, unit=None):
    """``|got - want| <= c unit S_d (1 + rho / g_n)``; ``unit`` defaults to ``sqrt(N) eps``."""
    got = np.asarray(got, dtype=np.float64)
    assert got.shape == want.shape, f"{what}: shape {got.shape} != {want.shape}"
    assert np.all(np.isfinite(got)), f"{what}: velocities not finite"
    w64 = np.asarray(w_exact, dtype=np.float64)
    n = w64.shape[-1]
    rho = float(np.abs(w64).max())
    g = np.array([vr.cluster_gaps(row, 1e-8) for row in w64])
    label = "sqrt(N) eps" if unit is None else f"{unit:g}"
    unit = np.sqrt(n) * EPS if unit is None else unit
    bound = unit * np.maximum(S, 1e-300)[None, None, :] * (1 + rho / g[:, :, None])
    ratio = float((np.abs(got.astype(np.longdouble) - want).astype(np.float64) / bound).max())
    print(f"[velocity] {what}: vel err {ratio:.3g} x {label} S_d (1 + rho / g)")
    assert ratio <= c, f"{what}: velocity error {ratio:.2f} > {c:g} units of S_d (1 + rho / g)"
    return ratio


# ------------------------------------------------------------------------- folded supercells through the default dispatch
# the (base, size) list of test_gpu_accuracy.py: trigonometric-product kernel (N <= 2), fused small kernel (N <= 8), GEMM
# + eigh up to N = 808; b1r has exactly degenerate folded spectra at Gamma and the zone boundary
FOLDED = [
    ("b1", (3, 1, 1)), ("b1", (2, 2, 1)), ("b1", (5, 1, 1)), ("b1", (3, 2, 1)), ("b1", (7, 1, 1)), ("b1", (2, 2, 2)),
    ("b1", (3, 3, 1)), ("b1", (3, 2, 2)), ("b1", (4, 4, 2)), ("b1", (11, 3, 1)), ("b1r", (3, 3, 4)), ("b1", (4, 4, 4)),
    ("b1", (41, 2, 1)), ("b1", (83, 1, 1)), ("b1r", (5, 5, 5)), ("b1", (8, 4, 4)), ("b1", (43, 3, 1)), ("b1", (5, 5, 8)),
    ("b1r", (8, 8, 4)), ("b1", (7, 7, 7)), ("b1", (8, 8, 8)), ("b1", (10, 10, 6)), ("b1", (9, 9, 9)), ("b1", (8, 101, 1)),
    ("b1", (1, 1, 1)), ("b2", (1, 1)), ("b2-3d", (1, 1, 1)), ("b2", (2, 2)), ("b2", (4, 4)), ("b2", (6, 6)), ("b2", (8, 8)), ("b2-3d", (2, 2, 2)), ("b2-3d", (3, 3, 2)),
    ("b2-3d", (4, 4, 4)),
] + [("b1-600", (3, 3, 1)), ("b2-1500", (2, 2, 2)), ("b1-3000", (3, 3, 4)), ("b2-3000", (3, 3, 2)), ("b1-4000", (4, 4, 4))]
# the last five: long-range bases whose supercells have 138 .. 309 stored R, so their H(k) runs on the INT8 digit GEMM by
# default (>= 81 stored R; tests/test_gpu_hk_int8_exact.py checks that it does)
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


def _fold_id(case):
    base, size = case
    return f"{base}-{'x'.join(map(str, size))}"


@pytest.mark.parametrize("case", FOLDED, ids=[_fold_id(c) for c in FOLDED])
def test_folded_supercell_velocities(tbk, case):
    """Device-packed (host and device entry points) and host-packed supercells against the exact velocities."""
    import torch

    name, size = case
    base = BASES[name]()
    sup = wl.supercell(base, size)
    n = sup.size
    K = kset(base.dim, n_random=9 if n <= 8 else (3 if n <= 300 else 1), seed=n)
    want_w, want_v = vr.folded_velocities(base, size, K)
    S = vr.velocity_budget(sup)
    dev = tbk.Evaluator.from_supercell(base, size)
    w, v = dev.band_velocity(K)
    check_eig(w, want_w, f"N={n} {name} device-packed")
    check_vel(v, want_v, want_w, S, f"N={n} {name} device-packed")
    wd, vd = dev.band_velocity_device(torch.from_numpy(K).cuda())
    dev.check()
    assert np.array_equal(wd.cpu().numpy(), w) and np.array_equal(vd.cpu().numpy(), v), "host and device entry points differ"
    dev.close()
    host = tbk.Evaluator(sup)
    w, v = host.band_velocity(K)
    host.close()
    check_eig(w, want_w, f"N={n} {name} host-packed")
    check_vel(v, want_v, want_w, S, f"N={n} {name} host-packed")


# ------------------------------------------------------------------------------------------------- oracle parity (goldens)
def _golden_models():
    d = load_golden("synthetic.npz")
    out = []
    for tag in ("n3", "n5", "n7", "n12", "n17", "n33", "c3", "c5s"):
        n_orb, n_half = (int(x) for x in d[f"{tag}_shape"])
        out.append((f"synthetic-{tag}", (wl.synthetic(n_orb, n_half, seed=1234), d[f"{tag}_k"][:8])))
    s = load_golden("silicon.npz")
    out.append(("silicon", (packed_from(s), s["k"][:16])))
    h = load_golden("haldane.npz")
    out.append(("haldane", (packed_from(h), h["k"][:64])))
    return out


GOLDEN = [m[0] for m in _golden_models()]


@pytest.mark.parametrize("name", GOLDEN)
def test_oracle_parity(tbk, name):
    p, k = dict(_golden_models())[name]
    ow, ov = vr.band_velocity(p.R, p.hop, p.pos, k)
    ev = tbk.Evaluator(p)
    w, v = ev.band_velocity(k)
    ev.close()
    rho = float(np.abs(ow).max())
    assert np.abs(w - ow).max() <= EIG_TOL * rho, f"{name}: eigenvalues beyond the north-star bound"
    check_vel(v, ov, ow, vr.velocity_budget(p), f"oracle {name}", c=1.0, unit=1e-10)


# ------------------------------------------------------------------------------------------------------------ consistency
CONSISTENCY = {
    "haldane-basis": lambda: packed_from(load_golden("haldane.npz")),
    "syn5-small": lambda: wl.synthetic(5, 13, seed=7),
    "syn12-gemm": lambda: wl.synthetic(12, 20, seed=8),
    "syn36-gemm": lambda: wl.synthetic(36, 60, seed=12),
    "syn90-gemm": lambda: wl.synthetic(90, 20, seed=13),
}


@pytest.mark.parametrize("name", list(CONSISTENCY))
def test_consistency(tbk, monkeypatch, name):
    """w bit-equal to eigh's; host and device entry points bit-equal; a 1 MB workspace (many chunks) bit-equal to the
    default; well-separated bands within 1e-6 S_d of central differences of eigenval (h = 1e-5)."""
    import torch

    p = CONSISTENCY[name]()
    k = np.random.default_rng(3).uniform(-1, 1, (37, p.dim))
    ev = tbk.Evaluator(p)
    w, v = ev.band_velocity(k)
    we, _ = ev.eigh(k)
    assert np.array_equal(w, we), f"{name}: w differs from eigh's"
    wd, vd = ev.band_velocity_device(torch.from_numpy(k).cuda())
    ev.check()
    assert np.array_equal(wd.cpu().numpy(), w) and np.array_equal(vd.cpu().numpy(), v), f"{name}: host != device"
    cols = []
    for d in range(p.dim):
        e = np.zeros(p.dim)
        e[d] = 1e-5
        cols.append((ev.eigenval_array(k + e) - ev.eigenval_array(k - e)) / 2e-5)
    ev.close()
    fd = np.stack(cols, axis=-1)
    gaps = np.minimum(np.diff(w, axis=1, prepend=-np.inf), np.diff(w, axis=1, append=np.inf))
    ok = gaps > 1e-2 * np.abs(w).max()
    S = vr.velocity_budget(p)
    ratio = float((np.abs(v - fd)[ok] / S).max())
    print(f"[velocity] {name}: vs finite differences of eigenval {ratio:.2e} S_d")
    assert ratio <= 1e-6
    monkeypatch.setenv("TBK_WORKSPACE_MB", "1")
    small = tbk.Evaluator(p)
    w1, v1 = small.band_velocity(k)
    small.close()
    assert np.array_equal(w1, w) and np.array_equal(v1, v), f"{name}: results depend on the chunk size"


# ---------------------------------------------------------------------------------------------------- degenerate models
def _doubled(p):
    hop = np.stack([np.kron(h, np.eye(2)) for h in p.hop])
    return pack_arrays(p.R, hop, np.repeat(p.pos, 2, axis=0))


@pytest.mark.parametrize("n", [8, 36, 128])
def test_doubled_model(tbk, n):
    """H (x) I_2: every eigenvalue exactly doubly degenerate; the velocities come in equal pairs, those of H."""
    base = wl.synthetic(n // 2, 13, seed=n)
    p = _doubled(base)
    k = np.random.default_rng(n).uniform(-1, 1, (5, 3))
    ev = tbk.Evaluator(p)
    w, v = ev.band_velocity(k)
    ev.close()
    bw, bv = vr.band_velocity(base.R, base.hop, base.pos, k)
    S = vr.velocity_budget(base)
    rho = float(np.abs(bw).max())
    assert np.abs(w[:, 0::2] - bw).max() <= EIG_TOL * rho and np.abs(w[:, 1::2] - bw).max() <= EIG_TOL * rho
    for half in (0, 1):
        check_vel(v[:, half::2], bv, bw, S, f"H x I2 N={n} member {half}", c=1.0, unit=1e-10)
    pair = float((np.abs(v[:, 0::2] - v[:, 1::2]) / S).max())
    print(f"[velocity] H x I2 N={n}: pair members differ by {pair:.2e} S_d")
    assert pair <= 64 * np.sqrt(n) * EPS


@pytest.mark.parametrize("n", [1, 4, 40])
def test_zero_model(tbk, n):
    """H = 0: one cluster of size N, all velocities zero."""
    p = pack_arrays(np.array([[0, 0, 0], [1, 0, 0]], np.int32), np.zeros((2, n, n), complex), np.zeros((n, 3)))
    ev = tbk.Evaluator(p)
    w, v = ev.band_velocity(np.random.default_rng(0).random((5, 3)))
    ev.close()
    assert w.shape == (5, n) and v.shape == (5, n, 3)
    assert not w.any() and not v.any()


# ----------------------------------------------------------------------------------------------------------------- scale
SCALE_MODELS = {
    "b1-2x2x2": lambda: wl.supercell(xs.band1(3), (2, 2, 2)),
    "b2-basis": lambda: xs.band2(2, 4),
    "syn36": lambda: wl.synthetic(36, 30, seed=4),
    "b1r-3x3x4": lambda: wl.supercell(xs.band1(3, real=True, seed=4), (3, 3, 4)),
}


@pytest.mark.parametrize("e", [-600, 600])
@pytest.mark.parametrize("name", list(SCALE_MODELS))
def test_scaled_models_bitwise(tbk, name, e):
    p = SCALE_MODELS[name]()
    k = kset(p.dim, n_random=5, seed=2)
    ev = tbk.Evaluator(p)
    w, v = ev.band_velocity(k)
    ev.close()
    ev = tbk.Evaluator(xs.scaled(p, e))
    ws, vs = ev.band_velocity(k)
    ev.close()
    assert np.array_equal(ws, np.ldexp(w, e)), f"{name} 2^{e}: eigenvalues are not 2^e times the unscaled ones"
    assert np.array_equal(vs, np.ldexp(v, e)), f"{name} 2^{e}: velocities are not 2^e times the unscaled ones"


# ---------------------------------------------------------------------------------------------------------------- errors
def test_errors(tbk):
    import torch

    kp = tbk.Evaluator.from_kdotp(np.array([[0, 0], [1, 0]], dtype=np.int32), np.stack([np.eye(2), np.diag([1.0, -1.0])]).astype(complex))
    with pytest.raises(tbk.TbkError):
        kp.band_velocity([0.1, 0.2])
    kp.close()
    ev = tbk.Evaluator(wl.synthetic(4, 6, seed=1))
    for bad in (-1e-8, float("nan")):
        with pytest.raises(ValueError):
            ev.band_velocity([0.1, 0.2, 0.3], degen_tol=bad)
        with pytest.raises(ValueError):
            ev.band_velocity_device(torch.zeros((2, 3), dtype=torch.float64, device="cuda"), degen_tol=bad)
    kd = torch.zeros((3, 3), dtype=torch.float64, device="cuda")
    with pytest.raises(ValueError):
        ev.band_velocity_device(kd, out_w=torch.empty((3, 5), dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        ev.band_velocity_device(kd, out_v=torch.empty((3, 4, 2), dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        ev.band_velocity_device(kd, out_v=torch.empty((3, 4, 3), dtype=torch.float32, device="cuda"))
    w, v = ev.band_velocity(np.zeros((0, 3)))
    assert w.shape == (0, 4) and v.shape == (0, 4, 3)
    w, v = ev.band_velocity([0.1, 0.2, 0.3])
    assert w.shape == (4,) and v.shape == (4, 3)
    ev.close()
