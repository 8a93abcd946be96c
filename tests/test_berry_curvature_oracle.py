"""The Berry-curvature references (tests/curvature_reference.py) pinned on the CPU: the numpy oracle against Berry phases
of small plaquettes of eigenvectors of ``hamilton(..., convention)`` (which fixes the sign and the convention-1 term), the
two-band closed forms against the oracle, the folded-supercell identity in longdouble, Chern numbers of the Haldane model,
the sum rule, the Cartesian conversion and the cluster semantics."""
import numpy as np
import pytest

from conftest import gpu_available, load_golden, packed_from
from oracle import exact_spectra as xs
from oracle import tb_oracle as orc
from oracle import workloads as wl
from tbmodels_b200 import pack_arrays

import curvature_reference as cr
import velocity_reference as vr

CONVENTIONS = (1, 2)


def _plaquette_curvature(p, k, convention, a, b, h=1e-4):
    """``[n_k, N]`` Berry phase of the counter-clockwise square of side h around k in the (a, b) plane, over h^2, from the
    eigenvectors of ``hamilton(k, convention)`` (A = i <u|grad u>: phase = -Im log prod <u_i|u_i+1>)."""
    ea = np.zeros(p.dim)
    eb = np.zeros(p.dim)
    ea[a] = h / 2
    eb[b] = h / 2
    corners = [-ea - eb, ea - eb, ea + eb, -ea + eb]
    vecs = [np.linalg.eigh(orc.hamilton(p.R, p.hop, p.pos, k + c, convention))[1] for c in corners]
    prod = np.ones((k.shape[0], p.size), dtype=complex)
    for i in range(4):
        prod *= np.einsum("kin,kin->kn", vecs[i].conj(), vecs[(i + 1) % 4])
    return -np.angle(prod) / (h * h)


def _curv_scale(p, convention, w, degen_tol=1e-8):
    """``[n_k, N, P]`` ``S_a S_b / g_n^2`` (g_n the gap from n's cluster to the next cluster)."""
    S = cr.curvature_budget(p, convention)
    g = np.array([vr.cluster_gaps(row, degen_tol) for row in np.asarray(w, dtype=np.float64)])
    sab = np.array([S[a] * S[b] for a, b in cr.pairs(p.dim)])
    return sab[None, None, :] / (g[:, :, None] ** 2)


PLAQUETTE_MODELS = {
    "haldane": lambda: packed_from(load_golden("haldane.npz")),
    "b2": lambda: xs.band2(2, 4),
    "b2-3d": lambda: xs.band2(3, 13, seed=4),
    "syn5": lambda: wl.synthetic(5, 9, seed=3),
    "syn12": lambda: wl.synthetic(12, 13, seed=5),
}


@pytest.mark.parametrize("convention", CONVENTIONS)
@pytest.mark.parametrize("name", list(PLAQUETTE_MODELS))
def test_oracle_against_plaquettes(name, convention):
    """Well-separated bands (gap to both neighbours > 1e-2 rho): oracle within 1e-5 S_a S_b / g^2 of the plaquette phase."""
    p = PLAQUETTE_MODELS[name]()
    k = np.random.default_rng(11).uniform(-1, 1, (4, p.dim))
    w, c = cr.berry_curvature(p.R, p.hop, p.pos, k, convention)
    gaps = np.minimum(np.diff(w, axis=1, prepend=-np.inf), np.diff(w, axis=1, append=np.inf))
    ok = gaps > 1e-2 * np.abs(w).max(axis=1, keepdims=True)
    assert ok.sum() >= w.size // 4, f"{name}: too few well-separated bands to test"
    scale = _curv_scale(p, convention, w)
    worst = 0.0
    for q, (a, b) in enumerate(cr.pairs(p.dim)):
        ph = _plaquette_curvature(p, k, convention, a, b)
        worst = max(worst, float((np.abs(c[:, :, q] - ph) / scale[:, :, q])[ok].max()))
    print(f"[curvature] {name} convention {convention}: oracle vs plaquettes {worst:.2e} S_a S_b / g^2")
    assert worst <= 1e-5


def test_conventions_differ():
    """band2 has distinct orbital positions: its local curvature depends on the convention."""
    p = xs.band2(2, 4)
    k = np.random.default_rng(5).uniform(-1, 1, (4, 2))
    _, c1 = cr.berry_curvature(p.R, p.hop, p.pos, k, 1)
    _, c2 = cr.berry_curvature(p.R, p.hop, p.pos, k, 2)
    assert np.abs(c1 - c2).max() > 1e-3 * np.abs(c2).max()


@pytest.mark.skipif(not xs.longdouble_is_extended(), reason="the exact references need an 80-bit np.longdouble")
@pytest.mark.parametrize("convention", CONVENTIONS)
@pytest.mark.parametrize("name", ["b2", "b2-3d"])
def test_closed_forms(name, convention):
    p = PLAQUETTE_MODELS[name]()
    k = np.random.default_rng(2).uniform(-1, 1, (6, p.dim))
    w, c = cr.berry_curvature(p.R, p.hop, p.pos, k, convention)
    exact = cr.base_curvature(p, k, convention).astype(np.float64)
    r = float((np.abs(c - exact) / _curv_scale(p, convention, w)).max())
    print(f"[curvature] closed form {name} convention {convention}: {r:.2e} S_a S_b / g^2")
    assert r <= 1e-12


FOLDED = [("b1", (3, 1, 1)), ("b1r", (3, 3, 2)), ("b2", (2, 2)), ("b2", (3, 1)), ("b2-3d", (2, 2, 1))]
BASES = {
    "b1": lambda: xs.band1(3),
    "b1r": lambda: xs.band1(3, real=True, seed=4),
    "b2": lambda: xs.band2(2, 4),
    "b2-3d": lambda: xs.band2(3, 13, seed=4),
}


@pytest.mark.skipif(not xs.longdouble_is_extended(), reason="the exact references need an 80-bit np.longdouble")
@pytest.mark.parametrize("convention", CONVENTIONS)
@pytest.mark.parametrize("case", FOLDED, ids=[f"{c[0]}-{'x'.join(map(str, c[1]))}" for c in FOLDED])
def test_folded_identity(case, convention):
    """folded_curvature against the oracle on the dense supercell: every member in convention 1 (X is block-diagonal in
    the base momentum), singletons and cluster traces in convention 2 (cross-block clusters have non-diagonal F)."""
    name, size = case
    base = BASES[name]()
    sup = wl.supercell(base, size)
    K = np.concatenate([np.zeros((1, base.dim)), np.full((1, base.dim), 0.5),
                        np.random.default_rng(7).uniform(-1, 1, (3, base.dim))])
    w, c = cr.folded_curvature(base, size, K, convention)
    ow, oc = cr.berry_curvature(sup.R, sup.hop, sup.pos, K, convention)
    scale = _curv_scale(sup, convention, w.astype(np.float64))
    err = np.abs((oc - c).astype(np.float64)) / scale
    if convention == 2:
        for i in range(K.shape[0]):
            for s, t in vr.clusters(w[i].astype(np.float64), 1e-8):
                if t - s > 1:
                    err[i, s:t] = np.abs((oc[i, s:t].sum(axis=0) - c[i, s:t].sum(axis=0)).astype(np.float64)) / scale[i, s]
    r = float(err.max())
    print(f"[curvature] folded {name} {size} convention {convention}: oracle {r:.2e} S_a S_b / g^2")
    assert r <= 1e-10
    assert np.abs(ow - w.astype(np.float64)).max() <= 1e-12 * np.abs(ow).max()


@pytest.mark.parametrize("convention", CONVENTIONS)
def test_haldane_chern_numbers(convention):
    """128^2 mid-point mesh: lower band C = -1, upper +1."""
    p = packed_from(load_golden("haldane.npz"))
    g = (np.arange(128) + 0.5) / 128
    k = np.stack(np.meshgrid(g, g, indexing="ij"), axis=-1).reshape(-1, 2)
    _, c = cr.berry_curvature(p.R, p.hop, p.pos, k, convention)
    chern = c[:, :, 0].sum(axis=0) / k.shape[0] / (2 * np.pi)
    print(f"[curvature] Haldane convention {convention}: Chern numbers {chern}")
    np.testing.assert_allclose(chern, [-1.0, 1.0], atol=1e-10)


@pytest.mark.parametrize("convention", CONVENTIONS)
@pytest.mark.parametrize("name", ["silicon", "syn12"])
def test_sum_rule(name, convention):
    p = packed_from(load_golden("silicon.npz")) if name == "silicon" else PLAQUETTE_MODELS[name]()
    k = np.random.default_rng(4).uniform(-1, 1, (5, p.dim))
    w, c = cr.berry_curvature(p.R, p.hop, p.pos, k, convention)
    r = float((np.abs(c.sum(axis=1)) / _curv_scale(p, convention, w).max(axis=1)).max())
    assert r <= 1e-12


def test_cartesian_conversion():
    """uc^T Omega_red uc / (4 pi^2) against plaquettes in Cartesian k on a sheared lattice (k_red = k_cart @ uc.T / (2 pi))."""
    p = packed_from(load_golden("haldane.npz"))
    uc = np.array([[1.0, 0.0], [0.45, 0.9]])
    kc = np.random.default_rng(8).uniform(-3, 3, (4, 2))
    w, c = cr.berry_curvature(p.R, p.hop, p.pos, kc @ uc.T / (2 * np.pi), 2)
    om = np.zeros((kc.shape[0], p.size, 2, 2))
    om[..., 0, 1] = c[..., 0]
    om[..., 1, 0] = -c[..., 0]
    cart = np.einsum("xa,knab,by->knxy", uc.T, om, uc) / (4 * np.pi ** 2)
    h = 1e-4
    corners = [np.array(v) * h / 2 for v in ((-1, -1), (1, -1), (1, 1), (-1, 1))]
    vecs = [np.linalg.eigh(orc.hamilton(p.R, p.hop, p.pos, (kc + d) @ uc.T / (2 * np.pi)))[1] for d in corners]
    prod = np.ones((kc.shape[0], p.size), dtype=complex)
    for i in range(4):
        prod *= np.einsum("kin,kin->kn", vecs[i].conj(), vecs[(i + 1) % 4])
    ph = -np.angle(prod) / (h * h)
    scale = np.abs(cart[..., 0, 1]).max()
    assert np.abs(cart[..., 0, 1] - ph).max() <= 1e-6 * scale
    np.testing.assert_allclose(cart[..., 1, 0], -cart[..., 0, 1])


def _doubled(p):
    """H (x) I_2: every orbital twice, every eigenvalue exactly doubly degenerate."""
    hop = np.stack([np.kron(h, np.eye(2)) for h in p.hop])
    return pack_arrays(p.R, hop, np.repeat(p.pos, 2, axis=0))


@pytest.mark.parametrize("convention", CONVENTIONS)
def test_cluster_semantics_doubled_model(convention):
    """H (x) I_2: the curvatures come in equal pairs, those of H."""
    p = wl.synthetic(5, 9, seed=3)
    k = np.random.default_rng(1).uniform(-1, 1, (5, 3))
    w, c = cr.berry_curvature(p.R, p.hop, p.pos, k, convention)
    q = _doubled(p)
    w2, c2 = cr.berry_curvature(q.R, q.hop, q.pos, k, convention)
    scale = _curv_scale(p, convention, w)
    assert np.abs(w2[:, 0::2] - w).max() <= 1e-13 * np.abs(w).max()
    for half in (0, 1):
        assert (np.abs(c2[:, half::2] - c) / scale).max() <= 1e-12


def test_zero_and_one_band_models():
    p = pack_arrays(np.array([[0, 0, 0], [1, 0, 0]], np.int32), np.zeros((2, 4, 4), complex), np.zeros((4, 3)))
    w, c = cr.berry_curvature(p.R, p.hop, p.pos, np.random.default_rng(0).random((3, 3)), 1)
    assert c.shape == (3, 4, 3) and not w.any() and not c.any()
    b = xs.band1(2)
    _, c = cr.berry_curvature(b.R, b.hop, b.pos, np.random.default_rng(0).random((3, 2)), 2)
    assert c.shape == (3, 1, 1) and not c.any()


def test_berry_curvature_without_gpu_is_an_error():
    """No CPU fallback: without a CUDA device the call fails with TBK_E_CUDA (the handle cannot be created)."""
    if gpu_available():
        pytest.skip("GPU present")
    import tbmodels_b200 as tbk
    from tbmodels_b200 import _capi

    with pytest.raises(tbk.TbkError) as exc:
        tbk.KModel.from_packed(packed_from(load_golden("haldane.npz"))).berry_curvature([0.1, 0.2])
    assert exc.value.code == _capi.TBK_E_CUDA
    with pytest.raises(tbk.TbkError) as exc:
        tbk.KModel.from_packed(packed_from(load_golden("haldane.npz"))).berry_curvature([0.1, 0.2], convention=1)
    assert exc.value.code == _capi.TBK_E_CUDA
