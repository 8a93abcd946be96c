"""The band-velocity references (tests/velocity_reference.py) pinned on the CPU: the numpy oracle against finite
differences of the eigenvalue oracle, the exact folded-supercell velocities against longdouble finite differences and
against the oracle, the cluster semantics on models with known degeneracies, and the Cartesian conversion."""
import numpy as np
import pytest

from conftest import gpu_available, load_golden, packed_from
from oracle import exact_spectra as xs
from oracle import tb_oracle as orc
from oracle import workloads as wl
from tbmodels_b200 import pack_arrays

import velocity_reference as vr

EPS = np.finfo(np.float64).eps


def _golden_models():
    out = []
    d = load_golden("synthetic.npz")
    for tag in ("n3", "n5", "n7", "n12", "n17", "n33", "c3", "c5s"):
        n_orb, n_half = (int(x) for x in d[f"{tag}_shape"])
        out.append((f"synthetic-{tag}", lambda n_orb=n_orb, n_half=n_half, tag=tag: (
            wl.synthetic(n_orb, n_half, seed=1234), load_golden("synthetic.npz")[f"{tag}_k"][:3])))
    out.append(("silicon", lambda: (packed_from(load_golden("silicon.npz")), load_golden("silicon.npz")["k"][:4])))
    out.append(("haldane", lambda: (packed_from(load_golden("haldane.npz")), load_golden("haldane.npz")["k"][:8])))
    return out


GOLDEN_MODELS = dict(_golden_models())


def _central_differences(eig_fn, k, h):
    """``[n_k, N, dim]`` central differences of ``eig_fn`` (``[n_k, dim] -> [n_k, N]``) in every direction."""
    cols = []
    for d in range(k.shape[1]):
        e = np.zeros(k.shape[1])
        e[d] = h
        cols.append((eig_fn(k + e) - eig_fn(k - e)) / (2 * h))
    return np.stack(cols, axis=-1)


@pytest.mark.parametrize("name", list(GOLDEN_MODELS))
def test_oracle_against_finite_differences(name):
    """Well-separated bands (gap to both neighbours > 1e-2 rho): oracle within 1e-7 S_d of central differences, h = 1e-5."""
    p, k = GOLDEN_MODELS[name]()
    w, v = vr.band_velocity(p.R, p.hop, p.pos, k)
    fd = _central_differences(lambda kk: orc.eigenval_array(p.R, p.hop, p.pos, kk), k, 1e-5)
    S = vr.velocity_budget(p)
    rho = np.abs(w).max(axis=1, keepdims=True)
    gaps = np.minimum(np.diff(w, axis=1, prepend=-np.inf), np.diff(w, axis=1, append=np.inf))
    ok = gaps > 1e-2 * rho
    assert ok.sum() >= w.size // 4, f"{name}: too few well-separated bands to test"
    ratio = float((np.abs(v - fd)[ok] / S).max())
    print(f"[velocity] {name}: oracle vs finite differences {ratio:.2e} S_d")
    assert ratio <= 1e-7


def _base_fd_longdouble(base, size, K, h):
    """Central differences in K of the folded spectrum with longdouble momenta (``[n_k, N, dim]``, longdouble)."""
    size_l = np.asarray(size, dtype=xs.LD)
    offs = xs.cell_offsets(size).astype(xs.LD)

    def spectrum(Kl):
        kb = ((Kl[:, None, :] + offs[None]) / size_l).reshape(-1, base.dim)
        return np.sort(xs.base_eigenvalues(base, kb).reshape(Kl.shape[0], -1), axis=1)

    Kl = np.asarray(K).astype(xs.LD)
    cols = []
    for d in range(base.dim):
        e = np.zeros(base.dim, dtype=xs.LD)
        e[d] = xs.LD(h)
        cols.append((spectrum(Kl + e) - spectrum(Kl - e)) / (2 * xs.LD(h)))
    return np.stack(cols, axis=-1)


BASES = {
    "b1": lambda: xs.band1(3),
    "b1r": lambda: xs.band1(3, real=True, seed=4),
    "b2": lambda: xs.band2(2, 4),
    "b2-3d": lambda: xs.band2(3, 13, seed=4),
}
FOLDED = [("b1", (3, 1, 1)), ("b1", (2, 2, 1)), ("b1r", (3, 3, 4)), ("b1r", (4, 4, 2)), ("b2", (1, 1)), ("b2", (2, 2)),
          ("b2-3d", (2, 2, 2))]


@pytest.mark.skipif(not xs.longdouble_is_extended(), reason="the exact references need an 80-bit np.longdouble")
@pytest.mark.parametrize("case", FOLDED, ids=[f"{c[0]}-{'x'.join(map(str, c[1]))}" for c in FOLDED])
def test_folded_velocities(case):
    """folded_velocities against longdouble central differences (random K, non-degenerate bands) and against the oracle
    on the dense supercell (K including Gamma and the zone boundary, where b1r's folded spectra are degenerate in pairs
    with velocities +-v)."""
    name, size = case
    base = BASES[name]()
    sup = wl.supercell(base, size)
    S = vr.velocity_budget(sup)
    K = np.random.default_rng(7).uniform(-1, 1, (4, base.dim))
    w, v = vr.folded_velocities(base, size, K)
    fd = _base_fd_longdouble(base, size, K, 1e-6)
    rho = np.abs(w.astype(np.float64)).max(axis=1, keepdims=True)
    wf = w.astype(np.float64)
    gaps = np.minimum(np.diff(wf, axis=1, prepend=-np.inf), np.diff(wf, axis=1, append=np.inf))
    ok = gaps > 1e-4 * rho
    ratio = float((np.abs((v - fd).astype(np.float64))[ok] / S).max())
    print(f"[velocity] folded {name} {size}: vs longdouble finite differences {ratio:.2e} S_d")
    assert ratio <= 1e-9

    K = np.concatenate([np.zeros((1, base.dim)), np.full((1, base.dim), 0.5), K])
    w, v = vr.folded_velocities(base, size, K)
    ow, ov = vr.band_velocity(sup.R, sup.hop, sup.pos, K)
    n = sup.size
    rho = float(np.abs(w.astype(np.float64)).max())
    g = np.array([vr.cluster_gaps(row, 1e-8) for row in w.astype(np.float64)])
    bound = np.sqrt(n) * EPS * S[None, None, :] * (1 + rho / g[:, :, None])
    r = float((np.abs((ov - v).astype(np.float64)) / bound).max())
    print(f"[velocity] folded {name} {size}: oracle {r:.2f} sqrt(N) eps S_d (1 + rho / g)")
    assert r <= 64
    if name == "b1r":  # degenerate pairs at Gamma: +-v
        assert np.any(np.abs(np.diff(w[0].astype(np.float64))) <= 1e-12 * rho)
        np.testing.assert_allclose(np.sort(v[0].astype(np.float64).sum(axis=0)), 0, atol=1e-9 * S.max() * n)


def _doubled(p):
    """H (x) I_2: every orbital twice, every eigenvalue exactly doubly degenerate."""
    hop = np.stack([np.kron(h, np.eye(2)) for h in p.hop])
    return pack_arrays(p.R, hop, np.repeat(p.pos, 2, axis=0))


def test_cluster_semantics_doubled_model():
    """H (x) I_2: the velocities come in equal pairs, those of H."""
    p = wl.synthetic(5, 9, seed=3)
    k = np.random.default_rng(1).uniform(-1, 1, (5, 3))
    w, v = vr.band_velocity(p.R, p.hop, p.pos, k)
    w2, v2 = vr.band_velocity(*(lambda q: (q.R, q.hop, q.pos))(_doubled(p)), k)
    S = vr.velocity_budget(p)
    assert np.abs(w2[:, 0::2] - w).max() <= 1e-13 * np.abs(w).max()
    assert np.abs(v2[:, 0::2] - v).max() <= 1e-12 * S.max()
    assert np.abs(v2[:, 1::2] - v).max() <= 1e-12 * S.max()


def test_cluster_semantics_zero_model():
    p = pack_arrays(np.zeros((1, 3), np.int32), np.zeros((1, 4, 4), complex), np.zeros((4, 3)))
    w, v = vr.band_velocity(p.R, p.hop, p.pos, np.random.default_rng(0).random((3, 3)))
    assert not w.any() and not v.any()


def test_cartesian_conversion():
    """v @ uc / (2 pi) against central differences in Cartesian k (k_red = k_cart @ uc.T / (2 pi))."""
    p = packed_from(load_golden("silicon.npz"))
    uc = np.array([[0.0, 2.7, 2.7], [2.7, 0.0, 2.7], [2.7, 2.7, 0.3]])
    kc = np.random.default_rng(2).uniform(-1, 1, (3, 3))
    w, v = vr.band_velocity(p.R, p.hop, p.pos, kc @ uc.T / (2 * np.pi))
    fd = _central_differences(lambda kk: orc.eigenval_array(p.R, p.hop, p.pos, kk @ uc.T / (2 * np.pi)), kc, 1e-5)
    gaps = np.minimum(np.diff(w, axis=1, prepend=-np.inf), np.diff(w, axis=1, append=np.inf))
    ok = gaps > 1e-3 * np.abs(w).max()
    scale = vr.velocity_budget(p).max() * np.abs(uc).max()
    assert np.abs((v @ uc / (2 * np.pi) - fd)[ok]).max() <= 1e-7 * scale


def test_band_velocity_without_gpu_is_an_error():
    """No CPU fallback: without a CUDA device the call fails with TBK_E_CUDA (the handle cannot be created)."""
    if gpu_available():
        pytest.skip("GPU present")
    import tbmodels_b200 as tbk
    from tbmodels_b200 import _capi

    with pytest.raises(tbk.TbkError) as exc:
        tbk.KModel.from_packed(packed_from(load_golden("haldane.npz"))).band_velocity([0.1, 0.2])
    assert exc.value.code == _capi.TBK_E_CUDA
