"""H(k) built from exact INT8 tensor-core digit products (hk_gemm_i8.cu), the default build of the explicit-k entry
points of phase handles with N > 8 and at least 81 stored R (``TBK_HK_FP64=0`` forces it for the smaller models here).
``test_gpu_hk_int8_exact.py`` holds the same kernel to its bit-exact restatement; the budgets here bound the scheme.

- Elementwise against the longdouble Fourier sum within the budget of ``test_gpu_accuracy.py``, dense (host-packed
  synthetic models) and block-sparse (device-packed supercells), N = 9 .. 512, |k| <= 2 and ~1e3.
- Against the FP64 DMMA build (``TBK_HK_FP64=1``): both read the same phase bits, so they differ by the roundings of the
  two GEMMs only, a few eps sum_R (|T_R,ij| + |T_R,ji|).
- The bits of a k-point do not depend on the batch, its position in it or the chunking; all-zero columns are exact
  zeros; a model scaled by 2^e gives the same bits times 2^e.
"""
import numpy as np
import pytest

from oracle import exact_spectra as xs
from oracle import workloads as wl
from oracle.accuracy import EPS, check_h

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


@pytest.fixture(autouse=True)
def int8_build(monkeypatch):
    monkeypatch.setenv("TBK_HK_FP64", "0")


DENSE = {
    "n9": lambda: wl.synthetic(9, 30, seed=31),
    "n36": lambda: wl.synthetic(36, 60, seed=32),
    "n64-2d": lambda: wl.synthetic(64, 20, seed=33, dim=2),
    "n128": lambda: wl.synthetic(128, 12, seed=34),
    "n512": lambda: wl.synthetic(512, 3, seed=35),
}
SPARSE = {"n128-b2x4x4x4": (lambda: xs.band2(3, 13, seed=4), (4, 4, 4)), "n512-b1x8x8x8": (lambda: xs.band1(3), (8, 8, 8))}


def _sum_abs(p):
    A = np.abs(np.asarray(p.hop))
    return (A + A.transpose(0, 2, 1)).sum(axis=0)


@pytest.mark.parametrize("kscale", [2.0, 1e3])
@pytest.mark.parametrize("name", list(DENSE) + list(SPARSE))
def test_int8_hamilton_against_longdouble(tbk, name, kscale):
    from oracle import tb_oracle as orc

    if name in DENSE:
        p = DENSE[name]()
        ev = tbk.Evaluator(p)
    else:
        base, size = SPARSE[name]
        p = wl.supercell(base(), size)
        ev = tbk.Evaluator.from_supercell(base(), size)
    k = np.random.default_rng(len(name)).uniform(-kscale, kscale, (5 if p.size >= 512 else 17, p.dim))
    for conv in (1, 2):
        want = orc.hamilton_longdouble(p.R, p.hop, p.pos, k, conv)
        check_h(ev.hamilton(k, convention=conv), want, xs.hamilton_scale(p, k, conv), f"INT8 H {name} conv{conv} |k|<={kscale:g}")
    ev.close()


@pytest.mark.parametrize("name", list(DENSE))
def test_int8_against_fp64_build(tbk, monkeypatch, name):
    p = DENSE[name]()
    k = np.random.default_rng(7).uniform(-2.0, 2.0, (33, p.dim))
    ev = tbk.Evaluator(p)
    got = ev.hamilton(k)
    ev.close()
    monkeypatch.setenv("TBK_HK_FP64", "1")
    ev = tbk.Evaluator(p)
    ref = ev.hamilton(k)
    ev.close()
    S = _sum_abs(p)
    ratio = float((np.abs(got - ref) / (EPS * np.maximum(S, 1e-300))[None]).max())
    print(f"[accuracy] INT8 vs FP64 build {name}: {ratio:.2f} eps sum|T|")
    assert ratio <= 8.0, f"{name}: INT8 and FP64 builds differ by {ratio:.2f} eps sum|T|"
    assert not np.array_equal(got, ref), f"{name}: the two builds agree bit for bit -- is the INT8 GEMM in use?"


def test_default_build_by_k(tbk, monkeypatch):
    """Without TBK_HK_FP64 the INT8 GEMM serves models with >= 6 K steps of 32 rows (81 stored R) and DMMA the rest (the edge
    itself, 80 and 81 stored R, is in test_gpu_hk_int8_exact.py)."""
    k = np.random.default_rng(11).uniform(-2.0, 2.0, (40, 3))
    for n_half, int8 in ((60, False), (100, True)):
        p = wl.synthetic(36, n_half, seed=37)
        got = {}
        for env in ("0", "1", None):
            if env is None:
                monkeypatch.delenv("TBK_HK_FP64")
            else:
                monkeypatch.setenv("TBK_HK_FP64", env)
            ev = tbk.Evaluator(p)
            got[env] = ev.hamilton(k)
            ev.close()
        assert not np.array_equal(got["0"], got["1"])
        assert np.array_equal(got[None], got["0" if int8 else "1"]), f"{n_half} R: default is not the {'INT8' if int8 else 'DMMA'} build"


def test_int8_bits_independent_of_batch_and_chunk(tbk, monkeypatch):
    p = wl.synthetic(36, 60, seed=32)
    k = np.random.default_rng(8).uniform(-3.0, 3.0, (1000, p.dim))
    ev = tbk.Evaluator(p)
    H = ev.hamilton(k)
    w = ev.eigenval_array(k)
    for sl in (slice(0, 1), slice(47, 48), slice(48, 49), slice(5, 101), slice(313, 1000)):
        assert np.array_equal(ev.hamilton(k[sl]), H[sl]), f"H of k[{sl.start}:{sl.stop}] differs from the whole batch"
        assert np.array_equal(ev.eigenval_array(k[sl]), w[sl])
    ev.close()
    monkeypatch.setenv("TBK_WORKSPACE_MB", "1")  # chunks of a few hundred k-points, not multiples of the 48-point tile
    ev = tbk.Evaluator(p)
    assert np.array_equal(ev.hamilton(k), H)
    assert np.array_equal(ev.eigenval_array(k), w)
    ev.close()


def test_int8_zero_columns_are_exact_zeros(tbk):
    p = wl.synthetic(36, 20, seed=36)
    hop = np.array(p.hop)
    hop[:, 7, :] = 0.0
    hop[:, :, 7] = 0.0
    hop[:, 20, 3] = 0.0
    hop[:, 3, 20] = 0.0
    q = xs.pack_arrays(p.R, hop, p.pos)
    k = np.random.default_rng(9).uniform(-2.0, 2.0, (50, q.dim))
    ev = tbk.Evaluator(q)
    H = ev.hamilton(k)
    ev.close()
    assert np.all(H[:, 7, :] == 0) and np.all(H[:, :, 7] == 0)
    assert np.all(H[:, 20, 3] == 0) and np.all(H[:, 3, 20] == 0)
    assert np.count_nonzero(H[:, 0, :]) == 50 * 35


@pytest.mark.parametrize("e", [-600, -64, 64, 600])
def test_int8_scaled_models_bit_equal(tbk, e):
    p = wl.synthetic(36, 60, seed=32)
    k = np.random.default_rng(10).uniform(-2.0, 2.0, (97, p.dim))
    ev = tbk.Evaluator(p)
    H = ev.hamilton(k)
    ev.close()
    ev = tbk.Evaluator(xs.scaled(p, e))
    Hs = ev.hamilton(k)
    ev.close()
    assert np.array_equal(np.ldexp(Hs.real, -e) + 1j * np.ldexp(Hs.imag, -e), H)
