"""The persistent INT8 digit GEMM (hk_gemm_i8.cu: one CTA per SM, tiles taken round-robin, tensor memory handed
between the MMA issuer and the epilogue once per tile) at the edges of its scheduler.  Each case must give the bits of
the same k-points built in chunks of a few hundred (``TBK_WORKSPACE_MB=1``), where every launch has other tiles:

- 1, 47, 48 and 49 k-points (one or two k tiles, fewer tiles than SMs);
- 150 k tiles of 11 column tiles, a tile count that no grid of 148 divides;
- N = 9 (one column tile) and N = 512 (2048 column tiles per k tile, checked point by point against the batch);
- a model of 33 K steps, above the 31 up to which the epilogue's two-part combination is correctly rounded; it must
  also stay within a few eps sum|T| of the FP64 DMMA build.
"""
import numpy as np
import pytest

from oracle import workloads as wl
from oracle.accuracy import EPS

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def tbk():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import tbmodels_b200

    return tbmodels_b200


@pytest.fixture(autouse=True)
def int8_build(monkeypatch):
    monkeypatch.setenv("TBK_HK_FP64", "0")


def _hamilton(tbk, p, k):
    ev = tbk.Evaluator(p)
    H = ev.hamilton(k)
    ev.close()
    return H


def _same_bits_as_small_chunks(tbk, monkeypatch, p, k, what):
    H = _hamilton(tbk, p, k)
    monkeypatch.setenv("TBK_WORKSPACE_MB", "1")
    ref = _hamilton(tbk, p, k)
    monkeypatch.delenv("TBK_WORKSPACE_MB")
    assert np.all(np.isfinite(H))
    assert np.array_equal(H, ref), f"{what}: the persistent GEMM's bits depend on the launch"
    return H


@pytest.mark.parametrize("nk", [1, 47, 48, 49])
def test_few_k_points(tbk, monkeypatch, nk):
    p = wl.synthetic(36, 120, seed=41)
    k = np.random.default_rng(nk).uniform(-2.0, 2.0, (nk, 3))
    _same_bits_as_small_chunks(tbk, monkeypatch, p, k, f"nk = {nk}")


def test_tile_count_not_divisible_by_grid(tbk, monkeypatch):
    p = wl.synthetic(36, 120, seed=42)
    k = np.random.default_rng(2).uniform(-2.0, 2.0, (150 * 48, 3))
    _same_bits_as_small_chunks(tbk, monkeypatch, p, k, "1650 tiles")


def test_one_column_tile(tbk, monkeypatch):
    p = wl.synthetic(9, 100, seed=43)
    k = np.random.default_rng(9).uniform(-2.0, 2.0, (97, 3))
    _same_bits_as_small_chunks(tbk, monkeypatch, p, k, "N = 9")


def test_many_column_tiles(tbk):
    """N = 512: a single k-point already has more tiles than the grid; each k-point alone must give the batch's bits."""
    p = wl.synthetic(512, 3, seed=43)
    k = np.random.default_rng(512).uniform(-2.0, 2.0, (5, 3))
    ev = tbk.Evaluator(p)
    H = ev.hamilton(k)
    for i in range(len(k)):
        assert np.array_equal(ev.hamilton(k[i : i + 1]), H[i : i + 1]), f"N = 512, k-point {i}"
    ev.close()


def test_above_31_k_steps(tbk, monkeypatch):
    p = wl.synthetic(36, 520, seed=44)  # 521 stored R: 33 K steps of 32 rows
    k = np.random.default_rng(3).uniform(-2.0, 2.0, (200, 3))
    H = _same_bits_as_small_chunks(tbk, monkeypatch, p, k, "33 K steps")
    monkeypatch.setenv("TBK_HK_FP64", "1")
    ref = _hamilton(tbk, p, k)
    A = np.abs(np.asarray(p.hop))
    S = (A + A.transpose(0, 2, 1)).sum(axis=0)
    ratio = float((np.abs(H - ref) / (EPS * np.maximum(S, 1e-300))[None]).max())
    print(f"[accuracy] INT8 vs FP64 build, 33 K steps: {ratio:.2f} eps sum|T|")
    assert ratio <= 8.0
