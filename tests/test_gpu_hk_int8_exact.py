"""The INT8 H(k) build (hk_gemm_i8.cu) bit for bit against its restatement ``hk_digits_reference.hamilton_int8``.

The digit scheme is exact by construction: the class sums are integers, whose value does not depend on the order of
summation, and the epilogue is one fma and two power-of-two scalings.  The kernel's output is therefore a deterministic
function of the phase bits and the weights, and ``ev.hamilton(k, convention=2)`` must equal the restatement under
``np.array_equal``.  A budget test cannot see a lost low digit class (class 9 weighs 2^-75 of s_j per row); this can.

- Phase probe (FP64 DMMA build): a model whose H00 is cos(2 pi k.R) and H10 is cos + i sin with nothing else added
  gives the phase kernel's bits, which must be those of the host restatement (fma chain of k.R, ``sincospi_lean``).  A
  failure of the INT8 tests below can then be told apart: phases or GEMM.
- INT8 bits for N = 9 .. 512, 1 .. 2047 K steps of 32 rows, batches around the 48-point tile and across chunks, weight
  columns that are zero, live at one R, span 12 decades, sit at the top of a binade or are powers of two, models scaled
  by 2^+-600, and device-packed block-sparse supercells against the host pack.
- Gate edges: 80 stored R (5 K steps) runs DMMA by default and 81 (6) INT8; 2047 K steps runs INT8; 2048 falls back to
  DMMA even when ``TBK_HK_FP64=0`` asks for INT8.
- Every long-range folded supercell that the consumer tests (accuracy, velocities, curvature) add really takes the INT8
  build by default.
"""
import itertools

import numpy as np
import pytest

import hk_digits_reference as hd
from oracle import exact_spectra as xs
from oracle import workloads as wl
from tbmodels_b200._pack import pack_arrays

pytestmark = [
    pytest.mark.gpu,
    pytest.mark.skipif(not xs.longdouble_is_extended(), reason="the restated phases need an 80-bit np.longdouble"),
]


@pytest.fixture(scope="module")
def tbk():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import tbmodels_b200

    return tbmodels_b200


def ksets(dim, n=9, seed=0):
    """{kind: k}: Gamma; half and quarter points; random at |k| <= 2 and ~1e3; dyadic (every k.R exact)."""
    rng = np.random.default_rng(seed)
    hq = np.array(list(itertools.product([0.5, 0.25, -0.75], repeat=dim)))
    dyadic = rng.integers(-(2**20), 2**20, (n, dim)) * 2.0**-17
    return {"gamma": np.zeros((1, dim)), "half-quarter": hq, "random2": rng.uniform(-2, 2, (n, dim)),
            "random1e3": rng.uniform(-1e3, 1e3, (n, dim)), "dyadic": dyadic}


def all_k(dim, n=9, seed=0, few=False):
    """Every kind of :func:`ksets` in one batch; ``few``: 7 points (N >= 128, where the restatement is large)."""
    ks = ksets(dim, n, seed)
    if few:
        ks["half-quarter"] = ks["half-quarter"][[0, len(ks["half-quarter"]) // 2, -1]]
        ks = {kind: k[:1] if kind != "half-quarter" else k for kind, k in ks.items()}
    return np.concatenate(list(ks.values()))


def hamilton(tbk, monkeypatch, p, k, fp64=None, supercell=None):
    """H(k) (convention 2) of ``p`` (or of ``Evaluator.from_supercell(*supercell)``) with TBK_HK_FP64 = ``fp64``
    (None: the default choice)."""
    if fp64 is None:
        monkeypatch.delenv("TBK_HK_FP64", raising=False)
    else:
        monkeypatch.setenv("TBK_HK_FP64", str(fp64))
    ev = tbk.Evaluator.from_supercell(*supercell) if supercell else tbk.Evaluator(p)
    H = ev.hamilton(k, convention=2)
    ev.close()
    monkeypatch.delenv("TBK_HK_FP64", raising=False)
    return H


def assert_bits(got, want, what):
    assert got.shape == want.shape, f"{what}: shape {got.shape} != {want.shape}"
    if not np.array_equal(got, want):
        bad = np.argwhere(got != want)
        i = tuple(bad[0])
        d = np.abs(got - want)
        raise AssertionError(f"{what}: {len(bad)} of {got.size} elements differ from hamilton_int8, first at {i}: "
                             f"{got[i]!r} != {want[i]!r}; largest difference {d.max():.3e}")


# ---------------------------------------------------------------------------------------------------------- phase probe
@pytest.mark.parametrize("R", [(1, 0, 0), (1, 2, -3), (7, -11, 5), (-29, 0, 31)], ids=lambda r: "R" + "_".join(map(str, r)))
def test_phase_probe_fp64_build(tbk, monkeypatch, R):
    """N = 9, one stored R, T_R[0, 0] = 0.5 and T_R[1, 0] = 1: the DMMA GEMM multiplies the phases by 1 and adds zeros,
    so H00 = cos and H10 = cos + i sin of 2 pi k.R exactly, which must be the restated phase bits."""
    hop = np.zeros((1, 9, 9), dtype=complex)
    hop[0, 0, 0] = 0.5
    hop[0, 1, 0] = 1.0
    p = pack_arrays(np.array([R]), hop, np.zeros((9, 3)))
    for kind, k in ksets(3, n=33, seed=sum(R) & 0xFF).items():
        H = hamilton(tbk, monkeypatch, p, k, fp64=1)
        sn, cs = hd.sincospi(hd.phase_args(k, p.R))
        assert np.array_equal(H[:, 0, 0].real, cs[:, 0]), f"R {R} {kind}: cos differs from the host phases"
        assert np.array_equal(H[:, 1, 0].real, cs[:, 0]), f"R {R} {kind}: cos of H10 differs from the host phases"
        assert np.array_equal(H[:, 1, 0].imag, sn[:, 0]), f"R {R} {kind}: sin differs from the host phases"


# ----------------------------------------------------------------------------------------------------------- INT8 bits
# (id, model, k-points per k-set kind): N and the K steps of 32 rows (16 stored R each) the kernel runs
MODELS = {
    "n9-ks2": (lambda: wl.synthetic(9, 30, seed=31), 9),
    "n36-ks4": (lambda: wl.synthetic(36, 60, seed=32), 9),
    "n64-2d-ks2": (lambda: wl.synthetic(64, 20, seed=33, dim=2), 9),
    "n128-ks1": (lambda: wl.synthetic(128, 12, seed=34), 1),
    "n512-ks1": (lambda: wl.synthetic(512, 3, seed=35), 1),
    "n9-ks5": (lambda: wl.synthetic(9, 79, seed=36), 9),
    "n36-ks6": (lambda: wl.synthetic(36, 80, seed=37), 9),
    "n36-ks16": (lambda: wl.synthetic(36, 255, seed=38), 9),
    "n9-ks31": (lambda: wl.synthetic(9, 495, seed=39), 9),
    "n9-ks32": (lambda: wl.synthetic(9, 511, seed=40), 9),
    "n36-ks33": (lambda: wl.synthetic(36, 520, seed=41), 9),
    "n9-ks2047": (lambda: wl.synthetic(9, 32751, seed=42), 2),
}


def _ksteps(p):
    return (p.n_R + 15) // 16


@pytest.mark.parametrize("name", list(MODELS))
def test_int8_bits(tbk, monkeypatch, name):
    make, n = MODELS[name]
    p = make()
    assert f"ks{_ksteps(p)}" in name
    k = all_k(p.dim, n, seed=len(name), few=p.size >= 128)
    assert_bits(hamilton(tbk, monkeypatch, p, k, fp64=0), hd.hamilton_int8(p, k), f"{name} (N = {p.size}, {p.n_R} R)")


@pytest.mark.parametrize("nk", [1, 47, 48, 49])
def test_int8_bits_batches(tbk, monkeypatch, nk):
    p = wl.synthetic(36, 120, seed=43)
    k = np.random.default_rng(nk).uniform(-3, 3, (nk, 3))
    assert_bits(hamilton(tbk, monkeypatch, p, k, fp64=0), hd.hamilton_int8(p, k), f"batch of {nk}")


def test_int8_bits_across_chunks(tbk, monkeypatch):
    """1 MB of workspace: chunks of a few hundred k-points, not multiples of the 48-point tile."""
    p = wl.synthetic(36, 120, seed=44)
    k = np.concatenate([all_k(3, 200, seed=5), np.random.default_rng(6).uniform(-2, 2, (600, 3))])
    monkeypatch.setenv("TBK_WORKSPACE_MB", "1")
    assert_bits(hamilton(tbk, monkeypatch, p, k, fp64=0), hd.hamilton_int8(p, k), "1 MB workspace")


def column_model():
    """N = 16, 101 stored R (7 K steps), with packed weight columns at the edges of the column scaling:
    (1, 0) all zero; (2, 0) non-zero at one R only; (3, 0) magnitudes over 12 decades; (4, 0) 1 - 2^-53 at every R, the
    top of a binade; (5, 0) and the diagonal (6, 6) exact powers of two; (7, 0) a single value of 1e-100 among zeros;
    everything else random."""
    p = wl.synthetic(16, 100, seed=45)
    hop = np.array(p.hop)
    rng = np.random.default_rng(46)
    n_R = p.n_R
    for i in range(1, 8):
        hop[:, i, 0] = 0.0
        hop[:, 0, i] = 0.0
    hop[37, 2, 0] = 0.3 - 0.7j
    hop[:, 3, 0] = (rng.normal(size=n_R) + 1j * rng.normal(size=n_R)) * 10.0 ** rng.integers(-12, 1, n_R)
    hop[:, 4, 0] = (1 - 2.0**-53) * (1 + 1j)
    hop[:, 5, 0] = 0.5 - 0.25j
    hop[:, 6, 6] = 0.25
    hop[11, 7, 0] = 1e-100j
    return pack_arrays(p.R, hop, p.pos)


def test_int8_bits_weight_columns(tbk, monkeypatch):
    p = column_model()
    k = all_k(3, 15, seed=7)
    H = hamilton(tbk, monkeypatch, p, k, fp64=0)
    assert_bits(H, hd.hamilton_int8(p, k), "weight-column model")
    assert np.all(H[:, 1, 0] == 0) and not np.signbit(H[:, 1, 0].real).any() and not np.signbit(H[:, 1, 0].imag).any()


@pytest.mark.parametrize("e", [-600, 600])
@pytest.mark.parametrize("name", ["n36-ks6", "weight-columns"])
def test_int8_bits_scaled_models(tbk, monkeypatch, name, e):
    p = xs.scaled(column_model() if name == "weight-columns" else MODELS[name][0](), e)
    k = all_k(3, 9, seed=8)
    assert_bits(hamilton(tbk, monkeypatch, p, k, fp64=0), hd.hamilton_int8(p, k), f"{name} scaled by 2^{e}")


# long-range bases whose folded supercells have >= 81 stored R (test_gpu_accuracy / velocity / curvature use them)
LONG_RANGE = {
    "b1-600-3x3x1": (lambda: xs.band1(3, 600), (3, 3, 1)),  # N 9, 139 R, 9 K steps
    "b2-1500-2x2x2": (lambda: xs.band2(3, 1500), (2, 2, 2)),  # N 16, 285 R, 18 K steps
    "b1-3000-3x3x4": (lambda: xs.band1(3, 3000), (3, 3, 4)),  # N 36, 186 R, 12 K steps
    "b2-3000-3x3x2": (lambda: xs.band2(3, 3000), (3, 3, 2)),  # N 36, 309 R, 20 K steps
    "b1-4000-4x4x4": (lambda: xs.band1(3, 4000), (4, 4, 4)),  # N 64, 138 R, 9 K steps
}


@pytest.mark.parametrize("name", list(LONG_RANGE) + ["b2-13-4x4x4"])
def test_int8_bits_device_packed_supercells(tbk, monkeypatch, name):
    """Block-sparse device-packed supercells (Evaluator.from_supercell) and the host-packed handle both give the bits
    of the restatement built from the host pack: every supercell hopping element comes from one base hopping, so the
    two packs agree bit for bit."""
    base, size = LONG_RANGE[name] if name in LONG_RANGE else (lambda: xs.band2(3, 13, seed=4), (4, 4, 4))
    b = base()
    sup = wl.supercell(b, size)
    k = all_k(3, 5, seed=9)
    want = hd.hamilton_int8(sup, k)
    assert_bits(hamilton(tbk, monkeypatch, sup, k, fp64=0), want, f"{name} host-packed")
    assert_bits(hamilton(tbk, monkeypatch, None, k, fp64=0, supercell=(b, size)), want, f"{name} device-packed")


@pytest.mark.parametrize("name", list(LONG_RANGE))
def test_long_range_supercells_run_int8_by_default(tbk, monkeypatch, name):
    """The default build of each long-range input (host- and device-packed) is the INT8 one: its bits equal the
    restatement and differ from the FP64 DMMA build."""
    base, size = LONG_RANGE[name]
    b = base()
    sup = wl.supercell(b, size)
    assert sup.n_R >= 81
    k = all_k(3, 5, seed=10)
    want = hd.hamilton_int8(sup, k)
    for what, p, sc in (("host-packed", sup, None), ("device-packed", None, (b, size))):
        got = hamilton(tbk, monkeypatch, p, k, supercell=sc)
        assert_bits(got, want, f"{name} {what}, default build")
        assert not np.array_equal(got, hamilton(tbk, monkeypatch, p, k, fp64=1, supercell=sc)), (
            f"{name} {what}: the default build equals the DMMA build")


def test_host_staging_model_runs_int8_by_default(tbk, monkeypatch):
    """c3-n36 of test_gpu_host_staging.py (251 stored R) stages its ``_host`` calls through the INT8 build."""
    p = wl.synthetic(36, 250, seed=1234)
    k = all_k(3, 5, seed=14)
    got = hamilton(tbk, monkeypatch, p, k)
    assert_bits(got, hd.hamilton_int8(p, k), "c3-n36, default build")
    assert not np.array_equal(got, hamilton(tbk, monkeypatch, p, k, fp64=1))


# ---------------------------------------------------------------------------------------------------------- gate edges
@pytest.mark.parametrize("n_half, int8", [(79, False), (80, True)], ids=["80R-dmma", "81R-int8"])
def test_gate_at_81_stored_r(tbk, monkeypatch, n_half, int8):
    """hk_i8_ksteps = (ceil(n_R / 8) + 1) / 2 K steps, INT8 by default from 6: the gate sits at 81 stored R."""
    p = wl.synthetic(36, n_half, seed=47)
    k = all_k(3, 9, seed=11)
    default = hamilton(tbk, monkeypatch, p, k)
    forced = {f: hamilton(tbk, monkeypatch, p, k, fp64=f) for f in (0, 1)}
    assert not np.array_equal(forced[0], forced[1])
    assert_bits(forced[0], hd.hamilton_int8(p, k), f"{p.n_R} R forced INT8")
    assert np.array_equal(default, forced[0 if int8 else 1]), f"{p.n_R} R: the default is not the {'INT8' if int8 else 'DMMA'} build"


def test_gate_at_2047_k_steps(tbk, monkeypatch):
    p = wl.synthetic(9, 32751, seed=48)  # 32 752 R: 2047 K steps, the most the int32 class sums allow
    k = all_k(3, 2, seed=12)
    assert_bits(hamilton(tbk, monkeypatch, p, k), hd.hamilton_int8(p, k), "2047 K steps, default build")


def test_2048_k_steps_fall_back_to_dmma(tbk, monkeypatch):
    p = wl.synthetic(9, 32767, seed=49)  # 32 768 R: 2048 K steps, past the int32 class sums
    k = all_k(3, 2, seed=13)
    forced = hamilton(tbk, monkeypatch, p, k, fp64=0)
    assert np.array_equal(forced, hamilton(tbk, monkeypatch, p, k, fp64=1)), "2048 K steps did not fall back to DMMA"
