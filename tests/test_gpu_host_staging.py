"""The vector ``_host`` entry points (``eigh``, ``band_velocity``, ``berry_curvature``, ``kdotp_coefficients``) stage
k-points and results through device buffers of one host chunk (``TBK_HOST_CHUNK_MB``).

* With 1 MB host chunks every op runs in at least three host chunks, the last one ragged, on one model per scratch
  regime: fused H(k) build; GEMM build with eigh in shared memory; eigh on global scratch; N > 128, where a host chunk
  holds a few k-points; and the INT8 H(k) build (c3-n36).  The results are bit-equal to the ``*_device`` call on the
  whole batch.
* With a 1 MB workspace as well, a host chunk holds a whole number of the op's device chunks: band velocities and Berry
  curvature run in exactly the device chunks of the ``*_device`` call (equal per-class launch counts), bit for bit.
* ``hamilton`` and ``hamilton_device`` reject a bad convention with the reference's message.
"""
import numpy as np
import pytest

from oracle import workloads as wl
from tbmodels_b200._evaluator import kdotp_powers

pytestmark = pytest.mark.gpu

MODELS = {  # name: (model, path); c3-n36 has 251 stored R (16 K steps), so its H(k) runs on the INT8 digit GEMM by default
    "n5-fused": (lambda: wl.synthetic(5, 13, seed=7), "fused-small"),
    "n12-gemm": (lambda: wl.synthetic(12, 20, seed=8), "gemm+tridiag-ql"),
    "c3-n36": (lambda: wl.synthetic(36, 250, seed=1234), "gemm+tridiag-ql"),
    "n130": (lambda: wl.synthetic(130, 6, seed=5), "gemm+tridiag-ql"),
}
OPS = ("eigh", "velocity", "curvature-1", "curvature-2", "kdotp")
KDOTP_ORDER = 2


@pytest.fixture(scope="module")
def tbk():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import tbmodels_b200

    return tbmodels_b200


def _op(op, n, dim):
    """(host call, device call, result doubles per k-point, kernel class counted, its launches per device chunk)."""
    if op == "eigh":
        return (lambda ev, k: ev.eigh(k)), (lambda ev, kd: ev.eigh_device(kd)), n + 2 * n * n, "eigh", 1
    if op == "velocity":
        return (lambda ev, k: ev.band_velocity(k)), (lambda ev, kd: ev.band_velocity_device(kd)), n + n * dim, "eigh", 2
    if op.startswith("curvature"):
        c = int(op[-1])
        return ((lambda ev, k: ev.berry_curvature(k, convention=c)),
                (lambda ev, kd: ev.berry_curvature_device(kd, convention=c)), n + n * dim * (dim - 1) // 2, "eigh", 3)
    terms = kdotp_powers(dim, KDOTP_ORDER).shape[0]
    return ((lambda ev, k: ev.kdotp_coefficients(k, KDOTP_ORDER)[1:]),
            (lambda ev, kd: ev.kdotp_coefficients_device(kd, KDOTP_ORDER)[1:]), terms * 2 * n * n, "expand", 1)


def _launches(ev):
    return {cls: n for cls, (_, n) in ev.profile_read().items()}


def _host_vs_device(tbk, name, op):
    """Results and per-class launch counts of the host call and of the device call on the same batch and handle; the batch
    is three and a half 1 MB host chunks."""
    import torch

    make, path = MODELS[name]
    p = make()
    host, dev, per_k, cls, per_chunk = _op(op, p.size, p.dim)
    hchunk = max(1, (1 << 20) // (8 * (p.dim + per_k)))  # before rounding to whole device chunks, which only shrinks it
    k = np.random.default_rng(11).uniform(-1, 1, (3 * hchunk + hchunk // 2 + 1, p.dim))
    ev = tbk.Evaluator(p)
    assert ev.path == path
    ev.profile(True)
    _launches(ev)
    got = host(ev, k)
    on_host = _launches(ev)
    want = dev(ev, torch.from_numpy(k).cuda())
    ev.check()
    on_device = _launches(ev)
    ev.close()
    for i, (g, w) in enumerate(zip(got, want)):
        assert np.array_equal(g, w.cpu().numpy()), f"{name} {op}: result {i} of the host call differs from the device call"
    return on_host, on_device, cls, per_chunk


@pytest.mark.parametrize("op", OPS)
@pytest.mark.parametrize("name", list(MODELS))
def test_host_chunks(tbk, monkeypatch, name, op):
    monkeypatch.setenv("TBK_HOST_CHUNK_MB", "1")
    on_host, _, cls, per_chunk = _host_vs_device(tbk, name, op)
    assert on_host[cls] >= 3 * per_chunk, f"{name} {op}: {on_host[cls] // per_chunk} chunk(s), expected at least 3"


@pytest.mark.parametrize("op", OPS)
@pytest.mark.parametrize("name", ["n5-fused", "n12-gemm", "c3-n36"])
def test_host_chunks_of_whole_device_chunks(tbk, monkeypatch, name, op):
    monkeypatch.setenv("TBK_HOST_CHUNK_MB", "1")
    monkeypatch.setenv("TBK_WORKSPACE_MB", "1")
    on_host, on_device, _, _ = _host_vs_device(tbk, name, op)
    if op in ("velocity", "curvature-1", "curvature-2"):  # (a 1 MB host chunk holds at most about one eigh or k.p chunk)
        assert on_host == on_device, f"{name} {op}: launches {on_host} through the host path, {on_device} on the device"


def test_hamilton_rejects_bad_convention(tbk):
    import torch

    ev = tbk.Evaluator(wl.haldane())
    with pytest.raises(ValueError, match="Invalid value '3' for 'convention'"):
        ev.hamilton([0.1, 0.2], convention=3)
    with pytest.raises(ValueError, match="Invalid value '3' for 'convention'"):
        ev.hamilton_device(torch.zeros((2, 2), dtype=torch.float64, device="cuda"), convention=3)
    ev.close()
