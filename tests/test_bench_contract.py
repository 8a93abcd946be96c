"""bench.py contract checks: the reference arm's JSON line, the fail-loud behaviour of the product arm without a CUDA
device, argument checks and the ``--dump-outputs`` files (on the GPU: that they hold what the timed path computed)."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT, assert_eig_close, gpu_available


def _run(args, timeout=240):
    env = dict(os.environ)
    env.pop("RANK", None)
    env.pop("WORLD_SIZE", None)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                          timeout=timeout, cwd=ROOT, env=env)


def test_reference_arm_prints_the_contract_line():
    r = _run(["--impl", "reference", "--workload", "c1", "--steps", "1", "--warmup", "1"])
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["impl"] == "reference" and line["metric"] == "kpoints_per_s_eigenval_fp64"
    for key in ("value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["vs_baseline"] is None and line["higher_is_better"] is True and line["dtype"] == "f64"
    from oracle import ref_shim

    want_kind = "reference" if ref_shim.reference_available() else "port"
    assert line["cpu_baseline"]["kind"] == want_kind and line["cpu_baseline"]["cores"] >= 1
    host = line["cpu_baseline"]["host"]
    assert host["numpy"] and host["scipy"] and "threadpool_info" in host
    for pool in host["worker_threadpool_info"] or []:  # BLAS threads = 1 in every worker (set before numpy is imported there)
        assert pool["num_threads"] == 1, pool
    assert line["scaling"] == "strong"
    assert line["cpu_baseline"]["value"] == line["value"] == line["e2e"]["value"] and line["value"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"] and "model" not in line["config"]


def test_product_arm_fails_loudly_without_a_gpu():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    r = _run(["--steps", "1", "--warmup", "1", "--nk", "1000"], timeout=120)
    assert r.returncode != 0
    assert "no CUDA device" in (r.stderr + r.stdout)


def test_reference_callable_is_the_same_model_as_the_packed_arrays():
    """bench.py builds a tbmodels.Model from the packed arrays for its CPU arms: same eigenvalues as the oracle."""
    import numpy as np

    import bench
    from oracle import ref_shim, tb_oracle as orc
    from oracle import workloads as wl

    if not ref_shim.reference_available():
        pytest.skip("reference package not available")
    tb = ref_shim.import_reference()
    for packed in (wl.haldane(), wl.synthetic(7, 9, seed=3)):
        fn, kind = bench._make_ref_callable(packed.R, packed.hop, packed.pos)
        assert kind == "reference"
        model = fn.__closure__[0].cell_contents if fn.__closure__ else None
        assert isinstance(model, tb.Model)
        k = np.random.default_rng(5).random((9, packed.dim))
        got = np.array(model.eigenval(k))
        want = orc.eigenval_array(packed.R, packed.hop, packed.pos, k)
        assert np.array_equal(got, want)


def test_bench_rejects_bad_arguments(tmp_path):
    assert _run(["--steps", "0"]).returncode == 2
    r = _run(["--impl", "reference", "--dump-outputs", str(tmp_path / "out")])
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and not (tmp_path / "out").exists()


def test_dump_outputs_writes_every_row_or_a_seeded_sample(tmp_path, monkeypatch):
    import numpy as np
    import torch

    import bench

    eig = torch.arange(1000 * 4, dtype=torch.float64).reshape(1000, 4)
    bench.dump_outputs(str(tmp_path / "all"), eig)
    assert np.array_equal(np.load(tmp_path / "all" / "eigenvalues.npy"), eig.numpy())
    monkeypatch.setattr(bench, "DUMP_BYTES", 100 * 4 * 8)
    for name in ("a", "b"):
        bench.dump_outputs(str(tmp_path / name), eig)
    a = np.load(tmp_path / "a" / "eigenvalues.npy")
    assert a.shape == (100, 4) and a.dtype == np.float64
    assert np.array_equal(a, np.load(tmp_path / "b" / "eigenvalues.npy"))
    rows = (a[:, 0] / 4).astype(np.int64)  # row i of eig starts with 4 i
    assert np.all(np.diff(rows) > 0) and np.array_equal(a, eig.numpy()[rows])


@pytest.mark.gpu
def test_dump_outputs_are_the_eigenvalues_of_the_timed_steps(tmp_path):
    """C1 (the 20^3 silicon grid, 8000 k-points: dumped whole) against the oracle on the same k-points."""
    if not gpu_available():
        pytest.skip("no CUDA device")
    import numpy as np

    import bench
    from oracle import tb_oracle as orc
    from oracle import workloads as wl

    r = _run(["--workload", "c1", "--steps", "2", "--warmup", "1", "--no-extra", "--no-cpu", "--no-peaks",
              "--dump-outputs", str(tmp_path)], timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    p = bench.build_model("c1")
    want = orc.eigenval_array(p.R, p.hop, p.pos, wl.kgrid_points((20, 20, 20)))
    assert_eig_close(np.load(tmp_path / "eigenvalues.npy"), want, "c1 --dump-outputs")
