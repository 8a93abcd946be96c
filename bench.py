#!/usr/bin/env python
"""bench.py -- k-points/s of Model.eigenval (H(k) build + eigenvalues, fp64) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3] [--impl ours|reference] [--dump-outputs DIR]

Default workload: BASELINE.json configs[2] (C3: synthetic 36-orbital Wannier model, 251 stored R-vectors, the
256^3 k-grid), the configuration the north_star target is quoted on.  One "step" = one pass of the hot path over the
WHOLE k-set of the configuration: the k-points are cut into contiguous shards, one per GPU (strong scaling: total work
is fixed as N grows), every rank evaluates its shard with the CUDA kernels and -- for N > 1 -- the eigenvalue shards
are exchanged so that every rank holds the full [N_k, N] result, INSIDE the timed region (SURVEY.md section 8 d1).
The exchange is fused behind the eigensolver: every finished chunk is stored straight into all peers' result buffers
over NVLink / NVSwitch (tbk_eigenval_push on a symmetric-memory buffer) while the next chunk computes, then one
device-side barrier; the plain "compute, then NCCL all_gather_into_tensor" variant is timed next to it
(`nccl_variant_ms_per_step`) and the two results are compared bit for bit.  Rank 0 prints ONE JSON line.

  value        device-resident throughput: k [N_k, D] already in HBM -> gathered eigenvalues in HBM; CUDA events on the
               launching stream, max over ranks
  e2e          same metric through the host-buffer C-ABI entry point (tbk_eigenval_host): pinned host k in, pinned host
               eigenvalues out, H2D / D2H inside the timed region (each rank its shard)
  roofline     dominant kernel: algorithmic flops (or bytes) per launch / CUDA-event duration of that kernel
  kernels      the same for every kernel class of the step
  cpu_baseline the UNMODIFIED reference (oracle/_ref, imported through oracle/ref_shim.py) -- or the numpy/scipy oracle
               port when the reference copy is absent -- timed on this box's host cores on a bounded sample
  extra        N = 1: the other BASELINE configs (C2 at 1e8 k-points, C1, C5 with its N_k sweep, C4 at 12 500 k-points),
               each with value / e2e / roofline / cpu_baseline, and C3 as a k-grid through eigenval_mesh;
               N > 1: the C5 strong-scaling sweep and C3 through eigenval_mesh, gathers included

``--impl reference`` times the reference's own ``Model.eigenval`` on all host cores (process pool over k-chunks,
BLAS threads = 1 each: the parallel mode the reference documents) with the same metric / unit / config.

``--dump-outputs DIR`` writes, after the timed steps of the main measurement, the eigenvalues its last step computed as
``DIR/eigenvalues.npy`` (float64): all rows of the [N_k, N] result, or a fixed seeded sample of rows when the whole array
exceeds 32 MiB.  The inputs depend only on the arguments, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import platform
import subprocess
import sys
import tempfile
import time

import numpy as np

# the tree may be read-only and must stay as build() left it: no bytecode caches written beside the sources
sys.dont_write_bytecode = True

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "kpoints_per_s_eigenval_fp64"
UNIT = "k-points/s"

# name: description, total k-points of the configuration, mesh dims (None = seeded random k-points),
#       default steps / warm-up, k-points of the single-process CPU sample
WORKLOADS = {
    "c1": dict(desc="silicon sp3 Wannier90 model N=8 95 stored R, 20^3 k-grid (8000 k-points)", total=8000,
               dims=(20, 20, 20), steps=50, warmup=5, cpu_sample=8000),
    "c2": dict(desc="2-band Haldane model N=2 D=2 4 stored R, 1e8 random k-points", total=10**8, dims=None,
               steps=20, warmup=5, cpu_sample=200_000),
    "c3": dict(desc="synthetic N=36 251 stored R (seed 1234), 256^3 k-grid (16 777 216 explicit k-points)",
               total=2**24, dims=(256, 256, 256), steps=3, warmup=3, cpu_sample=6000),
    "c4": dict(desc="silicon 4x4x4 supercell N=512 14 stored R, 1e5 random k-points", total=10**5, dims=None,
               steps=2, warmup=3, cpu_sample=60),
    "c5": dict(desc="synthetic N=128 1001 stored R (seed 1234), 2^17 k-points of a 32x64x64 k-grid", total=2**17,
               dims=(32, 64, 64), steps=3, warmup=3, cpu_sample=100),
}


def build_model(workload: str):
    from oracle import workloads as wl

    if workload == "c1":
        return wl.load_packed(os.path.join(ROOT, "tests", "golden", "silicon.npz"))
    if workload == "c2":
        return wl.haldane()
    if workload == "c3":
        return wl.synthetic(36, 250, seed=1234)
    if workload == "c4":
        return wl.supercell(wl.load_packed(os.path.join(ROOT, "tests", "golden", "silicon.npz")), (4, 4, 4))
    if workload == "c5":
        return wl.synthetic(128, 1000, seed=1234)
    raise SystemExit(f"unknown workload {workload}")


def workload_config(workload: str, packed, total: int) -> dict:
    """The `config` object of the JSON line: names the workload, identical for the GPU arm and the reference arm."""
    return {"workload": f"{workload}: {WORKLOADS[workload]['desc']}", "kpoints_total": int(total), "n_orb": packed.size,
            "n_R_stored": packed.n_R, "dim": packed.dim}


def mesh_dims_for(total: int, dims):
    """Mesh whose point count is ``total``: the configured one, or (for an --nk override / the C5 sweep) the
    power-of-two box (2^a, 2^b, 2^c), a <= b <= c as equal as possible.  None = seeded random k-points."""
    if dims is None:
        return None
    if int(np.prod(dims)) == total:
        return tuple(dims)
    if total < 8 or total & (total - 1) or len(dims) != 3:
        return None
    e = total.bit_length() - 1
    c = -(-e // 3)
    b = -(-(e - c) // 2)
    return (1 << (e - c - b), 1 << b, 1 << c)


def host_kpoints(workload: str, n_k: int, dim: int, seed: int = 0) -> np.ndarray:
    """A bounded CPU sample of the workload's k-set (mesh workloads: a seeded random subset of the mesh points)."""
    cfg = WORKLOADS[workload]
    rng = np.random.default_rng(seed)
    if cfg["dims"] is None:
        return rng.random((n_k, dim))
    dims = np.array(cfg["dims"], dtype=np.int64)
    total = int(np.prod(dims))
    if n_k >= total:
        idx = np.arange(total)
    else:
        idx = np.sort(rng.choice(total, size=n_k, replace=False))
    return np.stack(np.unravel_index(idx, dims), axis=1).astype(np.float64) / dims


# ------------------------------------------------------------------------------------------------ CPU reference
_REF_STATE = {}


def _ref_init(R, hop, pos, want_reference: bool):
    """Pool initialiser: BLAS threads = 1 (also set in the environment before the pool was spawned, so the BLAS
    library of this fresh interpreter never created a thread pool), then the evaluation callable."""
    try:
        import threadpoolctl

        _REF_STATE["limits"] = threadpoolctl.threadpool_limits(1)
    except Exception:  # noqa: BLE001
        pass
    _REF_STATE["fn"], _REF_STATE["kind"] = _make_ref_callable(R, hop, pos, want_reference)


def _make_ref_callable(R, hop, pos, want_reference: bool = True):
    """``fn(k[n,D]) -> None`` running Model.eigenval of the UNMODIFIED reference (kind "reference") when the package is
    importable (/root/reference or the verified copy under oracle/_ref), else the oracle port (kind "port")."""
    import warnings

    from oracle import ref_shim

    if want_reference and ref_shim.reference_available():
        tb = ref_shim.import_reference()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            model = tb.Model(hop={tuple(int(x) for x in r): np.array(h) for r, h in zip(R, hop)}, pos=np.array(pos),
                             size=pos.shape[0], dim=pos.shape[1], contains_cc=False)

        def fn(k, chunk=2048):  # chunked only to bound the two [n_k, N, N] temporaries of the reference
            for s in range(0, k.shape[0], chunk):
                model.eigenval(k[s : s + chunk])

        return fn, "reference"
    from oracle import tb_oracle as orc

    return (lambda k: orc.eigenval_array(R, hop, pos, k, chunk=2048)), "port"


def _ref_chunk(k):
    t0 = time.perf_counter()
    _REF_STATE["fn"](k)
    return time.perf_counter() - t0


def _ref_info(_):
    try:
        import threadpoolctl

        tp = [{k: d.get(k) for k in ("user_api", "internal_api", "version", "num_threads", "threading_layer")}
              for d in threadpoolctl.threadpool_info()]
    except Exception:  # noqa: BLE001
        tp = None
    return {"kind": _REF_STATE["kind"], "threadpool_info": tp}


def host_record() -> dict:
    """CPU model, library versions and BLAS thread pools of THIS process (SURVEY.md section 8 d4)."""
    import scipy

    rec = {"python": platform.python_version(), "numpy": np.__version__, "scipy": scipy.__version__,
           "host_cores": os.cpu_count()}
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.startswith("model name"):
                    rec["cpu_model"] = ln.split(":", 1)[1].strip()
                    break
    except OSError:
        pass
    try:
        import threadpoolctl

        rec["threadpool_info"] = [{k: d.get(k) for k in ("user_api", "internal_api", "version", "num_threads", "threading_layer")}
                                  for d in threadpoolctl.threadpool_info()]
    except Exception:  # noqa: BLE001
        rec["threadpool_info"] = None
    return rec


def cpu_baseline_single(workload: str, packed, budget_s: float = 8.0) -> dict:
    """The reference, single process as shipped (BLAS threads = library default), on a bounded sample."""
    fn, kind = _make_ref_callable(packed.R, packed.hop, packed.pos)
    cfg = WORKLOADS[workload]
    ks = host_kpoints(workload, min(cfg["cpu_sample"], cfg["total"]), packed.dim, seed=1)
    n_cal = max(4, min(ks.shape[0] // 20, 256))
    t0 = time.perf_counter()
    fn(ks[:n_cal])
    rate = n_cal / (time.perf_counter() - t0)
    n = int(min(ks.shape[0], max(n_cal, rate * budget_s)))
    ts = []
    for _ in range(3 if n * 3 / rate < 2 * budget_s else 1):
        t0 = time.perf_counter()
        fn(ks[:n])
        ts.append(time.perf_counter() - t0)
    rec = host_record()
    blas_threads = max([d.get("num_threads") or 1 for d in (rec.get("threadpool_info") or [])] or [1])
    return {
        "value": n / float(np.median(ts)),
        "unit": UNIT,
        "cores": int(blas_threads),
        "kind": kind,
        "sample": f"{n} k-points of the same workload (seeded subset), Model.eigenval of the "
                  f"{'unmodified reference (oracle/_ref via oracle/ref_shim.py)' if kind == 'reference' else 'numpy/scipy oracle port'}"
                  f", single process as the reference ships, BLAS threads = library default ({blas_threads}), median of {len(ts)}",
        "host": rec,
    }


def run_reference_arm(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp

    for var in ("OPENBLAS_NUM_THREADS", "OMP_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[var] = "1"  # before the workers are spawned: their BLAS reads it when numpy is first imported there
    packed = build_model(args.workload)
    cfg = WORKLOADS[args.workload]
    cores = os.cpu_count() or 1
    procs = max(1, min(cores, 64))
    steps = args.steps if args.steps is not None else 3
    warmup = args.warmup if args.warmup is not None else 1
    ctx = mp.get_context("spawn")
    with ctx.Pool(procs, initializer=_ref_init, initargs=(packed.R, packed.hop, packed.pos, True)) as pool:
        info = pool.map(_ref_info, range(procs))[0]

        def rate_of(k):
            parts = [p for p in np.array_split(k, procs) if p.shape[0]]
            t0 = time.perf_counter()
            pool.map(_ref_chunk, parts, chunksize=1)
            return k.shape[0] / (time.perf_counter() - t0)

        # calibrate on a small sample, then size each step so the whole run stays within ~2 minutes
        cal = host_kpoints(args.workload, min(cfg["total"], max(procs * 4, min(cfg["cpu_sample"], 2000) * procs // 8)), packed.dim, seed=2)
        rate_of(cal[: procs * 2])  # spin the workers up
        rate = rate_of(cal)
        step_s = min(12.0, max(1.0, 100.0 / max(steps + warmup, 1)))
        sample_k = int(min(cfg["total"], max(procs * 4, rate * step_s)))
        k = host_kpoints(args.workload, sample_k, packed.dim, seed=1)
        for _ in range(warmup):
            rate_of(k)
        t0 = time.perf_counter()
        for _ in range(steps):
            rate_of(k)
        dt = time.perf_counter() - t0
    value = steps * k.shape[0] / dt
    kind = info["kind"]
    line = {
        "impl": "reference",
        "metric": METRIC,
        "value": value,
        "unit": UNIT,
        "n_gpus": args.gpus,
        "steps": steps,
        "warmup": warmup,
        "ms_per_step": 1e3 * dt / steps,
        "higher_is_better": True,
        "scaling": "strong",
        "vs_baseline": None,
        "dtype": "f64",
        "data": "synthetic",
        "config": workload_config(args.workload, packed, cfg["total"]),
        "cpu_baseline": {
            "value": value,
            "unit": UNIT,
            "cores": procs,
            "kind": kind,
            "sample": f"{k.shape[0]} k-points of the same workload per step (seeded subset), Model.eigenval of the "
                      f"{'unmodified reference (oracle/_ref via oracle/ref_shim.py)' if kind == 'reference' else 'numpy/scipy oracle port'}"
                      f" in {procs} processes over contiguous k-chunks, BLAS threads = 1 each (set before the workers import "
                      f"numpy), host has {cores} cores",
            "host": {**host_record(), "worker_threadpool_info": info["threadpool_info"]},
        },
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    FIELDS = (
        "timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
        "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    )

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.proc = None
        self.marks = {}

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu)],
                stdout=self.tmp,
                stderr=subprocess.DEVNULL,
            )
        except OSError:
            self.proc = None

    def mark(self, name):
        self.marks[name] = time.time()

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        self.tmp.flush()
        rows = []
        import datetime

        for ln in open(self.tmp.name):
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 10:
                continue
            try:
                ts = datetime.datetime.strptime(parts[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(parts[2]), float(parts[3]), parts[4], parts[6:10]))
            except ValueError:
                continue
        os.unlink(self.tmp.name)
        t0, t1 = self.marks.get("timed_start", 0), self.marks.get("timed_end", 1e18)
        inside = [r for r in rows if t0 <= r[0] <= t1]
        window = "timed region"
        if len(inside) < 2:
            r0, r1 = self.marks.get("run_start", 0), self.marks.get("run_end", 1e18)
            inside = [r for r in rows if r0 <= r[0] <= r1]
            window = "warm-up + timed + e2e (timed region shorter than the 100 ms sampling period)"
        if not inside:
            inside = rows
            window = "whole run"
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in inside for n, v in zip(names, r[4]) if v.lower().startswith("active")})
        return {
            "sm_mhz": float(np.median([r[1] for r in inside])),
            "sm_max_mhz": float(max(r[2] for r in inside)),
            "reasons": reasons,
            "samples": len(inside),
            "window": window,
        }


# ------------------------------------------------------------------------------------------------ GPU arm
def measured_hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except Exception:  # noqa: BLE001
        return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


def ncu_traffic_table() -> dict:
    """DRAM bytes per k-point of the dominant kernels (dram__bytes_read.sum + dram__bytes_write.sum of one launch of
    an ``ncu --set full`` capture / the k-points of that launch): profiles/ncu_traffic.json, written by
    tools/ncu_traffic.py from the .ncu-rep files of the round."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            return json.load(f)
    except Exception:  # noqa: BLE001
        return {}


def flops_per_k(packed):
    n, nR = packed.size, packed.n_R
    return {"F_H": 8.0 * nR * n * n + 2.0 * n * n, "F_eig": (16.0 / 3.0) * n**3, "bytes": 8.0 * packed.dim + 8.0 * n}


def kernel_rooflines(workload, prof, steps, n_local, fl, peaks, path):
    """One roofline record per kernel class of the step (CUDA events around every launch, same timed region)."""
    hbm_peak, hbm_src = measured_hbm_peak()
    traffic = ncu_traffic_table()
    total_ms = sum(v[0] for v in prof.values()) or 1e-12
    out = {}
    for cls, (ms, cnt) in prof.items():
        if not cnt:
            continue
        per_launch_s = ms * 1e-3 / cnt
        k_per_launch = n_local * steps / cnt
        rec = {"kernel_ms_per_launch": per_launch_s * 1e3, "launches_per_step": cnt / steps,
               "kernel_share_of_step": ms / total_ms, "kpoints_per_launch": k_per_launch}
        if cls in ("hk_small", "expand"):
            a = fl["bytes"] * k_per_launch / per_launch_s / 1e9
            rec.update(kernel="hk_basis (profile class hk_small)" if path == "fused-product" else cls, bound="hbm", achieved=a,
                       peak=hbm_peak, unit="GB/s", frac=a / hbm_peak, peak_source=hbm_src,
                       algorithmic_bytes_per_kpoint=fl["bytes"],
                       note="fp64 sincospi/FMA work per k-point is co-limiting; see DESIGN.md")
        elif cls == "hk_gemm":
            a = fl["F_H"] * k_per_launch / per_launch_s / 1e12
            rec.update(kernel=cls, bound="tensor", achieved=a, peak=peaks["dmma"], unit="TFLOP/s", frac=a / peaks["dmma"],
                       peak_source="tbk_measure_fp64_peak: mma.sync.m8n8k4.f64 register loop on this GPU in this run",
                       algorithmic_flops_per_kpoint=fl["F_H"], executed_flops_per_kpoint=fl["F_H"] / 2.0,
                       frac_executed=a / 2.0 / peaks["dmma"],
                       note="achieved/frac count the ALGORITHMIC flops of the reference formulation (8 n_R N^2 per k-point); the "
                            "Hermitian split executes half of them, so frac_executed (= ncu tensor-pipe utilisation) is the "
                            "hardware utilisation and frac may legitimately reach 2.0")
        elif cls in ("tridiag", "ql"):
            # the eigensolver's algorithmic work, (16/3) N^3 flops per matrix, is charged to the tridiagonalisation;
            # the QL / bisection stage is O(N^2) latency-bound work with no meaningful flop roofline
            a = (fl["F_eig"] if cls == "tridiag" else 0.0) * k_per_launch / per_launch_s / 1e12
            rec.update(kernel=cls, bound="tensor", achieved=a, peak=peaks["dfma"], unit="TFLOP/s", frac=a / peaks["dfma"],
                       peak_source="tbk_measure_fp64_peak: DFMA register loop (the eigensolver runs on the FP64 FMA pipe, "
                                   "which shares its datapath with DMMA on B200)",
                       algorithmic_flops_per_kpoint=fl["F_eig"] if cls == "tridiag" else 0.0)
        else:
            rec.update(kernel=cls, bound="hbm", achieved=None, peak=hbm_peak, unit="GB/s", frac=None)
        tpk = traffic.get(f"{workload}:{cls}")
        rec["traffic"] = tpk["bytes_per_kpoint"] * k_per_launch if tpk else None
        if tpk:
            rec["traffic_source"] = tpk.get("source")
        out[cls] = rec
    return out


def time_device_steps(ev, step, steps, warmup, dist, dev, sampler=None):
    import torch

    for _ in range(warmup):
        step()
    ev.check()
    ev.profile_read()  # drop warm-up records
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    if sampler:
        sampler.mark("timed_start")
    l0 = ev.launch_count
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    if sampler:
        sampler.mark("timed_end")
    ms = e0.elapsed_time(e1)
    launches = ev.launch_count - l0
    prof = ev.profile_read()
    ev.check()
    if dist is not None:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms, launches, prof


def shard_k_device(workload, dims, total, lo, hi, dim, dev, seed_rank):
    """Explicit k-points [lo, hi) of the workload's k-set, generated on the device (mesh points in C order, or the
    rank's seeded random shard)."""
    import torch

    if dims is not None:
        idx = torch.arange(lo, hi, device=dev, dtype=torch.int64)
        cols = []
        stride = 1
        for d in reversed(range(len(dims))):
            cols.append(((idx // stride) % dims[d]).double() / dims[d])
            stride *= dims[d]
        return torch.stack(list(reversed(cols)), dim=1).contiguous()
    g = torch.Generator(device=dev).manual_seed(1234 + seed_rank)
    return torch.rand((hi - lo, dim), dtype=torch.float64, device=dev, generator=g)


DUMP_BYTES = 32 << 20


def dump_outputs(dump_dir, eig) -> None:
    """``DIR/eigenvalues.npy``: the rows of the device result ``eig`` [N_k, N], or a sample of DUMP_BYTES worth of rows
    chosen with a fixed seed (sorted), so that the same arguments always select the same k-points."""
    import torch

    total, n = eig.shape
    m = min(total, max(1, DUMP_BYTES // (8 * n)))
    rows = np.arange(total) if m == total else np.sort(np.random.default_rng(0).choice(total, size=m, replace=False))
    os.makedirs(dump_dir, exist_ok=True)
    np.save(os.path.join(dump_dir, "eigenvalues.npy"), eig[torch.from_numpy(rows).to(eig.device)].cpu().numpy())


def measure(workload, packed, total, steps, warmup, ctx, sampler=None, peaks=None, e2e_cap=None, use_mesh=False,
            dump_dir=None):
    """Strong-scaling measurement of one workload: shard, evaluate, gather (world > 1), all inside the timed region."""
    import torch

    import tbmodels_b200 as tbk
    from tbmodels_b200.sharded import shard_bounds

    dist, dev, rank, world = ctx["dist"], ctx["dev"], ctx["rank"], ctx["world"]
    cfg = WORKLOADS[workload]
    dims = mesh_dims_for(total, cfg["dims"])
    ev = tbk.Evaluator(packed, device=dev.index)
    ev.profile(True)
    fl = flops_per_k(packed)
    if total % world:
        raise SystemExit(f"{workload}: {total} k-points do not split evenly over {world} ranks")
    lo, hi = shard_bounds(total, world, rank)
    n_local = hi - lo
    k_dev = shard_k_device(workload, dims, total, lo, hi, packed.dim, dev, rank)
    out_dev = torch.empty((n_local, packed.size), dtype=torch.float64, device=dev)
    gathered = torch.empty((total, packed.size), dtype=torch.float64, device=dev) if world > 1 else None
    mesh_cfg = None
    if use_mesh:
        if dims is None:
            raise SystemExit("--mesh needs a k-grid workload (c1, c3, c5)")
        n_last = dims[-1]
        if lo % n_last or hi % n_last:
            raise SystemExit("--mesh: shard is not a whole number of mesh lines")
        mesh_cfg = {"dims": list(dims), "lines_per_gpu": n_local // n_last, "factorised": bool(ev.mesh_factorised(dims))}
        compute = lambda: ev.eigenval_mesh_device(dims, first_line=lo // n_last, n_lines=n_local // n_last, out=out_dev)  # noqa: E731
    else:
        compute = lambda: ev.eigenval_device(k_dev, out=out_dev)  # noqa: E731

    # N > 1: the exchange step.  Product path = FUSED gather: every chunk's rows are stored straight into all peers'
    # result buffers over NVLink while the next chunk computes (tbk_eigenval_push on a symmetric-memory buffer), then one
    # device-side barrier.  Baseline variant = compute, then NCCL all_gather_into_tensor; timed too and compared bit for bit.
    gather_kind, fused_err, pg = "none", None, None
    if world > 1 and not use_mesh and not args_no_fused():
        try:
            from tbmodels_b200.sharded import PeerGather

            pg = PeerGather(total, packed.size, device=dev)
            gather_kind = "fused peer stores (tbk_eigenval_push over symmetric memory) + device-side barrier"
        except Exception as e:  # noqa: BLE001 -- recorded in the JSON line, never silent
            fused_err = f"{type(e).__name__}: {e}"
            pg = None
    if world > 1 and pg is None:
        gather_kind = "NCCL all_gather_into_tensor after the local evaluation"

    def step_nccl():
        compute()
        dist.all_gather_into_tensor(gathered, out_dev)

    def step_fused():
        ev.eigenval_push_device(k_dev, pg.buffer[lo:hi], pg.peer_ptrs, lo)
        pg.barrier()

    step = compute if world == 1 else (step_fused if pg is not None else step_nccl)
    ms, launches, prof = time_device_steps(ev, step, steps, warmup, dist, dev, sampler)
    value = total * steps / (ms * 1e-3)
    if dump_dir and rank == 0:  # the last timed step's [total, N] result: this GPU's, or the buffer it was gathered into
        dump_outputs(dump_dir, out_dev if world == 1 else (pg.buffer if pg is not None else gathered))

    # the NCCL variant of the same step, for the record (and the gather alone)
    gather_ms = nccl_ms_per_step = None
    if world > 1:
        ms_n, _, _ = time_device_steps(ev, step_nccl, steps, 1, dist, dev, None)
        nccl_ms_per_step = ms_n / steps
        torch.cuda.synchronize()
        dist.barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        dist.all_gather_into_tensor(gathered, out_dev)
        g1.record()
        torch.cuda.synchronize()
        gather_ms = g0.elapsed_time(g1)
        if pg is not None:
            assert torch.equal(pg.buffer, gathered), "fused peer-store gather and NCCL all-gather disagree"
            out_dev.copy_(pg.buffer[lo:hi])

    # ---- parity inside the bench: sorted + finite; the NCCL-gathered rows of EVERY rank's shard against a single-rank
    # evaluation of the same k-points on this GPU (bit-exact: a k-point's bits do not depend on batch or shard) ----
    chk = out_dev[:: max(1, n_local // 1000)]
    assert bool(torch.isfinite(chk).all()) and bool((chk[:, 1:] >= chk[:, :-1]).all()), "bench output failed sanity check"
    gather_checked = 0
    if world > 1:
        assert torch.equal(gathered[lo:hi], out_dev), "all-gather misplaced this rank's own shard"
        m = min(256, n_local)
        for r in range(world):
            rlo, rhi = shard_bounds(total, world, r)
            if dims is not None:
                kr = shard_k_device(workload, dims, total, rlo, rlo + m, packed.dim, dev, r)
            else:
                kr = shard_k_device(workload, dims, total, rlo, rhi, packed.dim, dev, r)[:m].contiguous()
            want = ev.eigenval_device(kr)
            got = gathered[rlo : rlo + m]
            if use_mesh:
                scale = float(want.abs().max())
                assert float((got - want).abs().max()) <= 1e-10 * scale, f"gathered shard of rank {r} differs from a local evaluation"
            else:
                assert torch.equal(got, want), f"gathered shard of rank {r} differs from a local evaluation (not bit-equal)"
            gather_checked += m
        ev.check()
        ev.profile_read()

    kern = kernel_rooflines(workload, prof, steps, n_local, fl, peaks, ev.path) if peaks else {}
    dom = max(kern, key=lambda c: kern[c]["kernel_share_of_step"]) if kern else None
    if dom in ("hk_phase", "mesh_lines") and "hk_gemm" in kern:
        dom = "hk_gemm"

    # ---- end to end through the host-buffer C-ABI entry point (pinned host memory, copies inside) ----
    e2e_n = min(n_local, e2e_cap) if e2e_cap else n_local
    k_host = tbk.pinned_empty((e2e_n, packed.dim))
    k_host[:] = k_dev[:e2e_n].cpu().numpy()
    out_host = tbk.pinned_empty((e2e_n, packed.size))
    per_step_s = ms * 1e-3 / steps
    e2e_steps = int(max(1, min(steps, 10, 20.0 / max(per_step_s, 1e-3))))
    if use_mesh:  # the mesh has no k array: the host API is the pipelined kernels | D2H entry point, whole lines only
        n_last = dims[-1]
        e2e_n = max(n_last, e2e_n - e2e_n % n_last)
        out_host = tbk.pinned_empty((e2e_n, packed.size))
        host_call = lambda: ev.eigenval_mesh(dims, first_line=lo // n_last, n_lines=e2e_n // n_last, out=out_host)  # noqa: E731
    else:
        host_call = lambda: ev.eigenval_array(k_host, out=out_host)  # noqa: E731
    for _ in range(2 if per_step_s < 1.0 else 1):
        host_call()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        host_call()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if dist is not None:
        t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    ref_rows = out_dev[:64].cpu().numpy()
    assert np.array_equal(out_host[:64], ref_rows), "host and device entry points disagree"
    if use_mesh:  # mesh entry point vs explicit k-points: same values to rounding, not the same bits
        expl = ev.eigenval_device(k_dev[:64].contiguous()).cpu().numpy()
        assert np.abs(expl - ref_rows).max() <= 1e-10 * float(np.abs(ref_rows).max()), "mesh and explicit paths disagree"
    e2e = {
        "value": world * e2e_n * e2e_steps / e2e_s,
        "unit": UNIT,
        "h2d_bytes_per_step": 0 if use_mesh else int(e2e_n * packed.dim * 8),
        "d2h_bytes_per_step": int(e2e_n * packed.size * 8),
        "steps": e2e_steps,
        "kpoints_per_gpu_per_step": e2e_n,
        "api": ("Evaluator.eigenval_mesh -> tbk_eigenval_mesh_host (no k array; pinned host result, kernels | D2H pipeline); "
                if use_mesh else "Evaluator.eigenval_array -> tbk_eigenval_host (pinned host buffers, chunked 3-stream pipeline); ")
               + "every rank evaluates its shard into its own host buffer",
    }
    ev.profile_read()
    res = {
        "value": value,
        "unit": UNIT,
        "ms_per_step": ms / steps,
        "steps": steps,
        "warmup": warmup,
        "kpoints_total": total,
        "kpoints_per_gpu": n_local,
        "path": ev.path,
        "gpu_launches": int(launches),
        "e2e": e2e,
        "roofline": kern.get(dom),
        "kernels": kern,
        "kernel_ms_per_step": {c: v[0] / steps for c, v in prof.items() if v[1]},
        "allgather_ms": gather_ms,
        "gather": gather_kind,
        "gather_fallback_reason": fused_err,
        "nccl_variant_ms_per_step": nccl_ms_per_step,
        "gather_rows_checked": gather_checked,
        "fl": fl,
        "mesh": mesh_cfg,
    }
    ev.close()
    del k_dev, out_dev, gathered, k_host, out_host
    pg = None
    torch.cuda.empty_cache()
    return res


_NO_FUSED = [False]


def args_no_fused() -> bool:
    return _NO_FUSED[0]


def l2_note(res, packed):
    b = res["kpoints_per_gpu"] * res["fl"]["bytes"]
    scratch = res["kpoints_per_gpu"] * 8.0 * packed.size**2 if res["path"].startswith("gemm") else 0
    if b > 2 * 126e6 or scratch > 2 * 126e6:
        return "not flushed: inputs + outputs + H(k) scratch per step exceed the 126 MB L2 many times"
    return "not flushed: batch smaller than L2 (latency-bound parity config)"


def run_gpu_arm(args) -> None:
    import torch

    import tbmodels_b200 as tbk

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback; use --impl reference)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist = dist_mod
    if args.gpus != world and rank == 0:
        print(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={world}; reporting n_gpus={world}", file=sys.stderr)
    dev = torch.device("cuda", local_rank)
    ctx = {"dist": dist, "dev": dev, "rank": rank, "world": world}

    cfg = WORKLOADS[args.workload]
    total = args.nk or cfg["total"]
    steps = args.steps if args.steps is not None else cfg["steps"]
    warmup = max(args.warmup if args.warmup is not None else cfg["warmup"], 3)
    packed = build_model(args.workload)
    peaks = tbk.fp64_peaks() if not args.no_peaks else {"dmma": float("nan"), "dfma": float("nan")}

    sampler = ClockSampler(local_rank)
    sampler.start()
    sampler.mark("run_start")
    main = measure(args.workload, packed, total, steps, warmup, ctx, sampler, peaks, args.e2e_nk, use_mesh=args.mesh,
                   dump_dir=args.dump_outputs)

    def brief(res, workload, pk, with_cpu=True):
        rec = {k: res[k] for k in ("value", "unit", "ms_per_step", "steps", "warmup", "kpoints_total", "kpoints_per_gpu", "path",
                                   "gpu_launches", "e2e", "roofline", "kernel_ms_per_step", "allgather_ms", "gather",
                                   "nccl_variant_ms_per_step")}
        rec["workload"] = f"{workload}: {WORKLOADS[workload]['desc']}"
        if res.get("mesh"):
            rec["mesh"] = res["mesh"]
        if with_cpu and rank == 0 and world == 1 and not args.no_cpu:
            rec["cpu_baseline"] = cpu_baseline_single(workload, pk, budget_s=4.0)
        return rec

    extra = {}
    if not args.no_extra and args.workload == "c3" and not args.mesh and args.nk is None:
        # C3 as a k-grid through the mesh entry point (no k array; Fourier sum factorised over the last dimension)
        r = measure("c3", packed, total, steps, 3, ctx, None, peaks, args.e2e_nk, use_mesh=True)
        extra["c3_kgrid"] = brief(r, "c3", packed, with_cpu=False)
        extra["c3_kgrid"]["workload"] += " via eigenval_mesh"
        if world == 1:
            # eigenvalues + eigenvectors (SURVEY section 8 f4, extension API): 2^18 points of the same mesh
            import torch

            import tbmodels_b200 as tbk

            ev = tbk.Evaluator(packed, device=dev.index)
            n_e = 1 << 18
            k_e = shard_k_device("c3", cfg["dims"], total, 0, n_e, packed.dim, dev, 0)
            w_e = torch.empty((n_e, packed.size), dtype=torch.float64, device=dev)
            v_e = torch.empty((n_e, packed.size, packed.size), dtype=torch.complex128, device=dev)
            ev.profile(True)
            ms_e, l_e, prof_e = time_device_steps(ev, lambda: ev.eigh_device(k_e, out_w=w_e, out_v=v_e), 2, 3, None, dev)
            resid = (torch.linalg.norm(v_e[:8].mH @ v_e[:8] - torch.eye(packed.size, dtype=torch.complex128, device=dev)))
            assert float(resid) < 1e-10, "eigh: eigenvectors not orthonormal"
            extra["c3_eigh"] = {"workload": f"c3 model, eigenvalues AND eigenvectors (Evaluator.eigh_device) of {n_e} k-points per step",
                                "value": n_e * 2 / (ms_e * 1e-3), "unit": UNIT, "ms_per_step": ms_e / 2, "steps": 2, "warmup": 3,
                                "gpu_launches": int(l_e), "kernel_ms_per_step": {c: v[0] / 2 for c, v in prof_e.items() if v[1]},
                                "output_bytes_per_kpoint": 8 * packed.size + 16 * packed.size**2}
            # Model.hamilton (the other half of the reference API, row a1): complex128 [n_k, N, N] out, both conventions
            h_e = v_e  # same shape / dtype: reuse the buffer
            ham = {}
            for conv in (2, 1):
                ms_h, l_h, prof_h = time_device_steps(ev, lambda: ev.hamilton_device(k_e, convention=conv, out=h_e), 2, 3, None, dev)
                ham[f"convention_{conv}"] = {"value": n_e * 2 / (ms_h * 1e-3), "ms_per_step": ms_h / 2,
                                             "kernel_ms_per_step": {c: v[0] / 2 for c, v in prof_h.items() if v[1]}}
            extra["c3_hamilton"] = {"workload": f"c3 model, Model.hamilton of {n_e} k-points per step (device-resident in and out)",
                                    "unit": "k-points/s (hamilton)", "output_bytes_per_kpoint": 16 * packed.size**2, **ham}
            ev.close()
            del k_e, w_e, v_e, h_e
            torch.cuda.empty_cache()
        # C5: N_k sweep of the strong-scaling configuration (explicit k-points of 2^m-point meshes)
        p5 = build_model("c5")
        sweep = {}
        for e in (14, 16, 18, 20):
            if (1 << e) % world:
                continue
            r = measure("c5", p5, 1 << e, 3 if e <= 16 else 1, 3 if e <= 16 else 1, ctx, None, peaks, 1 << 14)
            sweep[f"2^{e}"] = {k: r[k] for k in ("value", "ms_per_step", "kpoints_per_gpu", "kernel_ms_per_step", "allgather_ms", "gather", "nccl_variant_ms_per_step", "steps", "warmup")}
            if e == 14 or (e == 16 and "c5" not in extra):
                extra["c5"] = brief(r, "c5", p5, with_cpu=(e == 14))
        extra["c5_sweep"] = {"workload": "c5: " + WORKLOADS["c5"]["desc"].split(",")[0] + ", N_k = 2^14 .. 2^20 (total, strong scaling)",
                             "unit": UNIT, "points": sweep}
        del p5
        if world >= 8 and 10**5 % world == 0:  # C4 at its stated size: 1e5 k-points over the 8 GPUs (12 500 each)
            pk = build_model("c4")
            r = measure("c4", pk, 10**5, 2, 1, ctx, None, peaks, 2048)
            extra["c4"] = brief(r, "c4", pk, with_cpu=False)
            del pk
        if world == 1:
            for name, tot, st, wu in (("c2", 10**8, 20, 5), ("c1", 8000, 50, 5), ("c4", 12500, 2, 1)):
                pk = build_model(name)
                r = measure(name, pk, tot, st, wu, ctx, None, peaks, None)
                extra[name] = brief(r, name, pk)
                if name == "c4":
                    extra[name]["workload"] += " -- 12 500 of them per step (one GPU's share of the 8-GPU configuration)"
                del pk
    sampler.mark("run_end")
    clocks = sampler.stop()

    # ---- CPU baseline: the reference on this box's host cores (rank 0, N = 1 only) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_baseline_single(args.workload, packed, budget_s=10.0)

    if rank == 0:
        line = {
            "metric": METRIC,
            "value": main["value"],
            "unit": UNIT,
            "n_gpus": world,
            "steps": steps,
            "warmup": warmup,
            "ms_per_step": main["ms_per_step"],
            "higher_is_better": True,
            "scaling": "strong",
            "vs_baseline": None,
            "dtype": "f64",
            "data": "synthetic",
            # `config` is identical in both arms (the driver compares them); what is specific to the GPU run is in `run`
            "config": workload_config(args.workload, packed, main["kpoints_total"]),
            "run": {
                "kpoints_per_gpu": main["kpoints_per_gpu"],
                "path": main["path"],
                "parallelism": f"contiguous k-shards x{world}" + (f", exchange inside the timed region: {main['gather']}" if world > 1 else ""),
                "l2": l2_note(main, packed),
                **({"mesh": main["mesh"]} if main.get("mesh") else {}),
            },
            "clocks": clocks,
            "e2e": main["e2e"],
            "gpu_launches": main["gpu_launches"],
            "roofline": main["roofline"],
            "kernels": main["kernels"],
            "cpu_baseline": cpu,
            "fp64_peak_tflops": peaks,
            "kernel_ms_per_step": main["kernel_ms_per_step"],
            "allgather_ms": main["allgather_ms"],
            "gather": main["gather"],
            "gather_fallback_reason": main["gather_fallback_reason"],
            "nccl_variant_ms_per_step": main["nccl_variant_ms_per_step"],
            "gather_rows_checked_bit_exact": main["gather_rows_checked"],
            "extra": extra,
        }
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", choices=sorted(WORKLOADS), default="c3")
    ap.add_argument("--nk", type=int, default=None, help="TOTAL k-points per step over all GPUs (default: the configuration's)")
    ap.add_argument("--e2e-nk", type=int, default=None, help="cap the k-points per GPU of an e2e step")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--no-peaks", action="store_true")
    ap.add_argument("--mesh", action="store_true", help="c1 / c3 / c5: evaluate the workload's k-grid through eigenval_mesh")
    ap.add_argument("--no-fused-gather", action="store_true", help="N > 1: NCCL all-gather after the evaluation instead of the fused peer stores")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the eigenvalues of the last timed step (seeded row sample above 32 MiB) to DIR/eigenvalues.npy")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU arm's results (--impl ours)")
    _NO_FUSED[0] = args.no_fused_gather
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
