"""Throughput of Evaluator.berry_curvature_device next to band_velocity_device and eigh_device (GPU box).

    python tools/berry_bench.py [--out profiles/berry_bench.json] [--steps 5]

Workloads (oracle/workloads.py, the models of bench.py): C3 (N = 36, 2^18 random k-points), C5 (N = 128, 2^15), C4
(silicon 4x4x4 supercell, N = 512, 512 k-points) and the 2-band C2 model (N = 2, 2^22).  C2 runs the FMA variant of the
product kernel, the others its DMMA variant.  k-points are seeded random points in [0, 1)^dim on the device.  Per workload
and entry point: k-points/s from CUDA events around `steps` calls after two warm-up calls, then the per-class device time
of one call (tbk_profile_read).  Kernel times come from one more call per entry point under torch.profiler, in a pass of
their own: the product kernel (berry_product_kernel / berry_product_small_kernel), the curvature kernel
(berry_curvature_kernel) and the velocity kernel (band_velocity_kernel).  The product kernel's FP64 rate counts the
flops of two complex N x N products per direction and k-point (16 dim N^3), over tbk_measure_fp64_peak(0) (DMMA) of this
run.  Writes one JSON line (GPU name and power limit read in the same run)."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

KERNELS = {"product": ("berry_product",), "curvature": ("berry_curvature_kernel",), "velocity": ("band_velocity_kernel",)}


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in out.split(","))
        return {"gpu": name, "power_limit": power, "clocks_max_sm": clock}
    except Exception as exc:  # noqa: BLE001 -- the numbers are still worth writing
        return {"gpu": "unknown", "error": str(exc)}


def kernel_ms(call):
    """Device milliseconds per kernel group of one call, from torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call()
        torch.cuda.synchronize()
    out = {g: 0.0 for g in KERNELS}
    for ev in prof.events():
        if str(getattr(ev, "device_type", "")).endswith("CUDA"):
            us = getattr(ev, "device_time", None)
            if us is None:
                us = getattr(ev, "cuda_time", 0.0)
            for g, keys in KERNELS.items():
                if any(k in ev.name for k in keys):
                    out[g] += us / 1e3
    return {g: round(v, 4) for g, v in out.items() if v}


def main():
    import numpy as np  # noqa: F401
    import torch

    import tbmodels_b200 as tbk
    from oracle import workloads as wl
    from tbmodels_b200 import _capi

    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "berry_bench.json"))
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--only", default="", help="comma-separated workload names (default: all)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("berry_bench.py needs a CUDA device")
    silicon = wl.load_packed(os.path.join(ROOT, "tests", "golden", "silicon.npz"))
    workloads = [
        ("c3", "synthetic N=36 251 stored R (seed 1234)", lambda: wl.synthetic(36, 250, seed=1234), 1 << 18),
        ("c5", "synthetic N=128 1001 stored R (seed 1234)", lambda: wl.synthetic(128, 1000, seed=1234), 1 << 15),
        ("c4", "silicon 4x4x4 supercell N=512", lambda: wl.supercell(silicon, (4, 4, 4)), 512),
        ("c2", "2-band Haldane model N=2 D=2", wl.haldane, 1 << 22),
    ]
    if args.only:
        workloads = [w for w in workloads if w[0] in args.only.split(",")]
    peak = float(_capi.load().tbk_measure_fp64_peak(0, 4000))
    rec = {"tool": "tools/berry_bench.py", "time": time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime()), **gpu_info(),
           "torch": torch.__version__, "steps": args.steps, "fp64_dmma_peak_tflops": round(peak, 3), "results": {}}
    for name, desc, make, nk in workloads:
        p = make()
        ev = tbk.Evaluator(p, device=0)
        gen = torch.Generator(device="cuda").manual_seed(1234)
        k = torch.rand((nk, p.dim), dtype=torch.float64, device="cuda", generator=gen)
        n, dim = p.size, p.dim
        w = torch.empty((nk, n), dtype=torch.float64, device="cuda")
        cbuf = torch.empty((nk, n, dim * (dim - 1) // 2), dtype=torch.float64, device="cuda")
        calls = {
            "eigh_device": (lambda v=torch.empty((nk, n, n), dtype=torch.complex128, device="cuda"):
                            ev.eigh_device(k, out_w=w, out_v=v)),
            "band_velocity_device": (lambda v=torch.empty((nk, n, dim), dtype=torch.float64, device="cuda"):
                                     ev.band_velocity_device(k, out_w=w, out_v=v)),
            "berry_curvature_device_c2": lambda: ev.berry_curvature_device(k, convention=2, out_w=w, out_c=cbuf),
            "berry_curvature_device_c1": lambda: ev.berry_curvature_device(k, convention=1, out_w=w, out_c=cbuf),
        }
        res = {"workload": f"{name}: {desc}, {nk} random k-points", "n_orb": n, "dim": dim, "kpoints": nk,
               "product_variant": "fma" if n <= 8 else "dmma"}
        for cname, call in calls.items():
            for _ in range(2):
                call()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(args.steps):
                call()
            b.record()
            torch.cuda.synchronize()
            ev.check()
            ms = a.elapsed_time(b) / args.steps
            ev.profile(True)
            call()
            prof = {c: round(t, 4) for c, (t, cnt) in ev.profile_read().items() if cnt}
            ev.profile(False)
            res[cname] = {"ms_per_call": round(ms, 4), "kpoints_per_s": nk / ms * 1e3, "profile_ms": prof}
            print(f"{name} {cname}: {ms:.3f} ms per call, {nk / ms * 1e3:.4g} k-points/s, classes {prof}", flush=True)
        for cname in ("band_velocity_device", "berry_curvature_device_c2", "berry_curvature_device_c1"):
            res[cname]["kernel_ms"] = kernel_ms(calls[cname])
            print(f"{name} {cname}: kernels {res[cname]['kernel_ms']}", flush=True)
        for cname in ("berry_curvature_device_c2", "berry_curvature_device_c1"):
            km = res[cname]["kernel_ms"]
            if km.get("product"):
                tf = 16.0 * dim * n ** 3 * nk / (km["product"] * 1e-3) / 1e12
                res[cname]["product_fp64_tflops"] = round(tf, 4)
                res[cname]["product_share_of_dmma_peak"] = round(tf / peak, 4) if peak > 0 else None
                res[cname]["product_ms_per_kpoint"] = km["product"] / nk
        vk = res["band_velocity_device"]["kernel_ms"].get("velocity")
        if vk:
            res["velocity_kernel_ms_per_kpoint"] = vk / nk
        rec["results"][name] = res
        ev.close()
        del k, w, cbuf, calls
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(json.dumps(rec) + "\n")
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
