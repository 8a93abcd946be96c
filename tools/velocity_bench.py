"""Throughput of Evaluator.band_velocity_device next to eigenval_device and eigh_device (GPU box).

    python tools/velocity_bench.py [--out profiles/velocity_bench.json] [--steps 5]

Workloads (oracle/workloads.py, the models of bench.py): C3 (N = 36, 2^18 random k-points), C5 (N = 128, 2^15),
C4 (silicon 4x4x4 supercell, N = 512, 512 k-points: a batch whose velocity scratch fits comfortably) and the 2-band C2
model (2^22).  k-points are seeded random points in [0, 1)^dim on the device.  Per workload and entry point: k-points/s
from CUDA events around `steps` calls after two warm-up calls, then, in separate profiled calls, the per-class device
time (tbk_profile_read).  The velocity kernel shares class 7 with eigh, so its time is the class-7 time of
band_velocity minus that of eigh on the same batch; the dH/dk build is class 2.  Writes one JSON line (GPU name and power
limit read in the same run)."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in out.split(","))
        return {"gpu": name, "power_limit": power, "clocks_max_sm": clock}
    except Exception as exc:  # noqa: BLE001 -- the numbers are still worth writing
        return {"gpu": "unknown", "error": str(exc)}


def main():
    import numpy as np
    import torch

    import tbmodels_b200 as tbk
    from oracle import workloads as wl

    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "velocity_bench.json"))
    ap.add_argument("--steps", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("velocity_bench.py needs a CUDA device")
    silicon = wl.load_packed(os.path.join(ROOT, "tests", "golden", "silicon.npz"))
    workloads = [
        ("c3", "synthetic N=36 251 stored R (seed 1234)", lambda: wl.synthetic(36, 250, seed=1234), 1 << 18),
        ("c5", "synthetic N=128 1001 stored R (seed 1234)", lambda: wl.synthetic(128, 1000, seed=1234), 1 << 15),
        ("c4", "silicon 4x4x4 supercell N=512", lambda: wl.supercell(silicon, (4, 4, 4)), 512),
        ("c2", "2-band Haldane model N=2 D=2", wl.haldane, 1 << 22),
    ]
    rec = {"tool": "tools/velocity_bench.py", "time": time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime()), **gpu_info(),
           "torch": torch.__version__, "steps": args.steps, "results": {}}
    for name, desc, make, nk in workloads:
        p = make()
        ev = tbk.Evaluator(p, device=0)
        gen = torch.Generator(device="cuda").manual_seed(1234)
        k = torch.rand((nk, p.dim), dtype=torch.float64, device="cuda", generator=gen)
        n = p.size
        w = torch.empty((nk, n), dtype=torch.float64, device="cuda")
        calls = {
            "eigenval_device": lambda: ev.eigenval_device(k, out=w),
            "eigh_device": (lambda v=torch.empty((nk, n, n), dtype=torch.complex128, device="cuda"):
                            ev.eigh_device(k, out_w=w, out_v=v)),
            "band_velocity_device": (lambda v=torch.empty((nk, n, p.dim), dtype=torch.float64, device="cuda"):
                                     ev.band_velocity_device(k, out_w=w, out_v=v)),
        }
        res = {"workload": f"{name}: {desc}, {nk} random k-points", "n_orb": n, "kpoints": nk}
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
        e7 = res["eigh_device"]["profile_ms"].get("eigh", 0.0)
        v7 = res["band_velocity_device"]["profile_ms"].get("eigh", 0.0)
        dk = res["band_velocity_device"]["profile_ms"].get("expand", 0.0)
        res["velocity_kernel_ms"] = round(v7 - e7, 4)
        res["dH_build_ms"] = dk
        res["velocity_kernel_over_eigh"] = round((v7 - e7) / e7, 4) if e7 else None
        res["dH_build_over_eigh"] = round(dk / e7, 4) if e7 else None
        rec["results"][name] = res
        ev.close()
        del k, w, calls
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(json.dumps(rec) + "\n")
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
