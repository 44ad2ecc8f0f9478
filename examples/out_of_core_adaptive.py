#!/usr/bin/env python
"""Out-of-core tracing with the per-ray adaptive solves against the in-core solve of the same grid: bench.py's C2 field
(turbulent 512^3), device-generated rays, RK45 per ray at SciPy's tolerances (the C4 workload's integrator) and Tsit5 at
1e-7 / 1e-9.  Slabs are cut from a resident device tensor, so the figures are the cost of the extra launches, the dropped
attempts and the re-packing, not of host I/O.  In-core and out-of-core runs alternate after a warm-up; times are host
clock ending in a synchronise.  One JSON line per method on stdout, with the card name and power limit.

    python examples/out_of_core_adaptive.py [--grid 512] [--rays 1e7] [--slab-planes 160] [--repeats 2]
"""
import argparse
import json
import os
import subprocess
import sys
from time import perf_counter

import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from synthpy_b200 import beam as B, domain as Dm, out_of_core as OC, propagator as P  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [v.strip() for v in q.split(",")]
        return name, power
    except Exception:
        return torch.cuda.get_device_name(0), "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grid", type=int, default=512)
    ap.add_argument("--rays", type=float, default=1e7)
    ap.add_argument("--slab-planes", type=int, default=160)
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--methods", default="rk45,tsit5")
    a = ap.parse_args()
    args = bench.parse(["--workload", "C2", "--grid", str(a.grid)])
    ne = bench.build_ne(args, "cuda")
    dom = Dm.ScalarDomain(bench.LENGTHS, a.grid)
    dom.external_ne(ne)
    s0 = B.Beam(int(a.rays), bench.BEAM_R, bench.BEAM_DIV, bench.EXTENT, device=True, seed=2).materialise()
    src = OC.array_source(ne)
    name, power = card()
    for method in a.methods.split(","):
        kw = dict(rtol=1e-7, atol=1e-9) if method == "tsit5" else {}

        def in_core():
            torch.cuda.synchronize()
            t0 = perf_counter()
            out = P.solve(s0, dom, bench.EXTENT, lwl=bench.LWL, method=method, return_state=True, **kw)
            torch.cuda.synchronize()
            return out, perf_counter() - t0

        def out_of_core():
            torch.cuda.synchronize()
            t0 = perf_counter()
            out = OC.solve_out_of_core(s0, src, bench.LENGTHS, a.grid, bench.EXTENT, slab_planes=a.slab_planes,
                                       max_slab_planes=a.grid, lwl=bench.LWL, method=method, return_state=True, **kw)
            torch.cuda.synchronize()
            return out, perf_counter() - t0

        in_core(), out_of_core()                                   # warm-up
        t_in, t_oc = [], []
        for _ in range(a.repeats):
            (rf, _, _, ex), t = in_core()
            t_in.append(t)
            (rf2, _, _, ex2), t = out_of_core()
            t_oc.append(t)
        slabs = ex2["slabs"]
        line = {"card": name, "power_limit": power, "method": method, "grid": a.grid, "rays": int(a.rays),
                "slab_planes": a.slab_planes, "launches": len(slabs),
                "slabs": [dict(planes=list(e["planes"]), launched=e["launched"], finished=e["finished"],
                               parked=e["parked"], parked_pending=e["parked_pending"], attempts=e["attempts"]) for e in slabs],
                "in_core_s": [round(t, 4) for t in t_in], "out_of_core_s": [round(t, 4) for t in t_oc],
                "attempts_in_core": ex["stats"]["ray_steps"], "attempts_out_of_core": ex2["stats"]["ray_steps"],
                "rhs_evals_in_core": ex["stats"]["rhs_evals"], "rhs_evals_out_of_core": ex2["stats"]["rhs_evals"],
                "identical_rf": bool(torch.equal(rf, rf2)), "identical_sf": bool(torch.equal(ex["sf"], ex2["sf"])),
                "identical_steps": bool(torch.equal(ex["steps"].long(), ex2["steps"].long()))}
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
