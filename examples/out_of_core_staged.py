#!/usr/bin/env python
"""Stage parking against attempt parking for the out-of-core adaptive solves, against the in-core solve of the same grid:
bench.py's C2 field (turbulent 512^3), 2e6 device-generated rays, slabs of 160 planes cut from a resident device tensor
(so the figures are the cost of the launches and the re-packing, not of host I/O).

Methods: RK45 at SciPy's tolerances (1e-3 / 1e-6), Tsit5 at upstream's controller (1 / 1e-5) and at 1e-7 / 1e-9, and RK45
with the Faraday channel (``B_on``, B from ``polarimetry_bench.analytic_B``).  Three runs each: in core,
``park='attempt'`` with ``max_slab_planes=512`` (the slab may grow to the whole grid) and ``park='stage'`` (it never
grows).  Each run is warmed up once, then timed ``--repeats`` times (host clock ending in a synchronise); its peak device
memory is the torch peak plus the largest slab field (in core: plus the whole field).  One JSON line per method on stdout
(and appended to ``--out``), with the card name and power limit.

    python examples/out_of_core_staged.py [--rays 2e6] [--slab-planes 160] [--repeats 2] [--out profiles/out_of_core_staged_b200.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
from time import perf_counter

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, ".."))
sys.path.insert(0, HERE)

import bench  # noqa: E402
from polarimetry_bench import analytic_B  # noqa: E402
from synthpy_b200 import beam as B, domain as Dm, out_of_core as OC, propagator as P  # noqa: E402

METHODS = {"rk45": ("rk45", {}, False), "tsit5_upstream": ("tsit5", dict(rtol=1.0, atol=1e-5), False),
           "tsit5_tight": ("tsit5", dict(rtol=1e-7, atol=1e-9), False), "rk45_B": ("rk45", {}, True)}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [v.strip() for v in q.split(",")]
        return name, power
    except Exception:
        return torch.cuda.get_device_name(0), "unknown"


def timed(fn, repeats):
    """Warm-up, then ``repeats`` timed calls; the last call's output, its times and its peak device memory."""
    fn()
    times = []
    for _ in range(repeats):
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        t0 = perf_counter()
        out = fn()
        torch.cuda.synchronize()
        times.append(round(perf_counter() - t0, 4))
        peak = torch.cuda.max_memory_allocated() - base
    return out, times, peak


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grid", type=int, default=512)
    ap.add_argument("--rays", type=float, default=2e6)
    ap.add_argument("--slab-planes", type=int, default=160)
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--methods", default=",".join(METHODS))
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    args = bench.parse(["--workload", "C2", "--grid", str(a.grid)])
    ne = bench.build_ne(args, "cuda")
    s0 = B.Beam(int(a.rays), bench.BEAM_R, bench.BEAM_DIV, bench.EXTENT, device=True, seed=2).materialise()
    src = OC.array_source(ne)
    name, power = card()
    for key in a.methods.split(","):
        method, kw, b_on = METHODS[key]
        ch = {}
        dom = Dm.ScalarDomain(bench.LENGTHS, a.grid, B_on=b_on)
        dom.external_ne(ne)
        if b_on:
            Bg = analytic_B(a.grid)
            dom.external_B(Bg)
            ch = dict(B_on=True, B=Bg)
        field_bytes = dom.device_field(bench.LWL).nbytes

        def in_core():
            return P.solve(s0, dom, bench.EXTENT, lwl=bench.LWL, method=method, return_state=True, **kw)

        def out_of_core(park):
            extra = dict(max_slab_planes=a.grid) if park == "attempt" else {}
            return OC.solve_out_of_core(s0, src, bench.LENGTHS, a.grid, bench.EXTENT, slab_planes=a.slab_planes, lwl=bench.LWL,
                                        method=method, return_state=True, park=park, **kw, **extra, **ch)

        (rf, _, _, ex), t_in, peak_in = timed(in_core, a.repeats)
        line = {"card": name, "power_limit": power, "method": key, "solver": method, **{k: v for k, v in kw.items()},
                "B_on": b_on, "grid": a.grid, "rays": int(a.rays), "slab_planes": a.slab_planes,
                "in_core": dict(s=t_in, peak_bytes=peak_in + field_bytes, rhs_evals=ex["stats"]["rhs_evals"],
                                attempts=ex["stats"]["ray_steps"])}
        for park in ("attempt", "stage"):
            (rf2, _, _, ex2), t, peak = timed(lambda: out_of_core(park), a.repeats)
            slabs = ex2["slabs"]
            run = dict(s=t, launches=len(slabs), max_planes=max(e["planes"][1] - e["planes"][0] + 1 for e in slabs),
                       peak_bytes=peak + max(e["field_bytes"] for e in slabs), rhs_evals=ex2["stats"]["rhs_evals"],
                       attempts=ex2["stats"]["ray_steps"], identical_rf=bool(torch.equal(rf, rf2)),
                       identical_sf=bool(torch.equal(ex["sf"], ex2["sf"])),
                       identical_steps=bool(torch.equal(ex["steps"].long(), ex2["steps"].long())),
                       slabs=[dict(planes=list(e["planes"]), launched=e["launched"], finished=e["finished"],
                                   parked=e["parked"], attempts=e["attempts"],
                                   **({"evals": e["evals"], "parked_mid": e["parked_mid"]} if park == "stage" else {}))
                              for e in slabs])
            line[park] = run
        print(json.dumps(line), flush=True)
        if a.out:
            with open(a.out, "a") as fh:
                fh.write(json.dumps(line) + "\n")
        del dom


if __name__ == "__main__":
    main()
