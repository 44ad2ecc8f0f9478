#!/usr/bin/env python
"""Faraday-rotation polarimetry out of core: the Faraday channel (ne and B) streamed slab by slab with the density.

(a) bench.py's C2 field (turbulent 512^3) with ``B_on=True``, B from ``polarimetry_bench.analytic_B`` and a fused Stokes
    image: RK4 in core against out of core (slabs of 160 planes cut from device tensors; both times, bit-identity of rf,
    Jf, sf and the Stokes planes), then per-ray RK45 at SciPy's tolerances on 2e6 rays with ``max_slab_planes=512``
    (every slab logged: SciPy's first attempts span about half the box, so the slab may have to grow).
(b) a 1536^3 ``turbulent_ne_slabs`` field (res 768) with the same B generated per slab on the device: an image that does
    not fit in core on one GPU (the packed field and the four float64 Faraday grids alone are 174 GB).  Construction time,
    time per slab, the 1e7-ray RK4 trace with its Stokes image, peak device memory (torch allocations plus the largest
    slab field), and whether the rotation angle is finite wherever a ray landed.

Times are host clock ending in a synchronise.  One JSON line per run on stdout (and appended to ``--out``), each with the
card name and power limit.

    python examples/out_of_core_polarimetry.py [--parts a,b] [--out profiles/out_of_core_polarimetry_b200.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
from time import perf_counter

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, ".."))
sys.path.insert(0, HERE)

import bench  # noqa: E402
from polarimetry_bench import analytic_B  # noqa: E402
from synthpy_b200 import beam as B, diagnostics as D, domain as Dm, field_generator as FG  # noqa: E402
from synthpy_b200 import out_of_core as OC, propagator as P  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [v.strip() for v in q.split(",")]
        return name, power
    except Exception:
        return torch.cuda.get_device_name(0), "unknown"


def emit(line, out):
    print(json.dumps(line), flush=True)
    if out:
        with open(out, "a") as fh:
            fh.write(json.dumps(line) + "\n")


def reset():
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    return torch.cuda.memory_allocated()


def timed(fn):
    torch.cuda.synchronize()
    t0 = perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, perf_counter() - t0


def part_a(a, name, power):
    grid = 512
    ne = bench.build_ne(bench.parse(["--workload", "C2", "--grid", str(grid)]), "cuda")
    Bf = analytic_B(grid)
    dom = Dm.ScalarDomain(bench.LENGTHS, grid, B_on=True)
    dom.external_ne(ne)
    dom.external_B(Bf)
    lines = []
    # RK4, in core against out of core
    s0 = B.Beam(int(a.rays), bench.BEAM_R, bench.BEAM_DIV, bench.EXTENT, device=True, seed=2).materialise()
    oc = dict(slab_planes=a.slab_planes, lwl=bench.LWL, return_E=True, return_state=True, B_on=True, B=Bf)
    src = OC.array_source(ne)

    def in_core(spec):
        out = P.solve(s0, dom, bench.EXTENT, lwl=bench.LWL, return_E=True, return_state=True)
        P.solve_and_image(dom, s0, bench.EXTENT, [spec], lwl=bench.LWL)
        return out

    def out_of_core(spec):
        return OC.solve_out_of_core(s0, src, bench.LENGTHS, grid, bench.EXTENT, diagnostics=[spec], **oc)

    in_core(D.spec("shadow_two", bin_scale=4, stokes=True)), out_of_core(D.spec("shadow_two", bin_scale=4, stokes=True))  # warm-up
    si, so = D.spec("shadow_two", bin_scale=4, stokes=True), D.spec("shadow_two", bin_scale=4, stokes=True)
    (rf, Jf, _, ex), t_in = timed(lambda: in_core(si))
    (rf2, Jf2, _, ex2), t_oc = timed(lambda: out_of_core(so))
    lines.append({"part": "a", "gpu": name, "power_limit": power, "method": "rk4", "grid": grid, "rays": int(a.rays),
                  "slab_planes": a.slab_planes, "slabs": len(ex2["slabs"]), "in_core_s": round(t_in, 4),
                  "out_of_core_s": round(t_oc, 4), "in_core_timing": "solve + solve_and_image",
                  "out_of_core_timing": "one solve_out_of_core with the fused Stokes image",
                  "identical_rf": bool(torch.equal(rf, rf2)), "identical_Jf": bool(torch.equal(Jf, Jf2)),
                  "identical_sf": bool(torch.equal(ex["sf"], ex2["sf"])),
                  "identical_steps": bool(torch.equal(ex["steps"].long(), ex2["steps"].long())),
                  "identical_stokes": bool(torch.equal(si.image.planes, so.image.planes)),
                  "max_abs_pol": float(ex["sf"][8].abs().max())})
    # RK45 per ray, 2e6 rays, the slab allowed to grow to the whole grid
    s1 = B.Beam(int(a.rays_rk45), bench.BEAM_R, bench.BEAM_DIV, bench.EXTENT, device=True, seed=3).materialise()
    (rf, Jf, _, ex), t_in = timed(lambda: P.solve(s1, dom, bench.EXTENT, lwl=bench.LWL, method="rk45", return_E=True,
                                                  return_state=True))
    (rf2, Jf2, _, ex2), t_oc = timed(lambda: OC.solve_out_of_core(s1, src, bench.LENGTHS, grid, bench.EXTENT, method="rk45",
                                                                  max_slab_planes=grid, **oc))
    slabs = ex2["slabs"]
    lines.append({"part": "a", "gpu": name, "power_limit": power, "method": "rk45", "grid": grid, "rays": int(a.rays_rk45),
                  "slab_planes": a.slab_planes, "max_slab_planes": grid, "launches": len(slabs),
                  "slabs": [dict(planes=list(e["planes"]), launched=e["launched"], finished=e["finished"], parked=e["parked"],
                                 parked_pending=e["parked_pending"], attempts=e["attempts"]) for e in slabs],
                  "largest_slab_planes": max(e["planes"][1] - e["planes"][0] + 1 for e in slabs),
                  "in_core_s": round(t_in, 4), "out_of_core_s": round(t_oc, 4),
                  "attempts_in_core": ex["stats"]["ray_steps"], "attempts_out_of_core": ex2["stats"]["ray_steps"],
                  "rhs_evals_in_core": ex["stats"]["rhs_evals"], "rhs_evals_out_of_core": ex2["stats"]["rhs_evals"],
                  "identical_rf": bool(torch.equal(rf, rf2)), "identical_Jf": bool(torch.equal(Jf, Jf2)),
                  "identical_sf": bool(torch.equal(ex["sf"], ex2["sf"])),
                  "identical_steps": bool(torch.equal(ex["steps"].long(), ex2["steps"].long()))})
    return lines


def part_b(a, name, power):
    n = 1536
    base = reset()
    t0 = perf_counter()
    src = FG.turbulent_ne_slabs(n // 2, seed=1, block_planes=64)
    torch.cuda.synchronize()
    build_s = perf_counter() - t0
    x, y = [torch.linspace(-L / 2, L / 2, n, dtype=torch.float64, device="cuda") for L in bench.LENGTHS[:2]]
    XX, YY = torch.meshgrid(x, y, indexing="ij")
    plane = torch.stack([5.0 * YY / 5e-3, -5.0 * XX / 5e-3, 10.0 * torch.exp(-(XX ** 2 + YY ** 2) / (3e-3) ** 2)], -1)
    del XX, YY

    def bsrc(k0, k1):                                    # analytic_B's field, one slab at a time
        return plane[:, :, None, :].expand(n, n, k1 - k0, 3).contiguous()
    s0 = B.Beam(int(a.rays), bench.BEAM_R, bench.BEAM_DIV, bench.EXTENT, device=True, seed=2).materialise()
    spec = D.spec("shadow_two", bin_scale=4, stokes=True)
    rf, _, trace_s, ex = OC.solve_out_of_core(s0, src, bench.LENGTHS, n, bench.EXTENT, slab_planes=a.slab_planes, lwl=bench.LWL,
                                              diagnostics=[spec], return_state=True, B_on=True, B=bsrc)
    torch_peak = torch.cuda.max_memory_allocated() - base
    field_peak = max(e["field_bytes"] for e in ex["slabs"])
    S = spec.image.stokes()
    ang = 0.5 * torch.atan2(-S["U"], -S["Q"])
    hit = S["N"] > 0
    return [{"part": "b", "gpu": name, "power_limit": power, "method": "rk4", "grid": n, "res": n // 2, "rays": int(a.rays),
             "slab_planes": a.slab_planes, "slabs": len(ex["slabs"]), "construct_s": round(build_s, 3),
             "trace_s": round(trace_s, 3), "s_per_slab": round(trace_s / len(ex["slabs"]), 3),
             "ray_steps": int(ex["stats"]["ray_steps"]), "torch_peak_bytes": int(torch_peak),
             "largest_slab_field_bytes": int(field_peak), "peak_device_bytes": int(torch_peak + field_peak),
             "pixels_hit": int(hit.sum()), "angle_finite_where_hit": bool(torch.isfinite(ang[hit]).all()),
             "max_abs_angle": float(ang[hit].abs().max()), "max_abs_pol": float(ex["sf"][8].abs().max()),
             "timing": "host clock ending in torch.cuda.synchronize(); trace_s includes generating and packing every slab"}]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parts", default="a,b")
    ap.add_argument("--rays", type=float, default=1e7)
    ap.add_argument("--rays-rk45", type=float, default=2e6)
    ap.add_argument("--slab-planes", type=int, default=160)
    ap.add_argument("--out", default=None, help="append the JSON lines to this file")
    a = ap.parse_args()
    name, power = card()
    parts = a.parts.split(",")
    if "a" in parts:
        for line in part_a(a, name, power):
            emit(line, a.out)
    if "b" in parts:
        for line in part_b(a, name, power):
            emit(line, a.out)


if __name__ == "__main__":
    main()
