#!/usr/bin/env python
"""Cost of the Stokes (polarimetry) detector image and of the Faraday-rotation integrator on bench.py's C2 field
(turbulent 512^3 by default): device-generated rays, fixed-step RK4 at half a cell, two-lens shadowgraphy train.
Three cases, alternated pass by pass after warm-up so that they see the same machine state:

  a  B_on=False, histogram channel                       (bench.py's fast path)
  b  a + a Stokes channel on the same rays                (cost of the Stokes epilogue)
  c  B_on=True, Stokes channel                            (the float64 RK4 kernel that integrates amp / pol)

The B field is smooth and analytic, built on the device: an azimuthal field of 5 T at 5 mm plus a 10 T axial column of
3 mm radius (golden g6's field, whose box has the same size).  One JSON line per case on stdout (and in ``--out``):
ms per pass (CUDA events; median and spread over the timed passes), rays*steps/s, HBM held by the packed field and
its channel grids, and the GPU's name and power limit read in the same run.

    python examples/polarimetry_bench.py [--grid 512] [--rays 1e7] [--passes 5] [--warmup 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from synthpy_b200 import beam as B, diagnostics as D, domain as Dm, engine, propagator as P  # noqa: E402


def gpu_identity():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [v.strip() for v in q.split(",")]
        return name, power
    except Exception:                                     # no nvidia-smi: name only
        return torch.cuda.get_device_name(), "unknown"


def analytic_B(grid):
    x, y, _ = [torch.linspace(-L / 2, L / 2, grid, dtype=torch.float64, device="cuda") for L in bench.LENGTHS]
    XX, YY = torch.meshgrid(x, y, indexing="ij")
    Bf = torch.empty((grid, grid, grid, 3), dtype=torch.float64, device="cuda")
    Bf[..., 0] = (5.0 * YY / 5e-3)[..., None]
    Bf[..., 1] = (-5.0 * XX / 5e-3)[..., None]
    Bf[..., 2] = (10.0 * torch.exp(-(XX ** 2 + YY ** 2) / (3e-3) ** 2))[..., None]
    return Bf


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grid", type=int, default=512)
    ap.add_argument("--rays", type=float, default=1e7)
    ap.add_argument("--passes", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="append the JSON lines to this file")
    a = ap.parse_args()
    if a.passes < 1 or a.warmup < 1:
        ap.error("--passes and --warmup must be at least 1")
    engine.require_cuda()
    ne = bench.build_ne(bench.parse(["--workload", "C2", "--grid", str(a.grid)]), "cuda")
    dom_plain = Dm.ScalarDomain(bench.LENGTHS, a.grid)
    dom_plain.external_ne(ne)
    dom_far = Dm.ScalarDomain(bench.LENGTHS, a.grid, B_on=True)
    dom_far.external_ne(ne)
    dom_far.external_B(analytic_B(a.grid))
    beam = B.Beam(int(a.rays), bench.BEAM_R, bench.BEAM_DIV, bench.EXTENT, device=True, seed=2)
    cases = {
        "a": (dom_plain, [D.spec("shadow_two")]),
        "b": (dom_plain, [D.spec("shadow_two"), D.spec("shadow_two", stokes=True)]),
        "c": (dom_far, [D.spec("shadow_two", stokes=True)]),
    }
    ms = {k: [] for k in cases}
    stats = {}
    for it in range(a.warmup + a.passes):
        for k, (dom, specs) in cases.items():
            for s in specs:
                s.image.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            st, _ = P.solve_and_image(dom, beam, bench.EXTENT, specs, lwl=bench.LWL, method="rk4", sync=False)
            e1.record()
            e1.synchronize()
            if it >= a.warmup:
                ms[k].append(e0.elapsed_time(e1))
            stats[k] = st
    name, power = gpu_identity()
    hist_a = cases["a"][1][0].image.counts
    checks = {"b": {"histogram_equals_a": bool(torch.equal(cases["b"][1][0].image.counts, hist_a)),
                    "stokes_N_equals_histogram": bool(torch.equal(cases["b"][1][1].image.planes[0], hist_a))}}
    lines = []
    for k, (dom, specs) in cases.items():
        s = engine.stats_dict(stats[k])
        med = float(np.median(ms[k]))
        field = dom.device_field(bench.LWL, phase=False)
        lines.append(dict(
            case=k, kinds=[sp.image.kind for sp in specs], B_on=bool(dom.B_on), grid=a.grid, rays=int(a.rays),
            integrator="rk4, ds = 0.5 cell, early exit", train="shadow_two", timing="CUDA events, alternated a/b/c",
            warmup_passes=a.warmup, timed_passes=a.passes, ms_per_pass=round(med, 3),
            ms_min=round(min(ms[k]), 3), ms_max=round(max(ms[k]), 3),
            ray_steps=s["ray_steps"], ray_steps_per_s=s["ray_steps"] / (med * 1e-3),
            field_hbm_bytes=field.nbytes, image_hbm_bytes=sum(sp.image.tensors()[0].numel() * 8 for sp in specs),
            rays_binned=s["rays_binned"], checks=checks.get(k, {}), gpu=name, power_limit=power))
    for line in lines:
        print(json.dumps(line))
    if a.out:
        with open(a.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
