#!/usr/bin/env python
"""Tracing a turbulent field that is never whole: ``field_generator.turbulent_ne_slabs`` makes the k^-11/3 field of
``turbulent_ne(res, noise='philox')`` slab by slab from one complex spectrum of about 8 bytes per grid point, and
``out_of_core.solve_out_of_core`` traces it.  At 2048^3 the float64 field alone would be 68.7 GB and its packed grid
137 GB; the source holds 68.8 GB, the trace one slab on top.

For each grid one JSON line on stdout (and in ``--out``):

  phase_a_s, max_pass_s   construction: the spectrum G with the inverse FFT along the probing axis, then one pass over
                          every block for max |f| (host clock ending in a device synchronise)
  block_ms                one block of ``--block-planes`` planes served from G (mean over all blocks, each made once)
  source_peak_bytes       torch.cuda.max_memory_allocated over construction and serving every block, above the baseline
  trace_s, rays_steps_per_s   solve_out_of_core of ``--rays`` device rays (engine.beam_generate, bench.py's C2 beam and
                          box) with a fused shadow_two image; rays·steps/s counts the launches' integrated ray steps
  trace_peak_bytes        max_memory_allocated over the trace, source included
  in_core                 grids up to ``--in-core-max``: the same trace through ``source(0, n)`` held whole
                          (propagator.solve_and_image / solve), and whether exit rays, states, steps and image are
                          bit-identical

and the GPU's name and power limit, read in the same run.

    python examples/out_of_core_turbulence.py [--grids 1024 2048] [--rays 1e7] [--slab-planes 256] [--block-planes 64]
                                              [--in-core-max 1024] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from synthpy_b200 import diagnostics as D, domain as Dm, engine, field_generator as FG, out_of_core as OC  # noqa: E402
from synthpy_b200 import propagator as P  # noqa: E402


def gpu_identity():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [v.strip() for v in q.split(",")]
        return name, power
    except Exception:                                     # no nvidia-smi: name only
        return torch.cuda.get_device_name(), "unknown"


def peak_since(base):
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def reset():
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    return torch.cuda.memory_allocated()


def run_grid(grid, a, name, power):
    n = grid
    base = reset()
    t0 = time.perf_counter()
    src = FG.turbulent_ne_slabs(n // 2, seed=a.seed, block_planes=a.block_planes)
    build_s = time.perf_counter() - t0
    times = []
    for k0 in range(0, n, a.block_planes):
        torch.cuda.synchronize()
        t = time.perf_counter()
        blk = src(k0, min(n, k0 + a.block_planes))
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t)
        del blk
    source_peak = peak_since(base)

    s0 = engine.beam_generate(engine.make_beam("circular", bench.BEAM_R, bench.BEAM_DIV, bench.EXTENT, "z", a.seed),
                              int(a.rays))
    reset()
    base_trace = 0                                        # the whole trace: the source's G counts
    spec = D.spec("shadow_two")
    rf, _, trace_s, ex = OC.solve_out_of_core(s0, src, bench.LENGTHS, n, bench.EXTENT, slab_planes=a.slab_planes,
                                              lwl=bench.LWL, diagnostics=[spec], return_state=True)
    trace_peak = peak_since(base_trace)
    ray_steps = ex["stats"]["ray_steps"]
    line = dict(grid=n, points=n ** 3, rays=int(a.rays), seed=a.seed, block_planes=a.block_planes,
                slab_planes=a.slab_planes, timing="host clock ending in torch.cuda.synchronize()",
                construct_s=round(build_s, 3), phase_a_s=round(src.build_seconds["phase_a"], 3),
                max_pass_s=round(src.build_seconds["max_pass"], 3), blocks=len(times),
                block_ms=round(1e3 * float(np.mean(times)), 2), block_ms_max=round(1e3 * max(times), 2),
                source_peak_bytes=int(source_peak), source_peak_bytes_per_point=round(source_peak / n ** 3, 3),
                trace_s=round(trace_s, 3), ray_steps=int(ray_steps), rays_steps_per_s=float(f"{ray_steps / trace_s:.4g}"),
                slabs=len(ex["slabs"]), trace_peak_bytes=int(trace_peak),
                trace_peak_bytes_per_point=round(trace_peak / n ** 3, 3), image_sum=float(spec.image.result().sum()),
                in_core=None, gpu=name, power_limit=power)
    if n <= a.in_core_max:
        ne = src(0, n)
        del src
        torch.cuda.empty_cache()
        dom = Dm.ScalarDomain(bench.LENGTHS, n)
        dom.external_ne(ne)
        del ne
        rf2, _, t_in, ex2 = P.solve(s0, dom, bench.EXTENT, lwl=bench.LWL, method="rk4", return_state=True)
        spec2 = D.spec("shadow_two")
        P.solve_and_image(dom, s0, bench.EXTENT, [spec2], lwl=bench.LWL, method="rk4")
        same = bool(torch.equal(rf, rf2) and torch.equal(ex["sf"], ex2["sf"]) and
                    torch.equal(ex["steps"].long(), ex2["steps"].long()) and
                    torch.equal(spec.image.result(), spec2.image.result()) and
                    ex["stats"]["ray_steps"] == ex2["stats"]["ray_steps"])
        line["in_core"] = dict(trace_s=round(t_in, 3), bit_identical=same)
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grids", type=int, nargs="+", default=[1024, 2048])
    ap.add_argument("--rays", type=float, default=1e7)
    ap.add_argument("--slab-planes", type=int, default=256)
    ap.add_argument("--block-planes", type=int, default=64)
    ap.add_argument("--in-core-max", type=int, default=1024, help="largest grid also traced in core for the identity check")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default=None, help="append the JSON lines to this file")
    a = ap.parse_args()
    if a.rays < 1 or a.slab_planes < 8 or a.block_planes < 1 or any(g < 8 or g % 2 for g in a.grids):
        ap.error("need --rays >= 1, --slab-planes >= 8, --block-planes >= 1 and even grids >= 8")
    engine.require_cuda()
    name, power = gpu_identity()
    warm = argparse.Namespace(**{**vars(a), "rays": 1e4, "slab_planes": 24})
    run_grid(64, warm, name, power)                       # module loads, cuFFT plans of the small shapes
    for grid in a.grids:
        line = run_grid(grid, a, name, power)
        print(json.dumps(line), flush=True)
        if a.out:
            with open(a.out, "a") as fh:
                fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
