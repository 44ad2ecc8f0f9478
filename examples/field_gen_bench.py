#!/usr/bin/env python
"""Cost of building the turbulent n_e field on the GPU with host-drawn noise (noise='torch') against device-drawn noise
(noise='philox': k_noise_spectrum writes the Hermitian half spectrum, then a real inverse FFT).

For each grid (512^3 = C2, 1024^3 = C5) the two modes alternate call by call after warm-up, so that they see the same
machine state.  One JSON line per (grid, mode) on stdout (and in ``--out``):

  wall_ms            field_generator.domain_fft(kolmogorov, 1, 0.01, 5, res) on a host clock ending in a device
                     synchronise (median, min, max over the timed calls)
  peak_alloc_bytes   torch.cuda.max_memory_allocated during one call, above what was allocated before it
  host_grid_bytes    host memory of grid size the call allocates, from the shapes: the float64 re and im noise arrays of
                     noise='torch' (16 bytes per point); 0 for noise='philox' (its host arrays are the two |k| axes)
  kernel_ms          philox only: CUDA-event time of one k_noise_spectrum launch (mean over --kernel-reps back-to-back
                     launches), next to hbm_floor_ms, its 20 bytes per half-grid point (4 read, 16 written) at the
                     B200 data sheet's 7.7 TB/s -- a bound, not a measured rate

and the GPU's name and power limit, read in the same run.

    python examples/field_gen_bench.py [--grids 512 1024] [--calls 2] [--warmup 1] [--kernel-reps 10] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)

from synthpy_b200 import _lib as L, engine, field_generator as FG  # noqa: E402

HBM_BYTES_PER_S = 7.7e12           # NVIDIA HGX B200 data sheet, one GPU
L_MAX, L_MIN, EXTENT = 1.0, 0.01, 5.0


def gpu_identity():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [v.strip() for v in q.split(",")]
        return name, power
    except Exception:                                     # no nvidia-smi: name only
        return torch.cuda.get_device_name(), "unknown"


def one_call(res, noise, seed):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    f = FG.domain_fft(FG.kolmogorov, L_MAX, L_MIN, EXTENT, res, noise=noise, seed=seed)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    return f, wall * 1e3, torch.cuda.max_memory_allocated() - base


def kernel_time(res, seed, reps):
    """k_noise_spectrum alone on the grid's half-grid S (CUDA events around `reps` launches)."""
    n = 2 * res
    k = 2 * np.pi * np.fft.fftfreq(n, d=EXTENT / res)
    S = FG.half_spectrum(FG.kolmogorov, L_MAX, L_MIN, (k, k, k))
    H = torch.empty(S.shape, dtype=torch.complex128, device="cuda")
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    launch = lambda: L.check(L.lib.sp_noise_spectrum(C.c_void_p(S.data_ptr()), n, n, n, seed, C.c_void_p(H.data_ptr()), stream))
    launch()                                              # warm-up (module load)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        launch()
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1) / reps
    half = S.numel()
    same = bool(torch.equal(H, engine.noise_spectrum(S, (n, n, n), seed)))
    del S, H
    return ms, half, same


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grids", type=int, nargs="+", default=[512, 1024])
    ap.add_argument("--calls", type=int, default=2, help="timed calls per mode and grid")
    ap.add_argument("--warmup", type=int, default=1, help="untimed calls per mode and grid first")
    ap.add_argument("--kernel-reps", type=int, default=10)
    ap.add_argument("--seed", type=int, default=3)
    ap.add_argument("--out", default=None, help="append the JSON lines to this file")
    a = ap.parse_args()
    if a.calls < 1 or a.warmup < 0 or a.kernel_reps < 1 or any(g < 2 or g % 2 for g in a.grids):
        ap.error("need --calls >= 1, --warmup >= 0, --kernel-reps >= 1 and even grids >= 2")
    engine.require_cuda()
    name, power = gpu_identity()
    lines = []
    for grid in a.grids:
        res, N = grid // 2, grid ** 3
        wall = {m: [] for m in ("torch", "philox")}
        peak = {m: 0 for m in wall}
        first_philox = None
        repeat_identical = True
        for it in range(a.warmup + a.calls):
            for mode in wall:
                f, ms, pk = one_call(res, mode, a.seed)
                if mode == "philox":
                    if first_philox is None:
                        first_philox = f.clone()
                    else:
                        repeat_identical &= bool(torch.equal(f, first_philox))
                del f
                if it >= a.warmup:
                    wall[mode].append(ms)
                    peak[mode] = max(peak[mode], pk)
        del first_philox
        k_ms, half, same = kernel_time(res, a.seed, a.kernel_reps)
        floor_ms = 20.0 * half / HBM_BYTES_PER_S * 1e3
        for mode in wall:
            lines.append(dict(
                grid=grid, points=N, mode=mode, call=f"domain_fft(kolmogorov, {L_MAX}, {L_MIN}, {EXTENT}, {res}, noise='{mode}')",
                timing="host clock ending in torch.cuda.synchronize(), modes alternated", warmup_calls=a.warmup,
                timed_calls=a.calls, wall_ms=round(float(np.median(wall[mode])), 3), wall_ms_min=round(min(wall[mode]), 3),
                wall_ms_max=round(max(wall[mode]), 3), peak_alloc_bytes=int(peak[mode]),
                peak_alloc_bytes_per_point=round(peak[mode] / N, 3), host_grid_bytes=16 * N if mode == "torch" else 0,
                kernel_ms=round(k_ms, 4) if mode == "philox" else None,
                hbm_floor_ms=round(floor_ms, 4) if mode == "philox" else None,
                half_grid_points=half if mode == "philox" else None,
                checks=dict(repeat_identical=repeat_identical, kernel_equals_wrapper=same) if mode == "philox" else {},
                gpu=name, power_limit=power))
    for line in lines:
        print(json.dumps(line))
    if a.out:
        with open(a.out, "a") as fh:
            for line in lines:
                fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
