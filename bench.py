#!/usr/bin/env python
"""Benchmark of the ray-propagation hot path (BASELINE.json metric: rays.steps/s, device-timed, max over ranks).

  python bench.py [--gpus N] [--steps K] [--warmup W]            our CUDA arm
  python bench.py --impl reference ...                           the reference's CPU algorithm (oracle port) on host cores
  torchrun --nproc-per-node N bench.py --gpus N ...              one rank per GPU, rays sharded, field replicated,
                                                                 detector images combined by one NCCL all-reduce

Default workload (BASELINE.json configs[1], "C2"): 1e7 rays per GPU through a 512^3 turbulent (k^-11/3 power spectrum,
field_generator.domain_fft) n_e field, lambda = 1064 nm, box 10 x 10 x 20 mm, circular beam r = 5 mm, divergence
5e-5; fixed-step RK4 with two steps per cell and early exit; shadowgraphy (two-lens) + dark-field schlieren
images at full 3448 x 2574 resolution fused into the propagation kernel.  One "step" = one pass of that whole
bundle.  Rays are generated on the device (Philox), so nothing but the replicated field is resident input.
--workload C1 / C3 / C4 / C5 select the other BASELINE configs (see ``workload_defaults``).

After the timed region rank 0 traces a sub-sample of the SAME rays through the SAME field with the CPU oracle
(oracle/, the checker) and prints the comparison under "parity".

--dump-outputs DIR: rank 0 writes what the last timed step handed its caller as DIR/<name>.npy (float64): one file per
detector channel (the image as ``image.result()`` returns it) and stats.npy (``engine.STAT_NAMES`` order), at most
64 MB in all (see ``dump_outputs``).  Field and rays are seeded, so two builds run with the same arguments can be
compared file for file.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LWL = 1064e-9
LENGTHS = (10e-3, 10e-3, 20e-3)
EXTENT = 10e-3
BEAM_R, BEAM_DIV = 5e-3, 5e-5
C_LIGHT = 299792458.0
# SURVEY.md 8d: one RHS evaluation gathers 8 corners x 16 B; RK4 = 4 evaluations, DP5 = 6
GATHER_BYTES = {"rk4": 512, "rk45": 768}
# Algorithmic FP64 work of one ray.step (DESIGN.md section 3 derives these): (instructions, flops with FMA = 2).
#   RK4:  4 x (3 sub + 3 mul + 3 x 7 fma) + Nystrom stage algebra (24 fma + 9 add)
#   +phase lane: 4 x 7 fma + 5
#   DP5:  6 x 27 + Nystrom stage positions (45 fma) + 5th-order update (33) + error estimate / norm (60)
FP64_WORK = {"rk4": (141, 249), "rk4_phase": (174, 312), "rk45": (300, 530)}


def parse(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C2", choices=["C1", "C2", "C3", "C4", "C5"],
                    help="C1 1e5 rays, 128^3 analytic Gaussian column, shadowgraphy (the reference's CPU-runnable case); "
                         "C2 shadowgraphy+schlieren on 512^3 turbulence (default, the headline); C3 interferometry with phase "
                         "accumulation; C4 refractometry + knife-edge schlieren with adaptive RK45, 1e8 rays; C5 shadowgraphy on a "
                         "1024^3 field, 1.25e8 rays per GPU (1e9 over 8)")
    ap.add_argument("--grid", type=int, default=None)
    ap.add_argument("--rays", type=float, default=None, help="rays per GPU per step")
    ap.add_argument("--bin-scale", type=int, default=None)
    ap.add_argument("--no-sort", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--parity-rays", type=int, default=2000, help="rays of the post-run oracle comparison (rank 0)")
    ap.add_argument("--cpu-rays-per-worker", type=int, default=4000)
    ap.add_argument("--fp32", action="store_true")
    ap.add_argument("--ds-frac", type=float, default=0.5, help="RK4 step as a fraction of the cell size along the probing axis")
    ap.add_argument("--start-offset-cells", type=float, default=0.0,
                    help="start the device beam this many cells further out along the probing axis (free flight outside the grid: "
                         "same physical rays, shifted fixed-step lattice)")
    ap.add_argument("--bundle", action="store_true", help="C4: one step size per 32-ray bundle instead of per ray")
    ap.add_argument("--extra-c5", choices=["auto", "on", "off"], default="auto",
                    help="after the timed region also run two passes of BASELINE configs[4] (1024^3, 1.25e8 rays per GPU) and "
                         "report them under extra.c5; auto = when 8 GPUs run the default C2 workload")
    ap.add_argument("--rtol", type=float, default=1e-3)
    ap.add_argument("--atol", type=float, default=1e-6)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the detector images and stats of the last timed step to DIR/<name>.npy (float64, <= 64 MB)")
    a = ap.parse_args(argv)
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA arm (--impl ours)")
    grid, rays, bs = workload_defaults(a.workload)
    a.grid = grid if a.grid is None else a.grid
    a.rays = rays if a.rays is None else a.rays
    a.bin_scale = bs if a.bin_scale is None else a.bin_scale
    if a.workload == "C5":
        a.no_cpu_baseline = True               # the CPU port on a 1024^3 grid needs tens of GB and minutes: C2 carries it
    return a


def workload_defaults(w):
    """(grid, rays per GPU, bin_scale) of the BASELINE.json configs (SURVEY.md 8d)."""
    return {"C1": (128, 1e5, 10), "C2": (512, 1e7, 1), "C3": (512, 1e7, 1), "C4": (512, 1e8, 1), "C5": (1024, 1.25e8, 1)}[w]


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def source_sha16():
    """Hash of the kernel sources: static ncu evidence in profiles/ is attached only while it matches."""
    h = hashlib.sha256()
    for f in ("ray_core.h", "synthpy_b200.cu"):
        h.update(open(os.path.join(ROOT, "synthpy_b200", "csrc", f), "rb").read())
    return h.hexdigest()[:16]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ workloads
def axes(grid):
    return [np.linspace(-L / 2, L / 2, grid) for L in LENGTHS]


def gaussian_column(grid):
    """C1 field A (SURVEY.md 8d): ne = 1e24 exp(-(x^2 + y^2) / (1 mm)^2), the formula of minimal_solver.test_lens
    (src/solvers-legacy/minimal_solver.py:192-201)."""
    x, y, z = axes(grid)
    XX, YY, _ = np.meshgrid(x, y, z, indexing="ij")
    return 1e24 * np.exp(-(XX ** 2 + YY ** 2) / (1e-3) ** 2)


def build_ne(a, device):
    """Our arm's field, built where it is used (synthpy_b200.field_generator: torch FFT on the GPU)."""
    if a.workload == "C1":
        return gaussian_column(a.grid)
    from synthpy_b200 import field_generator as fg
    return fg.turbulent_ne(a.grid // 2, noise="torch", seed=3 if a.workload == "C5" else 1, device=device)


def build_ne_reference(a):
    """The reference arm's field: the oracle's own NumPy restatement of gaussian3D.domain_fft (same noise stream), so
    that this process never imports the product package or maps its library."""
    if a.workload == "C1":
        return gaussian_column(a.grid)
    from oracle import field_gen
    return field_gen.turbulent_ne(a.grid // 2, noise="torch", seed=3 if a.workload == "C5" else 1)


def chain_names(a):
    """[(oracle chain name, kwargs)] of the workload's detector channels (rtm_solver.py:197-286,376-422)."""
    return {"C1": [("shadow_single", {})],
            "C2": [("shadow_two", {}), ("schlieren_DF", {"R_stop": 1})],
            "C3": [("interf_two", {})],
            "C4": [("refracto_incoherent", {}), ("schlieren_knife", {"offset": 0.1, "axis": 2, "direction": 1})],
            "C5": [("shadow_two", {})]}[a.workload]


def make_specs(a):
    from synthpy_b200 import diagnostics as D
    if a.workload == "C3":       # phase accumulation + 2-D interferogram (reference beam 10 fringes, 20 deg: diagnostics.py:616)
        return [D.spec("interf_two", bin_scale=a.bin_scale, interferogram=True, wavelength=LWL, ref_beam=(10, 20))]
    return [D.spec(name, bin_scale=a.bin_scale, **kw) for name, kw in chain_names(a)]


def solve_kw(a, dom):
    kw = dict(lwl=LWL, precision="fp32" if a.fp32 else "fp64", sort=not a.no_sort)
    if a.workload == "C4":       # adaptive RK45 (SciPy controller), the tolerance is the sweep parameter
        kw.update(method="rk45_bundle" if a.bundle else "rk45", rtol=a.rtol, atol=a.atol, max_steps=1000000)
    else:
        kw.update(method="rk4", ds=a.ds_frac * dom.cell_size())
    return kw


def rk4_lattice(a):
    """(h, n_steps) exactly as propagator._params derives them from ds."""
    h = a.ds_frac * (LENGTHS[2] / (a.grid - 1)) / C_LIGHT
    return h, int(np.ceil(np.sqrt(8.0) * EXTENT / C_LIGHT / h))


def workload_config(a):
    diag = {"C1": "shadowgraphy(single lens)", "C2": "shadowgraphy(two-lens) + schlieren(DF)",
            "C3": "interferometry(two-lens, phase accumulation, reference beam)",
            "C4": "refractometry(incoherent) + knife-edge schlieren", "C5": "shadowgraphy(two-lens)"}[a.workload]
    integ = (f"rk4, ds = {a.ds_frac:g} cell, early exit" if a.workload != "C4" else
             f"rk45 {'per 32-ray bundle' if a.bundle else 'per ray'} (SciPy controller), rtol {a.rtol:g} atol {a.atol:g}, early exit")
    field = "analytic Gaussian-column" if a.workload == "C1" else "turbulent (k^-11/3)"
    l2 = (f"inputs larger than L2 (packed field {16 * a.grid ** 3 / 1e9:.2f} GB vs 126 MB L2); no flush needed" if a.grid >= 256 else
          f"packed field {16 * a.grid ** 3 / 1e6:.0f} MB fits the 126 MB L2: the reference's own small case, L2-resident by design")
    rays = ("host-drawn legacy beam (np.random.seed(0), full_solver.init_beam order), resident in HBM" if a.workload == "C1" else
            "generated on device (Philox4x32-10)")
    return {"workload": f"{a.workload}: {int(a.rays):d} rays/GPU through a {a.grid}^3 {field} n_e field, {diag} at bin_scale {a.bin_scale}",
            "grid": a.grid, "rays_per_gpu": int(a.rays), "integrator": integ,
            "precision": "fp32" if a.fp32 else "fp64", "field_bytes": 16 * a.grid ** 3, "l2_policy": l2,
            "rays": rays + (", sorted into cell-column bundles" if not a.no_sort else ", unsorted")}


# ------------------------------------------------------------------------------------------------ CPU arms
_CPU = {}


def _cpu_worker(args):
    """One chunk of rays through the oracle's restatement of the shipped solver (joint RK45, full_solver.py:391) and the
    workload's first detector chain."""
    seed, n, chain = args
    from oracle import synthpy_oracle as O
    dom = _CPU["dom"]
    rng = np.random.RandomState(seed)
    s0 = O.init_beam(n, BEAM_R, BEAM_DIV, EXTENT, "circular", "z", rng=rng)
    t0 = time.perf_counter()
    sf, sol = dom.solve_joint(s0, return_stats=True)
    rf, J = O.ray_to_jones(sf, EXTENT)
    if chain[0] == "interf_two":
        r, E = O.run_chain(rf, O.chain("interf_two"), E=O.interfere_ref_beam(rf, J, 10, 20), wl=LWL)
        O.interferogram(r, E, bin_scale=chain[2])
    else:
        O.histogram(O.run_chain(rf, O.chain(chain[0], **chain[1])), bin_scale=chain[2])
    return n * (sol.nfev - 2) / 6.0, time.perf_counter() - t0


def _cpu_worker_rk4(args):
    """The GPU arm's own integrator on the CPU: fixed-step RK4 (same step, early exit) around the reference's RHS."""
    seed, n, h, n_steps, chain = args
    from oracle import synthpy_oracle as O
    dom = _CPU["dom"]
    s0 = O.init_beam(n, BEAM_R, BEAM_DIV, EXTENT, "circular", "z", rng=np.random.RandomState(seed))
    t0 = time.perf_counter()
    sf, steps = dom.solve_rk4(s0, n_steps, h=h, early_exit=True)
    rf, _ = O.ray_to_jones(sf, EXTENT)
    O.histogram(O.run_chain(rf, O.chain("shadow_two")), bin_scale=chain[2])
    return float(steps.sum()), time.perf_counter() - t0


def _pool_init():
    """One BLAS/OpenMP thread per worker process: the pool already uses every core (the reference's own
    config pins threads to 1 as well, src/simulator/config.py:80-122); without this np.dot inside solve_ivp
    oversubscribes the box and timings become erratic."""
    try:
        from threadpoolctl import threadpool_limits
        _CPU["tp"] = threadpool_limits(1)
    except Exception:
        pass


def cpu_setup(ne_host, a, phaseshift=None):
    from oracle import synthpy_oracle as O
    x, y, z = axes(a.grid)
    dom = O.Domain(x, y, z, EXTENT, phaseshift=(a.workload == "C3") if phaseshift is None else phaseshift)
    dom.external_ne(ne_host)
    dom.calc_dndr(LWL)
    if not dom.phaseshift:
        dom.ne = None
    _CPU["dom"] = dom
    return dom


def cpu_pass(pool, cores, rays_per_worker, seed0, chain):
    t0 = time.perf_counter()
    res = pool.map(_cpu_worker, [(seed0 + i, rays_per_worker, chain) for i in range(cores)])
    wall = time.perf_counter() - t0
    return sum(r[0] for r in res), wall


def first_chain(a):
    name, kw = chain_names(a)[0]
    return (name, kw, a.bin_scale)


def run_reference(a):
    """--impl reference: the reference's own CPU algorithm (NumPy/SciPy restatement in oracle/, pinned to the
    real reference by tests/golden -- /root/reference itself does not travel to the GPU box) on all host cores,
    mirroring the reference's multiprocessing driver (examples/jobs/run_scripts/pvti_trace_multiprocess.py:102-134).
    Nothing of the product package is imported here: the field comes from oracle/field_gen.py."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    if a.workload == "C5":
        try:
            import psutil
            avail = psutil.virtual_memory().available
        except Exception:
            avail = 0
        if avail < 120e9:
            print(json.dumps({"impl": "reference", "unavailable": "C5: the CPU port needs ~100 GB of host memory for a 1024^3 field "
                              "(float64 n_e + three float32 gradient grids + FFT workspace); C2 carries the CPU baseline"}))
            return
    ne = build_ne_reference(a)
    cpu_setup(ne, a)
    del ne
    chain = first_chain(a)
    rpw = min(a.cpu_rays_per_worker, max(1, int(a.rays) // cores))
    ctx = mp.get_context("fork")
    with ctx.Pool(cores, initializer=_pool_init) as pool:
        for w in range(a.warmup):
            cpu_pass(pool, cores, max(8, rpw // 8), 1000 + 100 * w, chain)
        t0 = time.perf_counter()
        units = 0.0
        for k in range(a.steps):
            u, _ = cpu_pass(pool, cores, rpw, 5000 + 100 * k, chain)
            units += u
        wall = time.perf_counter() - t0
    value = units / wall
    rays_per_s = cores * rpw * a.steps / wall
    sample = (f"{cores} workers x {rpw} rays per step, joint RK45 as shipped (rtol 1e-3, atol 1e-6, full_solver.py:391) + "
              f"{chain[0]} + image, same {a.grid}^3 field; a 'step' of this arm = one attempted joint-RK45 step of one ray "
              f"((nfev - 2) / 6), not the GPU arm's half-cell RK4 step: compare rays_per_s")
    line = {"impl": "reference", "metric": "rays*steps/s", "value": value, "unit": "rays*steps/s", "n_gpus": a.gpus,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * wall / max(1, a.steps), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(a), "rays_per_s": rays_per_s,
            "cpu_baseline": {"value": value, "unit": "rays*steps/s", "cores": cores, "kind": "port", "sample": sample,
                             "rays_per_s": rays_per_s},
            "e2e": {"value": value, "unit": "rays*steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def cpu_baseline(a, ne_host):
    """The oracle port of the shipped CPU solver, all host cores, bounded sample of the same workload; plus the GPU
    arm's own integrator (fixed-step RK4) around the reference's RHS on the same cores."""
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    cpu_setup(ne_host, a)
    chain = first_chain(a)
    ctx = mp.get_context("fork")
    h, n_steps = rk4_lattice(a)
    rpw = min(a.cpu_rays_per_worker, max(8, int(a.rays) // cores))
    n4 = max(8, rpw // 16)
    with ctx.Pool(cores, initializer=_pool_init) as pool:
        cpu_pass(pool, cores, 8, 100, chain)
        units, wall = cpu_pass(pool, cores, rpw, 200, chain)
        t0 = time.perf_counter()
        res = pool.map(_cpu_worker_rk4, [(300 + i, n4, h, n_steps, chain) for i in range(cores)])
        wall4 = time.perf_counter() - t0
    return {"value": units / wall, "unit": "rays*steps/s", "cores": cores, "kind": "port",
            "rays_per_s": cores * rpw / wall,
            "sample": f"{cores} workers x {rpw} rays, joint RK45 (SciPy defaults) + {chain[0]} + image on the same "
                      f"{a.grid}^3 field; {wall:.1f} s wall; a step here = one attempted joint-RK45 step ((nfev-2)/6)",
            "same_integrator": {"value": sum(r[0] for r in res) / wall4, "unit": "rays*steps/s", "rays_per_s": cores * n4 / wall4,
                                "sample": f"{cores} workers x {n4} rays, the GPU arm's fixed-step RK4 (ds = {a.ds_frac:g} cell, early "
                                          f"exit) around the reference's dsdt; {wall4:.1f} s wall"}}


# ------------------------------------------------------------------------------------------------ parity
def _rel(a_, b_, floor):
    """max over entries of |a - b| / max(|b|, floor); floor is a scalar or one value per row.  NaN patterns must agree."""
    a_, b_ = np.asarray(a_), np.asarray(b_)
    if not np.array_equal(np.isnan(a_), np.isnan(b_)):
        return float("inf")
    fl = np.broadcast_to(np.asarray(floor, dtype=np.float64).reshape(-1, *([1] * (b_.ndim - 1))) if np.ndim(floor) else floor, b_.shape)
    m = ~np.isnan(b_)
    return float(np.max(np.abs(a_[m] - b_[m]) / np.maximum(np.abs(b_[m]), fl[m]))) if m.any() else 0.0


def _row_scale(rf_o):
    """Natural scale of each exit-ray row [x, theta, y, phi]: its rms over the sample (beam size, deflection angle).
    'Relative 1e-9' (north_star) is taken against max(|value|, this scale): a coordinate that happens to be ~0 has no
    relative precision of its own, its error is 1e-9 of the beam like every other ray's."""
    return np.maximum(np.sqrt(np.nanmean(np.asarray(rf_o) ** 2, axis=1)), 1e-12)


def parity_check(a, dom, rays, odom, n, ray_offset=0, workers=None, conditioning=True):
    """The benchmarked configuration against the CPU oracle on a sub-sample of the very same rays: ``n`` rays starting at
    global index ``ray_offset`` of the device beam (or columns of the explicit bundle), through the same HBM-resident
    field and the same sort / early-exit / fused-epilogue path that produced the headline number.
    Compares exit rays (full_solver.py:838-894; relative to max(|value|, row rms), see _row_scale -- the old fixed 1e-7
    floor is reported too), steps per ray, and every detector image.  ``conditioning``: the oracle is also run on the same
    rays moved by ONE ulp, which shows how far rounding-level differences are amplified by the field itself.
    Adaptive (C4): on a grid-scale-rough field SciPy's step-size map is chaotic (DESIGN.md section 4), so step sequences
    fork between ANY two implementations; reported are the fraction of rays with identical nfev, the agreement of those
    rays, and the same two numbers for the oracle against its own one-ulp-perturbed run.
    ``odom``: oracle Domain prepared on the host copy of the same n_e grid (phaseshift=True for C3)."""
    from oracle import parallel as OP, synthpy_oracle as O
    from synthpy_b200 import propagator as P
    kw = solve_kw(a, dom)
    if a.workload == "C4":
        kw["early_exit"] = False       # solve_ivp integrates to t_end: keep the free-flight attempts so that step counts are comparable
    if hasattr(rays, "spec"):
        s0 = rays.materialise(n, ray_offset)
    else:
        s0 = rays[:, ray_offset:ray_offset + n].contiguous()
    s0_h = s0.cpu().numpy()
    out = {"n": int(n), "ray_offset": int(ray_offset),
           "oracle": "oracle/synthpy_oracle.py (golden-pinned port of full_solver / rtm_solver), same rays, same field"}
    c3 = a.workload == "C3"
    was = dom.phaseshift
    try:
        if c3:
            dom.phaseshift = True
        rf, Jf, _, ex = P.solve(s0, dom, EXTENT, return_E=c3, return_state=True, phase_f64=c3, **kw)
    finally:
        dom.phaseshift = was
    rf, steps, sf = rf.cpu().numpy(), ex["steps"].cpu().numpy().astype(np.int64), ex["sf"].cpu().numpy()
    s1_h = s0_h.copy()
    s1_h[0], s1_h[1] = np.nextafter(s1_h[0], np.inf), np.nextafter(s1_h[1], -np.inf)
    t0 = time.perf_counter()
    if a.workload == "C4":
        sf_o, nfev = OP.solve_per_ray(odom, s0_h, rtol=a.rtol, atol=a.atol, workers=workers)
        same = (6 * steps + 2) == nfev                                         # same accept / reject sequence as solve_ivp
        out["nfev_equal_frac"] = float(same.mean())
        out["steps_equal"] = bool(same.all())
        out["steps_per_ray"] = float(steps.mean())
        out["steps_per_ray_oracle"] = float((nfev - 2).mean() / 6.0)
    else:
        h, n_steps = rk4_lattice(a)
        sf_o, steps_o = OP.solve_rk4(odom, s0_h, n_steps, h=h, early_exit=True, workers=workers)
        out["steps_equal"] = bool(np.array_equal(steps, steps_o))
        out["steps_per_ray"] = float(steps_o.mean())
    out["oracle_seconds"] = round(time.perf_counter() - t0, 2)
    rf_o, J_o = O.ray_to_jones(sf_o, EXTENT)
    scale = _row_scale(rf_o)
    out["max_rel"] = _rel(rf, rf_o, scale)
    out["max_rel_floor_1e-7"] = _rel(rf, rf_o, 1e-7)
    out["max_abs"] = [float(v) for v in np.nanmax(np.abs(rf - rf_o), axis=1)]
    out["row_scale"] = [float(v) for v in scale]
    if a.workload == "C4":
        out["max_rel_same_sequence"] = _rel(rf[:, same], rf_o[:, same], scale) if same.any() else None
        out["median_rel"] = float(np.median(np.max(np.abs(rf - rf_o) / np.maximum(np.abs(rf_o), scale[:, None]), axis=0)))
    if conditioning:
        if a.workload == "C4":
            sf_1, nfev_1 = OP.solve_per_ray(odom, s1_h, rtol=a.rtol, atol=a.atol, workers=workers)
            rf_1 = O.ray_to_jones(sf_1, EXTENT)[0]
            out["oracle_one_ulp"] = {"nfev_equal_frac": float((nfev_1 == nfev).mean()), "max_rel": _rel(rf_1, rf_o, scale),
                                     "median_rel": float(np.median(np.max(np.abs(rf_1 - rf_o) / np.maximum(np.abs(rf_o), scale[:, None]), axis=0)))}
        else:
            sf_1, _ = OP.solve_rk4(odom, s1_h, n_steps, h=h, early_exit=True, workers=workers)
            rf_1 = O.ray_to_jones(sf_1, EXTENT)[0]
            out["oracle_one_ulp"] = {"max_rel": _rel(rf_1, rf_o, scale), "max_abs": [float(v) for v in np.nanmax(np.abs(rf_1 - rf_o), axis=1)]}
    if c3:
        out["phase_max_rel"] = float(np.max(np.abs(sf[7] - sf_o[7])) / np.abs(sf_o[7]).max())
    # fused images of the same sub-sample, in the benchmarked mode (C3: once more with the float64 phase grid)
    hist_equal, l1s = True, []
    for f64 in ((False, True) if c3 else (False,)):
        specs = make_specs(a)
        if hasattr(rays, "spec"):
            P.solve_and_image(dom, rays, EXTENT, specs, n_rays=n, ray_offset=ray_offset, phase_f64=f64, **kw)
        else:
            P.solve_and_image(dom, s0, EXTENT, specs, phase_f64=f64, **kw)
        for sp_, (name, ckw) in zip(specs, chain_names(a)):
            H = sp_.image.result().cpu().numpy()
            if c3:
                r_o, E_o = O.run_chain(rf_o, O.chain(name), E=O.interfere_ref_beam(rf_o, J_o, 10, 20), wl=LWL)
                H_o = O.interferogram(r_o, E_o, bin_scale=a.bin_scale)
                l1 = float(np.abs(H - H_o).sum() / H_o.sum())
                out["interferogram_l1_f64_phase" if f64 else "interferogram_l1_f32_phase"] = l1
            else:
                H_o = O.histogram(O.run_chain(rf_o, O.chain(name, **ckw)), bin_scale=a.bin_scale)
                hist_equal &= bool(np.array_equal(H, H_o))
                l1s.append(float(np.abs(H - H_o).sum() / max(1.0, H_o.sum())))
                out.setdefault("counts", []).append([int(H.sum()), int(H_o.sum())])
    if not c3:
        out["hist_equal"], out["hist_l1_max"] = hist_equal, max(l1s)
    return out


def attach_ncu_static(roof, a, n_rays):
    """Static ncu evidence of the same command (profiles/r2_<workload>_k_propagate_ncu_full.json, written by
    profiles/tools/ncu_extract.py --stamp): attached to the roofline only while the hash of the kernel sources equals the
    one stored in the capture, and its DRAM bytes reported as ``traffic`` only when the profiled launch had as many rays as
    a launch of this run -- so stale or mismatched evidence cannot ride on a changed kernel."""
    wd = workload_defaults(a.workload)
    ncu_file = os.path.join(ROOT, "profiles", f"r2_{a.workload.lower()}_k_propagate_ncu_full.json")
    if os.path.exists(ncu_file) and a.grid == wd[0] and not a.fp32 and not a.bundle:
        try:                                  # static evidence of the same command, attached only while the kernel source is unchanged
            m = json.load(open(ncu_file))
            if m.get("source_sha16") == source_sha16():
                unit = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}
                g = lambda k: float(str(m[k][0]).replace(",", "")) if k in m else None
                gb = lambda k: g(k) * unit.get(m[k][1], 1.0) if k in m else 0.0
                cap_rays = m.get("rays_per_launch")
                chunk = min(n_rays, 1 << 25)                                         # sp_propagate launches chunks of 2^25 rays
                if cap_rays == chunk:                                                # traffic is per launch: only a same-size launch counts
                    roof["traffic"] = gb("dram__bytes_read.sum") + gb("dram__bytes_write.sum") or None
                roof["ncu_static"] = {"source": os.path.relpath(ncu_file, ROOT), "source_sha16": m["source_sha16"],
                                      "rays_of_profiled_launch": cap_rays,
                                      "dram_bytes_of_profiled_launch": gb("dram__bytes_read.sum") + gb("dram__bytes_write.sum"),
                                      "fp64_pipe_pct": g("sm__pipe_fp64_cycles_active.avg.pct_of_peak_sustained_active"),
                                      "issue_active_pct": g("smsp__issue_active.avg.pct_of_peak_sustained_active"),
                                      "l2_hit_pct": g("lts__t_sector_hit_rate.pct"), "l1_hit_pct": g("l1tex__t_sector_hit_rate.pct"),
                                      "dram_throughput_pct": g("gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed"),
                                      "lanes_per_instruction": g("smsp__thread_inst_executed_per_inst_executed.ratio")}
            else:
                roof["ncu_static"] = {"stale": True, "source": os.path.relpath(ncu_file, ROOT)}
        except Exception:
            pass


# ------------------------------------------------------------------------------------------------- output dump
DUMP_BYTES = 64_000_000
_NPY_HEADER = 256          # upper bound of np.save's header for a 1-D or 2-D float64 array


def dump_outputs(out_dir, arrays, budget=DUMP_BYTES):
    """Write ``arrays`` (name -> array) as ``out_dir/<name>.npy`` in float64, ``budget`` bytes in all.  Arrays are
    taken smallest first and each gets an equal share of what is left; one that does not fit its share is replaced by
    its values at a fixed, seeded sample of flat indices (sorted, written beside it as ``<name>_index.npy``), so the
    same outputs always produce the same files."""
    os.makedirs(out_dir, exist_ok=True)
    items = sorted(((k, np.asarray(v, dtype=np.float64)) for k, v in arrays.items()), key=lambda kv: kv[1].size)
    left = budget
    for i, (name, v) in enumerate(items):
        share = left // (len(items) - i)
        if v.nbytes + _NPY_HEADER <= share:
            files = {name: v}
        else:
            k = (share - 2 * _NPY_HEADER) // 16                      # a float64 value and its float64 index per entry
            idx = np.sort(np.random.default_rng(0).choice(v.size, size=k, replace=False))
            files = {name: v.reshape(-1)[idx], name + "_index": idx.astype(np.float64)}
        for fn, arr in files.items():
            path = os.path.join(out_dir, fn + ".npy")
            np.save(path, arr)
            left -= os.path.getsize(path)


def last_step_outputs(a, specs, stats):
    """What one timed ``solve_and_image`` call hands its caller: each channel's image and the stats dict."""
    from synthpy_b200 import engine
    out = {name: s.image.result().cpu().numpy() for s, (name, _) in zip(specs, chain_names(a))}
    out["stats"] = np.array([stats[k] for k in engine.STAT_NAMES], dtype=np.float64)
    return out


# ------------------------------------------------------------------------------------------------- our arm
def run_c5_passes(a, rank, world, barrier, passes=2):
    """BASELINE configs[4] as a side measurement of a multi-GPU run: 1024^3 seed-3 field replicated on every GPU,
    1.25e8 device rays per GPU, two-lens shadowgraphy, images all-reduced; one warm-up pass, ``passes`` timed (device
    events, max over ranks).  Returns the dict printed under extra.c5."""
    import torch
    import torch.distributed as dist
    from synthpy_b200 import beam as B, distributed as SD, domain as Dm, engine, propagator as P
    c5 = parse(["--workload", "C5"])
    ne = build_ne(c5, "cuda")
    dom = Dm.ScalarDomain(LENGTHS, c5.grid)
    dom.external_ne(ne)
    dom.device_field(LWL)
    del ne
    dom.release_ne()
    torch.cuda.empty_cache()
    n_rays = int(c5.rays)
    beam = B.Beam(n_rays * world, BEAM_R, BEAM_DIV, EXTENT, device=True, seed=2, beam_type="circular")
    specs = make_specs(c5)
    kw = solve_kw(c5, dom)

    def one():
        for s_ in specs:
            s_.image.zero_()
        st_, _ = P.solve_and_image(dom, beam, EXTENT, specs, n_rays=n_rays, ray_offset=rank * n_rays, sync=False, **kw)
        if world > 1:
            SD.combine_images([s_.image for s_ in specs])
        return st_
    st_ = one()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(passes):
        st_ = one()
    e1.record()
    barrier()
    stats = engine.stats_dict(st_)
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    tot = torch.tensor([float(stats["ray_steps"]) * passes, float(stats["rays_binned"])], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms = float(t.item())
    img = int(specs[0].image.total().sum().item())
    return {"config": workload_config(c5), "value": float(tot[0].item()) / (ms * 1e-3), "unit": "rays*steps/s", "n_gpus": world,
            "passes": passes, "ms_per_pass": ms / passes, "rays_per_s": n_rays * world * passes / (ms * 1e-3),
            "allreduce_check": {"sum_image": img, "sum_rays_binned_over_ranks": int(tot[1].item()), "equal": img == int(tot[1].item())}}


def run_ours(a):
    import torch
    import torch.distributed as dist
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py (our arm) needs a CUDA device: there is no CPU fallback"
    torch.cuda.set_device(local)
    from synthpy_b200 import _lib, beam as B, distributed as SD, domain as Dm, engine, legacy, propagator as P
    numa = SD.bind_to_local_numa(local) if world > 1 else None     # pinned e2e buffers land on the GPU's own NUMA node
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    n_rays = int(a.rays)
    ne = build_ne(a, "cuda")
    dom = Dm.ScalarDomain(LENGTHS, a.grid)
    dom.external_ne(ne)
    dom.device_field(LWL)
    del ne
    torch.cuda.empty_cache()
    kw = solve_kw(a, dom)
    specs = make_specs(a)
    if a.workload == "C1":
        np.random.seed(0)
        rays = engine.to_device(legacy.init_beam(n_rays, BEAM_R, BEAM_DIV, EXTENT, "circular", "z"))
        call_kw = dict(kw)
    else:
        rays = B.Beam(n_rays * world, BEAM_R, BEAM_DIV, EXTENT + a.start_offset_cells * dom.cell_size(), device=True, seed=2,
                      beam_type="circular")
        call_kw = dict(kw, n_rays=n_rays, ray_offset=rank * n_rays)

    def one_pass(r, root_only=False):
        for s in specs:
            s.image.zero_()
        st, _ = P.solve_and_image(dom, r, EXTENT, specs, sync=False, **(call_kw if r is rays else kw))
        if world > 1:                         # the path's one exchange: sum of detector images (SURVEY.md 8e)
            SD.combine_images([s.image for s in specs], root=0 if root_only else None)
        return st

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, a.warmup)):
        st = one_pass(rays)
    barrier()
    steps_per_pass = engine.stats_dict(st)["ray_steps"]
    engine.propagate_kernel_ms()                       # reset the event log
    launches0 = _lib.launch_count()
    clocks = ClockSampler(local) if rank == 0 else None
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(a.steps):
        st = one_pass(rays)
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    clk = clocks.stop() if clocks else None
    launches = _lib.launch_count() - launches0
    kms, klaunch = engine.propagate_kernel_ms()
    stats = engine.stats_dict(st)
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    tot = torch.tensor([float(steps_per_pass) * a.steps, float(stats["rays_binned"])], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms = float(t.item())
    value = float(tot[0].item()) / (ms * 1e-3)
    # multi-GPU content check: the all-reduced images of the last pass hold exactly the rays every rank binned
    allreduce_check = None
    if world > 1 and a.workload != "C3":
        img_total = sum(int(s.image.total().sum().item()) for s in specs)
        allreduce_check = {"sum_images": img_total, "sum_rays_binned_over_ranks": int(tot[1].item()),
                           "equal": img_total == int(tot[1].item())}
    if a.dump_outputs and rank == 0:                   # before the e2e passes below reuse the image buffers
        dump_outputs(a.dump_outputs, last_step_outputs(a, specs, stats))

    # ---- e2e: host ray bundle in pinned memory -> H2D -> fused trace -> images D2H, every step
    e2e = None
    if not a.no_e2e:
        src = rays if a.workload == "C1" else rays.materialise(n_rays, rank * n_rays)
        s0_host = src.cpu().pin_memory()
        del src
        outs = ([torch.empty(s.image.tensors()[0].shape, dtype=s.image.tensors()[0].dtype).pin_memory() for s in specs]
                if rank == 0 else [])

        side = torch.cuda.Stream()
        snaps = []

        def e2e_pass(tok):
            st_ = one_pass(tok, root_only=True)          # like the reference's comm.reduce(H, root=0): one copy leaves the GPUs
            if outs:
                # the read-back of pass k overlaps the propagation of pass k+1: snapshot the image on the compute stream (the
                # accumulator is zeroed by the next pass), copy the snapshot to pinned memory on a side stream
                snaps[:] = [s.image.total().clone() for s in specs]
                done = torch.cuda.Event()
                done.record()
                side.wait_event(done)
                with torch.cuda.stream(side):
                    for o, t_ in zip(outs, snaps):
                        o.copy_(t_, non_blocking=True)
                        t_.record_stream(side)
            return st_
        # propagator.prefetch_rays: the host->device copy of step k+1's rays runs on a side stream while step k
        # propagates (two device buffers); every step's copy and image read-back is inside the timed region
        e2e_pass(P.prefetch_rays(s0_host))
        side.synchronize()
        barrier()
        t0 = time.perf_counter()
        nxt = P.prefetch_rays(s0_host)
        for k in range(a.steps):
            cur, nxt = nxt, (P.prefetch_rays(s0_host) if k + 1 < a.steps else None)
            st_ = e2e_pass(cur)
        side.synchronize()                               # the last image is in host memory before the clock stops
        barrier()
        wall = time.perf_counter() - t0
        tw = torch.tensor([wall], dtype=torch.float64, device="cuda")
        es = torch.tensor([float(engine.stats_dict(st_)["ray_steps"]) * a.steps], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tw, op=dist.ReduceOp.MAX)
            dist.all_reduce(es, op=dist.ReduceOp.SUM)
        e2e = {"value": float(es.item()) / float(tw.item()), "unit": "rays*steps/s",
               "rays_per_s": n_rays * world * a.steps / float(tw.item()),
               "h2d_bytes_per_step": int(s0_host.numel() * 8) * world, "d2h_bytes_per_step": int(sum(o.numel() * 8 for o in outs)),
               "api": "propagator.prefetch_rays(s0_host_pinned) -> propagator.solve_and_image(domain, handle, ...) -> "
                      "distributed.combine_images(root=0) -> image read-back on rank 0 (side stream, overlapping the next pass)", "numa_bind": numa}
        del s0_host

    # ---- BASELINE configs[4] beside the headline when the whole box is there: 1e9 rays through 1024^3 over 8 GPUs
    extra = None
    if a.extra_c5 == "on" or (a.extra_c5 == "auto" and world == 8 and a.workload == "C2"):
        extra = {"c5": run_c5_passes(a, rank, world, barrier)}

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    # ---- roofline of the dominant kernel (k_propagate): FP64 pipe, with the HBM-algorithmic figure beside it
    adaptive = a.workload == "C4"
    work_key = "rk45" if adaptive else ("rk4_phase" if a.workload == "C3" else "rk4")
    n_instr, n_flop = FP64_WORK[work_key]
    launch_s = kms / max(1, klaunch) * 1e-3
    per_launch_steps = steps_per_pass * a.steps / max(1, klaunch)
    fp64_peak = engine.fp64_peak()
    achieved_tf = per_launch_steps * n_flop / launch_s / 1e12 if launch_s > 0 else None
    hbm_peak, peak_src = peaks()
    gather_b = GATHER_BYTES["rk45" if adaptive else "rk4"]
    hbm_alg = per_launch_steps * gather_b / launch_s / 1e9 if launch_s > 0 else None
    roof = {"bound": "fp64_pipe", "achieved": achieved_tf, "peak": fp64_peak, "unit": "TFLOP/s",
            "frac": achieved_tf / fp64_peak if achieved_tf else None, "traffic": None,
            "kernel": "k_propagate<%s, %s>" % ("float" if a.fp32 else "double", "RK45" if adaptive else "RK4"),
            "kernel_ms_per_launch": kms / max(1, klaunch), "kernel_share_of_step": kms / ms if ms > 0 else None,
            "peak_source": "measured in this run: sp_fp64_peak (8 independent DFMA chains per thread, 2048 threads/SM, CUDA events)",
            "flops_per_ray_step": n_flop, "fp64_instructions_per_ray_step": n_instr,
            "issue_slot_frac": (per_launch_steps * n_instr / launch_s) / (fp64_peak * 1e12 / 2) if launch_s > 0 else None,
            "hbm_algorithmic": {"achieved_gbs": hbm_alg, "peak_gbs": hbm_peak, "frac": hbm_alg / hbm_peak if hbm_alg else None,
                                "frac_of_nominal_8TBps": hbm_alg / 8000.0 if hbm_alg else None,
                                "bytes_per_ray_step": gather_b, "peak_source": peak_src,
                                "note": "SURVEY.md 8d gather bytes over the HBM copy peak; gathers are served from registers / L1 / L2 "
                                        "(one fetch per cell, not per evaluation), so this exceeds 1 and is NOT the bound"},
            "dram_compulsory_bytes_per_launch": 16 * a.grid ** 3,
            "note": "achieved = algorithmic FP64 flops per ray.step (DESIGN.md section 3) x ray.steps per launch / event-timed launch "
                    "duration; frac < 1 is what reload divergence, address / control instructions and latency cost"}
    if a.fp32:
        roof["fp32_note"] = "fp32 mode: the same operation count runs on the FP32 pipe; the FP64 peak is kept as the common denominator"
    attach_ncu_static(roof, a, n_rays)
    # ---- CPU legs (rank 0): baseline timing and the oracle parity of the benchmarked configuration
    cpu, parity = None, None
    want_cpu = world == 1 and not a.no_cpu_baseline
    if (want_cpu or not a.no_parity) and a.workload != "C5":
        ne_host = dom.ne.cpu().numpy() if isinstance(dom.ne, torch.Tensor) else np.asarray(dom.ne)
        if want_cpu:
            cpu = cpu_baseline(a, ne_host)
            odom = _CPU["dom"]
        else:
            odom = cpu_setup(ne_host, a)
        del ne_host
        if not a.no_parity:
            n_par = min(a.parity_rays if a.workload != "C4" else min(a.parity_rays, 128), n_rays)
            parity = parity_check(a, dom, rays, odom, n_par, ray_offset=0)
    line = {"metric": "rays*steps/s", "value": value, "unit": "rays*steps/s", "n_gpus": world, "steps": a.steps,
            "warmup": max(3, a.warmup), "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32" if a.fp32 else "f64", "data": "synthetic", "config": workload_config(a),
            "rays_per_s": n_rays * world * a.steps / (ms * 1e-3),
            "roofline": roof, "cpu_baseline": cpu, "same_integrator": cpu["same_integrator"] if cpu else None,
            "e2e": e2e, "parity": parity, "allreduce_check": allreduce_check,
            "gpu_launches": int(launches), "clocks": clk, "extra": extra,
            "ray_steps_per_pass_per_gpu": int(steps_per_pass), "rays_binned_last_pass": stats["rays_binned"]}
    print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
