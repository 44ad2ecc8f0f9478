"""Tracing through a field that does not fit in HBM: the grid is streamed slab by slab along the probing axis.

The reference's counterpart is the domain batching of ``src/simulator/domain.py:137-243`` + ``propagator.py:366-450``
(``region_count`` sections of the domain, regenerated one after the other while the rays keep their state) -- work in
progress upstream (the section bounds are hard-coded, domain.py:247-252).  On a B200 a 1024^3 packed field is 17 GB of
180 GB, so this is needed only from ~2048^3 upwards (137 GB packed) or when several fields share a GPU; it is built so
that nothing about the result depends on it:

  * fixed-step RK4 only (the ray ODE has no explicit time dependence, so N steps through the whole grid are N_1 + N_2 +
    ... steps through consecutive slabs, the (9, N) state carried over exactly; an adaptive per-ray controller would see
    different step sequences);
  * a slab holds the planes [a, b] of the probing axis.  The float32 gradient stencil (field_prep.h) at plane k reads
    planes k-1 and k+1, so the edge planes of a slab carry one-sided differences that the whole grid would not: the
    planner keeps every RK stage of every live ray at least two planes inside (``plan_slab``), checks it afterwards on
    the actual positions, and re-runs the slab with fewer steps if a ray got further than planned.  Every field value a
    ray reads is then bit-identical to the one-region field, and so are the exit rays, the steps per ray and the images
    (tests/test_gpu_parity.py::test_out_of_core_equals_in_core; the same driver on the host build of the ray code:
    tests/test_core_host.py::test_out_of_core_planner_and_driver);
  * ``np.gradient`` switches to its uniform-spacing formula when all float32 spacings of an axis are equal; a slab is
    widened until its probing axis makes the same choice as the full axis.

The slab source is a callable ``source(k0, k1) -> ne[..., k0:k1 along the probing axis]`` (NumPy array, ``np.memmap`` of a
raw dump, or CUDA tensor): ``array_source`` wraps an array-like; ``field_generator.turbulent_ne_slabs`` generates a
turbulent field on the device slab by slab.  One slab is resident at a time; the next is packed after
the rays have left the current one.  ``PrefetchingSource`` overlaps the host-side read of the next slab with the tracing;
upload and packing are not overlapped yet.
"""
from time import time

import numpy as np

from . import engine

C_LIGHT = 299792458.0
MARGIN = 2                      # planes kept between any ray and a slab edge that is not a grid edge


def array_source(ne, probing_direction="z"):
    """``source(k0, k1)`` over an in-memory / memory-mapped (x_n, y_n, z_n) array."""
    axis = engine.AXIS[probing_direction]

    def source(k0, k1):
        idx = [slice(None)] * 3
        idx[axis] = slice(k0, k1)
        return ne[tuple(idx)]
    return source


class PrefetchingSource:
    """Wraps a HOST slab source so that the next slab is read (page faults, decoding, strided copy) on a worker thread while
    the GPU traces the current one.  After serving planes [k0, k1) it starts fetching the window the planner is expected to
    ask for next -- it begins ``back`` planes before k1 (the planner restarts MARGIN planes behind the slowest live ray, so
    consecutive slabs overlap by a few planes) -- and serves any later request that lies inside a window it holds by
    slicing it; anything else falls through to the wrapped source.  Pure data plumbing: what is returned is what the wrapped
    source would return.  Only for sources that return NumPy arrays (a worker thread must not touch the CUDA stream)."""

    def __init__(self, source, n_planes, axis, back=16):
        import threading
        self._source, self._n, self._axis, self._back = source, int(n_planes), int(axis), int(back)
        self._threading = threading
        self._job = None                    # (k0, k1, thread, result holder)
        self.hits = self.misses = 0

    def _start(self, k0, k1):
        box = {}

        def work():
            try:
                box["data"] = np.ascontiguousarray(self._source(k0, k1))
            except Exception as e:          # surfaced on the main thread when (if) the window is asked for
                box["error"] = e
        t = self._threading.Thread(target=work, daemon=True)
        t.start()
        self._job = (k0, k1, t, box)

    def __call__(self, k0, k1):
        k0, k1 = int(k0), int(k1)
        out = None
        if self._job is not None:
            j0, j1, t, box = self._job
            if j0 <= k0 and k1 <= j1:
                t.join()
                if "error" in box:
                    raise box["error"]
                idx = [slice(None)] * 3
                idx[self._axis] = slice(k0 - j0, k1 - j0)
                out = box["data"][tuple(idx)]
                self.hits += 1
            else:
                t.join()                    # a window nobody wants: let the read finish, then drop it
            self._job = None
        if out is None:
            out = self._source(k0, k1)
            self.misses += 1
            if getattr(out, "is_cuda", False):          # before any worker thread has called the source
                raise ValueError("prefetch=True is for host sources: this source returns CUDA tensors (use prefetch=False)")
        if k1 < self._n:
            n0 = max(0, k1 - self._back)
            self._start(n0, min(self._n, n0 + (k1 - k0) + self._back))
        return out

    def close(self):
        if self._job is not None:
            self._job[2].join()
            self._job = None


def axis_is_uniform(a32):
    """The test field_prep.h / np.gradient make on an axis: every float32 spacing equal to the first."""
    d = np.diff(np.asarray(a32, dtype=np.float32))
    return bool(np.all(d == d[0])) if d.size else True


def plan_slab(zc, zmin, zmax, vmax, h, steps_left, slab_planes):
    """Which planes [a, b] to load and how many RK4 steps to take in them.

    zc          the probing axis (float32 values as float64), n planes
    zmin, zmax  extreme probing-axis positions of the live rays now;  vmax  their largest speed along that axis
    Returns (a, b, m, z_stop): after m steps no live ray may be beyond z_stop (checked by the driver); ``b == n - 1``
    means the slab reaches the end of the grid and takes all remaining steps."""
    n = len(zc)
    cell = int(np.clip(np.searchsorted(zc, zmin, side="right") - 1, 0, n - 2))       # cell holding the last ray
    a = max(0, cell - MARGIN)
    b = min(n - 1, a + int(slab_planes) - 1)
    full_uniform = axis_is_uniform(zc)
    while axis_is_uniform(zc[a:b + 1]) != full_uniform and (b < n - 1 or a > 0):     # same stencil choice as the whole axis
        if b < n - 1:
            b += 1
        else:
            a -= 1
    if b == n - 1:
        return a, b, int(steps_left), np.inf
    z_stop = float(zc[b - MARGIN])
    m = int(np.floor((z_stop - zmax) / (h * vmax * 1.02))) if vmax > 0 else int(steps_left)
    if m < 1:
        raise ValueError(f"slab of {b - a + 1} planes is too thin for the spread of the rays along the probing axis "
                         f"({zmin:.4g} .. {zmax:.4g} m): increase slab_planes")
    return a, b, min(m, int(steps_left)), z_stop


class _DeviceBackend:
    """The product path: packed slab field in HBM, ``sp_propagate`` per slab."""

    def __init__(self, lwl, probing_direction, phase, phase_f64, out_axes, extent, sort):
        import torch
        self.torch = torch
        self.lwl, self.pd, self.phase, self.phase_f64 = lwl, probing_direction, phase, phase_f64
        self.out_axes, self.extent, self.sort = out_axes, extent, sort
        self.p = engine.AXIS[probing_direction]

    def to_state(self, s0):
        return engine.to_device(s0, self.torch.float64)

    def live_range(self, s, lo, hi):
        t = self.torch
        pos, vel = s[:3], s[3:6]
        lo_t, hi_t = (t.tensor(v, dtype=t.float64, device=s.device)[:, None] for v in (lo, hi))
        gone = (((pos > hi_t) & (vel >= 0)) | ((pos < lo_t) & (vel <= 0))).any(0)
        live = ~gone & t.isfinite(s[:6]).all(0)
        if not bool(live.any()):
            return None
        z, vz = pos[self.p][live], vel[self.p][live]
        return float(z.min()), float(z.max()), float(vz.abs().max())

    def field(self, ne_slab, axes):
        return engine.DeviceField.from_ne(ne_slab, axes[0], axes[1], axes[2], engine.omega_of(self.lwl), march_axis=self.p,
                                          phase=self.phase, phase_f64=self.phase_f64)

    def steps(self, field, s, m, h, last, want_jf, channels):
        P = engine.make_params("rk4", probing_direction=self.pd, extent=self.extent, omega=engine.omega_of(self.lwl), n_steps=m,
                               h=h, phase=self.phase, phase_f64=self.phase_f64, early_exit=True, sort=self.sort,
                               out_axes=self.out_axes)
        out = engine.propagate(field, P, s0=s, want_sf=True, want_rf=last, want_jf=last and want_jf, want_steps=True,
                               channels=channels if last else (), with_stats=True)
        return out["sf"], out["steps"].to(self.torch.int64), out["rf"], out["jf"], out["stats_dev"]

    def exit(self, s, want_jf):
        rf, jf, _ = engine.exit_plane(s, self.p, self.out_axes, self.extent, want_jf=want_jf)
        return rf, jf

    def release(self, field):
        self.torch.cuda.current_stream().synchronize()          # the launch that reads the slab has finished
        field.close()
        self.torch.cuda.empty_cache()


def trace_slabs(backend, s0, source, axes, probing_direction, n_steps, h, slab_planes, *, want_jf=False, channels=()):
    """The slab loop, independent of where the arithmetic runs (``backend``: the device, or the host build of the same ray
    code in the tests).  Returns (state, steps per ray, rf, jf, log, stats) with ``log`` one dict per slab (planes, steps taken,
    range of the live rays before it) and ``stats`` the launch counters summed over the slabs (None on the host build)."""
    p = engine.AXIS[probing_direction]
    ax64 = [np.asarray(np.float32(a), dtype=np.float64) for a in axes]
    zc = ax64[p]
    lo, hi = [float(a[0]) for a in ax64], [float(a[-1]) for a in ax64]
    s = backend.to_state(s0)
    steps_total, stats_total, done, log = None, None, 0, []
    rf = jf = None
    while True:
        if done == n_steps:                               # step budget spent before the end of the grid (short probing_depth)
            if channels:
                raise ValueError("the step budget ends inside the grid: fused diagnostics need the rays to reach its last slab")
            rf, jf = backend.exit(s, want_jf)
            return s, steps_total, rf, jf, log, stats_total
        rng = backend.live_range(s, lo, hi)
        if rng is None:                                   # every ray has left the grid for good: the rest are no-ops
            rng = (float(zc[-2]), float(zc[-2]), 0.0)
        zmin, zmax, vmax = rng
        a, b, m, z_stop = plan_slab(zc, zmin, zmax, vmax, h, n_steps - done, slab_planes)
        last = b == len(zc) - 1
        slab_axes = list(axes)
        slab_axes[p] = np.asarray(axes[p])[a:b + 1]
        field = backend.field(source(a, b + 1), slab_axes)
        while True:
            s_new, st, rf, jf, stats = backend.steps(field, s, m, h, last, want_jf, channels)
            after = None if last else backend.live_range(s_new, lo, hi)
            if last or after is None or after[1] <= z_stop:
                break
            if m == 1:
                raise RuntimeError("a ray crossed the slab margin in a single step: increase slab_planes")
            m = max(1, m // 2)                                # a ray got further than planned: redo with fewer steps
        backend.release(field)
        log.append(dict(planes=(a, b), steps=m, z_live=(zmin, zmax)))
        s, done = s_new, done + m
        steps_total = st if steps_total is None else steps_total + st
        if stats is not None:
            stats_total = stats if stats_total is None else stats_total + stats
        if last:
            return s, steps_total, rf, jf, log, stats_total


def solve_out_of_core(s0_import, source, lengths, dims, probing_depth, *, slab_planes, probing_direction="z", lwl=1064e-9,
                      return_E=False, phaseshift=False, phase_f64=False, n_steps=None, ds=None, sort=True,
                      axis_convention="current", diagnostics=(), return_state=False, prefetch=False):
    """``propagator.solve(..., method='rk4')`` for a grid delivered in slabs of ``slab_planes`` planes of the probing axis
    by ``source(k0, k1)``.  ``lengths`` / ``dims`` describe the whole grid as ``ScalarDomain`` takes them (axes
    ``linspace(-L/2, L/2, n)`` rounded to float32).  Same outputs as ``solve``: ``(rf, Jf, duration)`` (+ a dict with
    'sf', 'steps', 'slabs', 'stats' when ``return_state``); ``diagnostics`` (``DiagnosticSpec`` list) are binned by the
    last slab's launch, fused as in ``solve_and_image``.  ``prefetch=True`` (host sources only) reads the next slab on a
    worker thread while the current one is traced (``PrefetchingSource``)."""
    import torch
    from . import propagator
    engine.require_cuda()
    if np.ndim(lengths) == 0:
        lengths = [lengths] * 3
    if np.ndim(dims) == 0:
        dims = [dims] * 3
    axes = [np.float32(np.linspace(-float(L_) / 2, float(L_) / 2, int(n))) for L_, n in zip(lengths, dims)]
    extent = float(probing_depth)
    t_end = np.sqrt(8.0) * extent / C_LIGHT
    if ds is None and n_steps is None:
        pa = engine.AXIS[probing_direction]
        ds = 0.5 * float(lengths[pa]) / (int(dims[pa]) - 1)         # half a cell of the probing axis, as propagator.solve
    if ds is not None:
        h = float(ds) / C_LIGHT
        n_steps = int(np.ceil(t_end / h)) if n_steps is None else int(n_steps)
    else:
        n_steps, h = int(n_steps), t_end / int(n_steps)
    need_phase = any(d.image.kind == "interferogram" for d in diagnostics)
    phase = bool(phaseshift) or need_phase
    backend = _DeviceBackend(lwl, probing_direction, phase, phase_f64, propagator._out_axes(probing_direction, axis_convention),
                             extent, sort)
    chans = [(d.ops, d.image, d.wavelength if d.wavelength else lwl) for d in diagnostics]
    as_numpy = not isinstance(s0_import, torch.Tensor)
    if prefetch:
        pa = engine.AXIS[probing_direction]
        source = PrefetchingSource(source, int(dims[pa]), pa)
    torch.cuda.synchronize()
    start = time()
    try:
        sf, steps, rf, jf, log, stats = trace_slabs(backend, s0_import, source, axes, probing_direction, n_steps, h, slab_planes,
                                                    want_jf=return_E, channels=chans)
    finally:
        if prefetch:
            source.close()
    torch.cuda.synchronize()
    duration = time() - start
    if as_numpy:
        rf, jf = rf.cpu().numpy(), (None if jf is None else jf.cpu().numpy())
    if return_state:
        extra = dict(sf=sf.cpu().numpy() if as_numpy else sf, steps=steps.cpu().numpy() if as_numpy else steps, slabs=log,
                     stats=engine.stats_dict(stats))
        return rf, jf, duration, extra
    return rf, jf, duration


def solve_from_pvti(s0_import, filename, probing_depth, *, slab_planes, probing_direction="z", scale=1.0, **kw):
    """``solve_out_of_core`` on a ``.pvti`` / ``.vti`` dump that is never loaded whole: the box is the one the reference's
    drivers build from the file (half-lengths ``dim * spacing / 2``, pvti_trace_multiprocess.py:45-65 ==
    ``handle_filetypes.domain_from_pvti``), the slabs come from ``handle_filetypes.pvti_slab_source`` (a contiguous byte
    range of the mapped file per slab when probing along z)."""
    from . import handle_filetypes as hf
    source, dims, spacing = hf.pvti_slab_source(filename, probing_direction=probing_direction, device="cuda", scale=scale)
    lengths = [float(dims[a] * spacing[a]) for a in range(3)]
    return solve_out_of_core(s0_import, source, lengths, list(dims), probing_depth, slab_planes=slab_planes,
                             probing_direction=probing_direction, **kw)

