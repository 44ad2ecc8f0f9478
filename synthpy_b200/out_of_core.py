"""Tracing through a field that does not fit in HBM: the grid is streamed slab by slab along the probing axis.

The reference's counterpart is the domain batching of ``src/simulator/domain.py:137-243`` + ``propagator.py:366-450``
(``region_count`` sections of the domain, regenerated one after the other while the rays keep their state) -- work in
progress upstream (the section bounds are hard-coded, domain.py:247-252).  On a B200 a 1024^3 packed field is 17 GB of
180 GB, so this is needed only from ~2048^3 upwards (137 GB packed) or when several fields share a GPU; it is built so
that nothing about the result depends on it:

  * fixed-step RK4: the ray ODE has no explicit time dependence, so N steps through the whole grid are N_1 + N_2 + ...
    steps through consecutive slabs, the (9, N) state carried over exactly;
  * the per-ray adaptive solves (method='rk45', 'tsit5'; ``trace_slabs_adaptive`` over ``sp_propagate_window``): a ray
    parks when its next attempt would evaluate the field inside the grid but outside the slab's window, with its
    controller record as at the top of that loop iteration, and resumes in a later slab; every committed attempt is the
    in-core arithmetic (see ray_core.h dp5_window).  With ``park='stage'`` (``sp_propagate_window_staged``) a ray parks
    between stage evaluations instead, its attempt in progress kept in a per-ray stage store, so a window only has to
    hold the next point it evaluates: fixed-size slabs then serve SciPy's box-sized first attempts too, without growing,
    and every evaluation runs once, as in core.  Joint and bundle-step RK45 stay in core;
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

The attenuation and Faraday channels (``solve_out_of_core(..., inv_brems=True, B_on=True, B=..., Te=..., Z=...)``) stream
with the density: ``channel_source`` composes the ne source with slab sources of B, Te and Z into one that returns a
``ChannelSlab`` per slab -- the ne planes and the channel grids of the same planes, converted as ``ScalarDomain.device_field``
converts the whole grids (Te clamped to Te_min, kappa from ``engine.kappa_grid`` on the host: elementwise, so a slab's
kappa is the whole grid's kappa sliced).  The backends attach them to each slab's field; RK4 then runs sp_propagate's
RK4X kernel and RK45 sp_propagate_window_channels, with amp and pol carried in the (9, N) state.
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


class ChannelSlab:
    """One slab of ``channel_source``: the ne planes and the channel grids of the same planes (None where a channel is off):
    ``kappa`` (host float64), ``ne_faraday`` (the ne planes, for the Faraday term) and ``B`` (planes x 3)."""
    __slots__ = ("ne", "kappa", "ne_faraday", "B")

    def __init__(self, ne, kappa=None, ne_faraday=None, B=None):
        self.ne, self.kappa, self.ne_faraday, self.B = ne, kappa, ne_faraday, B

    def attach(self, field):
        if self.kappa is not None or self.B is not None:
            field.attach_channels(kappa=self.kappa, ne=self.ne_faraday, B=self.B)
        return field


def _host(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else a


def _slab_source(a, axis):
    """``f(k0, k1)`` over a slab callable (returned as is), an array-like over the whole grid (sliced along ``axis`` as
    ``array_source`` slices it; trailing axes kept) or a scalar (the same value for every slab)."""
    if callable(a):
        return a
    if getattr(a, "ndim", 0) == 0:
        return lambda k0, k1: a

    def source(k0, k1):
        idx = [slice(None)] * 3
        idx[axis] = slice(k0, k1)
        return a[tuple(idx)]
    return source


def _is_host_source(a):
    """Whether ``PrefetchingSource`` may wrap the slab source of ``a``: callables (refused later if they return CUDA tensors)
    and host arrays, not CUDA tensors or scalars."""
    return callable(a) or (getattr(a, "ndim", 0) > 0 and not getattr(a, "is_cuda", False))


def channel_source(source, probing_direction, omega, *, inv_brems=False, B_on=False, B=None, Te=None, Z=None, Te_min=1.0):
    """The slab source of a solve with the attenuation (``inv_brems``) and / or Faraday (``B_on``) channels: ``f(k0, k1)``
    returns a ``ChannelSlab`` of ``source(k0, k1)`` and the channel grids of those planes.  ``B`` ((..., 3) per point),
    ``Te`` and ``Z`` are slab callables or array-likes over the whole grid (NumPy, memmap, CUDA tensor); ``Te`` and ``Z``
    may be scalars.  Each slab is converted as ``ScalarDomain`` converts the whole grids: ``Te`` clamped with
    ``np.maximum(Te_min, Te)``, kappa = ``engine.kappa_grid(ne, Te, Z, omega)`` on the host, the ne planes themselves for
    the Faraday term.  A channel slab whose shape is not the ne slab's raises ``ValueError``."""
    axis = engine.AXIS[probing_direction]
    b_src = _slab_source(B, axis) if B_on else None
    te_src = _slab_source(Te, axis) if inv_brems else None
    z_src = _slab_source(Z, axis) if inv_brems else None

    def slab(k0, k1):
        ne = source(k0, k1)
        shape = tuple(ne.shape)
        kappa = b = None
        if inv_brems:
            te, z = te_src(k0, k1), z_src(k0, k1)
            for name, a in (("Te", te), ("Z", z)):
                if getattr(a, "ndim", 0) and tuple(a.shape) != shape:
                    raise ValueError(f"{name} slab has shape {tuple(a.shape)}, the ne slab {shape}")
            kappa = engine.kappa_grid(_host(ne), np.maximum(Te_min, _host(te)), _host(z), omega)
        if B_on:
            b = b_src(k0, k1)
            if tuple(b.shape) != shape + (3,):
                raise ValueError(f"B slab has shape {tuple(b.shape)}, expected {shape + (3,)} (the ne slab's, plus 3)")
        return ChannelSlab(ne, kappa, ne if B_on else None, b)
    return slab


def _field_of(backend, slab, axes):
    ne = slab.ne if isinstance(slab, ChannelSlab) else slab
    field = engine.DeviceField.from_ne(ne, axes[0], axes[1], axes[2], engine.omega_of(backend.lwl), march_axis=backend.p,
                                       phase=backend.phase, phase_f64=backend.phase_f64)
    return slab.attach(field) if isinstance(slab, ChannelSlab) else field


def axis_is_uniform(a32):
    """The test field_prep.h / np.gradient make on an axis: every float32 spacing equal to the first."""
    d = np.diff(np.asarray(a32, dtype=np.float32))
    return bool(np.all(d == d[0])) if d.size else True


def slab_planes_for(zc, zmin, slab_planes):
    """The planes [a, b] of the next slab: from MARGIN planes behind the cell holding ``zmin`` (the slowest live ray),
    ``slab_planes`` long, widened until its probing axis makes the same uniform / non-uniform stencil choice as the whole
    axis (zc: the probing axis, float32 values as float64)."""
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
    return a, b


def plan_slab(zc, zmin, zmax, vmax, h, steps_left, slab_planes):
    """Which planes [a, b] to load and how many RK4 steps to take in them.

    zc          the probing axis (float32 values as float64), n planes
    zmin, zmax  extreme probing-axis positions of the live rays now;  vmax  their largest speed along that axis
    Returns (a, b, m, z_stop): after m steps no live ray may be beyond z_stop (checked by the driver); ``b == n - 1``
    means the slab reaches the end of the grid and takes all remaining steps."""
    n = len(zc)
    a, b = slab_planes_for(zc, zmin, slab_planes)
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

    def __init__(self, lwl, probing_direction, phase, phase_f64, out_axes, extent, sort, atten=False, faraday=False):
        import torch
        self.torch = torch
        self.lwl, self.pd, self.phase, self.phase_f64 = lwl, probing_direction, phase, phase_f64
        self.out_axes, self.extent, self.sort = out_axes, extent, sort
        self.atten, self.faraday = atten, faraday
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
        return _field_of(self, ne_slab, axes)

    def steps(self, field, s, m, h, last, want_jf, channels):
        P = engine.make_params("rk4", probing_direction=self.pd, extent=self.extent, omega=engine.omega_of(self.lwl), n_steps=m,
                               h=h, phase=self.phase, phase_f64=self.phase_f64, early_exit=True, sort=self.sort,
                               out_axes=self.out_axes, atten=self.atten, faraday=self.faraday,
                               verdet=2.62e-13 * self.lwl ** 2 if self.faraday else 0.0)      # as propagator._solver_params
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
    range of the live rays before it, bytes of the slab's device field) and ``stats`` the launch counters summed over the slabs (None on the host build)."""
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
        nbytes = getattr(field, "nbytes", None)
        while True:
            s_new, st, rf, jf, stats = backend.steps(field, s, m, h, last, want_jf, channels)
            after = None if last else backend.live_range(s_new, lo, hi)
            if last or after is None or after[1] <= z_stop:
                break
            if m == 1:
                raise RuntimeError("a ray crossed the slab margin in a single step: increase slab_planes")
            m = max(1, m // 2)                                # a ray got further than planned: redo with fewer steps
        backend.release(field)
        log.append(dict(planes=(a, b), steps=m, z_live=(zmin, zmax), field_bytes=nbytes))
        s, done = s_new, done + m
        steps_total = st if steps_total is None else steps_total + st
        if stats is not None:
            stats_total = stats if stats_total is None else stats_total + stats
        if last:
            return s, steps_total, rf, jf, log, stats_total


class _AdaptiveDeviceBackend:
    """The product path of the adaptive solves: packed slab field in HBM, ``sp_propagate_window`` per slab
    (``sp_propagate_window_staged`` with ``park='stage'``)."""

    def __init__(self, params, lwl, probing_direction, phase, phase_f64, want_jf, park="attempt"):
        import torch
        self.torch, self.P, self.lwl, self.phase, self.phase_f64 = torch, params, lwl, phase, phase_f64
        self.p = engine.AXIS[probing_direction]
        self.want_jf, self.staged = want_jf, park == "stage"
        self.stats = torch.zeros(6, dtype=torch.int64, device="cuda")
        self.stages = None

    def to_state(self, s0):
        s = engine.to_device(s0, self.torch.float64)
        return s.clone() if isinstance(s0, self.torch.Tensor) else s        # advanced in place: never the caller's tensor

    def record(self, n):
        t = self.torch
        rec = engine.controller_record(n)
        rec["ctl"][2].fill_(np.inf)
        self.rf = t.empty((4, n), dtype=t.float64, device="cuda")
        self.jf = t.empty((2, n), dtype=t.complex128, device="cuda") if self.want_jf else None
        if self.staged:
            self.stages = engine.stage_store(n, self.P)
        return rec

    def _needed(self, s, rec):
        """Stage parking: the point a ray needs next -- where it parked, or its position before its first launch."""
        w = rec["ctl"][2]
        return self.torch.where(self.torch.isfinite(w), w, s[self.p])

    def slowest(self, s, rec):
        todo = (rec["flags"] & engine.L.CTL_FINISHED) == 0
        if not bool(todo.any()):
            return None
        z = self._needed(s, rec)[todo] if self.staged else self.torch.minimum(s[self.p][todo], rec["ctl"][2][todo])
        z = z[self.torch.isfinite(z)]
        return float(z.min()) if z.numel() else -np.inf

    def select(self, s, rec, w_lo, w_hi):
        w = self._needed(s, rec) if self.staged else s[self.p]
        ok = ((rec["flags"] & engine.L.CTL_FINISHED) == 0) & ~(w < w_lo) & ~(w > w_hi)      # NaN positions are inside
        return self.torch.nonzero(ok).squeeze(1).to(self.torch.int32)

    def summary(self, rec, idx, t_stop):
        f, c = rec["flags"][idx.long()], rec["ctl"][:, idx.long()]
        L = engine.L
        parked = (f & L.CTL_FINISHED) == 0
        out = dict(attempts=int(rec["steps"].sum()), finished=int(((rec["flags"] & L.CTL_FINISHED) != 0).sum()),
                   pending=int((parked & ((f & L.CTL_PENDING) != 0)).sum()),
                   clip=int((parked & (c[0] + c[1] - t_stop > 0)).sum()))
        if self.staged:
            mid = parked & ((f & L.CTL_STAGED) != 0) & (((f >> L.CTL_ROW_SHIFT) & 15) >= 1)
            out.update(evals=int(self.stats[5]), mid=int(mid.sum()))
        return out

    def field(self, ne_slab, axes):
        return _field_of(self, ne_slab, axes)

    def launch(self, field, s, rec, idx, w_lo, w_hi, grid_range, channels):
        engine.propagate_window(field, self.P, s, rec, w_lo, w_hi, grid_range, idx=idx, rf=self.rf, jf=self.jf, channels=channels,
                                stats=self.stats, stages=self.stages)

    def release(self, field):
        self.torch.cuda.current_stream().synchronize()
        field.close()
        self.torch.cuda.empty_cache()


def trace_slabs_adaptive(backend, s0, source, axes, probing_direction, slab_planes, t_stop, *, max_slab_planes=None,
                         channels=(), park="attempt"):
    """The slab loop of the adaptive solves (``backend``: the device, or the host build of the same ray code in the tests).
    Each pass loads the slab from MARGIN planes behind the slowest unfinished ray (or the lowest point a parked ray needs)
    and launches once over the unfinished rays inside its window; a ray runs until it finishes or parks at the window, and
    resumes in a later slab from its controller record.  Returns (state, record, log): ``log`` one dict per slab with its
    planes, window, rays launched, finished, parked, parked with a pending rejection ('parked_pending'), parked right
    before their final step, the one clipped to the end of the interval ('parked_clip'), committed attempts, and the bytes
    of the slab's device field ('field_bytes', channel grids included).
    ``t_stop`` is where that clip happens in the record's time (t_end for RK45, 1 for Tsit5's normalised time).

    A launch in which no ray commits an attempt or finishes leaves the state as it was: some attempt spans more planes than
    the window.  The slab then doubles, up to ``max_slab_planes`` (default ``slab_planes``: no growth), and returns to
    ``slab_planes`` after the next launch that makes progress.  SciPy's initial step is one such attempt: 100 h0 is of
    the order of the distance from the origin, so the first (rejected) attempts of RK45 span much of the box.  A second
    launch without progress at the largest slab raises ``ValueError`` instead of looping.

    ``park='stage'`` (a backend built for it: ``sp_propagate_window_staged``): rays park between stage evaluations and carry
    their attempt in progress in a stage store, so a window only has to hold the NEXT point a ray evaluates -- where it
    parked, or its position before its first launch (the ray's needed point).  ``slowest`` and ``select`` go by the needed
    point, and the window starts MARGIN planes behind the lowest one, so every launch evaluates at least that point: the
    slab never grows (``max_slab_planes`` is refused).  Each slab's log adds the field evaluations ('evals') and the rays
    parked mid-attempt ('parked_mid').  Two launches in a row that neither evaluate, commit nor finish anything raise
    ``RuntimeError`` (the first launch can evaluate only points outside the grid, which are not counted)."""
    if park not in ("attempt", "stage"):
        raise ValueError(f"park must be 'attempt' or 'stage', not {park!r}")
    staged = park == "stage"
    if staged and max_slab_planes is not None:
        raise ValueError("park='stage' never grows the slab: max_slab_planes does not apply")
    p = engine.AXIS[probing_direction]
    zc = np.asarray(np.float32(axes[p]), dtype=np.float64)
    n = len(zc)
    if int(slab_planes) < 2 * MARGIN + 2:
        raise ValueError(f"slab_planes must be at least {2 * MARGIN + 2}: the window is the slab less {MARGIN} planes per side")
    top = max(int(slab_planes), int(max_slab_planes or slab_planes))
    grid_range = (float(zc[0]), float(zc[-1]))
    s = backend.to_state(s0)
    rec = backend.record(s.shape[1])
    log, stalls, planes = [], 0, int(slab_planes)
    while True:
        zmin = backend.slowest(s, rec)
        if zmin is None:
            return s, rec, log
        a, b = slab_planes_for(zc, zmin, planes)
        w_lo = -np.inf if a == 0 else float(zc[a + MARGIN])
        w_hi = np.inf if b == n - 1 else float(zc[b - MARGIN])
        idx = backend.select(s, rec, w_lo, w_hi)
        before = backend.summary(rec, idx, t_stop)
        slab_axes = list(axes)
        slab_axes[p] = np.asarray(axes[p])[a:b + 1]
        field = backend.field(source(a, b + 1), slab_axes)
        nbytes = getattr(field, "nbytes", None)
        backend.launch(field, s, rec, idx, w_lo, w_hi, grid_range, channels)
        backend.release(field)
        after = backend.summary(rec, idx, t_stop)
        done, att = after["finished"] - before["finished"], after["attempts"] - before["attempts"]
        log.append(dict(planes=(a, b), window=(w_lo, w_hi), launched=len(idx), finished=done, parked=len(idx) - done,
                        parked_pending=after["pending"], parked_clip=after["clip"], attempts=att, field_bytes=nbytes))
        if staged:
            evals = after["evals"] - before["evals"]
            log[-1].update(evals=evals, parked_mid=after["mid"])
            stalls = 0 if (evals > 0 or att > 0 or done > 0) else stalls + 1
            if stalls >= 2:
                raise RuntimeError(f"stage parking: two launches over the window ({w_lo:.4g} .. {w_hi:.4g} m) evaluated "
                                   "nothing although it holds the lowest point a ray needs")
            continue
        # Nothing committed and nothing finished: the state is what it was, so the next window is this one or (once) the
        # one that holds the point a ray parked at below it.  Grow the slab; at the largest, a second such launch means an
        # attempt wider than the window.
        if att > 0 or done > 0:
            stalls, planes = 0, int(slab_planes)
        elif planes < top:
            planes = min(top, 2 * planes)
        else:
            stalls += 1
            if stalls >= 2:
                raise ValueError(f"slab of {b - a + 1} planes is too thin for the adaptive steps: no ray can take its next "
                                 f"attempt inside the window ({w_lo:.4g} .. {w_hi:.4g} m): increase slab_planes "
                                 "(or max_slab_planes)")


def solve_out_of_core(s0_import, source, lengths, dims, probing_depth, *, slab_planes, probing_direction="z", lwl=1064e-9,
                      return_E=False, phaseshift=False, phase_f64=False, n_steps=None, ds=None, sort=True,
                      axis_convention="current", diagnostics=(), return_state=False, prefetch=False, method="rk4",
                      rtol=None, atol=None, max_steps=None, precision="fp64", early_exit=True, save_steps=2,
                      max_slab_planes=None, inv_brems=False, B_on=False, B=None, Te=None, Z=None, park="attempt"):
    """``propagator.solve(..., method=...)`` for a grid delivered in slabs of ``slab_planes`` planes of the probing axis
    by ``source(k0, k1)``.  ``lengths`` / ``dims`` describe the whole grid as ``ScalarDomain`` takes them (axes
    ``linspace(-L/2, L/2, n)`` rounded to float32).  Same outputs as ``solve``: ``(rf, Jf, duration)`` (+ a dict with
    'sf', 'steps', 'slabs', 'stats' when ``return_state``); ``diagnostics`` (``DiagnosticSpec`` list) are binned fused as
    in ``solve_and_image`` (RK4: by the last slab's launch; adaptive: each ray by the launch it finishes in).
    ``prefetch=True`` (host sources only) reads the next slab on a worker thread while the current one is traced
    (``PrefetchingSource``).

    ``method='rk4'`` (default; ``n_steps`` / ``ds``) or the per-ray adaptive solves ``'rk45'`` and ``'tsit5'`` with
    ``rtol`` / ``atol`` / ``max_steps`` / ``precision`` / ``early_exit`` / ``save_steps`` as ``propagator.solve`` takes
    them; every result equals the in-core solve's bit for bit.  'rk45_joint' and 'rk45_bundle' are not available out of
    core (one step size per batch / per bundle).  ``max_slab_planes`` lets an adaptive solve grow a slab while no ray can
    take its next attempt inside it (``trace_slabs_adaptive``).

    The attenuation (``inv_brems``, with ``Te`` and ``Z``) and Faraday (``B_on``, with ``B``) channels are those of
    ``ScalarDomain(inv_brems=..., B_on=...)`` with ``external_Te`` / ``external_Z`` / ``external_B``: each of ``B`` ((..., 3)
    per point), ``Te`` and ``Z`` is an array-like over the whole grid (NumPy, memmap, CUDA tensor; sliced along the probing
    axis) or a slab callable ``f(k0, k1)`` like ``source``; ``Te`` and ``Z`` may be scalars (``channel_source``).  With
    the channels, RK4 and RK45 ('rk4', 'rk45') in float64; Tsit5 does not integrate them, in core or out of core.  RK45
    with ``park='attempt'`` saves memory only when ``max_slab_planes`` covers SciPy's first attempts, which span about half
    the box (DESIGN.md section 6).

    ``park`` (adaptive solves): 'attempt' (default) parks a ray a whole attempt at a time, so a window must hold the ray and
    every stage point of its next attempt (the slab grows up to ``max_slab_planes``); 'stage' parks it between stage
    evaluations with the attempt in progress kept in a per-ray stage store on the device (184 B per ray for RK45, 336 B
    for Tsit5, 432 B with the channels), so slabs of ``slab_planes`` planes serve every ray and the slab never grows --
    the same results, bit for bit, and the in-core evaluation count."""
    import torch
    from . import propagator
    if method in ("rk45_joint", "rk45_bundle"):
        raise ValueError(f"method={method!r} is not available out of core: its step size is shared by a whole batch / "
                         "bundle of rays; use 'rk45' (per ray), 'tsit5' or 'rk4'")
    if method not in ("rk4", "rk45", "tsit5"):
        raise ValueError(f"unknown method {method!r}")
    if park not in ("attempt", "stage"):
        raise ValueError(f"park must be 'attempt' or 'stage', not {park!r}")
    if park == "stage" and method == "rk4":
        raise ValueError("park='stage' is for the adaptive solves ('rk45', 'tsit5'): RK4 never parks mid-step")
    if park == "stage" and max_slab_planes is not None:
        raise ValueError("park='stage' never grows the slab: max_slab_planes does not apply")
    if method == "rk4" and (precision != "fp64" or not early_exit):
        raise ValueError("out-of-core RK4 runs in float64 with early exit (precision='fp64', early_exit=True)")
    inv_brems, B_on = bool(inv_brems), bool(B_on)
    if inv_brems or B_on:
        _check_channels(dims, probing_direction, method, precision, inv_brems, B_on, B, Te, Z)
    engine.require_cuda()
    if inv_brems or B_on:
        source = _channels_from(source, dims, probing_direction, lwl, prefetch, inv_brems, B_on, B, Te, Z)
        prefetch = False                          # each host source got its own PrefetchingSource
    if method in ("rk45", "tsit5"):
        return _solve_adaptive(s0_import, source, lengths, dims, probing_depth, slab_planes=slab_planes,
                               probing_direction=probing_direction, lwl=lwl, return_E=return_E, phaseshift=phaseshift,
                               phase_f64=phase_f64, axis_convention=axis_convention, diagnostics=diagnostics,
                               return_state=return_state, prefetch=prefetch, method=method, rtol=rtol, atol=atol,
                               max_steps=max_steps, precision=precision, early_exit=early_exit, save_steps=save_steps,
                               sort=sort, max_slab_planes=max_slab_planes, atten=inv_brems, faraday=B_on, park=park)
    lengths, dims, axes = _grid_axes(lengths, dims)
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
                             extent, sort, atten=inv_brems, faraday=B_on)
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
        _close(source)
    torch.cuda.synchronize()
    duration = time() - start
    if as_numpy:
        rf, jf = rf.cpu().numpy(), (None if jf is None else jf.cpu().numpy())
    if return_state:
        extra = dict(sf=sf.cpu().numpy() if as_numpy else sf, steps=steps.cpu().numpy() if as_numpy else steps, slabs=log,
                     stats=engine.stats_dict(stats))
        return rf, jf, duration, extra
    return rf, jf, duration


def _check_channels(dims, probing_direction, method, precision, inv_brems, B_on, B, Te, Z):
    """The refusals of a solve with channels, before anything touches the GPU."""
    if B_on and B is None:
        raise ValueError("B_on=True needs B (an array over the grid, (..., 3) per point, or a slab callable)")
    if inv_brems and (Te is None or Z is None):
        raise ValueError("inv_brems=True needs Te and Z (arrays over the grid, scalars or slab callables)")
    if method == "tsit5":
        raise ValueError("method='tsit5' does not integrate the attenuation / Faraday channels (in core neither): use 'rk4' "
                         "or 'rk45'")
    if precision != "fp64":
        raise ValueError("the attenuation / Faraday channels are float64 only (precision='fp64')")
    shape = tuple(int(n) for n in (dims if np.ndim(dims) else [dims] * 3))
    for name, a, want in (("B", B if B_on else None, shape + (3,)), ("Te", Te if inv_brems else None, shape),
                          ("Z", Z if inv_brems else None, shape)):
        if a is not None and not callable(a) and getattr(a, "ndim", 0) and tuple(a.shape) != want:
            raise ValueError(f"{name} has shape {tuple(a.shape)}, the grid needs {want}")


def _channels_from(source, dims, probing_direction, lwl, prefetch, inv_brems, B_on, B, Te, Z):
    """``channel_source`` over ``source`` and the channel inputs; with ``prefetch`` every host source (ne, B, Te, Z) is
    wrapped in its own ``PrefetchingSource`` first."""
    pa = engine.AXIS[probing_direction]
    n = int(dims[pa]) if np.ndim(dims) else int(dims)
    if prefetch:
        source = PrefetchingSource(source, n, pa)
        B, Te, Z = (PrefetchingSource(_slab_source(a, pa), n, pa) if (on and _is_host_source(a)) else a
                    for a, on in ((B, B_on), (Te, inv_brems), (Z, inv_brems)))
    slab = channel_source(source, probing_direction, engine.omega_of(lwl), inv_brems=inv_brems, B_on=B_on, B=B, Te=Te, Z=Z)
    slab.parts = [a for a in (source, B, Te, Z) if isinstance(a, PrefetchingSource)]
    return slab


def _close(source):
    """Stop the worker threads of the ``PrefetchingSource`` objects behind ``source``."""
    for s in [source] + list(getattr(source, "parts", ())):
        if isinstance(s, PrefetchingSource):
            s.close()


def _grid_axes(lengths, dims):
    if np.ndim(lengths) == 0:
        lengths = [lengths] * 3
    if np.ndim(dims) == 0:
        dims = [dims] * 3
    axes = [np.float32(np.linspace(-float(L_) / 2, float(L_) / 2, int(n))) for L_, n in zip(lengths, dims)]
    return list(lengths), list(dims), axes


def _solve_adaptive(s0_import, source, lengths, dims, probing_depth, *, slab_planes, probing_direction, lwl, return_E,
                    phaseshift, phase_f64, axis_convention, diagnostics, return_state, prefetch, method, rtol, atol,
                    max_steps, precision, early_exit, save_steps, sort, max_slab_planes, atten=False, faraday=False,
                    park="attempt"):
    import torch
    from . import propagator
    lengths, dims, axes = _grid_axes(lengths, dims)
    pa = engine.AXIS[probing_direction]
    need_phase = any(d.image.kind == "interferogram" for d in diagnostics)
    phase = bool(phaseshift) or need_phase
    P = propagator._solver_params(probing_direction, float(lengths[pa]) / (int(dims[pa]) - 1), atten, faraday, probing_depth,
                                  lwl, method, None, None, rtol, atol, precision, early_exit, phase, phase_f64, sort,
                                  axis_convention, max_steps, save_steps)
    backend = _AdaptiveDeviceBackend(P, lwl, probing_direction, phase, phase_f64, return_E, park=park)
    chans = [(d.ops, d.image, d.wavelength if d.wavelength else lwl) for d in diagnostics]
    as_numpy = not isinstance(s0_import, torch.Tensor)
    if prefetch:
        source = PrefetchingSource(source, int(dims[pa]), pa)
    torch.cuda.synchronize()
    start = time()
    try:
        sf, rec, log = trace_slabs_adaptive(backend, s0_import, source, axes, probing_direction, slab_planes,
                                            1.0 if method == "tsit5" else P.t_end, max_slab_planes=max_slab_planes,
                                            channels=chans, park=park)
    finally:
        _close(source)
    torch.cuda.synchronize()
    duration = time() - start
    rf, jf, steps = backend.rf, backend.jf, rec["steps"]
    if as_numpy:
        rf, jf = rf.cpu().numpy(), (None if jf is None else jf.cpu().numpy())
    if return_state:
        extra = dict(sf=sf.cpu().numpy() if as_numpy else sf, steps=steps.cpu().numpy() if as_numpy else steps, slabs=log,
                     stats=engine.stats_dict(backend.stats))
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

