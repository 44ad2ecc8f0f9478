"""``solve`` with the call shape of the reference's ``src/simulator/propagator.py::solve`` (propagator.py:351-702),
plus the fused ``solve_and_image`` fast path that never materialises exit rays.

Integrators (``method=``):
  'rk4'        fixed-step classical RK4, default ``ds`` = half a cell along the probing axis, early exit once a
               ray has left the grid.  The production default (SURVEY.md 7.3-7: the RHS is only C0, so ~2 steps
               per cell is where accuracy saturates).
  'rk45'       Dormand-Prince 5(4) with SciPy's controller and tolerances, step size chosen per ray
               (== the legacy solver run one ray at a time).
  'rk45_joint' the legacy solver exactly as shipped: one step size for the whole bundle
               (src/solvers-legacy/full_solver.py:391).  Explicit s0 only.
  'rk45_bundle' the same joint controller applied per 32-ray bundle (== the legacy solver called on 32-ray chunks):
               lanes stay in lock-step, ~2.5x the throughput of 'rk45'; results depend on bundle membership.
  'tsit5'      the current generation's solver (src/simulator/propagator.py:533-599): Tsitouras 5(4) per ray under
               diffrax's PID controller in normalised time, dt0 = T / save_steps, max_steps = 10000; rtol / atol default
               to upstream's shipped PIDController(rtol=1, atol=1e-5) -- pass 1e-7 / 1e-9 for the values upstream's
               evaluation scripts use.  PARITY UNPINNED (jax / diffrax are not installable where this was built): the
               published method and the controller's documented defaults, held to an independent NumPy restatement.
"""
from time import time

import numpy as np
import torch

from . import engine
from .engine import C_LIGHT as c


def _out_axes(probing_direction, convention):
    p = engine.AXIS[probing_direction]
    if convention == "legacy":            # full_solver.py:856-881
        return {0: (1, 2), 1: (0, 2), 2: (0, 1)}[p]
    return {0: (1, 2), 1: (2, 0), 2: (0, 1)}[p]      # propagator.py:222-262 ('y' swapped upstream)


def _params(domain, probing_depth, lwl, method, n_steps, ds, rtol, atol, precision, early_exit, phase, phase_f64,
            sort, convention, max_steps, save_steps=2):
    return _solver_params(domain.probing_direction, domain.cell_size(), bool(domain.inv_brems), bool(domain.B_on),
                          probing_depth, lwl, method, n_steps, ds, rtol, atol, precision, early_exit, phase, phase_f64,
                          sort, convention, max_steps, save_steps)


def _solver_params(probing_direction, cell_size, atten, faraday, probing_depth, lwl, method, n_steps, ds, rtol, atol,
                   precision, early_exit, phase, phase_f64, sort, convention, max_steps, save_steps=2):
    """``sp_params`` of a solve from what it reads of the domain: the probing direction, the cell size along it (RK4's
    default ``ds``) and whether the attenuation / Faraday channels are on (``out_of_core`` has no domain object)."""
    extent = float(probing_depth)
    t_end = np.sqrt(8.0) * extent / c
    h, n = 0.0, 0
    if rtol is None:
        rtol = 1.0 if method == "tsit5" else 1e-3              # propagator.py:557 / scipy's solve_ivp default
    if atol is None:
        atol = 1e-5 if method == "tsit5" else 1e-6
    if method == "tsit5":
        h = t_end / max(1, int(save_steps))                    # dt0 = (t1 - t0) * norm_factor / Nt with t1 - t0 = 1 (propagator.py:566)
        n = int(max_steps or 10000)                            # propagator.py:572
    elif method == "rk4":
        if ds is None and n_steps is None:
            ds = 0.5 * cell_size
        if ds is not None:
            h = float(ds) / c
            n = int(np.ceil(t_end / h)) if n_steps is None else int(n_steps)
        else:
            n = int(n_steps)
            h = t_end / n
    else:
        n = int(max_steps or 0)
    return engine.make_params(method, probing_direction=probing_direction, extent=extent,
                              omega=engine.omega_of(lwl), n_steps=n, h=h, t_end=t_end, rtol=rtol, atol=atol,
                              phase=phase, phase_f64=phase_f64, early_exit=early_exit, fp32=(precision == "fp32"),
                              sort=sort, out_axes=_out_axes(probing_direction, convention),
                              atten=atten, faraday=faraday,
                              verdet=2.62e-13 * lwl ** 2 if faraday else 0.0)      # propagator.py:353-355


def solve(s0_import, ScalarDomain, probing_depth, *, return_E=False, parallelise=True, jitted=True, save_steps=2,
          memory_debug=False, lwl=1064e-9, keep_domain=False,
          method="rk4", n_steps=None, ds=None, rtol=None, atol=None, precision="fp64", early_exit=True,
          phase_f64=False, sort=True, axis_convention="current", max_steps=None, return_stats=False,
          return_state=False):
    """Trace rays ``s0_import`` (9,N) through ``ScalarDomain``; returns ``(rf, Jf, duration)`` like the
    reference: rf (4,N) [x, theta, y, phi] at the exit plane (m, rad), Jf (2,N) complex or None.
    ``parallelise / jitted / save_steps / memory_debug / keep_domain`` are accepted for call compatibility.

    Call-compatible, not default-compatible: upstream integrates every ray with diffrax Tsit5 under
    ``PIDController(rtol=1, atol=1e-5)``, ``dt0 = (t1 - t0) / 2`` and ``max_steps=10000`` (propagator.py:533-599) -- a
    tolerance that lets the controller take the whole box in a handful of steps.  Here the default is fixed-step RK4 at
    half a cell (``method='rk4'``), and ``method='rk45'`` is SciPy's Dormand-Prince at 1e-3 / 1e-6 (the legacy
    generation's solver).  ``method='tsit5'`` restates upstream's solve itself (same tableau, controller constants, dt0
    and max_steps) but cannot be pinned against diffrax in this environment (DESIGN.md section 6).  ``parallelise`` / ``jitted`` have no effect: there is one code path.

    numpy in -> numpy out; CUDA tensors in -> CUDA tensors out (no host round trip).
    With ``return_stats`` / ``return_state`` a dict with 'stats', 'sf', 'steps' is appended to the tuple."""
    engine.require_cuda()
    as_numpy = not isinstance(s0_import, torch.Tensor)
    s0 = engine.to_device(s0_import, torch.float64)
    phase = bool(ScalarDomain.phaseshift)
    field = ScalarDomain.device_field(lwl, phase=phase, phase_f64=phase_f64)
    P = _params(ScalarDomain, probing_depth, lwl, method, n_steps, ds, rtol, atol, precision, early_exit, phase,
                phase_f64, sort, axis_convention, max_steps, save_steps)
    torch.cuda.synchronize()
    start = time()
    out = engine.propagate(field, P, s0=s0, want_rf=True, want_jf=return_E, want_sf=return_state,
                           want_steps=return_state, with_stats=True)
    torch.cuda.synchronize()
    duration = time() - start
    rf, jf = out["rf"], out["jf"]
    if as_numpy:
        rf = rf.cpu().numpy()
        jf = None if jf is None else jf.cpu().numpy()
    if return_stats or return_state:
        extra = {"stats": engine.stats_dict(out["stats_dev"])}
        if return_state:
            extra["sf"] = out["sf"].cpu().numpy() if as_numpy else out["sf"]
            extra["steps"] = out["steps"].cpu().numpy() if as_numpy else out["steps"]
        return rf, jf, duration, extra
    return rf, jf, duration


def solve_and_image(ScalarDomain, rays, probing_depth, diagnostics, *, lwl=1064e-9, n_rays=None, ray_offset=0,
                    method="rk4", n_steps=None, ds=None, rtol=None, atol=None, precision="fp64", early_exit=True,
                    phase_f64=False, sort=True, axis_convention="current", max_steps=None, sync=True):
    """Fused hot path: rays -> ODE -> exit plane -> optics -> detector images, in one kernel per chunk.

    rays         a (9,N) array/tensor, a ``prefetch_rays`` handle (host bundle whose copy overlaps the previous call), or
                 a ``Beam(device=True)`` whose rays are generated on the GPU
    diagnostics  list of ``DiagnosticSpec`` (see ``diagnostics.spec``); their images accumulate
    Returns (stats dict or None, elapsed seconds or None)."""
    engine.require_cuda()
    need_phase = any(d.image.kind == "interferogram" for d in diagnostics)
    phase = bool(ScalarDomain.phaseshift) or need_phase
    field = ScalarDomain.device_field(lwl, phase=phase, phase_f64=phase_f64)
    P = _params(ScalarDomain, probing_depth, lwl, method, n_steps, ds, rtol, atol, precision, early_exit, phase,
                phase_f64, sort, axis_convention, max_steps)
    chans = [(d.ops, d.image, d.wavelength if d.wavelength else lwl) for d in diagnostics]
    kw = dict(want_rf=False, channels=chans)
    if hasattr(rays, "spec"):                       # device Beam
        n = rays.Np if n_rays is None else n_rays
        kw.update(beam=rays.spec, n=n, ray_offset=ray_offset)
    elif isinstance(rays, PrefetchedRays):          # copy already in flight on the side stream
        torch.cuda.current_stream().wait_event(rays.copied)
        kw.update(s0=rays.tensor)
    else:
        kw.update(s0=engine.to_device(rays, torch.float64))
    if sync:
        torch.cuda.synchronize()
    start = time()
    out = engine.propagate(field, P, **kw)
    if isinstance(rays, PrefetchedRays):
        rays.release()
    if not sync:
        return out["stats_dev"], None
    torch.cuda.synchronize()
    return engine.stats_dict(out["stats_dev"]), time() - start


class PrefetchedRays:
    """Handle returned by ``prefetch_rays``: a (9,N) device buffer whose host->device copy may still be running."""

    def __init__(self, tensor, copied, state, slot):
        self.tensor, self.copied, self._state, self._slot = tensor, copied, state, slot

    def release(self):
        """Mark the buffer reusable once the work queued so far on the current stream has read it."""
        self._state["free"][self._slot].record(torch.cuda.current_stream())
        self._state["busy"][self._slot] = False


_PREFETCH = {}


def prefetch_rays(s0_host):
    """Start copying a (9,N) float64 ray bundle from PINNED host memory on a side stream and return a handle that
    ``solve_and_image`` accepts in place of the rays.  Two device buffers alternate, so the copy of the next bundle
    overlaps the propagation of the current one (the reference's drivers feed their workers chunk by chunk in the same
    way, pvti_trace_multiprocess.py:102-125):

        nxt = prefetch_rays(batches[0])
        for k in range(len(batches)):
            cur, nxt = nxt, (prefetch_rays(batches[k + 1]) if k + 1 < len(batches) else None)
            solve_and_image(domain, cur, depth, specs, sync=False)
    """
    engine.require_cuda()
    if not (isinstance(s0_host, torch.Tensor) and not s0_host.is_cuda and s0_host.is_pinned() and s0_host.dtype == torch.float64
            and s0_host.ndim == 2 and s0_host.shape[0] == 9 and s0_host.is_contiguous()):
        raise TypeError("prefetch_rays needs a contiguous (9, N) float64 tensor in pinned host memory")
    n = int(s0_host.shape[1])
    dev = torch.cuda.current_device()
    st = _PREFETCH.get(dev)
    if st is None or st["cap"] < 9 * n:
        st = dict(stream=st["stream"] if st else torch.cuda.Stream(), cap=9 * n, next=0,
                  bufs=[torch.empty(9 * n, dtype=torch.float64, device="cuda") for _ in range(2)],
                  free=[torch.cuda.Event() for _ in range(2)], busy=[False, False])
        _PREFETCH[dev] = st
    b = st["next"]
    if st["busy"][b]:
        raise RuntimeError("two prefetched bundles are already outstanding: pass one to solve_and_image first")
    st["next"] ^= 1
    st["busy"][b] = True
    dst = st["bufs"][b][:9 * n].view(9, n)
    copied = torch.cuda.Event()
    with torch.cuda.stream(st["stream"]):
        st["stream"].wait_event(st["free"][b])          # the propagation that last read this buffer has finished
        dst.copy_(s0_host, non_blocking=True)
        copied.record(st["stream"])
    return PrefetchedRays(dst, copied, st, b)


def ray_to_Jonesvector(rays, ne_extent, *, probing_direction="z", keep_current_plane=False, return_E=False,
                       axis_convention="current"):
    """propagator.py:178-298 (legacy: full_solver.py:838-894): (9,N) ODE states -> (ray_p (4,N), ray_J (2,N) or None)."""
    as_numpy = not isinstance(rays, torch.Tensor)
    sf = engine.to_device(rays, torch.float64)
    rf, jf, _ = engine.exit_plane(sf, engine.AXIS[probing_direction], _out_axes(probing_direction, axis_convention), ne_extent,
                                  keep_current_plane=keep_current_plane, want_jf=return_E)
    if as_numpy:
        rf, jf = rf.cpu().numpy(), (None if jf is None else jf.cpu().numpy())
    return rf, jf


def back_propogate(rays, ne_extent, probing_direction):
    """propagator.py:300-349 (spelling as upstream): move (9,N) states along their straight lines onto the exit plane.
    (Upstream additionally permutes the rows for 'y'; here rows keep their x, y, z meaning.)"""
    as_numpy = not isinstance(rays, torch.Tensor)
    sf = engine.to_device(rays, torch.float64)
    p = engine.AXIS[probing_direction]
    _, _, sb = engine.exit_plane(sf, p, _out_axes(probing_direction, "legacy"), ne_extent, want_rf=False, want_state=True)
    return sb.cpu().numpy() if as_numpy else sb


def rhs(s, ScalarDomain, *, lwl=1064e-9, phase_f64=False):
    """d(state)/dt of the ray ODE (propagator.py:94-175 / full_solver.py:516-544) for a (9,N) state."""
    as_numpy = not isinstance(s, torch.Tensor)
    sd = engine.to_device(s, torch.float64)
    phase = bool(ScalarDomain.phaseshift)
    field = ScalarDomain.device_field(lwl, phase=phase, phase_f64=phase_f64)
    P = engine.make_params("rk4", probing_direction=ScalarDomain.probing_direction, extent=1.0,
                           omega=engine.omega_of(lwl), n_steps=1, h=1.0, phase=phase, phase_f64=phase_f64)
    out = engine.rhs(field, P, sd)
    return out.cpu().numpy() if as_numpy else out
