"""Out-of-core tracing with the per-ray adaptive solves (out_of_core.trace_slabs_adaptive, sp_propagate_window).

CPU: the slab driver run over the host build of the windowed controller loops (ray_core.h dp5_window / tsit5_window,
compiled with g++ in tests/window_harness.cpp) against one unbounded launch over the whole grid, which is the in-core
kernel's arithmetic.  GPU: solve_out_of_core against propagator.solve / solve_and_image, bit for bit."""
import ctypes as C

import numpy as np
import pytest

from window_harness import WindowHarness, window_record

C_LIGHT = 299792458.0


def omega_of(lwl):
    return 2 * np.pi * (C_LIGHT / lwl)


@pytest.fixture(scope="module")
def H():
    return WindowHarness()


class _HostAdaptiveBackend:
    """``out_of_core.trace_slabs_adaptive`` on the host build of the windowed loops: same driver as the device path."""

    def __init__(self, H, omega, p, phase, **kw):
        self.H, self.omega, self.p, self.phase, self.kw = H, omega, p, phase, kw
        self.launches = []

    def to_state(self, s0):
        return np.array(s0, dtype=np.float64)

    def record(self, n):
        return window_record(n)

    def slowest(self, s, rec):
        todo = (rec["flags"] & 4) == 0
        if not todo.any():
            return None
        z = np.minimum(s[self.p][todo], rec["ctl"][2][todo])
        z = z[np.isfinite(z)]
        return float(z.min()) if z.size else -np.inf

    def select(self, s, rec, w_lo, w_hi):
        w = s[self.p]
        return np.nonzero(((rec["flags"] & 4) == 0) & ~(w < w_lo) & ~(w > w_hi))[0]

    def summary(self, rec, idx, t_stop):
        f, c = rec["flags"][idx], rec["ctl"][:, idx]
        parked = (f & 4) == 0
        return dict(attempts=int(rec["steps"].sum()), finished=int(((rec["flags"] & 4) != 0).sum()),
                    pending=int((parked & ((f & 2) != 0)).sum()), clip=int((parked & (c[0] + c[1] - t_stop > 0)).sum()))

    def field(self, ne_slab, axes):
        return self.H.field(np.ascontiguousarray(ne_slab), axes[0], axes[1], axes[2], self.omega, march_axis=self.p,
                            phase=self.phase, f64=self.phase)

    def launch(self, field, s, rec, idx, w_lo, w_hi, grid_range, channels):
        self.launches.append(len(idx))
        sub = np.ascontiguousarray(s[:, idx])
        r = {k: np.ascontiguousarray(v[..., idx]) for k, v in rec.items()}
        self.H.window(field, sub, r, w_lo, w_hi, grid_range, **self.kw)
        s[:, idx] = sub
        for k, v in rec.items():
            v[..., idx] = r[k]

    def release(self, field):
        pass


def _whole(H, g, axes, p, phase, s0, **kw):
    """One launch over the whole grid with an unbounded window: the in-core solve."""
    omega = kw.pop("omega")
    f = H.field(g["ne"], *axes, omega, march_axis=p, phase=phase, f64=phase)
    s = np.array(s0, dtype=np.float64)
    rec = window_record(s.shape[1])
    H.window(f, s, rec, -np.inf, np.inf, **kw)
    assert ((rec["flags"] & 4) != 0).all()
    return s, rec


def _case(H, golden, pd, method, phase, planes, *, depth_scale=1.0, early=False, cap=0, rtol=None, atol=None):
    from synthpy_b200 import out_of_core as OC
    g = golden("g3_turb")
    p = "xyz".index(pd)
    pre = "" if pd == "z" else pd + "_"
    axes = [g[pre + k] for k in "xyz"]
    s0 = g[pre + "s0"]
    omega, ext = omega_of(float(g["lwl"])), float(g["extent"]) * depth_scale
    t_end = np.sqrt(8.0) * ext / C_LIGHT
    if method == "tsit5":
        kw = dict(method="tsit5", t_end=t_end, dt0=0.5, rtol=rtol or 1e-7, atol=atol or 1e-9, cap=cap)
        t_stop = 1.0
    else:
        kw = dict(method="rk45", t_end=t_end, rtol=rtol or 1e-3, atol=atol or 1e-6, cap=cap, early=early)
        t_stop = t_end
    sw, rw = _whole(H, g, axes, p, phase, s0, omega=omega, **kw)
    be = _HostAdaptiveBackend(H, omega, p, phase, **kw)
    s, rec, log = OC.trace_slabs_adaptive(be, s0, OC.array_source(g["ne"], pd), axes, pd, planes, t_stop, max_slab_planes=32)
    assert np.array_equal(s, sw, equal_nan=True), (pd, method)
    assert np.array_equal(rec["steps"], rw["steps"]) and np.array_equal(rec["flags"], rw["flags"])
    assert np.array_equal(rec["ctl"][:2], rw["ctl"][:2], equal_nan=True)
    rf = H.field(g["ne"], *axes, omega, march_axis=p).exit(s, p, *{0: (1, 2), 1: (2, 0), 2: (0, 1)}[p], ext)
    rf_w = H.field(g["ne"], *axes, omega, march_axis=p).exit(sw, p, *{0: (1, 2), 1: (2, 0), 2: (0, 1)}[p], ext)
    assert np.array_equal(rf, rf_w, equal_nan=True)
    assert sum(e["attempts"] for e in log) == int(rw["steps"].sum())             # committed attempts are the in-core ones
    assert (rec["evals"] >= rw["evals"]).all()                                    # plus the evaluations of dropped attempts
    assert sum(e["finished"] for e in log) == s0.shape[1]
    assert log[0]["planes"][1] - log[0]["planes"][0] + 1 <= planes + 1                # slabs grow only while no ray can go on
    return g, s, rec, rw, log


@pytest.mark.parametrize("pd,method,phase,planes", [("z", "rk45", False, 9), ("z", "rk45", True, 14), ("x", "rk45", False, 11),
                                                    ("y", "rk45", True, 12), ("z", "tsit5", False, 9), ("z", "tsit5", True, 13),
                                                    ("x", "tsit5", True, 11), ("y", "tsit5", False, 12)])
def test_adaptive_slabs_equal_whole_grid(H, golden, pd, method, phase, planes):
    """Slabs of 9 .. 14 of 32 planes reproduce the whole-grid solve bit for bit: full states, attempts per ray, controller
    records and exit rays; parks happen, some of them with a rejected attempt pending (RK45).  On this 32-plane box the
    first attempts (SciPy's initial step, diffrax's dt0) span most of it, so the slab grows to the whole grid before the
    rays can finish."""
    g, s, rec, rw, log = _case(H, golden, pd, method, phase, planes)
    assert len(log) >= 3 and log[0]["planes"][0] == 0 and log[-1]["planes"][1] == 31, log
    assert sum(e["parked"] for e in log) > 0
    if method == "rk45":
        assert sum(e["parked_pending"] for e in log) > 0, log
    if phase:
        assert np.nanmax(np.abs(s[7])) > 1.0


def test_adaptive_slabs_host_references(H, golden):
    """The unbounded-window loop is the harness's whole-grid hh_rk45 up to its error norm (it divides by
    n_state where the kernels multiply by its reciprocal, and an ulp there can change a later step): most rays agree bit
    for bit (72 % for RK45 on this field)."""
    g = golden("g3_turb")
    axes = [g[k] for k in "xyz"]
    omega, ext = omega_of(float(g["lwl"])), float(g["extent"])
    t_end = np.sqrt(8.0) * ext / C_LIGHT
    f = H.field(g["ne"], *axes, omega)
    sw, rw = _whole(H, g, axes, 2, False, g["s0"], omega=omega, method="rk45", t_end=t_end)
    sf, att, _ = f.rk45(g["s0"], t_end)
    assert np.mean(att == rw["steps"]) > 0.9 and np.mean((sf == sw).all(0)) > 0.6


def test_adaptive_slabs_short_depth_early_exit_and_cap(H, golden):
    """A short probing depth (rays reach t_end inside the grid), early exit, and a small attempt cap (capped rays) give the
    whole-grid result too."""
    _case(H, golden, "z", "rk45", False, 9, depth_scale=0.5)
    _case(H, golden, "z", "rk45", True, 10, early=True)
    g, s, rec, rw, log = _case(H, golden, "z", "rk45", False, 10, cap=12)
    assert ((rec["flags"] & 8) != 0).any() and rec["steps"].max() == 12
    g, s, rec, rw, log = _case(H, golden, "z", "tsit5", False, 10, cap=9)
    assert ((rec["flags"] & 8) != 0).any()


def test_adaptive_slab_too_thin_raises(H, golden):
    """Tsit5 at upstream's rtol=1 takes steps far wider than a thin slab's window: the driver raises instead of looping."""
    from synthpy_b200 import out_of_core as OC
    g = golden("g3_turb")
    axes = [g[k] for k in "xyz"]
    omega, ext = omega_of(float(g["lwl"])), float(g["extent"])
    be = _HostAdaptiveBackend(H, omega, 2, False, method="tsit5", t_end=np.sqrt(8.0) * ext / C_LIGHT, dt0=0.5, rtol=1.0, atol=1e-5)
    with pytest.raises(ValueError, match="increase slab_planes"):
        OC.trace_slabs_adaptive(be, g["s0"], OC.array_source(g["ne"]), axes, "z", 8, 1.0)
    assert len(be.launches) == 2
    with pytest.raises(ValueError, match="slab_planes must be at least"):
        OC.trace_slabs_adaptive(be, g["s0"], OC.array_source(g["ne"]), axes, "z", 5, 1.0)


def test_adaptive_methods_refused():
    """Joint and bundle-step RK45 cannot run out of core (one step size per batch / bundle); out-of-core RK4 stays float64
    with early exit.  Refused before anything touches the GPU."""
    from synthpy_b200 import out_of_core as OC
    for m in ("rk45_joint", "rk45_bundle"):
        with pytest.raises(ValueError, match="not available out of core"):
            OC.solve_out_of_core(np.zeros((9, 1)), None, 1.0, 8, 1.0, slab_planes=8, method=m)
    with pytest.raises(ValueError, match="unknown method"):
        OC.solve_out_of_core(np.zeros((9, 1)), None, 1.0, 8, 1.0, slab_planes=8, method="euler")
    with pytest.raises(ValueError, match="float64 with early exit"):
        OC.solve_out_of_core(np.zeros((9, 1)), None, 1.0, 8, 1.0, slab_planes=8, precision="fp32")


def test_propagate_window_validation():
    """sp_propagate_window: every invalid argument is SP_EINVAL with a message, before any CUDA call."""
    from synthpy_b200 import _lib as L, engine
    lib = L.lib
    buf = (C.c_double * 16)()
    u32 = (C.c_uint32 * 4)()
    fake = C.cast(buf, C.c_void_p)

    def call(P, state=fake, ctl=fake, flags=u32, steps=u32, lo=0.0, hi=1.0, field=fake, ws=fake):
        return lib.sp_propagate_window(field, C.byref(P), ws, state, 1, None, 0, ctl, C.cast(flags, C.c_void_p) if flags is not None else None,
                                       C.cast(steps, C.c_void_p) if steps is not None else None, lo, hi, -1.0, 1.0, None, None, None, 0, None,
                                       None)

    def P(method="rk45", **kw):
        return engine.make_params(method, extent=1e-2, omega=1e15, h=0.5, **kw)
    cases = [(P("rk4"), {}), (P("rk45_joint"), {}), (P("rk45_bundle"), {}), (P(atten=True), {}), (P(faraday=True), {}),
             (P(), dict(lo=1.0, hi=0.0)), (P(), dict(lo=float("nan"))), (P(), dict(state=None)), (P(), dict(ctl=None)),
             (P(), dict(flags=None)), (P(), dict(steps=None)), (P(), dict(field=None)), (P(), dict(ws=None))]
    for params, kw in cases:
        rc = call(params, **kw)
        assert rc == -1, (params.method, kw)                                      # SP_EINVAL
        assert lib.sp_last_error().decode()
