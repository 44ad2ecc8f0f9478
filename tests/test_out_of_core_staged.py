"""Out-of-core adaptive solves with stage parking (out_of_core.trace_slabs_adaptive(park='stage'),
sp_propagate_window_staged).

CPU: the slab driver over the host build of the windowed loops with STAGED on (ray_core.h dp5_window / tsit5_window /
dp5x_window, compiled with g++ in tests/stage_harness.cpp) against one unbounded launch over the whole grid, which is the
in-core arithmetic; the refusals of solve_out_of_core and of the C ABI."""
import ctypes as C

import numpy as np
import pytest

from stage_harness import CTL_STAGED, ROW_SHIFT, StageHarness, stage_record

C_LIGHT = 299792458.0


def omega_of(lwl):
    return 2 * np.pi * (C_LIGHT / lwl)


@pytest.fixture(scope="module")
def H():
    return StageHarness()


class _HostStagedBackend:
    """``out_of_core.trace_slabs_adaptive(park='stage')`` on the host build of the staged loops: the device backend's rules
    (needed point, selection, summary) over NumPy arrays.  ``served_away`` counts launched rays whose own position was
    outside the window (served only because their next point was inside)."""

    def __init__(self, H, omega, p, phase, channels=None, **kw):
        self.H, self.omega, self.p, self.phase, self.channels, self.kw = H, omega, p, phase, channels, kw
        self.launches, self.served_away = [], 0

    def to_state(self, s0):
        return np.array(s0, dtype=np.float64)

    def record(self, n):
        return stage_record(n, self.kw["method"])

    def _needed(self, s, rec):
        w = rec["ctl"][2]
        return np.where(np.isfinite(w), w, s[self.p])

    def slowest(self, s, rec):
        todo = (rec["flags"] & 4) == 0
        if not todo.any():
            return None
        z = self._needed(s, rec)[todo]
        z = z[np.isfinite(z)]
        return float(z.min()) if z.size else -np.inf

    def select(self, s, rec, w_lo, w_hi):
        w = self._needed(s, rec)
        return np.nonzero(((rec["flags"] & 4) == 0) & ~(w < w_lo) & ~(w > w_hi))[0]

    def summary(self, rec, idx, t_stop):
        f, c = rec["flags"][idx], rec["ctl"][:, idx]
        parked = (f & 4) == 0
        mid = parked & ((f & CTL_STAGED) != 0) & (((f >> ROW_SHIFT) & 15) >= 1)
        return dict(attempts=int(rec["steps"].sum()), finished=int(((rec["flags"] & 4) != 0).sum()),
                    pending=int((parked & ((f & 2) != 0)).sum()), clip=int((parked & (c[0] + c[1] - t_stop > 0)).sum()),
                    evals=int(rec["evals"].sum()), mid=int(mid.sum()))

    def field(self, slab, axes):
        if self.channels is None:
            return self.H.field(np.ascontiguousarray(slab), axes[0], axes[1], axes[2], self.omega, march_axis=self.p,
                                phase=self.phase, f64=self.phase)
        f = self.H.field(np.ascontiguousarray(slab.ne), axes[0], axes[1], axes[2], self.omega, march_axis=self.p, phase=True,
                         f64=True)
        z = np.zeros(slab.ne.shape)
        f.attach(z if slab.kappa is None else slab.kappa, z if slab.ne_faraday is None else slab.ne_faraday,
                 np.zeros(slab.ne.shape + (3,)) if slab.B is None else slab.B)
        return f

    def launch(self, field, s, rec, idx, w_lo, w_hi, grid_range, channels):
        self.launches.append(len(idx))
        w = s[self.p][idx]
        self.served_away += int((((rec["flags"][idx] & CTL_STAGED) != 0) & ((w < w_lo) | (w > w_hi))).sum())
        sub = np.ascontiguousarray(s[:, idx])
        r = {k: np.ascontiguousarray(v[..., idx]) for k, v in rec.items()}
        self.H.staged(field, sub, r, w_lo, w_hi, grid_range, **self.kw)
        s[:, idx] = sub
        for k, v in rec.items():
            v[..., idx] = r[k]

    def release(self, field):
        pass


def _widest(zc, planes):
    """The widest slab slab_planes_for gives for ``planes``: ``planes`` unless the uniform-axis widening adds some."""
    from synthpy_b200 import out_of_core as OC
    return max(b - a + 1 for a, b in (OC.slab_planes_for(zc, z, planes) for z in zc))


def _check(H, be, field_whole, s0, sources, axes, pd, planes, t_stop, ext):
    """The staged slab driver against one unbounded launch over the whole grid, bit for bit."""
    from synthpy_b200 import out_of_core as OC
    p = "xyz".index(pd)
    sw, rw = np.array(s0, dtype=np.float64), stage_record(s0.shape[1], be.kw["method"])
    H.staged(field_whole, sw, rw, -np.inf, np.inf, **be.kw)
    assert ((rw["flags"] & 4) != 0).all() and ((rw["flags"] & CTL_STAGED) == 0).all()
    s, rec, log = OC.trace_slabs_adaptive(be, s0, sources, axes, pd, planes, t_stop, park="stage")
    assert np.array_equal(s, sw, equal_nan=True), (pd, be.kw)
    assert np.array_equal(rec["steps"], rw["steps"]) and np.array_equal(rec["flags"], rw["flags"])
    assert np.array_equal(rec["ctl"][:2], rw["ctl"][:2], equal_nan=True)
    assert np.array_equal(rec["evals"], rw["evals"])                              # every evaluation ran exactly once
    out = {0: (1, 2), 1: (2, 0), 2: (0, 1)}[p]
    assert np.array_equal(field_whole.exit(s, p, *out, ext), field_whole.exit(sw, p, *out, ext), equal_nan=True)
    zc = np.float64(np.float32(axes[p]))
    assert max(e["planes"][1] - e["planes"][0] + 1 for e in log) <= _widest(zc, planes)      # the slab never grows
    assert sum(e["evals"] for e in log) == int(rw["evals"].sum())
    assert sum(e["attempts"] for e in log) == int(rw["steps"].sum()) and sum(e["finished"] for e in log) == s0.shape[1]
    return s, rec, log


def _case(H, golden, pd, method, phase, planes, *, depth_scale=1.0, early=False, cap=0, rtol=None, atol=None, nan=False):
    from synthpy_b200 import out_of_core as OC
    g = golden("g3_turb")
    p = "xyz".index(pd)
    pre = "" if pd == "z" else pd + "_"
    axes = [g[pre + k] for k in "xyz"]
    s0 = np.array(g[pre + "s0"], dtype=np.float64)
    if nan:
        s0[:3, 5] = np.nan
    omega, ext = omega_of(float(g["lwl"])), float(g["extent"]) * depth_scale
    t_end = np.sqrt(8.0) * ext / C_LIGHT
    if method == "tsit5":
        kw = dict(method="tsit5", t_end=t_end, dt0=0.5, rtol=rtol or 1e-7, atol=atol or 1e-9, cap=cap)
        t_stop = 1.0
    else:
        kw = dict(method="rk45", t_end=t_end, rtol=rtol or 1e-3, atol=atol or 1e-6, cap=cap, early=early)
        t_stop = t_end
    whole = H.field(g["ne"], *axes, omega, march_axis=p, phase=phase, f64=phase)
    be = _HostStagedBackend(H, omega, p, phase, **kw)
    s, rec, log = _check(H, be, whole, s0, OC.array_source(g["ne"], pd), axes, pd, planes, t_stop, ext)
    return g, s, rec, log, be


@pytest.mark.parametrize("pd,method,phase,planes,tol", [("z", "rk45", False, 8, None), ("z", "rk45", True, 10, None),
                                                        ("x", "rk45", False, 9, None), ("x", "rk45", True, 12, None),
                                                        ("y", "rk45", False, 11, None), ("y", "rk45", True, 8, None),
                                                        ("z", "tsit5", False, 9, (1e-7, 1e-9)), ("x", "tsit5", True, 10, (1e-7, 1e-9)),
                                                        ("z", "tsit5", True, 12, (1.0, 1e-5)), ("y", "tsit5", False, 10, (1.0, 1e-5))])
def test_staged_slabs_equal_whole_grid(H, golden, pd, method, phase, planes, tol):
    """Fixed slabs of 8 .. 12 of 32 planes reproduce the whole-grid solve bit for bit (states, the record's t and h, flags,
    attempts, exit rays) with the whole grid's evaluation count; rays park mid-attempt and are served by windows that do not
    hold their own position (SciPy's first attempts span most of this box)."""
    rtol, atol = tol or (None, None)
    g, s, rec, log, be = _case(H, golden, pd, method, phase, planes, rtol=rtol, atol=atol)
    assert len(log) >= 3 and sum(e["parked_mid"] for e in log) > 0, log
    assert be.served_away > 0
    if phase:
        assert np.nanmax(np.abs(s[7])) > 1.0


def test_staged_tsit5_rtol1_in_thin_slabs(H, golden):
    """Tsit5 at upstream's controller (rtol 1, atol 1e-5) in 8-plane slabs -- where attempt parking raises 'increase
    slab_planes' -- completes and equals the whole grid."""
    g, s, rec, log, be = _case(H, golden, "z", "tsit5", False, 8, rtol=1.0, atol=1e-5)
    assert max(e["planes"][1] - e["planes"][0] + 1 for e in log) == 8


def test_staged_short_depth_early_exit_cap_nan(H, golden):
    """A short probing depth (rays reach t_end inside the grid), early exit, an attempt cap (capped rays) and a NaN ray give
    the whole-grid result too."""
    _case(H, golden, "z", "rk45", False, 9, depth_scale=0.5)
    _case(H, golden, "z", "tsit5", True, 9, depth_scale=0.5)
    _case(H, golden, "x", "rk45", True, 10, early=True)
    g, s, rec, log, be = _case(H, golden, "z", "rk45", False, 10, cap=12)
    assert ((rec["flags"] & 8) != 0).any() and rec["steps"].max() == 12
    g, s, rec, log, be = _case(H, golden, "z", "tsit5", False, 10, cap=9)
    assert ((rec["flags"] & 8) != 0).any() and rec["steps"].max() == 9
    g, s, rec, log, be = _case(H, golden, "z", "rk45", False, 9, nan=True)
    assert (rec["flags"][5] & 8) != 0 and not np.isfinite(s[:3, 5]).any()


@pytest.mark.parametrize("method", ["rk45", "rk45x"])
def test_staged_resume_outside_slab_early_exit(H, golden, method):
    """Early exit of a resumed ray whose position lies outside the slab: rays launched slowly up a steep density ramp turn
    back, so an attempt can park at a stage point below the window while the ray itself is above the next slab, moving up.
    The escape test of such a ray uses the whole grid's w bounds, not the slab's, so it does not finish early and the
    driver equals the whole grid."""
    from synthpy_b200 import out_of_core as OC
    g = golden("g3_turb")
    axes = [g[k] for k in "xyz"]
    z = np.float64(np.float32(axes[2]))
    ne = np.broadcast_to(3e26 * (1 + 4 * (z - z[0]) / (z[-1] - z[0]))[None, None, :], g["ne"].shape).copy()
    omega, ext = omega_of(float(g["lwl"])), float(g["extent"])
    rng = np.random.default_rng(1)
    n = 64
    s0 = np.zeros((9, n))
    s0[0], s0[1], s0[2] = rng.uniform(-3e-3, 3e-3, n), rng.uniform(-3e-3, 3e-3, n), rng.uniform(z[4], z[-4], n)
    s0[5], s0[6] = C_LIGHT * 0.02 * rng.uniform(0.5, 1.5, n), 1.0
    t_end = np.sqrt(8.0) * ext / C_LIGHT

    class Watch(_HostStagedBackend):
        """Counts resumed rays whose position is past the window on the side their w velocity points to."""
        ahead = 0

        def launch(self, field, s, rec, idx, w_lo, w_hi, grid_range, channels):
            w, v = s[2][idx], s[5][idx]
            held = (rec["flags"][idx] & CTL_STAGED) != 0
            self.ahead += int((held & (((w > w_hi) & (v >= 0)) | ((w < w_lo) & (v <= 0)))).sum())
            super().launch(field, s, rec, idx, w_lo, w_hi, grid_range, channels)
    src, whole = OC.array_source(ne), H.field(ne, *axes, omega, phase=method == "rk45x", f64=method == "rk45x")
    kw = dict(method=method, t_end=t_end, early=True)
    if method == "rk45x":                         # the nine-row loop, with an attenuation channel on the same ramp
        from synthpy_b200 import engine
        src = OC.channel_source(src, "z", omega, inv_brems=True, Te=100.0, Z=1.0)
        whole.attach(engine.kappa_grid(ne, 100.0, 1.0, omega), np.zeros(ne.shape), np.zeros(ne.shape + (3,)))
        kw.update(verdet=0.0, atten=True)
    be = Watch(H, omega, 2, False, channels=True if method == "rk45x" else None, **kw)
    _check(H, be, whole, s0, src, axes, "z", 8, t_end, ext)
    assert be.ahead > 0


@pytest.mark.parametrize("atten,faraday,pd,planes", [(False, True, "z", 8), (True, False, "z", 10), (True, True, "z", 9),
                                                     (True, True, "x", 8)])
def test_staged_channels_equal_whole_grid(H, golden, atten, faraday, pd, planes):
    """The staged nine-row RK45 (dp5x_window) over slabs with the ChannelSlab grids attached (Te clamped to Te_min) equals
    the unbounded launch on all nine rows, attempts and evaluations; with both channels also the whole-grid hh_rk45_ext."""
    from synthpy_b200 import engine, out_of_core as OC
    from test_out_of_core_channels import _along
    g = golden("g6_channels")
    lwl, ext = float(g["lwl"]), float(g["extent"])
    omega, verdet = omega_of(lwl), 2.62e-13 * lwl ** 2
    p = "xyz".index(pd)
    axes = [g[k] for k in "xyz"]
    Te = g["Te"].copy()
    Te.reshape(-1)[::17] = 0.25
    kappa = engine.kappa_grid(g["ne"], np.maximum(1.0, Te), g["Z"], omega)
    s0 = _along(g, pd)
    t_end = np.sqrt(8.0) * ext / C_LIGHT
    whole = H.field(g["ne"], *axes, omega, march_axis=p, phase=True, f64=True)
    whole.attach(kappa, g["ne"], g["B"])
    src = OC.channel_source(OC.array_source(g["ne"], pd), pd, omega, inv_brems=atten, B_on=faraday, B=g["B"], Te=Te, Z=g["Z"])
    be = _HostStagedBackend(H, omega, p, True, channels=True, method="rk45x", t_end=t_end, verdet=verdet, atten=atten,
                            faraday=faraday)
    s, rec, log = _check(H, be, whole, s0, src, axes, pd, planes, t_end, ext)
    assert sum(e["parked_mid"] for e in log) > 0 and be.served_away > 0, log
    if atten:
        assert np.ptp(s[6]) > 1e-4
    if faraday:
        assert np.abs(s[8] - s0[8]).max() > 1e-7
    if atten and faraday:
        sf, nfev = whole.rk45_ext(s0, t_end, verdet)
        assert np.array_equal(s, sf, equal_nan=True) and np.array_equal(rec["steps"], (nfev - 2) // 6)


def test_staged_refusals():
    """park='stage' refusals: ValueError before anything touches the GPU."""
    from synthpy_b200 import out_of_core as OC
    s0 = np.zeros((9, 1))
    for extra, msg in [(dict(park="stage"), "RK4 never parks"), (dict(park="stage", method="rk45", max_slab_planes=16), "never grows"),
                       (dict(park="ray", method="rk45"), "park must be"), (dict(park="stage", method="tsit5", B_on=True, B=np.zeros((8, 8, 8, 3))), "tsit5")]:
        with pytest.raises(ValueError, match=msg):
            OC.solve_out_of_core(s0, None, 1.0, 8, 1.0, slab_planes=8, **extra)
    with pytest.raises(ValueError, match="park must be"):
        OC.trace_slabs_adaptive(None, s0, None, [np.zeros(8)] * 3, "z", 8, 1.0, park="whole")
    with pytest.raises(ValueError, match="never grows"):
        OC.trace_slabs_adaptive(None, s0, None, [np.zeros(8)] * 3, "z", 8, 1.0, park="stage", max_slab_planes=16)


def test_propagate_window_staged_validation():
    """sp_propagate_window_staged: a null stage store and everything the two other windowed entry points refuse is SP_EINVAL
    with a message, before any CUDA call."""
    from synthpy_b200 import _lib as L, engine
    lib = L.lib
    buf = (C.c_double * 4096)()
    u32 = (C.c_uint32 * 4)()
    fake = C.cast(buf, C.c_void_p)

    def call(P, state=fake, ctl=fake, flags=u32, steps=u32, stage=fake, lo=0.0, hi=1.0, g_lo=-1.0, field=fake, ws=fake, n_ch=0):
        return lib.sp_propagate_window_staged(field, C.byref(P), ws, state, 1, None, 0, ctl,
                                              C.cast(flags, C.c_void_p) if flags is not None else None,
                                              C.cast(steps, C.c_void_p) if steps is not None else None, stage, lo, hi, g_lo,
                                              1.0, None, None, None, n_ch, None, None)

    def P(method="rk45", **kw):
        return engine.make_params(method, extent=1e-2, omega=1e15, h=0.5, **kw)
    ch = dict(atten=True, faraday=True)
    cases = [(P(), dict(stage=None)), (P("tsit5"), dict(stage=None)), (P(**ch), dict(stage=None)),
             (P("rk4"), {}), (P("rk45_joint"), {}), (P("rk45_bundle"), {}), (P("rk4", **ch), {}), (P("tsit5", **ch), {}),
             (P("tsit5", faraday=True), {}), (P(fp32=True, **ch), {}), (P(fp32=True, atten=True), {}),
             (P("rk45_bundle", **ch), {}), (P(), dict(lo=1.0, hi=0.0)), (P(**ch), dict(lo=float("nan"))),
             (P(), dict(g_lo=2.0)), (P(), dict(state=None)), (P(**ch), dict(ctl=None)), (P(), dict(flags=None)),
             (P("tsit5"), dict(steps=None)), (P(), dict(field=None)), (P(**ch), dict(ws=None)), (P(), dict(n_ch=5)),
             (engine.make_params("rk45", extent=1e-2, omega=1e15, probing_direction="z"), {})]
    for params, kw in cases:
        rc = call(params, **kw)
        assert rc == -1, (params.method, params.flags, kw)                     # SP_EINVAL
        assert lib.sp_last_error().decode()
    params = P()
    params.probing_axis = 3
    assert call(params) == -1
