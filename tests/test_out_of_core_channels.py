"""Out-of-core tracing with the attenuation and Faraday channels (out_of_core.channel_source, sp_propagate_window_channels).

CPU: the slab drivers run over the host build of the ray code with each slab's kappa, ne and B attached (RK4: rk4_step_ext;
RK45: ray_core.h dp5x_window, compiled with g++ in tests/channel_harness.cpp) against the whole-grid solves hh_rk4_ext /
hh_rk45_ext, bit for bit; the slab conversions; the refusals of the C ABI and of solve_out_of_core."""
import ctypes as C

import numpy as np
import pytest

from channel_harness import ChannelHarness
from window_harness import window_record

C_LIGHT = 299792458.0


def omega_of(lwl):
    return 2 * np.pi * (C_LIGHT / lwl)


@pytest.fixture(scope="module")
def H():
    return ChannelHarness()


def _grids(g, omega):
    """g6's channel inputs, with Te pushed below Te_min at a few points (the clamp must act), and the whole-grid kappa."""
    from synthpy_b200 import engine
    Te = g["Te"].copy()
    Te.reshape(-1)[::17] = 0.25
    kappa = engine.kappa_grid(g["ne"], np.maximum(1.0, Te), g["Z"], omega)
    return Te, kappa


def _along(g, pd):
    """g6's rays, or (pd='x') rays along x through the same box."""
    if pd == "z":
        return g["s0"]
    from synthpy_b200 import legacy
    np.random.seed(4)
    s0 = legacy.init_beam(96, 3e-3, 2e-3, float(g["x"][-1]), "circular", "x")
    s0[6] = np.linspace(0.5, 1.5, s0.shape[1])             # amp and pol start away from 1 / 0: carried from slab to slab
    s0[8] = np.linspace(-0.1, 0.1, s0.shape[1])
    return s0


class _HostRK4ChannelBackend:
    """``out_of_core.trace_slabs`` on the host build: each slab's field gets the ChannelSlab's grids attached."""

    def __init__(self, H, omega, p, out_axes, extent, verdet):
        self.H, self.omega, self.p, self.out_axes, self.extent, self.verdet = H, omega, p, out_axes, extent, verdet
        self.launches, self.vscale = [], 1.0

    def to_state(self, s0):
        return np.array(s0, dtype=np.float64)

    def live_range(self, s, lo, hi):
        pos, vel = s[:3], s[3:6]
        lo, hi = np.array(lo)[:, None], np.array(hi)[:, None]
        gone = (((pos > hi) & (vel >= 0)) | ((pos < lo) & (vel <= 0))).any(0)
        live = ~gone & np.isfinite(s[:6]).all(0)
        if not live.any():
            return None
        z, vz = pos[self.p][live], vel[self.p][live]
        return float(z.min()), float(z.max()), float(np.abs(vz).max()) * self.vscale

    def field(self, slab, axes):
        f = self.H.field(np.ascontiguousarray(slab.ne), axes[0], axes[1], axes[2], self.omega, march_axis=self.p, phase=True,
                         f64=True)
        f.attach(slab.kappa, slab.ne_faraday, slab.B)
        return f

    def steps(self, field, s, m, h, last, want_jf, channels):
        self.launches.append(m)
        sf, st = self.H.rk4_ext_steps(field, s, m, h, self.verdet)
        rf = field.exit(sf, self.p, self.out_axes[0], self.out_axes[1], self.extent) if last else None
        return sf, st.astype(np.int64), rf, None, None

    def release(self, field):
        pass


@pytest.mark.parametrize("pd", ["z", "x"])
def test_rk4_channel_slabs_equal_whole_grid(H, golden, pd):
    """RK4 with kappa, ne and B attached to every slab: all nine state rows, steps per ray and exit rays equal the whole-grid
    hh_rk4_ext bit for bit -- along z and x, with the planner's forced redo, and with every source prefetched."""
    from synthpy_b200 import out_of_core as OC
    g = golden("g6_channels")
    lwl, ext = float(g["lwl"]), float(g["extent"])
    omega, verdet = omega_of(lwl), 2.62e-13 * lwl ** 2
    p = "xyz".index(pd)
    out_axes = {0: (1, 2), 1: (2, 0), 2: (0, 1)}[p]
    axes = [g[k] for k in "xyz"]
    Te, kappa = _grids(g, omega)
    s0 = _along(g, pd)
    cell = np.diff(np.float32(axes[p])).min()
    h = 0.5 * float(cell) / C_LIGHT
    n = int(np.ceil(np.sqrt(8.0) * ext / C_LIGHT / h))
    whole = H.field(g["ne"], *axes, omega, march_axis=p, phase=True, f64=True)
    whole.attach(kappa, g["ne"], g["B"])
    sf, steps = H.rk4_ext_steps(whole, s0, n, h, verdet)
    rf = whole.exit(sf, p, out_axes[0], out_axes[1], ext)
    assert np.ptp(sf[6]) > 1e-3 and np.abs(sf[8] - s0[8]).max() > 1e-6                 # both channels are live
    src = OC.channel_source(OC.array_source(g["ne"], pd), pd, omega, inv_brems=True, B_on=True, B=g["B"], Te=Te, Z=g["Z"])
    for vscale in (1.0, 0.45):
        be = _HostRK4ChannelBackend(H, omega, p, out_axes, ext, verdet)
        be.vscale = vscale
        s_sl, st_sl, rf_sl, _, log, _ = OC.trace_slabs(be, s0, src, axes, pd, n, h, 9)
        assert len(log) >= 3 and log[-1]["planes"][1] == len(axes[p]) - 1, log
        assert np.array_equal(s_sl, sf, equal_nan=True) and np.array_equal(st_sl, steps), (pd, vscale)
        assert np.array_equal(rf_sl, rf, equal_nan=True)
        assert (len(be.launches) > len(log)) == (vscale < 1.0)                          # the redo happened (only) when forced
    # every host source behind its own PrefetchingSource, composed after wrapping (as solve_out_of_core(prefetch=True))
    pre = [OC.PrefetchingSource(OC._slab_source(a, p), len(axes[p]), p) for a in (g["ne"], g["B"], Te, g["Z"])]
    src = OC.channel_source(pre[0], pd, omega, inv_brems=True, B_on=True, B=pre[1], Te=pre[2], Z=pre[3])
    be = _HostRK4ChannelBackend(H, omega, p, out_axes, ext, verdet)
    s_pf, st_pf, rf_pf, _, log, _ = OC.trace_slabs(be, s0, src, axes, pd, n, h, 9)
    for q in pre:
        q.close()
        assert q.misses == 1 and q.hits == len(log) - 1
    assert np.array_equal(s_pf, sf, equal_nan=True) and np.array_equal(st_pf, steps) and np.array_equal(rf_pf, rf, equal_nan=True)


class _HostChannelWindowBackend:
    """``out_of_core.trace_slabs_adaptive`` on the host build of dp5x_window, the slabs' channel grids attached."""

    def __init__(self, H, omega, p, **kw):
        self.H, self.omega, self.p, self.kw = H, omega, p, kw
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

    def field(self, slab, axes):
        f = self.H.field(np.ascontiguousarray(slab.ne), axes[0], axes[1], axes[2], self.omega, march_axis=self.p, phase=True,
                         f64=True)
        f.attach(slab.kappa, slab.ne_faraday, slab.B)
        return f

    def launch(self, field, s, rec, idx, w_lo, w_hi, grid_range, channels):
        self.launches.append(len(idx))
        sub = np.ascontiguousarray(s[:, idx])
        r = {k: np.ascontiguousarray(v[..., idx]) for k, v in rec.items()}
        self.H.window_ext(field, sub, r, w_lo, w_hi, grid_range, **self.kw)
        s[:, idx] = sub
        for k, v in rec.items():
            v[..., idx] = r[k]

    def release(self, field):
        pass


@pytest.mark.parametrize("pd,planes", [("z", 8), ("z", 12), ("x", 10)])
def test_rk45_channel_window_equals_whole_grid(H, golden, pd, planes):
    """dp5x_window over slabs of 8 .. 12 planes (growing while no ray can go on) equals hh_rk45_ext on the whole grid bit
    for bit: all nine rows, attempts per ray, the committed attempts of the slab log; rays park, some with a rejection
    pending."""
    from synthpy_b200 import out_of_core as OC
    g = golden("g6_channels")
    lwl, ext = float(g["lwl"]), float(g["extent"])
    omega, verdet = omega_of(lwl), 2.62e-13 * lwl ** 2
    p = "xyz".index(pd)
    axes = [g[k] for k in "xyz"]
    Te, kappa = _grids(g, omega)
    s0 = _along(g, pd)
    t_end = np.sqrt(8.0) * ext / C_LIGHT
    whole = H.field(g["ne"], *axes, omega, march_axis=p, phase=True, f64=True)
    whole.attach(kappa, g["ne"], g["B"])
    sf, nfev = whole.rk45_ext(s0, t_end, verdet)
    attempts = (nfev - 2) // 6
    # one unbounded launch is the whole-grid loop
    s1, r1 = np.array(s0, dtype=np.float64), window_record(s0.shape[1])
    H.window_ext(whole, s1, r1, -np.inf, np.inf, t_end=t_end, verdet=verdet)
    assert np.array_equal(s1, sf, equal_nan=True) and np.array_equal(r1["steps"], attempts)
    src = OC.channel_source(OC.array_source(g["ne"], pd), pd, omega, inv_brems=True, B_on=True, B=g["B"], Te=Te, Z=g["Z"])
    be = _HostChannelWindowBackend(H, omega, p, t_end=t_end, verdet=verdet)
    s, rec, log = OC.trace_slabs_adaptive(be, s0, src, axes, pd, planes, t_end, max_slab_planes=len(axes[p]))
    assert np.array_equal(s, sf, equal_nan=True), pd
    assert np.array_equal(rec["steps"], attempts) and ((rec["flags"] & 4) != 0).all()
    assert sum(e["attempts"] for e in log) == int(attempts.sum()) and sum(e["finished"] for e in log) == s0.shape[1]
    assert (rec["evals"] >= r1["evals"]).all()
    assert len(log) >= 3 and sum(e["parked"] for e in log) > 0 and sum(e["parked_pending"] for e in log) > 0, log
    assert np.ptp(s[6]) > 1e-4 and np.abs(s[8] - s0[8]).max() > 1e-7                    # both channels are live


def test_ext_eval_cached_equals_fresh(H, golden):
    """A resumed ray recomputes its derivative through a fresh cell cache: deriv9 after a walk through one cache (kappa,
    ne and B interpolated with the cached cell's weights) equals fresh lookups bit for bit away from nodes."""
    g = golden("g6_channels")
    lwl = float(g["lwl"])
    omega, verdet = omega_of(lwl), 2.62e-13 * lwl ** 2
    f = H.field(g["ne"], g["x"], g["y"], g["z"], omega, phase=True, f64=True)
    f.attach(g["kappa"], g["ne"], g["B"])
    ax = [np.float64(np.float32(g[k])) for k in "xyz"]
    rng = np.random.default_rng(5)
    n = 20000
    pts = np.zeros((3, n))
    q = np.array([a[len(a) // 2] for a in ax]) + 1e-7
    for i in range(n):
        u = rng.random()
        if u < 0.8:
            k = rng.integers(3)
            q[k] += rng.normal() * 0.6 * np.median(np.diff(ax[k]))
        elif u < 0.95:
            q = np.array([rng.uniform(a[0] - 0.2 * (a[-1] - a[0]), a[-1] + 0.2 * (a[-1] - a[0])) for a in ax])
        else:
            k = rng.integers(3)
            q[k] = ax[k][rng.integers(len(ax[k]))]
        pts[:, i] = q
    s = np.zeros((9, n))
    s[0:3] = pts
    s[3:6] = rng.normal(size=(3, n)) * C_LIGHT
    s[6] = 1.0 + rng.random(n)
    fresh, walk = f.rhs_ext(s, verdet), H.rhs_ext_walk(f, s, verdet)
    on_node = np.zeros(n, dtype=bool)
    for k in range(3):
        on_node |= np.abs(pts[k][:, None] - ax[k][None, :]).min(axis=1) <= 4 * np.spacing(np.abs(pts[k]))
    off = ~on_node
    assert off.mean() > 0.8 and (fresh[6][off] != 0).mean() > 0.3 and (fresh[8][off] != 0).mean() > 0.3
    for row in (3, 4, 5, 6, 8):
        assert np.array_equal(walk[row][off], fresh[row][off]), row
    assert np.allclose(walk[[6, 8]], fresh[[6, 8]], rtol=1e-12, atol=0)


@pytest.mark.parametrize("pd", ["z", "x"])
def test_slab_kappa_equals_whole_grid(golden, pd):
    """Each ChannelSlab holds the whole grid's kappa (Te clamped to Te_min first), ne and B sliced, bit for bit; scalar Te
    and Z broadcast as engine.kappa_grid broadcasts them; a channel slab of another shape is refused."""
    from synthpy_b200 import engine, out_of_core as OC
    g = golden("g6_channels")
    omega = omega_of(float(g["lwl"]))
    p = "xyz".index(pd)
    Te, kappa = _grids(g, omega)
    ne_src = OC.array_source(g["ne"], pd)
    src = OC.channel_source(ne_src, pd, omega, inv_brems=True, B_on=True, B=g["B"], Te=Te, Z=g["Z"])
    kappa_s = engine.kappa_grid(g["ne"], np.maximum(1.0, 0.5), 3.0, omega)
    src_s = OC.channel_source(ne_src, pd, omega, inv_brems=True, Te=0.5, Z=3.0)
    n = g["ne"].shape[p]
    for k0, k1 in ((0, 7), (5, 13), (n - 9, n)):
        idx = [slice(None)] * 3
        idx[p] = slice(k0, k1)
        idx = tuple(idx)
        sl = src(k0, k1)
        assert np.array_equal(sl.kappa, kappa[idx]) and np.array_equal(sl.ne, g["ne"][idx])
        assert np.array_equal(sl.ne_faraday, g["ne"][idx]) and np.array_equal(sl.B, g["B"][idx])
        sl = src_s(k0, k1)
        assert np.array_equal(sl.kappa, kappa_s[idx]) and sl.B is None and sl.ne_faraday is None
    assert (Te < 1.0).any() and not np.array_equal(kappa, engine.kappa_grid(g["ne"], Te, g["Z"], omega))
    bad = OC.channel_source(ne_src, pd, omega, B_on=True, B=lambda k0, k1: np.zeros((2, 2, 2, 3)))
    with pytest.raises(ValueError, match="B slab has shape"):
        bad(0, 4)
    bad = OC.channel_source(ne_src, pd, omega, inv_brems=True, Te=lambda k0, k1: np.ones((2, 2, 2)), Z=1.0)
    with pytest.raises(ValueError, match="Te slab has shape"):
        bad(0, 4)


def test_propagate_window_channels_validation():
    """sp_propagate_window_channels: every invalid argument is SP_EINVAL with a message, before any CUDA call."""
    from synthpy_b200 import _lib as L, engine
    lib = L.lib
    buf = (C.c_double * 4096)()
    u32 = (C.c_uint32 * 4)()
    fake = C.cast(buf, C.c_void_p)

    def call(P, state=fake, ctl=fake, flags=u32, steps=u32, lo=0.0, hi=1.0, g_lo=-1.0, field=fake, ws=fake, n_ch=0):
        return lib.sp_propagate_window_channels(field, C.byref(P), ws, state, 1, None, 0, ctl,
                                                C.cast(flags, C.c_void_p) if flags is not None else None,
                                                C.cast(steps, C.c_void_p) if steps is not None else None, lo, hi, g_lo, 1.0,
                                                None, None, None, n_ch, None, None)

    def P(method="rk45", atten=True, faraday=True, **kw):
        return engine.make_params(method, extent=1e-2, omega=1e15, h=0.5, atten=atten, faraday=faraday, **kw)
    cases = [(P("rk4"), {}), (P("tsit5"), {}), (P("rk45_joint"), {}), (P("rk45_bundle"), {}), (P(atten=False, faraday=False), {}),
             (P(fp32=True), {}), (P(faraday=False, fp32=True), {}), (P(), dict(lo=1.0, hi=0.0)), (P(), dict(lo=float("nan"))),
             (P(), dict(g_lo=2.0)), (P(), dict(state=None)), (P(), dict(ctl=None)), (P(), dict(flags=None)),
             (P(), dict(steps=None)), (P(), dict(field=None)), (P(), dict(ws=None)), (P(), dict(n_ch=5)),
             (engine.make_params("rk45", extent=1e-2, omega=1e15, faraday=True, probing_direction="z"), {})]
    for params, kw in cases:
        rc = call(params, **kw)
        assert rc == -1, (params.method, params.flags, kw)                     # SP_EINVAL
        assert lib.sp_last_error().decode()
    params = P()
    params.probing_axis = 3
    assert call(params) == -1


def test_solve_out_of_core_channel_refusals():
    """Every refusal of a solve with channels is a ValueError raised before anything touches the GPU."""
    from synthpy_b200 import out_of_core as OC
    s0 = np.zeros((9, 1))
    B, T = np.zeros((8, 8, 8, 3)), np.ones((8, 8, 8))
    kw = dict(slab_planes=8)
    cases = [(dict(B_on=True), "needs B"), (dict(inv_brems=True), "needs Te and Z"), (dict(inv_brems=True, Te=T), "needs Te and Z"),
             (dict(inv_brems=True, Z=T), "needs Te and Z"), (dict(B_on=True, B=B, method="tsit5"), "tsit5"),
             (dict(inv_brems=True, Te=T, Z=1.0, method="rk45", precision="fp32"), "float64 only"),
             (dict(B_on=True, B=np.zeros((8, 8, 7, 3))), "B has shape"), (dict(B_on=True, B=np.zeros((8, 8, 8))), "B has shape"),
             (dict(inv_brems=True, Te=np.ones((8, 8, 9)), Z=1.0), "Te has shape"),
             (dict(inv_brems=True, Te=1.0, Z=np.ones((7, 8, 8))), "Z has shape")]
    for extra, msg in cases:
        with pytest.raises(ValueError, match=msg):
            OC.solve_out_of_core(s0, None, 1.0, 8, 1.0, **kw, **extra)
