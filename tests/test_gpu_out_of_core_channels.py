"""Out-of-core tracing with the attenuation and Faraday channels on the GPU against the in-core solves, bit for bit:
RK4 (sp_propagate's RK4X kernel per slab) and per-ray RK45 (sp_propagate_window_channels)."""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

C_LIGHT = 299792458.0
CHANNELS = {"B": dict(B_on=True), "brems": dict(inv_brems=True), "both": dict(B_on=True, inv_brems=True)}


def _g6(golden):
    g = golden("g6_channels")
    lengths = [float(g[k][-1] - g[k][0]) for k in "xyz"]
    Te = g["Te"].copy()
    Te.reshape(-1)[::17] = 0.25                      # below Te_min: the clamp acts
    return g, lengths, list(g["ne"].shape), Te


def _domain(g, lengths, dims, Te, pd="z", **ch):
    from synthpy_b200 import domain as Dm
    dom = Dm.ScalarDomain(lengths, dims, phaseshift=True, probing_direction=pd, **ch)
    dom.external_ne(g["ne"])
    dom.external_B(g["B"])
    dom.external_Te(Te)
    dom.external_Z(g["Z"])
    return dom


def _rays(g, pd):
    from synthpy_b200 import legacy
    if pd == "z":
        s0 = np.array(g["s0"])
    else:
        np.random.seed(4)
        s0 = legacy.init_beam(96, 3e-3, 2e-3, float(g["x"][-1]), "circular", "x")
    s0[6] = np.linspace(0.5, 1.5, s0.shape[1])
    s0[8] = np.linspace(-0.1, 0.1, s0.shape[1])
    s0[0, 3] = np.nan
    return s0


def _check(ex, ex2, rf, rf2, Jf, Jf2, adaptive):
    assert np.array_equal(rf2, rf, equal_nan=True)
    assert np.array_equal(Jf2, Jf, equal_nan=True)
    assert np.array_equal(ex2["sf"], ex["sf"], equal_nan=True) and np.array_equal(ex2["steps"], ex["steps"])
    for k in ("ray_steps", "ray_steps_acc", "rays_capped"):
        assert ex2["stats"][k] == ex["stats"][k], k
    if adaptive:
        assert ex2["stats"]["rhs_evals"] >= ex["stats"]["rhs_evals"]


@pytest.mark.parametrize("method", ["rk4", "rk45"])
@pytest.mark.parametrize("chan", ["B", "brems", "both"])
def test_channels_out_of_core_equals_in_core(golden, tmp_path, method, chan):
    """solve_out_of_core with the channels equals propagator.solve on ScalarDomain(inv_brems, B_on): exit rays, Jones
    vectors, all nine state rows, steps per ray and the committed-work stats, with a NaN ray; along z and x; the channel
    inputs from arrays, from memory-mapped files and with prefetch=True; RK45 also with a small max_steps."""
    from synthpy_b200 import out_of_core as OC, propagator as P
    g, lengths, dims, Te = _g6(golden)
    lwl, ext = float(g["lwl"]), float(g["extent"])
    ch = CHANNELS[chan]
    mm = {}
    for k, a in (("ne", g["ne"]), ("B", g["B"]), ("Te", Te), ("Z", g["Z"])):
        m = np.memmap(str(tmp_path / f"{k}.raw"), dtype=np.float64, mode="w+", shape=a.shape)
        m[:] = a
        m.flush()
        mm[k] = np.memmap(str(tmp_path / f"{k}.raw"), dtype=np.float64, mode="r", shape=a.shape)
    adaptive = method == "rk45"
    oc = dict(slab_planes=10, max_slab_planes=dims[2], lwl=lwl, method=method, return_E=True, phaseshift=True,
              return_state=True, **ch)
    for pd in ("z", "x"):
        s0 = _rays(g, pd)
        depth = ext if pd == "z" else float(g["x"][-1])
        dom = _domain(g, lengths, dims, Te, pd, **ch)
        for extra in ({}, dict(max_steps=15)) if adaptive else ({},):
            rf, Jf, _, ex = P.solve(s0, dom, depth, return_E=True, lwl=lwl, method=method, return_state=True, **extra)
            if chan != "brems":
                assert np.abs(ex["sf"][8] - s0[8])[np.isfinite(ex["sf"][8])].max() > 1e-7
            if chan != "B":
                assert np.nanmax(np.abs(ex["sf"][6] - s0[6])) > 1e-4
            runs = [dict(src=OC.array_source(g["ne"], pd), B=g["B"], Te=Te, Z=g["Z"]),
                    dict(src=OC.array_source(mm["ne"], pd), B=mm["B"], Te=mm["Te"], Z=mm["Z"]),
                    dict(src=OC.array_source(mm["ne"], pd), B=mm["B"], Te=mm["Te"], Z=mm["Z"], prefetch=True)]
            for r in runs if not extra else runs[:1]:
                src = r.pop("src")
                rf2, Jf2, _, ex2 = OC.solve_out_of_core(s0, src, lengths, dims, depth, probing_direction=pd, **oc, **extra, **r)
                _check(ex, ex2, rf, rf2, Jf, Jf2, adaptive)
                assert len(ex2["slabs"]) >= 2
            if extra:
                assert ex["stats"]["rays_capped"] > 0


@pytest.mark.parametrize("method", ["rk4", "rk45"])
def test_channels_out_of_core_fused_stokes(golden, method):
    """A fused Stokes image (diagnostics=[spec(..., stokes=True)]) out of core equals solve_and_image's planes."""
    from synthpy_b200 import diagnostics as D, legacy, out_of_core as OC, propagator as P
    g, lengths, dims, Te = _g6(golden)
    lwl, ext = float(g["lwl"]), float(g["extent"])
    dom = _domain(g, lengths, dims, Te, B_on=True, inv_brems=True)
    np.random.seed(8)
    s0 = legacy.init_beam(20000, 3e-3, 2e-3, ext, "circular", "z")
    a, b = D.spec("shadow_two", bin_scale=16, stokes=True), D.spec("shadow_two", bin_scale=16, stokes=True)
    st, _ = P.solve_and_image(dom, s0, ext, [a], lwl=lwl, method=method)
    _, _, _, ex = OC.solve_out_of_core(s0, OC.array_source(g["ne"]), lengths, dims, ext, slab_planes=10, max_slab_planes=dims[2],
                                       lwl=lwl, phaseshift=True, method=method, diagnostics=[b], return_state=True,
                                       B_on=True, inv_brems=True, B=g["B"], Te=Te, Z=g["Z"])
    assert torch.equal(a.image.planes, b.image.planes)                             # count, I, Q, U: integer planes
    sa = a.image.stokes()
    assert sa["N"].sum() > 200 and float(sa["U"].abs().max()) > 0                   # a non-trivial image
    assert ex["stats"]["rays_binned"] == st["rays_binned"]


def _slab_B(n, lengths, axis=2):
    """A z-invariant B on the device (the field of examples/polarimetry_bench.analytic_B), as a slab source."""
    x, y = [torch.linspace(-L / 2, L / 2, n, dtype=torch.float64, device="cuda") for L in lengths[:2]]
    XX, YY = torch.meshgrid(x, y, indexing="ij")
    plane = torch.stack([5.0 * YY / 5e-3, -5.0 * XX / 5e-3, 10.0 * torch.exp(-(XX ** 2 + YY ** 2) / (3e-3) ** 2)], -1)
    return lambda k0, k1: plane[:, :, None, :].expand(n, n, k1 - k0, 3).contiguous()


@pytest.mark.parametrize("method", ["rk4", "rk45"])
def test_channels_out_of_core_turbulent_source(method):
    """128^3 turbulent_ne_slabs with a device B slab source, traced out of core: equals the in-core trace of source(0, n)
    with the whole B."""
    from synthpy_b200 import domain as Dm, field_generator as FG, legacy, out_of_core as OC, propagator as P
    n, lwl, ext = 128, 1064e-9, 10e-3
    lengths = (10e-3, 10e-3, 10e-3)
    src = FG.turbulent_ne_slabs(n // 2, seed=6, block_planes=16)
    bsrc = _slab_B(n, lengths)
    dom = Dm.ScalarDomain(lengths, n, B_on=True, phaseshift=True)
    dom.external_ne(src(0, n))
    dom.external_B(bsrc(0, n))
    np.random.seed(10)
    s0 = legacy.init_beam(4000, 4e-3, 1e-3, ext, "circular", "z")
    rf, Jf, _, ex = P.solve(s0, dom, ext, lwl=lwl, method=method, return_E=True, return_state=True)
    rf2, Jf2, _, ex2 = OC.solve_out_of_core(s0, src, lengths, (n, n, n), ext, slab_planes=40, max_slab_planes=n, lwl=lwl,
                                            method=method, return_E=True, phaseshift=True, return_state=True, B_on=True, B=bsrc)
    _check(ex, ex2, rf, rf2, Jf, Jf2, method == "rk45")
    assert len(ex2["slabs"]) >= 2 and np.abs(ex["sf"][8]).max() > 1e-6


def test_channels_out_of_core_peak_memory():
    """256^3 with all channels in 32-plane slabs: the out-of-core peak (torch allocations plus the largest slab field) is
    below the in-core peak (torch allocations plus the field with its five float64 grids) by at least half."""
    from synthpy_b200 import domain as Dm, legacy, out_of_core as OC, propagator as P
    n, lwl, ext = 256, 1064e-9, 5e-3
    lengths = (10e-3, 10e-3, 10e-3)
    rng = np.random.default_rng(3)
    ne = 1e24 * (1.0 + 0.1 * rng.random((n, n, n)))
    B = np.zeros((n, n, n, 3))
    B[..., 2] = 5.0
    Te, Z = 100.0, 3.0
    np.random.seed(11)
    s0 = legacy.init_beam(20000, 3e-3, 1e-3, ext, "circular", "z")
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    dom = Dm.ScalarDomain(lengths, n, B_on=True, inv_brems=True, phaseshift=True)
    dom.external_ne(ne)
    dom.external_B(B)
    dom.external_Te(Te)
    dom.external_Z(Z)
    rf, _, _ = P.solve(s0, dom, ext, lwl=lwl)
    in_core = torch.cuda.max_memory_allocated() - base + dom.device_field(lwl).nbytes
    del dom
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    rf2, _, _, ex2 = OC.solve_out_of_core(s0, OC.array_source(ne), lengths, n, ext, slab_planes=32, lwl=lwl, phaseshift=True,
                                          return_state=True, B_on=True, inv_brems=True, B=B, Te=Te, Z=Z)
    out_core = torch.cuda.max_memory_allocated() - base + max(e["field_bytes"] for e in ex2["slabs"])
    assert np.array_equal(rf2, rf, equal_nan=True)
    assert out_core < 0.5 * in_core, (out_core, in_core)


def test_propagate_window_channels_estate(golden):
    """sp_propagate_window_channels on a real field without the grids: SP_ESTATE, for each flag."""
    from synthpy_b200 import _lib as L, engine
    g = golden("g6_channels")
    lwl = float(g["lwl"])
    f = engine.DeviceField.from_ne(g["ne"], g["x"], g["y"], g["z"], engine.omega_of(lwl), phase=True)
    s = torch.zeros((9, 4), dtype=torch.float64, device="cuda")
    rec = engine.controller_record(4)
    for flags in (dict(atten=True), dict(faraday=True), dict(atten=True, faraday=True)):
        P = engine.make_params("rk45", extent=1e-2, omega=engine.omega_of(lwl), phase=True, verdet=1.0, **flags)
        rc = L.lib.sp_propagate_window_channels(f._h, C.byref(P), engine.workspace(), C.c_void_p(s.data_ptr()), 4, None, 0,
                                                C.c_void_p(rec["ctl"].data_ptr()), C.c_void_p(rec["flags"].data_ptr()),
                                                C.c_void_p(rec["steps"].data_ptr()), -np.inf, np.inf, -1.0, 1.0, None, None,
                                                None, 0, None, C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == -4, flags                                                     # SP_ESTATE
        assert "sp_field_attach_channels" in L.lib.sp_last_error().decode()
    f.attach_channels(kappa=np.ones(g["ne"].shape))
    P = engine.make_params("rk45", extent=1e-2, omega=engine.omega_of(lwl), phase=True, faraday=True, verdet=1.0)
    with pytest.raises(Exception):
        engine.propagate_window(f, P, s, rec, -np.inf, np.inf, (-1.0, 1.0))
