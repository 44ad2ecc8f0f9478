"""Out-of-core RK45 / Tsit5 with stage parking on the GPU (sp_propagate_window_staged) against the in-core solves, bit for
bit, with the in-core evaluation count."""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

C_LIGHT = 299792458.0
CHANNELS = {"B": dict(B_on=True), "brems": dict(inv_brems=True), "both": dict(B_on=True, inv_brems=True)}


def _check(ex, ex2, rf, rf2, Jf, Jf2, planes):
    assert np.array_equal(rf2, rf, equal_nan=True)
    assert np.array_equal(Jf2, Jf, equal_nan=True)
    assert np.array_equal(ex2["sf"], ex["sf"], equal_nan=True) and np.array_equal(ex2["steps"], ex["steps"])
    for k in ("ray_steps", "ray_steps_acc", "rays_capped", "rhs_evals"):
        assert ex2["stats"][k] == ex["stats"][k], k                   # rhs_evals too: every evaluation runs once
    assert max(e["planes"][1] - e["planes"][0] + 1 for e in ex2["slabs"]) <= planes
    assert sum(e["evals"] for e in ex2["slabs"]) == ex["stats"]["rhs_evals"]


@pytest.mark.parametrize("method,kw", [("rk45", {}), ("tsit5", dict(rtol=1e-7, atol=1e-9)), ("tsit5", dict(rtol=1.0, atol=1e-5))])
def test_staged_out_of_core_equals_in_core(golden, tmp_path, method, kw):
    """solve_out_of_core(park='stage') against propagator.solve: exit rays, Jones vectors, states, attempts per ray and the
    stats, rhs_evals equal; slabs of 8 planes that never grow; from an array, a memmap and with prefetch; along x; float32
    and a small max_steps; a NaN ray."""
    from synthpy_b200 import domain as Dm, legacy, out_of_core as OC, propagator as P
    g = golden("g3_turb")
    lwl, ext, ne = float(g["lwl"]), float(g["extent"]), g["ne"]
    lengths, dims = (10e-3, 10e-3, 20e-3), (32, 32, 32)
    np.random.seed(8)
    s0 = legacy.init_beam(3000, 3e-3, 2e-3, ext, "circular", "z")
    s0[0, 5] = np.nan
    dom = Dm.ScalarDomain(lengths, dims, phaseshift=True)
    dom.external_ne(ne)
    mm = np.memmap(str(tmp_path / "ne.raw"), dtype=np.float64, mode="w+", shape=ne.shape)
    mm[:] = ne
    mm.flush()
    mm = np.memmap(str(tmp_path / "ne.raw"), dtype=np.float64, mode="r", shape=ne.shape)
    oc = dict(slab_planes=8, lwl=lwl, method=method, park="stage", return_E=True, phaseshift=True, return_state=True)
    for extra in ({}, dict(max_steps=20), dict(precision="fp32")):
        rf, Jf, _, ex = P.solve(s0, dom, ext, return_E=True, lwl=lwl, method=method, return_state=True, **kw, **extra)
        runs = [dict(src=OC.array_source(ne)), dict(src=OC.array_source(mm)), dict(src=OC.array_source(mm), prefetch=True)]
        for r in runs if not extra else runs[:1]:
            src = r.pop("src")
            rf2, Jf2, _, ex2 = OC.solve_out_of_core(s0, src, lengths, dims, ext, **oc, **kw, **extra, **r)
            _check(ex, ex2, rf, rf2, Jf, Jf2, 8)
            if not extra:
                assert len(ex2["slabs"]) >= 3 and sum(e["parked_mid"] for e in ex2["slabs"]) > 0
    domx = Dm.ScalarDomain(lengths, dims, probing_direction="x", phaseshift=True)
    domx.external_ne(ne)
    np.random.seed(9)
    sx = legacy.init_beam(1000, 3e-3, 1e-3, 5e-3, "circular", "x")
    rf, Jf, _, ex = P.solve(sx, domx, 5e-3, return_E=True, lwl=lwl, method=method, return_state=True, **kw)
    rf2, Jf2, _, ex2 = OC.solve_out_of_core(sx, OC.array_source(ne, "x"), lengths, dims, 5e-3, probing_direction="x", **oc, **kw)
    _check(ex, ex2, rf, rf2, Jf, Jf2, 8)


@pytest.mark.parametrize("method,kw", [("rk45", {}), ("tsit5", dict(rtol=1e-7, atol=1e-9))])
@pytest.mark.parametrize("phase", ["off", "f64"])
def test_staged_phase_variants_equal_in_core(golden, method, kw, phase):
    """The staged kernels without the phase lane and with the float64 aux grid (phase_f64) equal in core bit for bit, in
    float64 and float32: nvcc contracts each instantiation on its own, so each is held against in core on the device."""
    from synthpy_b200 import domain as Dm, legacy, out_of_core as OC, propagator as P
    g = golden("g3_turb")
    lwl, ext, ne = float(g["lwl"]), float(g["extent"]), g["ne"]
    lengths, dims = (10e-3, 10e-3, 20e-3), (32, 32, 32)
    np.random.seed(8)
    s0 = legacy.init_beam(3000, 3e-3, 2e-3, ext, "circular", "z")
    ph = dict(phaseshift=phase == "f64", phase_f64=phase == "f64")
    dom = Dm.ScalarDomain(lengths, dims, phaseshift=ph["phaseshift"])
    dom.external_ne(ne)
    for precision in ("fp64", "fp32"):
        if precision == "fp32" and phase == "f64":
            continue                                  # the float64 aux grid is a float64 option
        rf, Jf, _, ex = P.solve(s0, dom, ext, return_E=True, lwl=lwl, method=method, return_state=True, precision=precision,
                                phase_f64=ph["phase_f64"], **kw)
        rf2, Jf2, _, ex2 = OC.solve_out_of_core(s0, OC.array_source(ne), lengths, dims, ext, slab_planes=8, lwl=lwl, method=method,
                                                park="stage", return_E=True, return_state=True, precision=precision, **ph, **kw)
        _check(ex, ex2, rf, rf2, Jf, Jf2, 8)
        if ph["phaseshift"]:
            assert np.nanmax(np.abs(ex["sf"][7])) > 1.0


@pytest.mark.parametrize("chan", ["B", "brems", "both"])
def test_staged_channels_equal_in_core(golden, chan):
    """RK45 with each channel combination (Te clamped) out of core with stage parking equals the in-core solve: all nine rows,
    exit rays, Jones vectors, attempts and rhs_evals; along z and x."""
    from synthpy_b200 import domain as Dm, legacy, out_of_core as OC, propagator as P
    g = golden("g6_channels")
    lengths = [float(g[k][-1] - g[k][0]) for k in "xyz"]
    dims = list(g["ne"].shape)
    Te = g["Te"].copy()
    Te.reshape(-1)[::17] = 0.25
    lwl, ext = float(g["lwl"]), float(g["extent"])
    ch = CHANNELS[chan]
    for pd in ("z", "x"):
        if pd == "z":
            s0 = np.array(g["s0"])
        else:
            np.random.seed(4)
            s0 = legacy.init_beam(96, 3e-3, 2e-3, float(g["x"][-1]), "circular", "x")
        s0[6] = np.linspace(0.5, 1.5, s0.shape[1])
        s0[8] = np.linspace(-0.1, 0.1, s0.shape[1])
        s0[0, 3] = np.nan
        depth = ext if pd == "z" else float(g["x"][-1])
        dom = Dm.ScalarDomain(lengths, dims, phaseshift=True, probing_direction=pd, **ch)
        dom.external_ne(g["ne"])
        dom.external_B(g["B"])
        dom.external_Te(Te)
        dom.external_Z(g["Z"])
        rf, Jf, _, ex = P.solve(s0, dom, depth, return_E=True, lwl=lwl, method="rk45", return_state=True)
        rf2, Jf2, _, ex2 = OC.solve_out_of_core(s0, OC.array_source(g["ne"], pd), lengths, dims, depth, probing_direction=pd,
                                                slab_planes=8, lwl=lwl, method="rk45", park="stage", return_E=True,
                                                phaseshift=True, return_state=True, B=g["B"], Te=Te, Z=g["Z"], **ch)
        _check(ex, ex2, rf, rf2, Jf, Jf2, 8)


def test_staged_fused_images(golden):
    """Fused histogram and Stokes images of a staged out-of-core solve equal solve_and_image's."""
    from synthpy_b200 import diagnostics as D, domain as Dm, legacy, out_of_core as OC, propagator as P
    g = golden("g6_channels")
    lengths = [float(g[k][-1] - g[k][0]) for k in "xyz"]
    dims = list(g["ne"].shape)
    lwl, ext = float(g["lwl"]), float(g["extent"])
    dom = Dm.ScalarDomain(lengths, dims, phaseshift=True, B_on=True)
    dom.external_ne(g["ne"])
    dom.external_B(g["B"])
    np.random.seed(8)
    s0 = legacy.init_beam(20000, 3e-3, 2e-3, ext, "circular", "z")
    for stokes, kw in ((False, {}), (True, dict(B_on=True, B=g["B"]))):
        a, b = (D.spec("shadow_two", bin_scale=16, stokes=stokes) for _ in range(2))
        if stokes:
            P.solve_and_image(dom, s0, ext, [a], lwl=lwl, method="rk45")
        else:
            d0 = Dm.ScalarDomain(lengths, dims, phaseshift=True)
            d0.external_ne(g["ne"])
            P.solve_and_image(d0, s0, ext, [a], lwl=lwl, method="rk45")
        OC.solve_out_of_core(s0, OC.array_source(g["ne"]), lengths, dims, ext, slab_planes=8, lwl=lwl, phaseshift=True,
                             method="rk45", park="stage", diagnostics=[b], **kw)
        if stokes:
            assert torch.equal(a.image.planes, b.image.planes)
        else:
            ra, rb = a.image.result(), b.image.result()
            assert torch.equal(ra, rb) and float(ra.sum()) > 100


def test_staged_turbulent_source():
    """128^3 turbulent_ne_slabs, RK45 in 32-plane slabs: attempt parking without growth raises, stage parking finishes and
    equals the in-core trace of source(0, n)."""
    from synthpy_b200 import domain as Dm, field_generator as FG, legacy, out_of_core as OC, propagator as P
    n, lwl, ext = 128, 1064e-9, 10e-3
    lengths = (10e-3, 10e-3, 10e-3)
    src = FG.turbulent_ne_slabs(n // 2, seed=6, block_planes=16)
    dom = Dm.ScalarDomain(lengths, n, phaseshift=True)
    dom.external_ne(src(0, n))
    np.random.seed(10)
    s0 = legacy.init_beam(4000, 4e-3, 1e-3, ext, "circular", "z")
    rf, Jf, _, ex = P.solve(s0, dom, ext, lwl=lwl, method="rk45", return_E=True, return_state=True)
    with pytest.raises(ValueError, match="increase slab_planes"):
        OC.solve_out_of_core(s0, src, lengths, (n, n, n), ext, slab_planes=32, max_slab_planes=32, lwl=lwl, method="rk45",
                             phaseshift=True)
    rf2, Jf2, _, ex2 = OC.solve_out_of_core(s0, src, lengths, (n, n, n), ext, slab_planes=32, lwl=lwl, method="rk45",
                                            park="stage", return_E=True, phaseshift=True, return_state=True)
    _check(ex, ex2, rf, rf2, Jf, Jf2, 32)


def test_staged_peak_memory():
    """256^3 with all channels, RK45 in 32-plane slabs with stage parking: the out-of-core peak (torch allocations plus the
    largest slab field) is below half the in-core peak (torch allocations plus the field with its channel grids)."""
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
    rf, _, _, ex = P.solve(s0, dom, ext, lwl=lwl, method="rk45", return_state=True)
    in_core = torch.cuda.max_memory_allocated() - base + dom.device_field(lwl).nbytes
    del dom
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    rf2, _, _, ex2 = OC.solve_out_of_core(s0, OC.array_source(ne), lengths, n, ext, slab_planes=32, lwl=lwl, phaseshift=True,
                                          method="rk45", park="stage", return_state=True, B_on=True, inv_brems=True, B=B,
                                          Te=Te, Z=Z)
    out_core = torch.cuda.max_memory_allocated() - base + max(e["field_bytes"] for e in ex2["slabs"])
    assert np.array_equal(rf2, rf, equal_nan=True) and ex2["stats"]["rhs_evals"] == ex["stats"]["rhs_evals"]
    assert max(e["planes"][1] - e["planes"][0] + 1 for e in ex2["slabs"]) <= 32
    assert out_core < 0.5 * in_core, (out_core, in_core)


def test_propagate_window_staged_estate(golden):
    """sp_propagate_window_staged on a real field without the channel grids: SP_ESTATE, for each flag."""
    from synthpy_b200 import _lib as L, engine
    g = golden("g6_channels")
    lwl = float(g["lwl"])
    f = engine.DeviceField.from_ne(g["ne"], g["x"], g["y"], g["z"], engine.omega_of(lwl), phase=True)
    s = torch.zeros((9, 4), dtype=torch.float64, device="cuda")
    rec = engine.controller_record(4)
    for flags in (dict(atten=True), dict(faraday=True), dict(atten=True, faraday=True)):
        P = engine.make_params("rk45", extent=1e-2, omega=engine.omega_of(lwl), phase=True, verdet=1.0, **flags)
        st = engine.stage_store(4, P)
        assert tuple(st.shape) == (54, 4)
        rc = L.lib.sp_propagate_window_staged(f._h, C.byref(P), engine.workspace(), C.c_void_p(s.data_ptr()), 4, None, 0,
                                              C.c_void_p(rec["ctl"].data_ptr()), C.c_void_p(rec["flags"].data_ptr()),
                                              C.c_void_p(rec["steps"].data_ptr()), C.c_void_p(st.data_ptr()), -np.inf, np.inf,
                                              -1.0, 1.0, None, None, None, 0, None,
                                              C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == -4, flags                                                     # SP_ESTATE
        assert "sp_field_attach_channels" in L.lib.sp_last_error().decode()
