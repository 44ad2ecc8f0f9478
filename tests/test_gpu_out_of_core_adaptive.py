"""Out-of-core RK45 / Tsit5 on the GPU (sp_propagate_window) against the in-core solves, bit for bit."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

C_LIGHT = 299792458.0


@pytest.fixture(scope="module")
def beam():
    from synthpy_b200 import legacy
    return legacy


def _check(ex, ex2, rf, rf2, Jf=None, Jf2=None):
    assert np.array_equal(rf2, rf, equal_nan=True)
    if Jf is not None:
        assert np.array_equal(Jf2, Jf, equal_nan=True)
    assert np.array_equal(ex2["sf"], ex["sf"], equal_nan=True) and np.array_equal(ex2["steps"], ex["steps"])
    for k in ("ray_steps", "ray_steps_acc", "rays_capped"):
        assert ex2["stats"][k] == ex["stats"][k], k
    assert ex2["stats"]["rhs_evals"] >= ex["stats"]["rhs_evals"]


@pytest.mark.parametrize("method,kw", [("rk45", {}), ("tsit5", dict(rtol=1e-7, atol=1e-9))])
def test_adaptive_out_of_core_equals_in_core(beam, golden, tmp_path, method, kw):
    """solve_out_of_core(method=...) against propagator.solve: exit rays, Jones vectors, full states, attempts per ray and
    the committed-work stats, with a NaN ray and a sideways ray; from an array and a memory-mapped file, along x,
    early_exit=False, a small max_steps (capped rays) and float32."""
    from synthpy_b200 import domain as Dm, out_of_core as OC, propagator as P
    g = golden("g3_turb")
    lwl, ext, ne = float(g["lwl"]), float(g["extent"]), g["ne"]
    lengths, dims = (10e-3, 10e-3, 20e-3), (32, 32, 32)
    np.random.seed(8)
    s0 = beam.init_beam(3000, 3e-3, 2e-3, ext, "circular", "z")
    s0[0, 5] = np.nan
    s0[3, 6] = 0.5 * C_LIGHT
    dom = Dm.ScalarDomain(lengths, dims, phaseshift=True)
    dom.external_ne(ne)
    mm = np.memmap(str(tmp_path / "ne.raw"), dtype=np.float64, mode="w+", shape=ne.shape)
    mm[:] = ne
    mm.flush()
    oc = dict(slab_planes=10, max_slab_planes=32, lwl=lwl, method=method)
    for extra in ({}, dict(early_exit=False), dict(max_steps=20), dict(precision="fp32")):
        rf, Jf, _, ex = P.solve(s0, dom, ext, return_E=True, lwl=lwl, method=method, return_state=True, **kw, **extra)
        srcs = (OC.array_source(ne), OC.array_source(np.memmap(str(tmp_path / "ne.raw"), dtype=np.float64, mode="r", shape=ne.shape)))
        for src in srcs[:2 if not extra else 1]:
            rf2, Jf2, _, ex2 = OC.solve_out_of_core(s0, src, lengths, dims, ext, return_E=True, phaseshift=True, return_state=True,
                                                    **oc, **kw, **extra)
            _check(ex, ex2, rf, rf2, Jf, Jf2)
            if "max_steps" not in extra:                  # with a small cap every ray may finish (capped) in the first slab
                assert len(ex2["slabs"]) >= 2 and sum(e["parked"] for e in ex2["slabs"]) > 0
        if "max_steps" in extra:
            assert ex["stats"]["rays_capped"] > 0
    domx = Dm.ScalarDomain(lengths, dims, probing_direction="x")
    domx.external_ne(ne)
    np.random.seed(9)
    sx = beam.init_beam(1000, 3e-3, 1e-3, 5e-3, "circular", "x")
    rfx, _, _, exx = P.solve(sx, domx, 5e-3, lwl=lwl, method=method, return_state=True, **kw)
    rfx2, _, _, exx2 = OC.solve_out_of_core(sx, OC.array_source(ne, "x"), lengths, dims, 5e-3, probing_direction="x",
                                            return_state=True, slab_planes=11, max_slab_planes=32, lwl=lwl, method=method, **kw)
    _check(exx, exx2, rfx, rfx2)


def test_adaptive_out_of_core_fused_image(beam, golden):
    """A fused detector image (diagnostics=[spec]) equals solve_and_image's: each ray binned by the launch it finishes in."""
    from synthpy_b200 import diagnostics as D, domain as Dm, out_of_core as OC, propagator as P
    g = golden("g3_turb")
    lwl, ext, ne = float(g["lwl"]), float(g["extent"]), g["ne"]
    lengths, dims = (10e-3, 10e-3, 20e-3), (32, 32, 32)
    np.random.seed(8)
    s0 = beam.init_beam(6000, 3e-3, 2e-3, ext, "circular", "z")
    dom = Dm.ScalarDomain(lengths, dims, phaseshift=True)
    dom.external_ne(ne)
    for method in ("rk45", "tsit5"):
        a, b = D.spec("shadow_two", bin_scale=16), D.spec("shadow_two", bin_scale=16)
        st, _ = P.solve_and_image(dom, s0, ext, [a], lwl=lwl, method=method)
        _, _, _, ex = OC.solve_out_of_core(s0, OC.array_source(ne), lengths, dims, ext, slab_planes=10, max_slab_planes=32,
                                           lwl=lwl, phaseshift=True, method=method, diagnostics=[b], return_state=True)
        assert a.image.result().sum() > 1000 and torch.equal(a.image.result(), b.image.result())
        assert ex["stats"]["rays_binned"] == st["rays_binned"]


def test_adaptive_out_of_core_turbulent_slabs():
    """128^3 turbulent_ne_slabs source traced with RK45: equals the in-core RK45 trace of the same planes held whole."""
    from synthpy_b200 import domain as Dm, field_generator as FG, legacy, out_of_core as OC, propagator as P
    n, lwl, ext = 128, 1064e-9, 10e-3
    lengths = (10e-3, 10e-3, 10e-3)
    src = FG.turbulent_ne_slabs(n // 2, seed=6, block_planes=16)
    dom = Dm.ScalarDomain(lengths, n)
    dom.external_ne(src(0, n))
    np.random.seed(10)
    s0 = legacy.init_beam(4000, 4e-3, 1e-3, ext, "circular", "z")
    rf, _, _, ex = P.solve(s0, dom, ext, lwl=lwl, method="rk45", return_state=True)
    rf2, _, _, ex2 = OC.solve_out_of_core(s0, src, lengths, (n, n, n), ext, slab_planes=40, max_slab_planes=n, lwl=lwl,
                                          method="rk45", return_state=True)
    _check(ex, ex2, rf, rf2)
    assert len(ex2["slabs"]) >= 2
