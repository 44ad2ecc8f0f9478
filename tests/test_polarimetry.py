"""Faraday-rotation polarimetry: Stokes-parameter detector images (SP_IMG_STOKES) on the fused and stand-alone paths.

Parity rests on the reference's own exit rays and Jones vectors (golden g6: attenuation + Faraday channels), carried
through the oracle's optical train and binned by ``np.histogram2d(..., weights=)`` on the histogram's edges."""
import ctypes as C
import os
import re
import socket
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")
HEADER = os.path.join(ROOT, "include", "synthpy_b200.h")
C_LIGHT = 299792458.0
Q32 = 2.0 ** -32
BS = 100                                   # bin scale of the g6 comparisons: 34 x 25 pixels for 128 rays
R = 100                                    # aperture radius, mm: g6's column deflects rays by up to 6.4 degrees, and the
                                           # default 25 mm apertures would let 3 of its 128 rays reach the detector


@pytest.fixture(scope="module")
def g6():
    return dict(np.load(os.path.join(GOLDEN, "g6_channels.npz")))


# ---- NumPy restatement -------------------------------------------------------------------------------------------
def stokes_of(J):
    """Per-ray Stokes I, Q, U of (2, N) Jones vectors."""
    xx, yy = np.abs(J[0]) ** 2, np.abs(J[1]) ** 2
    return xx + yy, xx - yy, 2.0 * np.real(J[0] * np.conj(J[1]))


def stokes_images(r_det, J, bin_scale=BS, pix_x=3448, pix_y=2574, Lx=18, Ly=13.5):
    """N, I, Q, U (ny, nx): np.histogram2d of the detector rays (mm, NaN = rejected) with weights I, Q, U."""
    ok = ~np.isnan(r_det[0]) & ~np.isnan(r_det[2])
    kw = dict(bins=[pix_x // bin_scale, pix_y // bin_scale], range=[[-Lx / 2, Lx / 2], [-Ly / 2, Ly / 2]])
    out = [np.histogram2d(r_det[0][ok], r_det[2][ok], **kw)[0].T]
    for w in stokes_of(J):
        out.append(np.histogram2d(r_det[0][ok], r_det[2][ok], weights=w[ok], **kw)[0].T)
    return out


def reference_images(rf, J):
    from oracle import synthpy_oracle as O
    return stokes_images(O.run_chain(rf, O.chain("shadow_two", R=R)), J)


def _pixels(N, I, Q, U):
    """A Polarimetry whose 'pixels' are given arrays (its angle / analyser algebra needs no device)."""
    from synthpy_b200.diagnostics import Polarimetry
    p = Polarimetry.__new__(Polarimetry)
    p.N, p.I, p.Q, p.U = N, I, Q, U
    return p


# ---- CPU ---------------------------------------------------------------------------------------------------------
def test_abi_constants_match_header_and_structs_unchanged():
    from synthpy_b200 import _lib as L
    src = open(HEADER).read()
    define = lambda name: int(re.search(rf"#define {name} (\d+)", src).group(1))
    assert L.IMG_STOKES == define("SP_IMG_STOKES") == 2
    assert L.STOKES_FRAC_BITS == define("SP_STOKES_FRAC_BITS") == 32
    assert C.sizeof(L.Image) == 64 and C.sizeof(L.Channel) == 88
    assert L.lib.sp_version() == 4


def _stokes_channel(ops=(), planes=True):
    from synthpy_b200 import _lib as L
    arr = (L.OpticOp * max(1, len(ops)))(*[L.OpticOp(kind=k, p0=a, p1=b) for k, a, b in ops])
    img = L.Image(kind=L.IMG_STOKES, nx=8, ny=6, x_lo=-9.0, x_hi=9.0, y_lo=-6.75, y_hi=6.75,
                  planes_dev=8 if planes else None)
    return L.Channel(ops_host=arr, n_ops=len(ops), wavelength=1064e-9, image=img), arr


def test_validation_before_any_cuda_call():
    from synthpy_b200 import _lib as L
    lib, d = L.lib, C.c_void_p(8)                       # never dereferenced: every call must fail validation first
    ch, keep = _stokes_channel()
    assert lib.sp_optics_image(d, None, 16, C.byref(ch), None, None, None) == -1
    assert b"Stokes image needs Jones vectors" in lib.sp_last_error()
    ch, keep = _stokes_channel(planes=False)
    assert lib.sp_optics_image(d, d, 16, C.byref(ch), None, None, None) == -1
    assert b"Stokes channel without planes buffer" in lib.sp_last_error()
    ch, keep = _stokes_channel(ops=[(L.OP_REF_BEAM, 10.0, 20.0), (L.OP_TRAVEL, 400.0, 0.0)])
    assert lib.sp_optics_image(d, d, 16, C.byref(ch), None, None, None) == -1
    assert b"reference beam" in lib.sp_last_error()
    P = L.Params(method=0, n_steps=10, h=1e-12, probing_axis=2, out_axis_a=0, out_axis_b=1)
    chans = (L.Channel * 1)(ch)
    assert lib.sp_propagate(d, C.byref(P), d, d, None, 16, 0, None, None, None, None, chans, 1, None, None) == -1
    assert b"reference beam" in lib.sp_last_error()


def test_spec_and_constructor_argument_errors():
    from synthpy_b200 import diagnostics as D
    with pytest.raises(ValueError, match="not both"):
        D.spec("shadow_two", stokes=True, interferogram=True)
    with pytest.raises(ValueError, match="reference beam"):
        D.spec("shadow_two", stokes=True, ref_beam=(10, 20))
    with pytest.raises(ValueError, match="Jf"):
        D.Polarimetry(1064e-9, np.zeros((4, 3)))


def test_restatement_identities_on_reference_jones_vectors(g6):
    for sf, J in ((g6["rk4_sf"], g6["rk4_Jf"]), (g6["joint_sf"], g6["joint_Jf"])):
        amp, pol = sf[6], sf[8]
        assert np.ptp(pol) > 1e-3 and np.ptp(amp) > 1e-3        # both channels are live in g6
        I, Q, U = stokes_of(J)                                   # amp reaches ~12 in g6: relative to I
        assert np.max(np.abs(I - amp ** 2) / I) < 1e-12
        assert np.max(np.abs(Q * Q + U * U - I * I) / I ** 2) < 1e-12
        assert np.max(np.abs(Q + amp ** 2 * np.cos(2 * pol)) / I) < 1e-12
        assert np.max(np.abs(U + amp ** 2 * np.sin(2 * pol)) / I) < 1e-12
        p = _pixels(np.ones_like(I), I, Q, U)
        d = np.angle(np.exp(2j * (p.rotation_angle() - pol))) / 2          # difference modulo pi
        assert np.max(np.abs(d)) < 1e-12
        assert np.max(np.abs(p.analyser_image(pol) - I) / I) < 1e-12
        assert np.max(np.abs(p.analyser_image(pol + np.pi / 2)) / I) < 1e-12
    p = _pixels(np.array([0.0, 1.0]), np.array([0.0, 1.0]), np.array([0.0, -1.0]), np.array([0.0, 0.0]))
    a = p.rotation_angle()
    assert np.isnan(a[0]) and a[1] == 0.0


# ---- GPU ---------------------------------------------------------------------------------------------------------
def _g6_domain(g, *, B_on=True, inv_brems=True, phaseshift=False):
    from synthpy_b200 import domain as Dm
    dom = Dm.ScalarDomain([10e-3, 10e-3, 20e-3], [24, 20, 28], phaseshift=phaseshift, B_on=B_on, inv_brems=inv_brems)
    dom.external_ne(g["ne"]); dom.external_B(g["B"]); dom.external_Te(g["Te"]); dom.external_Z(g["Z"])
    return dom


def _polarimetry(lwl, rf, J, bin_scale=BS):
    from synthpy_b200 import diagnostics as D
    p = D.Polarimetry(lwl, rf, J, R=R)
    p.two_lens_solve()
    p.polarimetry(bin_scale=bin_scale)
    return [np.asarray(v) for v in (p.N, p.I, p.Q, p.U)]


def _assert_images(got, want, rel_tol):
    """Counts identical; I, Q, U within the fixed-point quantisation (2^-32 per ray) plus rel_tol of the pixel's I."""
    N = want[0]
    assert np.array_equal(got[0], N)
    for a, b in zip(got[1:], want[1:]):
        assert np.all(np.abs(a - b) <= N * Q32 + rel_tol * want[1] + 1e-15)


@pytest.mark.gpu
def test_pinned_to_reference_jones_vectors(g6):
    lwl = float(g6["lwl"])
    for rf, J in ((g6["rk4_rf"], g6["rk4_Jf"]), (g6["joint_rf"], g6["joint_Jf"])):
        want = reference_images(rf, J)
        assert want[0].sum() == 128
        _assert_images(_polarimetry(lwl, rf, J), want, 0.0)


@pytest.mark.gpu
def test_histogram_edges_right_edge_inclusive():
    """Stokes images use np.histogram2d's edges: a ray on the right-most edge lands in the last bin."""
    from synthpy_b200 import engine
    rng = np.random.default_rng(4)
    n = 4000
    r = np.zeros((4, n))
    r[0], r[2] = rng.uniform(-10, 10, n), rng.uniform(-7.5, 7.5, n)
    r[0, :8], r[2, :8] = [9.0, -9.0, 9.0, 0.0, 9.0, 9.5, np.nan, 0.0], [0.0, 6.75, 6.75, -6.75, -7.0, 0.0, 0.0, np.nan]
    pol, amp = rng.uniform(-2, 2, n), rng.uniform(0.5, 2, n)
    J = amp * np.stack([-np.sin(pol), np.cos(pol)]) * np.exp(1j * rng.uniform(0, 6, n))
    img = engine.ImageBuffer.for_stokes(bin_scale=BS)
    engine.optics_image(engine.to_device(r), [], jf=engine.to_device(J, torch.complex128), image=img, input_mm=True,
                        want_rays=False)
    got = [v.cpu().numpy() for v in img.stokes().values()]
    want = stokes_images(r, J)
    assert got[0][-1, -1] >= 1 and got[0][-1, 0] >= 1           # (9, 6.75) and (-9, 6.75) are binned
    _assert_images(got, want, 1e-15)


@pytest.mark.gpu
def test_end_to_end_matches_reference(g6):
    from synthpy_b200 import propagator as P
    lwl, ext, n = float(g6["lwl"]), float(g6["extent"]), int(g6["rk4_nsteps"])
    dom = _g6_domain(g6, phaseshift=True)
    rf, Jf, _ = P.solve(g6["s0"], dom, ext, lwl=lwl, return_E=True, method="rk4", n_steps=n, early_exit=False, phase_f64=True)
    _assert_images(_polarimetry(lwl, rf, Jf), reference_images(g6["rk4_rf"], g6["rk4_Jf"]), 1e-7)


@pytest.mark.gpu
@pytest.mark.parametrize("method", ["rk4", "rk45"])
def test_fused_equals_two_stage(g6, method):
    from synthpy_b200 import diagnostics as D, propagator as P
    lwl, ext, n = float(g6["lwl"]), float(g6["extent"]), int(g6["rk4_nsteps"])
    dom = _g6_domain(g6)
    kw = dict(lwl=lwl, method=method, early_exit=False, **({"n_steps": n} if method == "rk4" else {}))
    spec = D.spec("shadow_two", bin_scale=BS, R=R, stokes=True)
    stats, _ = P.solve_and_image(dom, g6["s0"], ext, [spec], **kw)
    fused = {k: v.cpu().numpy() for k, v in spec.image.stokes().items()}
    rf, Jf, _ = P.solve(g6["s0"], dom, ext, return_E=True, **kw)
    two = _polarimetry(lwl, rf, Jf)
    assert stats["rays_binned"] == int(fused["N"].sum()) == 128
    for k, v in zip("NIQU", two):
        assert np.array_equal(fused[k], v), k
    assert np.array_equal(spec.image.result().cpu().numpy(), fused["I"])


def _device_case(g, *, B_on=True, inv_brems=True, precision="fp64", chunks=((0, 100000),), sort=True, bin_scale=20):
    from synthpy_b200 import beam as B, diagnostics as D, propagator as P
    dom = _g6_domain(g, B_on=B_on, inv_brems=inv_brems)
    beam = B.Beam(100000, 4e-3, 5e-5, float(g["extent"]), device=True, seed=11)
    spec = D.spec("shadow_two", bin_scale=bin_scale, R=R, stokes=True)
    for off, cnt in chunks:
        P.solve_and_image(dom, beam, float(g["extent"]), [spec], lwl=float(g["lwl"]), n_rays=cnt, ray_offset=off,
                          sort=sort, precision=precision)
    return spec.image


@pytest.mark.gpu
def test_partition_and_order_invariance(g6):
    ref = _device_case(g6).planes.cpu().numpy()
    assert ref[0].sum() > 50000
    assert np.array_equal(_device_case(g6, sort=False).planes.cpu().numpy(), ref)
    assert np.array_equal(_device_case(g6, chunks=((0, 40000), (40000, 60000))).planes.cpu().numpy(), ref)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp64", "fp32"])
def test_exact_unattenuated_unrotated(g6, precision):
    img = _device_case(g6, B_on=False, inv_brems=False, precision=precision)
    N, I, Q, U = img.planes.cpu().numpy()
    assert N.sum() > 50000
    assert np.array_equal(I, N << 32) and np.array_equal(Q, -I) and not U.any()
    S = img.stokes()
    assert torch.equal(S["I"], S["N"]) and torch.equal(img.result(), S["N"])


@pytest.mark.gpu
def test_inverse_bremsstrahlung_channel_weights_intensity(g6):
    """The reference integrates amp' = +kappa amp (full_solver.py:540) and g6's kappa is positive everywhere, so every
    ray's amp grows from 1 (g6: 1.19 to 11.8 after the box) and I = sum amp^2 exceeds the ray count on every lit pixel."""
    assert g6["kappa"].min() > 0
    S = {k: v.cpu().numpy() for k, v in _device_case(g6, B_on=False, inv_brems=True).stokes().items()}
    lit = S["N"] > 0
    assert lit.sum() > 100 and np.all(S["I"][lit] > S["N"][lit]) and not S["I"][~lit].any()


@pytest.mark.gpu
def test_faraday_rotation_known_answer():
    """Uniform ne = n0 (no refraction: straight rays) and B = B0 z: every ray turns by V n0 B0 Lz."""
    from synthpy_b200 import beam as B, diagnostics as D, domain as Dm, propagator as P
    lwl, ext, dims = 1064e-9, 10e-3, (16, 16, 33)
    n0, B0 = 1e24, 50.0
    V, Lz = 2.62e-13 * lwl ** 2, 2 * ext
    dom = Dm.ScalarDomain([10e-3, 10e-3, Lz], dims, B_on=True)
    dom.external_ne(np.full(dims, n0))
    Bf = np.zeros(dims + (3,))
    Bf[..., 2] = B0
    dom.external_B(Bf)
    beam = B.Beam(20000, 3e-3, 0.0, ext, device=True, seed=5)
    s0 = beam.materialise()
    rf, Jf, _ = P.solve(s0, dom, ext, lwl=lwl, return_E=True, method="rk4")
    p = D.Polarimetry(lwl, rf, Jf)
    p.two_lens_solve()
    p.polarimetry(bin_scale=20)
    N, I, Q, U = (np.asarray(v.cpu()) for v in (p.N, p.I, p.Q, p.U))
    lit = N > 0
    rot = V * n0 * B0 * Lz
    ds = 0.5 * dom.cell_size()
    assert 0.25 < rot < 0.35 and lit.sum() > 100
    ang = p.rotation_angle().cpu().numpy()
    assert np.all(np.isnan(ang[~lit]))
    assert np.max(np.abs(ang[lit] - rot)) <= 2 * V * n0 * B0 * C_LIGHT * (ds / C_LIGHT)
    for a in (0.0, 0.4, -1.1, np.pi / 3):
        s = (p.analyser_image(a) + p.analyser_image(a + np.pi / 2)).cpu().numpy()
        assert np.all(np.abs(s[lit] - I[lit]) <= 1e-12 * I[lit])
    best = p.analyser_image(p.rotation_angle()).cpu().numpy()
    assert np.all(best[lit] >= (1 - 1e-6) * I[lit])


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _multi_setup():
    from synthpy_b200 import beam as B, diagnostics as D
    g = dict(np.load(os.path.join(GOLDEN, "g6_channels.npz")))
    dom = _g6_domain(g)
    beam = B.Beam(200000, 4e-3, 5e-5, float(g["extent"]), device=True, seed=3)
    return g, dom, beam, [D.spec("shadow_two", bin_scale=20, R=R, stokes=True)]


def _multi_worker(rank, world, port, out_path):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    sys.path.insert(0, ROOT)
    from synthpy_b200 import distributed as Dist
    Dist.init(backend="nccl")
    g, dom, beam, specs = _multi_setup()
    Dist.solve_and_image_sharded(dom, beam, float(g["extent"]), specs, lwl=float(g["lwl"]))
    torch.cuda.synchronize()
    if rank == 0:
        np.save(out_path, specs[0].image.total().cpu().numpy())
    torch.distributed.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_stokes_image_equals_one_gpu(tmp_path):
    import torch.multiprocessing as mp
    from synthpy_b200 import propagator as P
    out = str(tmp_path / "stokes.npy")
    mp.spawn(_multi_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    g, dom, beam, specs = _multi_setup()
    P.solve_and_image(dom, beam, float(g["extent"]), specs, lwl=float(g["lwl"]))
    assert np.array_equal(np.load(out), specs[0].image.planes.cpu().numpy())
