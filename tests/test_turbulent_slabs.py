"""Out-of-core turbulent fields: the k^-11/3 philox field generated slab by slab (field_generator.domain_fft_slabs /
turbulent_ne_slabs over sp_noise_spectrum_box / k_noise_spectrum_box).

CPU: the box noise of the host build is the Hermitian extension of the half spectrum, bit for bit; spectrum_box is the
half / full-grid |k| expression; the C ABI validates before any CUDA call; the slab decomposition (phases A and B) run
on the CPU over the host build reproduces irfftn of the half spectrum.  GPU (-m gpu): the kernel against the host build
and against sp_noise_spectrum, the field against turbulent_ne(noise='philox'), window independence, out-of-core tracing
bit-identical to in-core tracing of the same planes, and memory / host-to-device traffic at 256^3."""
import ctypes as C
import itertools
import json
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

SHAPES = [(16, 16, 16), (16, 16, 15), (8, 12, 10)]
ORDERS = list(itertools.permutations(range(3)))
BAND = (4.0, 1.0)           # l_max, l_min: a band that cuts both ends of the small grids' |k| range


@pytest.fixture(scope="module")
def H():
    """The host builds of noise_core.h: noise_half / noise_full (noise_harness) and noise_box (noise_box_harness)."""
    from noise_box_harness import NoiseBoxHarness
    from noise_harness import NoiseHarness
    h = NoiseHarness()
    h.noise_box = NoiseBoxHarness().noise_box
    return h


def _k(shape, extent=5.0):
    """2 pi fftfreq axes of domain_fft for a (n0, n1, n2) grid, dx = extent / (n0 / 2)."""
    dx = extent / (shape[0] / 2)
    return [2 * np.pi * np.fft.fftfreq(n, d=dx) for n in shape]


def _steep(k):
    """k^-4 from correctly rounded float32 operations only.  torch's CPU pow (kolmogorov) rounds the same |k|
    differently in the vectorised body and the scalar tail of a loop, so its S depends on the layout on the CPU; these
    operations do not, and S(-k) == S(k) holds bit for bit in every box."""
    return 1.0 / ((k * k) * (k * k))


def _boxes(shape):
    """(lo, cnt) per grid axis: the whole grid, an interior box, the Nyquist / upper planes and the zero planes."""
    n0, n1, n2 = shape
    return [((0, 0, 0), shape),
            ((1, 2, 3), (n0 - 3, n1 - 5, n2 - 4)),
            ((n0 // 2, 0, n2 // 2), (n0 - n0 // 2, n1, n2 - n2 // 2)),
            ((0, 0, 0), (1, 1, n2)),
            ((0, n1 // 2, 0), (n0, 1, 1))]


def _box_index(lo, cnt, order):
    return np.ix_(*[np.arange(lo[o], lo[o] + cnt[o]) for o in order])


def _hermitian_full(Hh, shape):
    """The full grid of a half spectrum: H(k) for l <= n2 / 2, conj H(-k) above."""
    n0, n1, n2 = shape
    up = np.arange(n2 // 2 + 1, n2)
    upper = np.conj(Hh[np.ix_((-np.arange(n0)) % n0, (-np.arange(n1)) % n1, n2 - up)])
    return np.concatenate([Hh, upper], axis=2)


def _host_noise_box(Hn):
    """engine.noise_spectrum_box's signature over the host build, for the decomposition on the CPU."""
    def write(S, shape, order, lo, cnt, seed, out):
        out.copy_(torch.from_numpy(Hn.noise_box(S.numpy(), shape, order, lo, cnt, seed)))
        return out
    return write


# ------------------------------------------------------------------------------------------------------------ CPU

@pytest.mark.parametrize("shape", SHAPES)
def test_box_is_hermitian_extension_of_half(H, shape):
    """hh_noise_box on any box in any order == the Hermitian extension of hh_noise_half, bit for bit (signed zeros too)."""
    from synthpy_b200 import field_generator as FG
    n2h = shape[2] // 2 + 1
    S_full = FG.spectrum_box(_steep, *BAND, _k(shape), (0, 1, 2), (0, 0, 0), shape, "cpu").numpy()
    S_half = np.ascontiguousarray(S_full[..., :n2h])
    assert 0.2 < (S_full > 0).mean() < 0.9 and S_full[0, 0, 0] == 0
    full = _hermitian_full(H.noise_half(S_half, shape, 7), shape)
    for order in ORDERS:
        for lo, cnt in _boxes(shape):
            idx = _box_index(lo, cnt, order)
            S_box = np.ascontiguousarray(S_full.transpose(order)[idx])
            out = H.noise_box(S_box, shape, order, lo, cnt, 7)
            ref = np.ascontiguousarray(full.transpose(order)[idx])
            assert np.array_equal(out.view(np.uint64), ref.view(np.uint64)), (order, lo, cnt)


@pytest.mark.parametrize("shape", SHAPES + [(64, 64, 64)])
def test_spectrum_box_is_the_half_and_full_grid_S(shape):
    """spectrum_box's |k| is half_spectrum's / domain_fft's expression bit for bit in every order and box (checked
    through an exact k_func); with kolmogorov, on the CPU, it agrees to torch's CPU pow rounding (1 ulp) and is
    identical to half_spectrum on the half box."""
    from synthpy_b200 import field_generator as FG
    ks = _k(shape)
    n2h = shape[2] // 2 + 1
    ky, kx, kz = (torch.from_numpy(a) for a in ks)
    k_full = torch.sqrt((kx[None, :, None] ** 2 + ky[:, None, None] ** 2 + kz[None, None, :] ** 2).to(torch.float32))
    k_full = k_full.masked_fill(~((k_full >= 2 * np.pi / BAND[0]) & (k_full <= 2 * np.pi / BAND[1])), 0.0)
    ident = lambda k: k
    assert torch.equal(FG.half_spectrum(ident, *BAND, ks, "cpu"), k_full[..., :n2h])
    half = FG.half_spectrum(FG.kolmogorov, *BAND, ks, "cpu")
    assert torch.equal(FG.spectrum_box(FG.kolmogorov, *BAND, ks, (0, 1, 2), (0, 0, 0), shape[:2] + (n2h,), "cpu"), half)
    for order in ORDERS:
        for lo, cnt in _boxes(shape):
            ref = k_full.permute(order)[_box_index(lo, cnt, order)]
            assert torch.equal(FG.spectrum_box(ident, *BAND, ks, order, lo, cnt, "cpu"), ref), (order, lo, cnt)
            kol = FG.spectrum_box(FG.kolmogorov, *BAND, ks, order, lo, cnt, "cpu")
            ref_kol = FG.kolmogorov(ref).masked_fill(ref == 0, 0.0)
            torch.testing.assert_close(kol, ref_kol, rtol=2.5e-7, atol=0)


def test_abi_validation_without_cuda():
    """sp_noise_spectrum_box refuses null pointers, n < 2, an order that is not a permutation, a box outside the grid
    and a misaligned output before any CUDA call; the slab sources have no CPU path."""
    from synthpy_b200 import _lib as L, field_generator as FG
    lib = L.lib
    d, odd = C.c_void_p(256), C.c_void_p(264)
    i3 = lambda *v: (C.c_int * 3)(*v)
    ok = dict(order=i3(2, 0, 1), lo=i3(0, 1, 2), cnt=i3(4, 3, 2))

    def call(S=d, n=(4, 4, 4), out=d, **kw):
        a = dict(ok, **kw)
        return lib.sp_noise_spectrum_box(S, *n, a["order"], a["lo"], a["cnt"], 1, out, None)

    assert call(S=None) == -1 and b"null" in lib.sp_last_error()
    assert call(out=None) == -1 and b"null" in lib.sp_last_error()
    for k in ("order", "lo", "cnt"):
        assert call(**{k: None}) == -1 and b"null" in lib.sp_last_error(), k
    for n in [(1, 4, 4), (4, 1, 4), (4, 4, 1), (0, 4, 4), (4, 4, -3)]:
        assert call(n=n) == -1 and b">= 2" in lib.sp_last_error(), n
    for o in [(0, 0, 1), (0, 1, 3), (-1, 1, 2), (2, 2, 2)]:
        assert call(order=i3(*o)) == -1 and b"permutation" in lib.sp_last_error(), o
    for lo, cnt in [((-1, 0, 0), (2, 2, 2)), ((0, 0, 0), (0, 2, 2)), ((0, 0, 0), (2, -1, 2)), ((3, 0, 0), (2, 2, 2)),
                    ((0, 0, 4), (1, 1, 1)), ((0, 2**31 - 1, 0), (1, 2, 1))]:
        assert call(lo=i3(*lo), cnt=i3(*cnt)) == -1 and b"box" in lib.sp_last_error(), (lo, cnt)
    assert call(out=odd) == -1 and b"aligned" in lib.sp_last_error()
    with pytest.raises(RuntimeError, match="no CPU path"):
        FG.domain_fft_slabs(FG.kolmogorov, 1, 0.01, 5, 4, axis=2, seed=1, device="cpu")
    with pytest.raises(RuntimeError, match="no CPU path"):
        FG.turbulent_ne_slabs(4, device="cpu")


@pytest.mark.parametrize("shape", SHAPES + [(12, 12, 7)])
def test_slab_decomposition_on_host_build(H, shape):
    """Phases A and B (inverse FFT along p chunk by chunk, then along r and the C2R along q per block) over the host
    build's box noise reproduce irfftn of the host build's half spectrum to 1e-13 of max |f|, for every probing axis;
    every window is the same bits as the slice of the whole; ne0 + dne f is formed per block as turbulent_ne forms it."""
    from synthpy_b200 import field_generator as FG
    ks = _k(shape)
    S_half = FG.half_spectrum(_steep, *BAND, ks, "cpu").numpy()
    f_ref = np.fft.irfftn(H.noise_half(S_half, shape, 5), s=shape, axes=(0, 1, 2))
    m = max(f_ref.max(), -f_ref.min())
    rng = np.random.default_rng(0)
    for axis in range(3):
        src = FG._FieldSlabs(_steep, *BAND, ks, axis=axis, seed=5, block_planes=3, device=torch.device("cpu"),
                             noise_box=_host_noise_box(H))
        n = shape[axis]
        whole = src(0, n)
        assert whole.dtype == torch.float64 and tuple(whole.shape) == shape and src.shape == shape
        assert abs(src.max_abs - m) <= 1e-13 * m
        assert float(np.abs(whole.numpy() - f_ref / m).max()) <= 1e-13, axis
        for _ in range(6):
            k0 = int(rng.integers(0, n - 1))
            k1 = int(rng.integers(k0 + 1, n + 1))
            assert torch.equal(src(k0, k1), whole.narrow(axis, k0, k1 - k0)), (axis, k0, k1)
        ne = FG._FieldSlabs(_steep, *BAND, ks, axis=axis, seed=5, block_planes=3, device=torch.device("cpu"),
                            noise_box=_host_noise_box(H), ne0=1e25, dne=9e24)
        assert torch.equal(ne(0, n), 1e25 + 9e24 * whole)
        with pytest.raises(ValueError):
            src(0, n + 1)
        with pytest.raises(ValueError):
            src(2, 2)


# ------------------------------------------------------------------------------------------------------------ GPU

def _ulp_error(dev, host, scale):
    return np.maximum(np.abs(dev.real - host.real), np.abs(dev.imag - host.imag)) / np.spacing(scale)


@pytest.mark.gpu
def test_device_box_equals_host_build_and_half_kernel(H):
    """k_noise_spectrum_box against the host build (the 8-ulp allowance of test_field_noise's device test), and bit for
    bit against k_noise_spectrum wherever both write -- and against its conjugate mirror everywhere else.  spectrum_box on
    the device is half_spectrum's S exactly, in every order."""
    from synthpy_b200 import engine, field_generator as FG
    for shape in SHAPES + [(128, 128, 99)]:
        ks = _k(shape)
        n2h = shape[2] // 2 + 1
        S_full = FG.spectrum_box(FG.kolmogorov, 100.0, 0.01, ks, (0, 1, 2), (0, 0, 0), shape, "cuda")
        S_half = FG.half_spectrum(FG.kolmogorov, 100.0, 0.01, ks, "cuda")
        assert torch.equal(S_full[..., :n2h], S_half)
        full_dev = _hermitian_full(engine.noise_spectrum(S_half, shape, 42).cpu().numpy(), shape)
        full_host = _hermitian_full(H.noise_half(S_half.cpu().numpy(), shape, 42), shape)
        Z = H.noise_full(shape, 42)
        r = np.abs(Z)
        mirror = np.ix_(*[(-np.arange(n)) % n for n in shape])
        scale = np.sqrt(S_full.cpu().numpy()).astype(np.float64) * 0.5 * (r + r[mirror])
        for order in ORDERS:
            for lo, cnt in _boxes(shape)[:3]:
                S_box = FG.spectrum_box(FG.kolmogorov, 100.0, 0.01, ks, order, lo, cnt, "cuda")
                idx = _box_index(lo, cnt, order)
                assert torch.equal(S_box.cpu(), S_full.cpu().permute(order)[idx])
                Hb = engine.noise_spectrum_box(S_box, shape, order, lo, cnt, 42)
                out = torch.empty_like(Hb)
                assert engine.noise_spectrum_box(S_box, shape, order, lo, cnt, 42, out=out) is out and torch.equal(out, Hb)
                Hb = Hb.cpu().numpy()
                host = np.ascontiguousarray(full_host.transpose(order)[idx])
                sc = np.maximum(np.ascontiguousarray(scale.transpose(order)[idx]), np.finfo(np.float64).tiny)
                assert _ulp_error(Hb, host, sc).max() <= 8, (shape, order, lo, cnt)
                # the same device math as k_noise_spectrum at k and -k: the Hermitian extension of its half, bit for bit
                ref = np.ascontiguousarray(full_dev.transpose(order)[idx])
                assert np.array_equal(Hb.view(np.uint64), ref.view(np.uint64)), (shape, order, lo, cnt)


@pytest.mark.gpu
@pytest.mark.parametrize("pd", ["x", "y", "z"])
def test_slab_field_equals_turbulent_ne(pd):
    """source(0, n) of turbulent_ne_slabs against turbulent_ne(noise='philox') at 64^3, to 1e-12 of max |ne - ne0|."""
    from synthpy_b200 import field_generator as FG
    ref = FG.turbulent_ne(32, noise="philox", seed=9)
    src = FG.turbulent_ne_slabs(32, probing_direction=pd, seed=9, block_planes=16)
    ne = src(0, 64)
    assert ne.is_cuda and ne.dtype == torch.float64 and tuple(ne.shape) == src.shape == (64, 64, 64)
    dev = float((ref - 1e25).abs().max())
    assert float((ne - ref).abs().max()) <= 1e-12 * dev


@pytest.mark.gpu
def test_slab_field_odd_nz_and_window_independence():
    """domain_fft_slabs against domain_fft(noise='philox') at 32 x 32 x 24 and 32 x 32 x 25 (odd n_q when probing z:
    the half is along y then), 20 random windows bit-identical to slices of the whole, two constructions identical."""
    from synthpy_b200 import field_generator as FG
    for factor in (0.75, 0.78125):
        ref = FG.domain_fft(FG.kolmogorov, 1, 0.01, 5, 16, factor, noise="philox", seed=4)
        for axis in range(3):
            src = FG.domain_fft_slabs(FG.kolmogorov, 1, 0.01, 5, 16, factor, axis=axis, seed=4, block_planes=5)
            whole = src(0, ref.shape[axis])
            assert float((whole - ref).abs().max()) <= 1e-12, (factor, axis)
    rng = np.random.default_rng(1)
    for axis in (0, 2):
        a = FG.turbulent_ne_slabs(32, probing_direction="xyz"[axis], seed=2, block_planes=7)
        b = FG.turbulent_ne_slabs(32, probing_direction="xyz"[axis], seed=2, block_planes=7)
        whole = a(0, 64)
        assert torch.equal(whole, b(0, 64)) and a.max_abs == b.max_abs
        for _ in range(20):
            k0 = int(rng.integers(0, 63))
            k1 = int(rng.integers(k0 + 1, min(64, k0 + 40) + 1))
            assert torch.equal(a(k0, k1), whole.narrow(axis, k0, k1 - k0)), (axis, k0, k1)


@pytest.mark.gpu
def test_out_of_core_trace_of_slab_field_is_in_core_trace():
    """128^3, probing z and x: solve_out_of_core on turbulent_ne_slabs against propagator.solve on the same planes
    source(0, n) held whole -- exit rays, Jones vectors, states, steps per ray, launch stats and a fused shadow_two
    image bit for bit.  prefetch=True refuses the device source."""
    from synthpy_b200 import diagnostics as D, domain as Dm, legacy, out_of_core as OC, propagator as P
    from synthpy_b200 import field_generator as FG
    n, lwl, ext = 128, 1064e-9, 10e-3
    lengths = (10e-3, 10e-3, 10e-3)
    for pd in ("z", "x"):
        src = FG.turbulent_ne_slabs(n // 2, probing_direction=pd, seed=6, block_planes=16)
        dom = Dm.ScalarDomain(lengths, n, probing_direction=pd, phaseshift=True)
        dom.external_ne(src(0, n))
        np.random.seed(10)
        s0 = legacy.init_beam(8000, 4e-3, 1e-3, ext, "circular", pd)
        steps = 2 * (n - 1)
        rf, Jf, _, ex = P.solve(s0, dom, ext, lwl=lwl, return_E=True, method="rk4", n_steps=steps, return_state=True)
        rf2, Jf2, _, ex2 = OC.solve_out_of_core(s0, src, lengths, (n, n, n), ext, slab_planes=40, probing_direction=pd,
                                                lwl=lwl, return_E=True, phaseshift=True, n_steps=steps, return_state=True)
        assert len(ex2["slabs"]) >= 3 and sum(e["steps"] for e in ex2["slabs"]) == steps
        assert np.isfinite(rf).all(axis=0).sum() > 0.5 * s0.shape[1]
        assert np.array_equal(rf2, rf, equal_nan=True) and np.array_equal(Jf2, Jf, equal_nan=True)
        assert np.array_equal(ex2["sf"], ex["sf"], equal_nan=True) and np.array_equal(ex2["steps"], ex["steps"])
        assert ex2["stats"]["ray_steps"] == ex["stats"]["ray_steps"]
        a, b = D.spec("shadow_two", bin_scale=16), D.spec("shadow_two", bin_scale=16)
        P.solve_and_image(dom, s0, ext, [a], lwl=lwl, method="rk4", n_steps=steps)
        OC.solve_out_of_core(s0, src, lengths, (n, n, n), ext, slab_planes=40, probing_direction=pd, lwl=lwl,
                             phaseshift=True, n_steps=steps, diagnostics=[b])
        assert a.image.result().sum() > 1000 and torch.equal(a.image.result(), b.image.result())
        with pytest.raises(ValueError, match="host sources"):
            OC.solve_out_of_core(s0, src, lengths, (n, n, n), ext, slab_planes=40, probing_direction=pd, lwl=lwl,
                                 n_steps=steps, prefetch=True)


def _h2d_bytes(trace_path):
    with open(trace_path) as fh:
        events = json.load(fh)["traceEvents"]
    return sum(int(e.get("args", {}).get("bytes", 0)) for e in events
               if e.get("cat") == "gpu_memcpy" and "HtoD" in e.get("name", ""))


@pytest.mark.gpu
def test_slab_source_memory_and_host_copies_256(tmp_path):
    """256^3, block_planes=16: the peak allocation over the source's whole life (construction and every block served
    once) is at most 12 bytes per grid point (G alone is 8.06), and it copies less than 1 MB host to device."""
    from synthpy_b200 import field_generator as FG
    n, N = 256, 256 ** 3

    def life():
        src = FG.turbulent_ne_slabs(n // 2, seed=1, block_planes=16)
        for k0 in range(0, n, 16):
            blk = src(k0, k0 + 16)
            del blk
        torch.cuda.synchronize()
        return src

    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    src = life()
    peak = torch.cuda.max_memory_allocated() - base
    del src
    assert peak <= 12 * N, peak / N
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        src = life()
    del src
    path = str(tmp_path / "slabs.json")
    prof.export_chrome_trace(path)
    assert _h2d_bytes(path) < 1 << 20
