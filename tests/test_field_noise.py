"""Turbulent-field noise drawn on the device (field_generator noise='philox', sp_noise_spectrum / k_noise_spectrum).

CPU: the per-element source (noise_core.h) built by g++ (tests/noise_harness.cpp): the Hermitian half spectrum it writes is
the full complex path's field after irfftn, its noise is N(0, 1) and independent, and the C ABI validates its arguments
before any CUDA call.  GPU (-m gpu): the kernel against the host build, the product path against the full complex path,
the spectrum at 512^3, memory and host-to-device traffic at 256^3, a traced field, and two GPUs."""
import ctypes as C
import json
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

SHAPES = [(16, 16, 16), (16, 16, 15), (8, 12, 10)]
NOISE_TAG = 0xF1E1D
BEAM_TAG = 0x5EED
BAND = (4.0, 1.0)           # l_max, l_min: a band that cuts both ends of the small grids' |k| range


@pytest.fixture(scope="module")
def H():
    from noise_harness import NoiseHarness
    return NoiseHarness()


@pytest.fixture(scope="module")
def philox():
    """The Philox4x32-10 block function of the host build (ray_core.h)."""
    from harness import Harness
    return Harness().philox


def _k(shape, extent=5.0):
    """2 pi fftfreq axes of domain_fft for a (n0, n1, n2) grid, dx = extent / (n0 / 2)."""
    dx = extent / (shape[0] / 2)
    return [2 * np.pi * np.fft.fftfreq(n, d=dx) for n in shape]


def _full_S(shape, device, l_max=1.0, l_min=0.01):
    """S on the full grid with domain_fft's own expression (float32 |k|, k_func on the band only)."""
    from synthpy_b200 import field_generator as FG
    ky, kx, kz = (torch.from_numpy(a).to(device) for a in _k(shape))
    k = torch.sqrt((kx[None, :, None] ** 2 + ky[:, None, None] ** 2 + kz[None, None, :] ** 2).to(torch.float32))
    mask = (k >= 2 * np.pi / l_max) & (k <= 2 * np.pi / l_min)
    S = torch.zeros_like(k)
    S[mask] = FG.kolmogorov(k[mask])
    return S


def _half_S(shape, device, l_max=1.0, l_min=0.01):
    from synthpy_b200 import field_generator as FG
    return FG.half_spectrum(FG.kolmogorov, l_max, l_min, _k(shape), device)


def _mirror(shape):
    return np.ix_(*[(-np.arange(n)) % n for n in shape])


def _mirrored(S_half, shape):
    """The full grid of a half-grid S: S(i, j, l) = S(-i, -j, n2 - l) for l > n2 // 2."""
    n0, n1, n2 = shape
    upper = S_half[np.ix_((-np.arange(n0)) % n0, (-np.arange(n1)) % n1, n2 - np.arange(n2 // 2 + 1, n2))]
    return np.concatenate([S_half, upper], axis=2)


def _self_conjugate(shape):
    n0, n1, n2 = shape
    I, J, L = np.meshgrid(np.arange(n0), np.arange(n1), np.arange(n2 // 2 + 1), indexing="ij")
    return ((-I) % n0 == I) & ((-J) % n1 == J) & ((-L) % n2 == L)


def _box_muller(block):
    u = lambda hi, lo: float(((int(hi) << 32) | int(lo)) >> 11) / 2.0 ** 53
    U0, U1 = u(block[0], block[1]), u(block[2], block[3])
    r = np.sqrt(-2.0 * np.log(1.0 - U0))
    return r * np.cos(2 * np.pi * U1) + 1j * r * np.sin(2 * np.pi * U1)


# ------------------------------------------------------------------------------------------------------------ CPU

@pytest.mark.parametrize("shape", SHAPES)
def test_half_spectrum_is_the_full_complex_path(H, shape):
    """irfftn of the half spectrum == Re ifftn(Z sqrt(S)) for the same Z, to FFT rounding; Im H == +0 exactly at the
    self-conjugate points (odd n2 has them on the l = 0 plane only)."""
    n2h = shape[2] // 2 + 1
    S_half = _half_S(shape, "cpu", *BAND).numpy()
    # the kernel reads S on the half grid and relies on S(-k) == S(k); the full grid is that half mirrored.  domain_fft's
    # full-grid S agrees to float32 rounding (CPU torch's vectorised pow may round k^-11/3 differently at mirrored points)
    S_ref = _full_S(shape, "cpu", *BAND).numpy()
    S = _mirrored(S_half, shape)
    assert np.array_equal(S, S[_mirror(shape)]) and np.array_equal(S[..., :n2h], S_half)
    np.testing.assert_allclose(S, S_ref, rtol=2.5e-7, atol=0)
    assert 0.2 < (S > 0).mean() < 0.9 and S[0, 0, 0] == 0                      # band-limited at both ends
    Hh = H.noise_half(S_half, shape, 7)
    Z = H.noise_full(shape, 7)
    f_half = np.fft.irfftn(Hh, s=shape, axes=(0, 1, 2))
    f_full = np.fft.ifftn(Z * np.sqrt(S).astype(np.float64)).real
    assert np.max(np.abs(f_half - f_full)) <= 1e-13 * np.max(np.abs(f_full))
    sc = _self_conjugate(shape)
    assert sc.sum() == (8 if shape[2] % 2 == 0 else 4)
    assert np.all(Hh.imag[sc] == 0) and not np.signbit(Hh.imag[sc]).any()
    # H is Hermitian on the planes that are their own mirror (l = 0, and l = n2/2 for even n2)
    planes = [0] + ([shape[2] // 2] if shape[2] % 2 == 0 else [])
    for l in planes:
        P = Hh[..., l]
        assert np.array_equal(P, np.conj(P[np.ix_(*[(-np.arange(n)) % n for n in shape[:2]])]))


@pytest.mark.parametrize("shape", SHAPES + [(40, 40, 3), (64, 64, 63)])
def test_slab_wise_inverse_fft_is_irfftn(shape):
    """The philox path's inverse FFT (C2C over axes 0, 1 in place slab by slab, then C2R slab by slab) is
    torch.fft.irfftn, also for a half spectrum that is not Hermitian on its self-mirrored planes."""
    from synthpy_b200.field_generator import _irfftn_slabs
    g = torch.Generator().manual_seed(3)
    H = torch.randn(shape[:2] + (shape[2] // 2 + 1,), dtype=torch.complex128, generator=g)
    ref = torch.fft.irfftn(H, s=shape, dim=(0, 1, 2))
    out = _irfftn_slabs(H.clone(), shape)
    assert out.dtype == torch.float64 and tuple(out.shape) == shape
    assert float((out - ref).abs().max()) <= 1e-15 * float(ref.abs().max())


def test_noise_definition(H, philox):
    """Z at flat index f is Box-Muller of one Philox4x32-10 block, key = seed, counter = (f lo, f hi, 0, 0xf1e1d)."""
    seed = 0x123456789ABCDEF
    shape = (4, 6, 7)
    Z = H.noise_full(shape, seed).ravel()
    key = (seed & 0xFFFFFFFF, seed >> 32)
    for f in range(Z.size):
        z = _box_muller(philox(key, (f, 0, 0, NOISE_TAG)))
        assert abs(Z[f] - z) <= 4e-15 * max(1.0, abs(z)), f


def test_noise_statistics(H):
    """1.2e6 host-build draws: Re and Im are N(0, 1) (moments, KS), uncorrelated with each other and along the index."""
    from scipy import stats
    z = H.noise_full((128, 96, 100), 2024).ravel()
    assert z.size >= 1_000_000
    for x in (z.real, z.imag):
        assert abs(x.mean()) < 5e-3 and abs(x.var() - 1) < 5e-3
        assert stats.kstest(x, "norm").pvalue > 1e-3
        assert abs(np.corrcoef(x[:-1], x[1:])[0, 1]) < 5e-3
    assert abs(np.corrcoef(z.real, z.imag)[0, 1]) < 5e-3


def test_streams_differ_by_seed_and_from_the_beam(H, philox):
    """Two seeds give unrelated noise; the field stream and the beam stream of the same seed are unrelated too."""
    shape = (64, 64, 64)
    a, b = H.noise_full(shape, 5).ravel(), H.noise_full(shape, 6).ravel()
    assert not np.any(a == b)
    assert abs(np.corrcoef(a.real, b.real)[0, 1]) < 5e-3 and abs(np.corrcoef(a.imag, b.imag)[0, 1]) < 5e-3
    # beam ray i uses counter (i, 0, 0, 0x5eed) for its first block; the field uses (i, 0, 0, 0xf1e1d)
    n = 4096
    field = np.array([philox((5, 0), (i, 0, 0, NOISE_TAG)) for i in range(n)], dtype=np.float64)
    beam = np.array([philox((5, 0), (i, 0, 0, BEAM_TAG)) for i in range(n)], dtype=np.float64)
    assert not np.any(field == beam)
    for w in range(4):
        assert abs(np.corrcoef(field[:, w], beam[:, w])[0, 1]) < 0.06          # 1/sqrt(4096) = 0.016


def test_abi_validation_without_cuda():
    """sp_noise_spectrum refuses null pointers, dimensions below 2 and a misaligned output before any CUDA call;
    noise='philox' has no CPU path."""
    from synthpy_b200 import _lib as L, field_generator as FG
    lib = L.lib
    d, odd = C.c_void_p(256), C.c_void_p(264)
    assert lib.sp_noise_spectrum(None, 4, 4, 4, 1, d, None) == -1 and b"null" in lib.sp_last_error()
    assert lib.sp_noise_spectrum(d, 4, 4, 4, 1, None, None) == -1 and b"null" in lib.sp_last_error()
    for n in [(1, 4, 4), (4, 1, 4), (4, 4, 1), (0, 4, 4), (4, 4, -3)]:
        assert lib.sp_noise_spectrum(d, *n, 1, d, None) == -1 and b">= 2" in lib.sp_last_error(), n
    assert lib.sp_noise_spectrum(d, 4, 4, 4, 1, odd, None) == -1 and b"aligned" in lib.sp_last_error()
    with pytest.raises(RuntimeError, match="no CPU path"):
        FG.domain_fft(FG.kolmogorov, 1, 0.01, 5, 4, noise="philox", device="cpu")
    with pytest.raises(RuntimeError, match="no CPU path"):
        FG.turbulent_ne(4, noise="philox", device="cpu")


# ------------------------------------------------------------------------------------------------------------ GPU

def _ulp_error(dev, host, Hh_scale):
    return np.maximum(np.abs(dev.real - host.real), np.abs(dev.imag - host.imag)) / np.spacing(Hh_scale)


@pytest.mark.gpu
def test_device_spectrum_equals_host_build(H):
    """k_noise_spectrum against the host build of the same source on the same S: equal to a few ulp of the element's
    scale sqrt(S) (|Z| + |Z(-k)|) / 2 (CUDA's log and sincos against glibc's: 1 and 2 ulp documented bounds), and
    bit-identical from call to call.  The last shape has more half-grid elements than one launch has threads, so the
    grid-stride loop's index carries are exercised."""
    from synthpy_b200 import engine
    for shape in SHAPES + [(128, 128, 99)]:
        S = _half_S(shape, "cuda", 100.0, 0.01)                    # S > 0 everywhere but k = 0
        Hd = engine.noise_spectrum(S, shape, 42)
        assert torch.equal(Hd, engine.noise_spectrum(S, shape, 42))
        Hd = Hd.cpu().numpy()
        S_h = S.cpu().numpy()
        Hh = H.noise_half(S_h, shape, 42)
        Z = H.noise_full(shape, 42)
        n2h = shape[2] // 2 + 1
        r = np.abs(Z)
        scale = np.sqrt(S_h).astype(np.float64) * 0.5 * (r[..., :n2h] + r[_mirror(shape)][..., :n2h])
        err = _ulp_error(Hd, Hh, np.maximum(scale, np.finfo(np.float64).tiny))
        assert err.max() <= 8, (shape, float(err.max()))
        assert np.all(Hd[S_h == 0] == 0) and np.all(Hd.imag[_self_conjugate(shape)] == 0)
        assert not np.isnan(Hd).any()


@pytest.mark.gpu
@pytest.mark.parametrize("res,factor", [(16, 1), (16, 0.78125)])
def test_philox_field_equals_full_complex_path(H, res, factor):
    """domain_fft(noise='philox') against Re ifftn(Z sqrt(S)) on the full grid, with Z from the host build and S from
    domain_fft's own full-grid expression on the device: 32^3 and 32 x 32 x 25 (odd nz)."""
    from synthpy_b200 import field_generator as FG
    shape = (2 * res, 2 * res, int(2 * res * factor))
    f = FG.domain_fft(FG.kolmogorov, 1, 0.01, 5, res, factor, noise="philox", seed=11)
    assert f.is_cuda and f.dtype == torch.float64 and tuple(f.shape) == shape
    S_full = _full_S(shape, "cuda")
    S_half = _half_S(shape, "cuda")
    assert torch.equal(S_half, S_full[..., : shape[2] // 2 + 1])                # same S, bit for bit
    mirrored = torch.roll(torch.flip(S_full, dims=(0, 1, 2)), shifts=(1, 1, 1), dims=(0, 1, 2))    # S(-k)
    assert torch.equal(S_full, mirrored)
    Z = torch.from_numpy(H.noise_full(shape, 11)).cuda()
    ref = torch.fft.ifftn(Z * torch.sqrt(S_full).to(torch.float64)).real
    ref = ref / ref.abs().max()
    assert float((f - ref).abs().max()) <= 1e-12
    assert float(f.abs().max()) == 1.0
    g = FG.domain_fft(FG.kolmogorov, 1, 0.01, 5, res, factor, noise="philox", seed=11)
    assert torch.equal(f, g)
    assert not torch.equal(f, FG.domain_fft(FG.kolmogorov, 1, 0.01, 5, res, factor, noise="philox", seed=12))


@pytest.mark.gpu
def test_philox_field_spectrum_512():
    """At the C2 size the philox field is band-limited and follows k^-11/3 inside the band, as the torch-noise field
    does (test_gpu_configs::test_field_generator_on_device)."""
    from synthpy_b200 import field_generator as FG
    n, res, extent = 512, 256, 5.0
    f = (FG.turbulent_ne(res, noise="philox", seed=1) - 1e25) / 9e24
    P = torch.fft.fftn(f).abs() ** 2
    del f
    k1 = 2 * np.pi * torch.fft.fftfreq(n, d=extent / res, device="cuda", dtype=torch.float64)
    k = torch.sqrt(k1[:, None, None] ** 2 + k1[None, :, None] ** 2 + k1[None, None, :] ** 2)
    k_min, k_max = 2 * np.pi / 1.0, 2 * np.pi / 0.01
    inside = (k >= k_min) & (k <= k_max)
    assert float(P[~inside].sum()) < 1e-20 * float(P[inside].sum())
    edges = torch.logspace(np.log10(k_min * 1.5), np.log10(float(k.max()) * 0.5), 13, device="cuda", dtype=torch.float64)
    kc, pk = [], []
    for lo, hi in zip(edges[:-1], edges[1:]):
        m = (k >= lo) & (k < hi)
        kc.append(float(k[m].mean())); pk.append(float(P[m].mean()))
    slope = np.polyfit(np.log(kc), np.log(pk), 1)[0]
    assert abs(slope + 11.0 / 3.0) < 0.1, slope


def _h2d_bytes(trace_path):
    with open(trace_path) as fh:
        events = json.load(fh)["traceEvents"]
    return sum(int(e.get("args", {}).get("bytes", 0)) for e in events
               if e.get("cat") == "gpu_memcpy" and "HtoD" in e.get("name", ""))


@pytest.mark.gpu
def test_philox_memory_and_host_copies_256(tmp_path):
    """256^3: the philox path's peak allocation is at most 20 bytes per grid point (H, the field and one slab of FFT
    temporaries: about 17.5) and below the torch-noise path's (about 60);
    it copies less than 1 MB host to device (the torch path copies its 16 bytes per point of noise)."""
    from synthpy_b200 import field_generator as FG
    res, N = 128, 256 ** 3
    peaks = {}
    for noise in ("philox", "torch"):
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        f = FG.domain_fft(FG.kolmogorov, 1, 0.01, 5, res, noise=noise, seed=1)
        torch.cuda.synchronize()
        peaks[noise] = torch.cuda.max_memory_allocated() - base
        del f
    assert peaks["philox"] <= 20 * N, peaks["philox"] / N
    assert peaks["philox"] < peaks["torch"], peaks
    h2d = {}
    for noise in ("philox", "torch"):
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            f = FG.domain_fft(FG.kolmogorov, 1, 0.01, 5, res, noise=noise, seed=1)
            torch.cuda.synchronize()
        del f
        path = str(tmp_path / f"{noise}.json")
        prof.export_chrome_trace(path)
        h2d[noise] = _h2d_bytes(path)
    assert h2d["torch"] >= 16 * N                                    # the trace does list the copies
    assert h2d["philox"] < 1 << 20, h2d


@pytest.mark.gpu
def test_philox_field_traced_end_to_end():
    """A philox n_e grid, handed over as a CUDA tensor, through propagator.solve and a shadowgraphy histogram."""
    from synthpy_b200 import diagnostics as D, domain as Dm, field_generator as FG, legacy, propagator as P
    n, ext, lwl = 64, 10e-3, 1064e-9
    ne = FG.turbulent_ne(n // 2, noise="philox", seed=3)
    assert ne.is_cuda and torch.isfinite(ne).all()
    dom = Dm.ScalarDomain((10e-3, 10e-3, 20e-3), n)
    dom.external_ne(ne)
    np.random.seed(4)
    s0 = legacy.init_beam(20000, 4e-3, 5e-5, ext, "circular", "z")
    rf, _, _ = P.solve(s0, dom, ext, lwl=lwl, method="rk4", n_steps=2 * (n - 1), early_exit=False)
    assert np.isfinite(rf).all(axis=0).sum() > 0.9 * s0.shape[1]
    sh = D.Shadowgraphy(lwl, rf)
    sh.single_lens_solve()
    sh.histogram(bin_scale=10)
    assert np.isfinite(sh.H).all() and 0.5 * s0.shape[1] < sh.H.sum() <= s0.shape[1]


@pytest.mark.gpu
def test_philox_spectrum_identical_on_two_gpus():
    """The noise is a function of (seed, index) only: H on cuda:1 is bit-identical to H on cuda:0."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from synthpy_b200 import engine
    shape = (64, 64, 63)
    out = []
    for dev in ("cuda:0", "cuda:1"):
        S = _half_S(shape, dev)
        Hd = engine.noise_spectrum(S, shape, 77)
        assert Hd.device == torch.device(dev)
        out.append(Hd.cpu())
    assert torch.equal(out[0], out[1])
