"""Band-limited Gaussian random field on the GPU: restates ``gaussian3D.domain_fft``
(reference: src/field_generator/gaussian3D.py:215-271) so that 512^3 / 1024^3 turbulent n_e grids can be built
where they are used (SURVEY.md 8f-1).  Input producer for the ray path, not part of it; torch.fft is the
library FFT here (plumbing), the ray kernels are in csrc/.

noise='numpy' draws the complex noise with NumPy's legacy global RNG in the reference's order (same field as
the reference for the same ``np.random.seed``): the parity path.  noise='torch' draws it with torch's (multi-threaded)
CPU generator -- fast enough for 1024^3, but the noise (16 bytes per grid point) lives in host memory and is copied to
the device.

noise='philox' draws nothing on the host.  The library's ``k_noise_spectrum`` makes the noise at every grid index from
(seed, index) with Philox4x32-10 and writes the Hermitian half spectrum sqrt(S) (Z(k) + conj Z(-k)) / 2 directly;
``torch.fft.irfftn`` of it is Re ifftn(Z sqrt(S)), the reference's expression.  The field is a function of the seed
alone (any GPU, any launch), its distribution is the reference's, its noise stream is not (no seed reproduces a NumPy or
torch realisation).  It needs no host memory or host-to-device copy of grid size, half the spectrum memory of the
other modes and a real inverse FFT, run slab by slab: 17.5 bytes per grid point at the peak (the half spectrum, the
field and one slab of FFT temporaries) against 60 (measured on a B200 at 512^3 and 1024^3).  CUDA only.

domain_fft_slabs / turbulent_ne_slabs make the same philox field as a slab source for out_of_core.solve_out_of_core,
for grids (2048^3) where the generator and the tracer cannot both hold a grid-sized field: ``k_noise_spectrum_box``
writes H straight into one complex array of about 8 bytes per grid point with the Hermitian half along an axis other
than the probing one, and every slab is inverse-transformed from it when asked for.  CUDA only.
"""
import numpy as np
import torch


def domain_fft(k_func, l_max, l_min, extent, res, factor=1, *, noise="numpy", seed=0, device="cuda"):
    """Returns the (2res, 2res, int(2res*factor)) field as a float64 torch tensor on ``device``, normalised to
    max |f| = 1.  k_func maps a float32 torch tensor of |k| to the power spectrum."""
    k_axes = _k_axes(extent, res, factor)
    dev = torch.device(device)
    if noise == "philox":
        return _philox_field(k_func, l_max, l_min, k_axes, seed, dev)
    kx, _, kz = k_axes
    kxt, kzt = torch.from_numpy(kx).to(dev), torch.from_numpy(kz).to(dev)
    # np.meshgrid(kx, ky, kz) uses 'xy' indexing: axis 0 <- ky, axis 1 <- kx   (gaussian3D.py:238)
    k2 = kxt[None, :, None] ** 2 + kxt[:, None, None] ** 2 + kzt[None, None, :] ** 2
    k = torch.sqrt(k2.to(torch.float32))                       # np.sqrt(..., dtype=np.float32)
    del k2
    k_min, k_max = 2 * np.pi / l_max, 2 * np.pi / l_min
    mask = (k >= k_min) & (k <= k_max)
    S = torch.zeros_like(k)
    S[mask] = k_func(k[mask])
    del mask, k
    shape = (len(kx), len(kx), len(kz))                        # (ny, nx, nz)
    if noise == "numpy":
        re = torch.from_numpy(np.random.normal(0, 1, shape)).to(dev)
        im = torch.from_numpy(np.random.normal(0, 1, shape)).to(dev)
    else:
        # drawn with torch's CPU generator so that the realisation does not depend on where the FFT runs
        gen = torch.Generator(device="cpu").manual_seed(int(seed))
        re = torch.randn(shape, generator=gen, dtype=torch.float64).to(dev)
        im = torch.randn(shape, generator=gen, dtype=torch.float64).to(dev)
    spec = torch.complex(re, im) * torch.sqrt(S).to(torch.float64)
    del re, im, S
    field = torch.fft.ifftn(spec).real
    del spec
    return field / field.abs().max()


def _k_axes(extent, res, factor):
    """The 2 pi fftfreq axes (kx, ky, kz) of domain_fft's (2res, 2res, int(2res * factor)) grid, spacing extent / res."""
    dx = extent / res
    kx = 2 * np.pi * np.fft.fftfreq(2 * res, d=dx)
    return kx, kx, 2 * np.pi * np.fft.fftfreq(int(2 * res * factor), d=dx)


def half_spectrum(k_func, l_max, l_min, k_axes, device="cuda"):
    """The power spectrum S on the half grid of a (n0, n1, n2) grid as a float32 tensor (n0, n1, n2 // 2 + 1).
    k_axes = (k0, k1, k2): the 2 pi fftfreq arrays of the three axes (domain_fft: (kx, kx, kz)).  Same float32 |k|
    expression as domain_fft, so the result equals its S[..., : n2 // 2 + 1] element for element.  k_func is evaluated on
    every |k| and kept inside the band only (no index list of the band is built)."""
    n0, n1, n2 = (len(k) for k in k_axes)
    return spectrum_box(k_func, l_max, l_min, k_axes, (0, 1, 2), (0, 0, 0), (n0, n1, n2 // 2 + 1), device)


def spectrum_box(k_func, l_max, l_min, k_axes, order, lo, cnt, device="cuda"):
    """The power spectrum S on the box [lo, lo + cnt) (per grid axis) of the grid of ``k_axes``, stored with box axis t
    along grid axis order[t]: a float32 tensor (cnt[order[0]], cnt[order[1]], cnt[order[2]]), the layout
    ``engine.noise_spectrum_box`` reads.  Every element is the one ``half_spectrum`` / domain_fft computes at that grid
    index, bit for bit: the float32 |k| of (k1^2 + k0^2) + k2^2 in that order whatever the box order is."""
    kt = []
    for a in range(3):
        v = torch.from_numpy(np.ascontiguousarray(k_axes[a][lo[a]: lo[a] + cnt[a]])).to(device)
        view = [1, 1, 1]
        view[list(order).index(a)] = int(cnt[a])
        kt.append(v.view(view))
    ksq = kt[1] ** 2 + kt[0] ** 2 + kt[2] ** 2
    k = torch.sqrt(ksq.to(torch.float32))
    del ksq
    k_min, k_max = 2 * np.pi / l_max, 2 * np.pi / l_min
    mask = (k >= k_min) & (k <= k_max)
    S = k_func(k).to(torch.float32)                            # domain_fft stores k_func's values in a float32 S
    del k
    return S.masked_fill_(~mask, 0.0)


def _philox_field(k_func, l_max, l_min, k_axes, seed, dev):
    if dev.type != "cuda":
        raise RuntimeError("noise='philox' is generated by a CUDA kernel and has no CPU path: use device='cuda' "
                           "(or noise='torch' / 'numpy' on the CPU)")
    from . import engine
    shape = tuple(len(k) for k in k_axes)
    S = half_spectrum(k_func, l_max, l_min, k_axes, dev)
    H = engine.noise_spectrum(S, shape, seed)
    del S
    field = _irfftn_slabs(H, shape)
    del H
    return field.div_(torch.maximum(field.max(), -field.min()))     # max |f| without a grid-sized |f|


def _irfftn_slabs(H, shape, slabs=16):
    """torch.fft.irfftn(H, s=shape) holding only H and the output at grid size.  One irfftn call keeps about four
    H-sized buffers alive at once (its input, a permuted copy, the inverse C2C's output and the output field).  Here
    the inverse C2C over axes 0 and 1 overwrites H one slab of axis 2 at a time, then the C2R along axis 2 writes the
    field one slab of axis 0 at a time, so every FFT temporary is one slab."""
    n0, _, n2 = shape
    nh = H.shape[2]
    step = -(-nh // slabs)
    for a in range(0, nh, step):
        H[..., a:a + step] = torch.fft.ifftn(H[..., a:a + step], dim=(0, 1))
    field = torch.empty(shape, dtype=torch.float64, device=H.device)
    step = -(-n0 // slabs)
    for a in range(0, n0, step):
        torch.fft.irfft(H[a:a + step], n=n2, dim=2, out=field[a:a + step])
    return field


class _FieldSlabs:
    """Slab source of the field ``domain_fft(..., noise='philox')`` makes, for grids whose field does not fit in device
    memory next to what traces it (``out_of_core.solve_out_of_core``).  Only one complex array G of about 8 bytes per
    grid point is held, never the field.

    p is the probing axis, q the axis that carries the Hermitian half (2, or 1 when p == 2), r the third.  G is complex128
    [n_r][n_p][n_q // 2 + 1]: H (k_noise_spectrum_box) with the inverse FFT along p already done, built chunk by chunk of
    r at construction.  A block of planes [a, b) of p is then ifft along r and irfft along q of G[:, a:b, :].  Blocks sit
    on a fixed grid of ``block_planes`` planes, so the values of a plane do not depend on the window asked for.  The
    normalisation max |f| needs the whole field: construction runs over every block once and keeps only the maximum.

    ``noise_box`` writes H for a box (engine.noise_spectrum_box's signature); tests substitute the host build of the
    same source to run the decomposition on the CPU."""

    def __init__(self, k_func, l_max, l_min, k_axes, *, axis, seed, block_planes, device, noise_box, ne0=None, dne=None):
        from time import perf_counter
        self.shape = tuple(len(k) for k in k_axes)
        self.axis, self.block_planes = int(axis), int(block_planes)
        if self.axis not in (0, 1, 2) or self.block_planes < 1:
            raise ValueError("axis must be 0, 1 or 2 and block_planes >= 1")
        self._affine = None if ne0 is None else (ne0, dne)
        p = self.axis
        q = 2 if p != 2 else 1
        r = 3 - p - q
        self._order, self._q = (r, p, q), q
        n_r, n_p, n_q = self.shape[r], self.shape[p], self.shape[q]
        nqh = n_q // 2 + 1
        self._G = torch.empty((n_r, n_p, nqh), dtype=torch.complex128, device=device)
        t0 = perf_counter()
        for c0 in range(0, n_r, self.block_planes):                                    # phase A
            c1 = min(n_r, c0 + self.block_planes)
            lo, cnt = [0, 0, 0], [0, 0, 0]
            lo[r], cnt[r], cnt[p], cnt[q] = c0, c1 - c0, n_p, nqh
            S = spectrum_box(k_func, l_max, l_min, k_axes, self._order, lo, cnt, device)
            noise_box(S, self.shape, self._order, lo, cnt, seed, out=self._G[c0:c1])
            del S
            self._G[c0:c1] = torch.fft.ifft(self._G[c0:c1], dim=1)
        self._sync()
        t1 = perf_counter()
        self._max, self._cache = None, None
        m = None
        for ib in range(self.n_blocks):                                                   # max pass
            f = self._raw_block(ib)
            b = torch.maximum(f.max(), -f.min())
            m = b if m is None else torch.maximum(m, b)
            del f
        self._max = m                          # 0-d device tensor: f / max is a true division, as in domain_fft
        self.max_abs = float(m)
        self.build_seconds = dict(phase_a=t1 - t0, max_pass=perf_counter() - t1)

    def _sync(self):
        if self._G.is_cuda:
            torch.cuda.synchronize(self._G.device)

    @property
    def n_blocks(self):
        return -(-self.shape[self.axis] // self.block_planes)

    def _raw_block(self, ib):
        """Unnormalised f on planes [ib * block_planes, ...) of p, in grid order."""
        a = ib * self.block_planes
        b = min(self.shape[self.axis], a + self.block_planes)
        T = torch.fft.ifft(self._G[:, a:b, :], dim=0)
        q = self._q
        f = torch.empty((T.shape[0], b - a, self.shape[q]), dtype=torch.float64, device=T.device)
        torch.fft.irfft(T, n=self.shape[q], dim=2, out=f)
        del T
        return f.permute([self._order.index(g) for g in range(3)]).contiguous()

    def _block(self, ib):
        if self._cache is not None and self._cache[0] == ib:
            return self._cache[1]
        self._cache = None                     # free the previous block before making the next
        f = self._raw_block(ib).div_(self._max)
        if self._affine is not None:
            f = self._affine[0] + self._affine[1] * f
        self._cache = (ib, f)
        return f

    def __call__(self, k0, k1):
        """Planes [k0, k1) of the probing axis, float64 in grid order on the device."""
        k0, k1, n = int(k0), int(k1), self.shape[self.axis]
        if not 0 <= k0 < k1 <= n:
            raise ValueError(f"planes [{k0}, {k1}) are not inside [0, {n})")
        bp, p = self.block_planes, self.axis
        shape = list(self.shape)
        shape[p] = k1 - k0
        out = torch.empty(shape, dtype=torch.float64, device=self._G.device)     # never the cached block itself
        for ib in range(k0 // bp, (k1 - 1) // bp + 1):
            a, b = max(k0, ib * bp), min(k1, (ib + 1) * bp)
            out.narrow(p, a - k0, b - a).copy_(self._block(ib).narrow(p, a - ib * bp, b - a))
        return out


def domain_fft_slabs(k_func, l_max, l_min, extent, res, factor=1, *, axis, seed, block_planes=64, device="cuda"):
    """The field of ``domain_fft(k_func, l_max, l_min, extent, res, factor, noise='philox', seed=seed)`` as a slab source
    ``source(k0, k1)`` -> planes [k0, k1) along grid axis ``axis`` (float64 CUDA tensor, normalised to max |f| = 1),
    without the field ever existing whole.  Equal to domain_fft's to FFT rounding (the inverse FFT is decomposed in
    another order); every plane is the same bits whatever window it is asked in.  ``source.shape`` is the grid,
    ``source.max_abs`` the normalisation, ``source.build_seconds`` the two construction passes.  Device memory: about 8
    bytes per grid point for the life of the source, plus a few blocks of ``block_planes`` planes.  CUDA only."""
    return _slabs(k_func, l_max, l_min, _k_axes(extent, res, factor), axis, seed, block_planes, device)


def _slabs(k_func, l_max, l_min, k_axes, axis, seed, block_planes, device, **kw):
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("out-of-core philox fields are generated by a CUDA kernel and have no CPU path: use "
                           "device='cuda'")
    from . import engine
    return _FieldSlabs(k_func, l_max, l_min, k_axes, axis=axis, seed=seed, block_planes=block_planes, device=dev,
                       noise_box=engine.noise_spectrum_box, **kw)


def kolmogorov(k):
    return k ** (-11.0 / 3.0)                                   # examples/.../turb_gen.py:36-50


def turbulent_ne(res, *, ne0=1e25, dne=9e24, l_max=1, l_min=0.01, extent=5, noise="torch", seed=1, device="cuda"):
    """ne = ne0 + dne * f with f the k^-11/3 field of ``domain_fft`` on a (2res)^3 grid (BASELINE config C2/C5)."""
    f = domain_fft(kolmogorov, l_max, l_min, extent, res, 1, noise=noise, seed=seed, device=device)
    return ne0 + dne * f


def turbulent_ne_slabs(res, *, probing_direction="z", ne0=1e25, dne=9e24, l_max=1, l_min=0.01, extent=5, seed=1,
                       block_planes=64, device="cuda"):
    """``turbulent_ne(res, noise='philox', seed=seed)`` as the slab source ``out_of_core.solve_out_of_core`` takes:
    ``source(k0, k1)`` is ne on planes [k0, k1) of the probing axis, float64 on the device, with nothing of grid size
    held but ``domain_fft_slabs``'s spectrum (about 8 bytes per point: 68.8 GB at 2048^3).  The values agree with
    turbulent_ne's to FFT rounding and are the same bits whatever window is asked for."""
    from . import engine
    return _slabs(kolmogorov, l_max, l_min, _k_axes(extent, res, 1), engine.AXIS[probing_direction], seed,
                  block_planes, device, ne0=ne0, dne=dne)
