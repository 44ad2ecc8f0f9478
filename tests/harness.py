"""ctypes loader of tests/host_harness.cpp (CPU self-test build of the product's per-ray math)."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "_build", "libhost_harness.so")
SRC = os.path.join(HERE, "host_harness.cpp")
DEPS = [SRC, os.path.join(HERE, "..", "synthpy_b200", "csrc", "ray_core.h"),
        os.path.join(HERE, "..", "synthpy_b200", "csrc", "field_prep.h"),
        os.path.join(HERE, "..", "synthpy_b200", "csrc", "fresnel_core.h"),
        os.path.join(HERE, "..", "synthpy_b200", "csrc", "noise_core.h")]

OPK = {"travel": 0, "travel_noE": 1, "lens": 2, "circ_ap": 3, "circ_stop": 4, "rect_ap": 5, "knife": 6, "ref_beam": 7}


def build():
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    if os.path.exists(SO) and all(os.path.getmtime(SO) >= os.path.getmtime(d) for d in DEPS):
        return SO
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", SRC, "-o", SO], check=True)
    return SO


class HOp(C.Structure):
    _fields_ = [("kind", C.c_int32), ("pad", C.c_int32), ("p0", C.c_double), ("p1", C.c_double), ("p2", C.c_double)]


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class Harness:
    def __init__(self):
        self.lib = C.CDLL(build())
        self.lib.hh_field_create.restype = C.c_void_p

    def field(self, ne, x, y, z, omega, march_axis=2, phase=False, f64=False):
        ne = np.ascontiguousarray(ne, dtype=np.float64)
        ax = [np.ascontiguousarray(np.float32(a)) for a in (x, y, z)]
        h = self.lib.hh_field_create(_p(ne), _p(ax[0]), _p(ax[1]), _p(ax[2]), C.c_int(len(ax[0])), C.c_int(len(ax[1])),
                                     C.c_int(len(ax[2])), C.c_double(omega), C.c_int(march_axis),
                                     C.c_int((1 if phase else 0) | (2 if f64 else 0)))
        assert h
        return HField(self, C.c_void_p(h), ne.shape, omega, phase, f64)

    def optics(self, rf, ops, jf=None, wavelength=0.0, input_mm=False):
        rf = np.ascontiguousarray(rf, dtype=np.float64)
        n = rf.shape[1]
        arr = (HOp * max(1, len(ops)))()
        for i, op in enumerate(ops):
            v = list(op[1:]) + [0.0] * (4 - len(op))
            arr[i] = HOp(OPK[op[0]], 0, float(v[0]), float(v[1]), float(v[2]))
        out = np.empty_like(rf)
        jo = None
        if jf is not None:
            jf = np.ascontiguousarray(jf, dtype=np.complex128)
            jo = np.empty_like(jf)
        self.lib.hh_optics(_p(rf), _p(jf), C.c_uint64(n), arr, C.c_int(len(ops)), C.c_double(wavelength),
                           C.c_int(int(input_mm)), _p(out), _p(jo))
        return (out, jo) if jf is not None else out

    def bins(self, v, lo, hi, nb, right_inclusive):
        v = np.ascontiguousarray(v, dtype=np.float64)
        out = np.empty(v.shape, dtype=np.int32)
        self.lib.hh_bin(_p(v), C.c_uint64(v.size), C.c_double(lo), C.c_double(hi), C.c_int(nb), C.c_int(int(right_inclusive)),
                        _p(out))
        return out

    def beam(self, beam_type, probing_axis, size_a, size_b, divergence, start, seed, off, n):
        s0 = np.empty((9, n))
        self.lib.hh_beam(C.c_int(beam_type), C.c_int(probing_axis), C.c_double(size_a), C.c_double(size_b),
                         C.c_double(divergence), C.c_double(start), C.c_uint64(seed), C.c_uint64(off), C.c_uint64(n), _p(s0))
        return s0

    def philox(self, key, ctr):
        out = np.empty(4, dtype=np.uint32)
        self.lib.hh_philox(*(C.c_uint32(k) for k in key), *(C.c_uint32(c) for c in ctr), _p(out))
        return out

    def noise_full(self, shape, seed):
        """Z of the turbulent-field noise at every full-grid index: complex128 of ``shape``."""
        out = np.empty(shape, dtype=np.complex128)
        self.lib.hh_noise_full(*(C.c_int(n) for n in shape), C.c_uint64(seed), _p(out))
        return out

    def noise_half(self, S, shape, seed):
        """The half spectrum k_noise_spectrum writes: complex128 (n0, n1, n2 // 2 + 1) from float32 S of that shape."""
        n0, n1, n2 = shape
        S = np.ascontiguousarray(S, dtype=np.float32)
        assert S.shape == (n0, n1, n2 // 2 + 1)
        out = np.empty(S.shape, dtype=np.complex128)
        self.lib.hh_noise_half(_p(S), *(C.c_int(n) for n in shape), C.c_uint64(seed), _p(out))
        return out

    def noise_box(self, S, shape, order, lo, cnt, seed):
        """The box k_noise_spectrum_box writes: complex128 of shape (cnt[order[0]], cnt[order[1]], cnt[order[2]]) from
        float32 S of that shape; lo, cnt per grid axis."""
        S = np.ascontiguousarray(S, dtype=np.float32)
        assert S.shape == tuple(cnt[o] for o in order)
        ints = lambda v: (C.c_int * 3)(*(int(x) for x in v))
        out = np.empty(S.shape, dtype=np.complex128)
        self.lib.hh_noise_box(_p(S), *(C.c_int(n) for n in shape), ints(order), ints(lo), ints(cnt), C.c_uint64(seed),
                              _p(out))
        return out


class Fresnel:
    """The wave-optics kernels' per-sample code (fresnel_core.h) run serially on the host; FFT by NumPy."""

    def __init__(self, H):
        self.lib = H.lib

    def scatter_to_grid(self, px, py, values, tri, gx, gy, fill=0.0):
        px, py, gx, gy = (np.ascontiguousarray(a, dtype=np.float64) for a in (px, py, gx, gy))
        vals = np.ascontiguousarray(np.stack(values), dtype=np.float64)
        tri = np.ascontiguousarray(tri, dtype=np.int32)
        out = np.empty((vals.shape[0], len(gy), len(gx)))
        self.lib.hh_scatter_to_grid(_p(px), _p(py), _p(vals), C.c_int(vals.shape[0]), C.c_uint64(len(px)), _p(tri),
                                    C.c_uint64(len(tri)), _p(gx), _p(gy), C.c_int(len(gx)), C.c_int(len(gy)), C.c_double(fill), _p(out))
        return out

    def prepare(self, a, b=None, pad=2, alpha=0.4):
        mode = 0 if b is None else 1
        a = np.ascontiguousarray(a, dtype=np.complex128 if mode == 0 else np.float64)
        b = None if b is None else np.ascontiguousarray(b, dtype=np.float64)
        n0, n1 = a.shape
        out = np.empty(((2 * pad + 1) * n0, (2 * pad + 1) * n1), dtype=np.complex128)
        self.lib.hh_fresnel_prepare(_p(a), _p(b), C.c_int(mode), C.c_int(n0), C.c_int(n1), C.c_int(pad), C.c_double(alpha), _p(out))
        return out

    def propagate(self, prepared, L, wavelength, z, original_shape, pad=2, sigma=0.0):
        n0, n1 = original_shape
        spec = np.ascontiguousarray(np.fft.fft2(prepared))
        self.lib.hh_fresnel_transfer(_p(spec), C.c_int(spec.shape[0]), C.c_int(spec.shape[1]), C.c_double(L[0] / n0),
                                     C.c_double(L[1] / n1), C.c_double(wavelength), C.c_double(z), C.c_double(sigma))
        back = np.fft.ifft2(spec)
        scale = np.exp(1j * (2 * np.pi / wavelength) * z) / (1j * wavelength * z)
        return back[pad * n0:(pad + 1) * n0, pad * n1:(pad + 1) * n1] * scale

    def window(self, M, alpha):
        w = np.empty(M)
        self.lib.hh_window(C.c_int(M), C.c_double(alpha), _p(w))
        return w

    def reflect(self, n, lo, hi):
        out = np.empty(hi - lo, dtype=np.int32)
        self.lib.hh_reflect(C.c_int(n), C.c_int(lo), C.c_int(hi), _p(out))
        return out


class HField:
    def __init__(self, H, h, shape, omega, phase, f64):
        self.H, self.h, self.shape, self.omega, self.phase, self.f64 = H, h, shape, omega, phase, f64

    def __del__(self):
        self.H.lib.hh_field_destroy(self.h)

    def attach(self, kappa, ne, B):
        self._ext = [np.ascontiguousarray(a, dtype=np.float64) for a in (kappa, ne, B[..., 0], B[..., 1], B[..., 2])]
        self.H.lib.hh_attach(self.h, *[_p(a) for a in self._ext])

    def rhs_ext(self, s, verdet):
        s = np.ascontiguousarray(s, dtype=np.float64)
        out = np.empty_like(s)
        self.H.lib.hh_rhs_ext(self.h, _p(s), C.c_uint64(s.shape[1]), _p(out), C.c_double(self.omega), C.c_double(verdet))
        return out

    def rk4_ext(self, s0, n_steps, h, verdet, early=False):
        s0 = np.ascontiguousarray(s0, dtype=np.float64)
        sf = np.empty_like(s0)
        self.H.lib.hh_rk4_ext(self.h, _p(s0), C.c_uint64(s0.shape[1]), C.c_int(n_steps), C.c_double(h), C.c_double(self.omega),
                              C.c_double(verdet), C.c_int(int(early)), _p(sf))
        return sf

    def rk45_ext(self, s0, t_end, verdet, rtol=1e-3, atol=1e-6):
        s0 = np.ascontiguousarray(s0, dtype=np.float64)
        sf = np.empty_like(s0)
        nfev = np.empty(s0.shape[1], dtype=np.uint32)
        self.H.lib.hh_rk45_ext(self.h, _p(s0), C.c_uint64(s0.shape[1]), C.c_double(t_end), C.c_double(rtol), C.c_double(atol),
                               C.c_double(self.omega), C.c_double(verdet), _p(sf), _p(nfev))
        return sf, nfev

    def export(self):
        outs = [np.empty(self.shape, dtype=np.float32) for _ in range(4)]
        self.H.lib.hh_field_export(self.h, *[_p(o) for o in outs])
        return outs

    def rhs(self, s, aux64=None):
        s = np.ascontiguousarray(s, dtype=np.float64)
        out = np.empty_like(s)
        self.H.lib.hh_rhs(self.h, _p(s), C.c_uint64(s.shape[1]), _p(out), C.c_double(self.omega), C.c_int(int(self.phase)),
                          C.c_int(int(self.f64 if aux64 is None else aux64)))
        return out

    def rhs_direct(self, s):
        s = np.ascontiguousarray(s, dtype=np.float64)
        out = np.empty_like(s)
        self.H.lib.hh_rhs_direct(self.h, _p(s), C.c_uint64(s.shape[1]), _p(out), C.c_double(self.omega), C.c_int(int(self.phase)),
                                 C.c_int(int(self.f64)))
        return out

    def rhs_walk(self, s, near):
        s = np.ascontiguousarray(s, dtype=np.float64)
        out = np.empty_like(s)
        self.H.lib.hh_rhs_walk(self.h, _p(s), C.c_uint64(s.shape[1]), _p(out), C.c_int(int(near)))
        return out

    def rk4(self, s0, n_steps, h, early=False, fp32=False, aux64=None):
        s0 = np.ascontiguousarray(s0, dtype=np.float64)
        sf = np.empty_like(s0)
        steps = np.empty(s0.shape[1], dtype=np.uint32)
        self.H.lib.hh_rk4(self.h, _p(s0), C.c_uint64(s0.shape[1]), C.c_int(n_steps), C.c_double(h), C.c_double(self.omega),
                          C.c_int(int(self.phase)), C.c_int(int(self.f64 if aux64 is None else aux64)), C.c_int(int(early)),
                          C.c_int(int(fp32)), _p(sf), _p(steps))
        return sf, steps

    def rk45(self, s0, t_end, rtol=1e-3, atol=1e-6, n_state=9, cap=0, aux64=None):
        s0 = np.ascontiguousarray(s0, dtype=np.float64)
        sf = np.empty_like(s0)
        att = np.empty(s0.shape[1], dtype=np.uint32)
        nfev = np.empty(s0.shape[1], dtype=np.uint32)
        self.H.lib.hh_rk45(self.h, _p(s0), C.c_uint64(s0.shape[1]), C.c_double(t_end), C.c_double(rtol), C.c_double(atol),
                           C.c_double(self.omega), C.c_int(int(self.phase)), C.c_int(int(self.f64 if aux64 is None else aux64)),
                           C.c_int(n_state), C.c_int(cap), _p(sf), _p(att), _p(nfev))
        return sf, att, nfev

    def tsit5(self, s0, T_norm, dt0, rtol=1.0, atol=1e-5, n_state=9, cap=0, aux64=None):
        s0 = np.ascontiguousarray(s0, dtype=np.float64)
        sf = np.empty_like(s0)
        att = np.empty(s0.shape[1], dtype=np.uint32)
        acc = np.empty(s0.shape[1], dtype=np.uint32)
        self.H.lib.hh_tsit5(self.h, _p(s0), C.c_uint64(s0.shape[1]), C.c_double(T_norm), C.c_double(dt0), C.c_double(rtol),
                            C.c_double(atol), C.c_double(self.omega), C.c_int(int(self.phase)),
                            C.c_int(int(self.f64 if aux64 is None else aux64)), C.c_int(n_state), C.c_int(cap), _p(sf), _p(att), _p(acc))
        return sf, att, acc

    def exit(self, sf, p, a, b, extent):
        sf = np.ascontiguousarray(sf, dtype=np.float64)
        rf = np.empty((4, sf.shape[1]))
        self.H.lib.hh_exit(self.h, _p(sf), C.c_uint64(sf.shape[1]), C.c_int(p), C.c_int(a), C.c_int(b), C.c_double(extent), _p(rf))
        return rf
