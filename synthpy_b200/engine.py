"""Thin host-side engine over the C ABI: owns device buffers (as torch tensors) and handles, nothing else.

torch is used for buffer ownership, streams and (in ``distributed.py``) NCCL plumbing only; every
computation on the ray path is a kernel in ``csrc/synthpy_b200.cu`` reached through ``_lib``.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib as L

AXIS = {"x": 0, "y": 1, "z": 2}
C_LIGHT = 299792458.0          # scipy.constants.c, as used by the reference (full_solver.py:93)

OP_KINDS = {"travel": L.OP_TRAVEL, "travel_noE": L.OP_TRAVEL_NOE, "lens": L.OP_LENS, "circ_ap": L.OP_CIRC_AP,
            "circ_stop": L.OP_CIRC_STOP, "rect_ap": L.OP_RECT_AP, "knife": L.OP_KNIFE, "ref_beam": L.OP_REF_BEAM}
METHODS = {"rk4": L.METHOD_RK4, "rk45": L.METHOD_RK45, "rk45_joint": L.METHOD_RK45_JOINT, "rk45_bundle": L.METHOD_RK45,
           "tsit5": L.METHOD_TSIT5}
BEAM_TYPES = {"circular": L.BEAM_CIRCULAR_POW2, "circular_legacy": L.BEAM_CIRCULAR_FOLD, "square": L.BEAM_SQUARE,
              "rectangular": L.BEAM_RECTANGULAR, "rect_trackers": L.BEAM_RECTANGULAR, "linear": L.BEAM_LINEAR}


def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("synthpy_b200 needs a CUDA device: the hot path has no CPU fallback")


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def to_device(a, dtype=torch.float64):
    """numpy / torch -> contiguous CUDA tensor of ``dtype`` (no copy when already there)."""
    require_cuda()
    if isinstance(a, torch.Tensor):
        t = a
    else:
        t = torch.from_numpy(np.ascontiguousarray(a))
    return t.to(device="cuda", dtype=dtype).contiguous()


def kappa_grid(ne, Te, Z, omega):
    """Inverse-bremsstrahlung rate grid, NRL formulary as coded in the reference (ScalarDomain.kappa,
    src/solvers-legacy/full_solver.py:243-268; src/simulator/propagator.py:27-58).  Host NumPy float64: field
    preparation, evaluated once per domain like the analytic profiles."""
    e = 1.602176634e-19
    ne_cc = np.asarray(ne, dtype=np.float64) * 1e-6
    Te, Z = np.asarray(Te, dtype=np.float64), np.asarray(Z, dtype=np.float64)
    o_pe = 5.64e4 * np.sqrt(ne_cc)
    o_max = np.copy(o_pe)
    o_max[o_pe < omega] = omega
    L_max = np.maximum(Z * e / Te, 2.760428269727312e-10 / np.sqrt(Te))
    CL = np.maximum(2.0, np.log(4.19e5 * np.sqrt(Te) / (o_max * L_max)))
    return 3.1e-5 * Z * C_LIGHT * np.power(ne_cc / omega, 2) * CL * np.power(Te, -1.5)


def omega_of(lwl):
    return 2 * np.pi * (C_LIGHT / lwl)          # full_solver.py:218, propagator.py:357


def critical_density(omega):
    """n_c in m^-3 as the reference writes it (full_solver.py:220)."""
    return 3.14207787e-4 * omega ** 2


class DeviceField:
    """Owner of an ``sp_field`` handle (packed float4 grid + axis tables in HBM)."""

    def __init__(self, handle, shape, march_axis, has_phase, has_f64):
        self._h = handle
        self.shape, self.march_axis, self.has_phase, self.has_f64 = tuple(shape), march_axis, has_phase, has_f64

    @classmethod
    def from_ne(cls, ne, x, y, z, omega, march_axis=2, phase=False, phase_f64=False):
        """ne: (nx,ny,nz) numpy/torch, float64 or float32; x,y,z: coordinate axes (rounded to float32 here,
        full_solver.py:119 / domain.py:230-232)."""
        require_cuda()
        ax = [np.ascontiguousarray(np.float32(a)) for a in (x, y, z)]
        is64 = (ne.dtype in (np.float64, torch.float64))
        ne_d = to_device(ne, torch.float64 if is64 else torch.float32)
        if tuple(ne_d.shape) != tuple(len(a) for a in ax):
            raise ValueError(f"ne shape {tuple(ne_d.shape)} does not match axes {[len(a) for a in ax]}")
        flags = (L.FIELD_PHASE if phase else 0) | (L.FIELD_PHASE_F64 if phase_f64 else 0)
        h = C.c_void_p()
        L.check(L.lib.sp_field_create(C.byref(h), _ptr(ne_d), int(is64), ax[0].ctypes.data, ax[1].ctypes.data,
                                      ax[2].ctypes.data, len(ax[0]), len(ax[1]), len(ax[2]), float(omega),
                                      int(march_axis), flags, _stream()))
        return cls(h, ne_d.shape, march_axis, phase or phase_f64, phase_f64)

    @classmethod
    def from_gradients(cls, gx, gy, gz, x, y, z, march_axis=2, aux32=None, aux64=None):
        require_cuda()
        ax = [np.ascontiguousarray(np.float32(a)) for a in (x, y, z)]
        g = [to_device(a, torch.float32) for a in (gx, gy, gz)]
        a32 = None if aux32 is None else to_device(aux32, torch.float32)
        a64 = None if aux64 is None else to_device(aux64, torch.float64)
        h = C.c_void_p()
        L.check(L.lib.sp_field_create_from_gradients(C.byref(h), _ptr(g[0]), _ptr(g[1]), _ptr(g[2]), _ptr(a32),
                                                     _ptr(a64), ax[0].ctypes.data, ax[1].ctypes.data,
                                                     ax[2].ctypes.data, len(ax[0]), len(ax[1]), len(ax[2]),
                                                     int(march_axis), _stream()))
        torch.cuda.current_stream().synchronize()       # inputs may be temporaries
        return cls(h, g[0].shape, march_axis, a32 is not None or a64 is not None, a64 is not None)

    def attach_channels(self, kappa=None, ne=None, B=None):
        """Attenuation / Faraday grids (float64, (nx,ny,nz); B is (nx,ny,nz,3)): see sp_field_attach_channels."""
        k = None if kappa is None else to_device(kappa)
        n = None if ne is None else to_device(ne)
        b = [None] * 3 if B is None else [to_device(B[..., c]) for c in range(3)]
        L.check(L.lib.sp_field_attach_channels(self._h, _ptr(k), _ptr(n), _ptr(b[0]), _ptr(b[1]), _ptr(b[2]), _stream()))
        torch.cuda.current_stream().synchronize()
        self.has_kappa, self.has_faraday = k is not None, (n is not None and B is not None)

    def export_gradients(self):
        outs = [torch.empty(self.shape, dtype=torch.float32, device="cuda") for _ in range(4)]
        L.check(L.lib.sp_field_export_gradients(self._h, *[_ptr(o) for o in outs], _stream()))
        return outs

    @property
    def nbytes(self):
        return int(L.lib.sp_field_bytes(self._h))

    def close(self):
        if self._h is not None and self._h.value:
            L.lib.sp_field_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_workspaces = {}


def workspace():
    """The ``sp_workspace`` of the current (device, stream).  A workspace holds the bundle dispenser, the sort scratch and
    the joint-solve buffers of the launches in flight, so two streams (or threads with their own streams) must never
    share one: each (device, stream) pair gets its own, created on first use."""
    require_cuda()
    key = (torch.cuda.current_device(), int(torch.cuda.current_stream().cuda_stream))
    if key not in _workspaces:
        h = C.c_void_p()
        L.check(L.lib.sp_workspace_create(C.byref(h)))
        _workspaces[key] = h
    return _workspaces[key]


def propagate_kernel_ms():
    """(total ms, launches) of the k_propagate launches since the last call -- CUDA events on the launch stream."""
    ms, n = C.c_double(), C.c_int()
    L.check(L.lib.sp_workspace_propagate_ms(workspace(), C.byref(ms), C.byref(n)))
    return ms.value, n.value


def fp64_peak(iters=20000, repeats=5):
    """Measured FP64 FMA peak of the current GPU in TFLOP/s (2 flops per DFMA): best of ``repeats`` launches of the
    library's DFMA microbenchmark, CUDA-event timed.  bench.py's roofline denominator for the integrator."""
    require_cuda()
    out = torch.empty(148 * 8 * 256 * 2, dtype=torch.float64, device="cuda")
    n = C.c_uint64()
    best = None
    for _ in range(repeats + 1):                                 # first launch = warm-up
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        L.check(L.lib.sp_fp64_peak(int(iters), _ptr(out), out.numel(), C.byref(n), _stream()))
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1)
        best = ms if best is None else min(best, ms)
    return 2.0 * n.value / (best * 1e-3) / 1e12


def joint_log():
    """(h, error_norm) arrays of every attempted step of the last 'rk45_joint' solve."""
    n = C.c_int()
    L.check(L.lib.sp_workspace_joint_log(workspace(), None, None, 0, C.byref(n)))
    h, en = np.empty(n.value), np.empty(n.value)
    L.check(L.lib.sp_workspace_joint_log(workspace(), h.ctypes.data, en.ctypes.data, n.value, C.byref(n)))
    return h, en


def make_params(method="rk4", *, probing_direction="z", extent, omega, n_steps=0, h=0.0, t_end=None, rtol=1e-3,
                atol=1e-6, phase=False, phase_f64=False, early_exit=True, fp32=False, sort=True, n_state=9,
                out_axes=None, atten=False, faraday=False, verdet=0.0):
    p = AXIS[probing_direction]
    if out_axes is None:
        # legacy ray_to_Jonesvector conventions (full_solver.py:856-881): x->(y,z), y->(x,z), z->(x,y)
        out_axes = {0: (1, 2), 1: (0, 2), 2: (0, 1)}[p]
    flags = ((L.FLAG_PHASE if phase else 0) | (L.FLAG_PHASE_F64 if (phase and phase_f64) else 0) |
             (L.FLAG_EARLY_EXIT if early_exit else 0) | (L.FLAG_FP32 if fp32 else 0) | (0 if sort else L.FLAG_NO_SORT) |
             (L.FLAG_ATTEN if atten else 0) | (L.FLAG_FARADAY if faraday else 0) |
             (L.FLAG_BUNDLE_STEP if method == "rk45_bundle" else 0))
    if t_end is None:
        t_end = np.sqrt(8.0) * extent / C_LIGHT       # full_solver.py:381, propagator.py:454
    return L.Params(method=METHODS[method], flags=flags, n_steps=int(n_steps), n_state=int(n_state), h=float(h),
                    t_end=float(t_end), rtol=float(rtol), atol=float(atol), omega=float(omega), extent=float(extent),
                    probing_axis=p, out_axis_a=out_axes[0], out_axis_b=out_axes[1], verdet=float(verdet))


def make_beam(beam_type, size, divergence, ne_extent, probing_direction="z", seed=0):
    if isinstance(beam_type, str):
        beam_type = BEAM_TYPES[beam_type]
    if np.ndim(size) == 0:
        sa = sb = float(size)
    else:
        sa, sb = float(size[0]), float(size[1])
    return L.Beam(beam_type=beam_type, probing_axis=AXIS[probing_direction], size_a=sa, size_b=sb,
                  divergence=float(divergence), start=-float(ne_extent), seed=int(seed))


IMAGE_KINDS = {"histogram": L.IMG_HISTOGRAM, "interferogram": L.IMG_INTERFEROGRAM, "stokes": L.IMG_STOKES}


class ImageBuffer:
    """Detector image accumulator in HBM.  ``kind`` 'histogram' -> uint64 counts (np.histogram2d semantics),
    'interferogram' -> four int64 fixed-point planes (2^-40 units) of summed complex E (digitize semantics), 'stokes' ->
    int64 ray count plus Stokes I, Q, U of the rays' Jones vectors in fixed point (2^-32 units; histogram semantics):
    integer sums are exact, so the image is identical from run to run and for any partition of the rays over GPUs."""

    def __init__(self, kind, nx, ny, x_range, y_range):
        require_cuda()
        self.kind, self.nx, self.ny = kind, int(nx), int(ny)
        self.x_range, self.y_range = (float(x_range[0]), float(x_range[1])), (float(y_range[0]), float(y_range[1]))
        self.counts = self.planes = None
        self._global = None            # sum over ranks attached by distributed.combine_images (out of place)
        if kind == "histogram":
            self.counts = torch.zeros((self.ny, self.nx), dtype=torch.int64, device="cuda")
        elif kind in ("interferogram", "stokes"):
            self.planes = torch.zeros((4, self.ny, self.nx), dtype=torch.int64, device="cuda")
        else:
            raise ValueError(kind)

    @classmethod
    def for_histogram(cls, bin_scale=1, pix_x=3448, pix_y=2574, Lx=18, Ly=13.5):
        # diagnostics.py:349 / rtm_solver.py:170-172
        return cls("histogram", pix_x // bin_scale, pix_y // bin_scale, (-Lx / 2, Lx / 2), (-Ly / 2, Ly / 2))

    @classmethod
    def for_interferogram(cls, bin_scale=1, pix_x=3448, pix_y=2574, Lx=18, Ly=13.5):
        # diagnostics.py:362-363 / rtm_solver.py:436-437: edges linspace(-Lx//2, Lx//2, pix//bs)  (floor division!)
        return cls("interferogram", pix_x // bin_scale - 1, pix_y // bin_scale - 1, (-Lx // 2, Lx // 2),
                   (-Ly // 2, Ly // 2))

    @classmethod
    def for_stokes(cls, bin_scale=1, pix_x=3448, pix_y=2574, Lx=18, Ly=13.5):
        # the histogram's edges: np.histogram2d(..., weights=) of I, Q, U is the image
        return cls("stokes", pix_x // bin_scale, pix_y // bin_scale, (-Lx / 2, Lx / 2), (-Ly / 2, Ly / 2))

    def struct(self):
        return L.Image(kind=IMAGE_KINDS[self.kind], nx=self.nx,
                       ny=self.ny, x_lo=self.x_range[0], x_hi=self.x_range[1], y_lo=self.y_range[0],
                       y_hi=self.y_range[1], counts_dev=None if self.counts is None else self.counts.data_ptr(),
                       planes_dev=None if self.planes is None else self.planes.data_ptr())

    def zero_(self):
        (self.counts if self.counts is not None else self.planes).zero_()
        self._global = None

    def tensors(self):
        """This rank's accumulator (what the kernels add to)."""
        return [self.counts] if self.counts is not None else [self.planes]

    def set_global(self, tensors):
        """Attach (or drop, with None) the sum over ranks; see distributed.combine_images."""
        self._global = None if tensors is None else tensors[0]

    def touched(self):
        """The accumulator is about to change: a previously attached global sum no longer describes it."""
        self._global = None

    def total(self):
        """The global image if one is attached (after combine_images), else this rank's accumulator."""
        return self._global if self._global is not None else self.tensors()[0]

    def result(self):
        """H as the reference returns it: float64 counts (ny, nx), or sqrt(Re(sum Ex)^2 + Re(sum Ey)^2); for a Stokes
        image the intensity I (ny, nx), i.e. the attenuation-weighted shadowgram."""
        if self.counts is not None:
            return self.total().to(torch.float64)
        if self.kind == "stokes":
            return self.stokes()["I"]
        return self._finalize((self.ny, self.nx))

    def stokes(self):
        """Stokes image as float64 (ny, nx) tensors: {'N': ray count, 'I', 'Q', 'U'} (include/synthpy_b200.h SP_IMG_STOKES)."""
        if self.kind != "stokes":
            raise ValueError(f"stokes() needs a 'stokes' image, this one is '{self.kind}'")
        H = self._finalize((4, self.ny, self.nx))
        return dict(zip("NIQU", H.unbind(0)))

    def _finalize(self, shape):
        H = torch.empty(shape, dtype=torch.float64, device="cuda")
        img = self.struct()
        img.planes_dev = self.total().data_ptr()
        L.check(L.lib.sp_image_finalize(C.byref(img), _ptr(H), _stream()))
        return H


def _null_image():
    return L.Image(kind=L.IMG_HISTOGRAM, nx=0, ny=0)


def make_channel(ops, image=None, wavelength=0.0, input_mm=False):
    """ops: list of (kind, params...) tuples, e.g. [("travel", 300.0), ("circ_ap", 25), ...].
    Returns (Channel struct, keepalive)."""
    arr = (L.OpticOp * max(1, len(ops)))()
    for i, op in enumerate(ops):
        vals = list(op[1:]) + [0.0] * (4 - len(op))
        arr[i] = L.OpticOp(kind=OP_KINDS[op[0]], p0=float(vals[0]), p1=float(vals[1]), p2=float(vals[2]))
    ch = L.Channel(ops_host=arr, n_ops=len(ops), input_mm=int(bool(input_mm)), wavelength=float(wavelength or 0.0),
                   image=image.struct() if image is not None else _null_image())
    return ch, (arr, image)


def propagate(field, params, *, s0=None, beam=None, n=None, ray_offset=0, want_sf=False, want_rf=True,
              want_jf=False, want_steps=False, channels=(), with_stats=True):
    """One call of ``sp_propagate``.  s0: (9,N) CUDA float64 tensor, or ``beam`` (L.Beam) + n.
    channels: list of (ops, ImageBuffer, wavelength).  Returns dict of tensors + stats (no sync)."""
    require_cuda()
    if s0 is not None:
        if not (isinstance(s0, torch.Tensor) and s0.is_cuda and s0.dtype == torch.float64 and s0.is_contiguous()):
            raise TypeError("s0 must be a contiguous CUDA float64 tensor of shape (9, N)")
        if s0.ndim != 2 or s0.shape[0] != 9:
            raise ValueError("s0 must have shape (9, N)")
        n = s0.shape[1]
    elif beam is None or n is None:
        raise ValueError("need s0 or (beam, n)")
    n = int(n)
    f64 = dict(dtype=torch.float64, device="cuda")
    out = {
        "sf": torch.empty((9, n), **f64) if want_sf else None,
        "rf": torch.empty((4, n), **f64) if want_rf else None,
        "jf": torch.empty((2, n), dtype=torch.complex128, device="cuda") if want_jf else None,
        "steps": torch.empty((n,), dtype=torch.int32, device="cuda") if want_steps else None,
    }
    stats = torch.zeros(6, dtype=torch.int64, device="cuda") if with_stats else None
    out["stats_dev"], out["n"] = stats, n
    if n == 0:                                  # empty bundle: nothing to launch
        return out
    keep, structs = [], []
    for ops, image, wl in channels:
        if image is not None:
            image.touched()
        ch, k = make_channel(ops, image, wl)
        structs.append(ch)
        keep.append(k)
    ch_arr = (L.Channel * max(1, len(structs)))(*structs)
    L.check(L.lib.sp_propagate(field._h, C.byref(params), workspace(), _ptr(s0),
                               C.byref(beam) if beam is not None else None, n, int(ray_offset), _ptr(out["sf"]),
                               _ptr(out["rf"]), _ptr(out["jf"]), _ptr(out["steps"]), ch_arr, len(structs),
                               _ptr(stats), _stream()))
    out["stats_dev"] = stats
    out["n"] = n
    return out


def controller_record(n):
    """Zeroed controller record of ``propagate_window`` for n rays: 'ctl' (3, n) float64 (t or tau, h_abs or dt, w of the
    point that parked the ray), 'flags' (n,) int32 of SP_CTL_* bits, 'steps' (n,) int32 attempts so far."""
    require_cuda()
    return dict(ctl=torch.zeros((3, n), dtype=torch.float64, device="cuda"),
                flags=torch.zeros(n, dtype=torch.int32, device="cuda"), steps=torch.zeros(n, dtype=torch.int32, device="cuda"))


def stage_store(n, params):
    """Zeroed stage store of ``propagate_window(..., stages=...)`` for n rays solved with ``params``: (values, n) CUDA,
    float32 with ``FLAG_FP32`` and float64 otherwise, values = ``STAGE_RK45`` (23), ``STAGE_TSIT5`` (42) or, with a channel
    flag, ``STAGE_RK45X`` (54) -- the layout of sp_propagate_window_staged in include/synthpy_b200.h."""
    require_cuda()
    dtype = torch.float32 if params.flags & L.FLAG_FP32 else torch.float64
    return torch.zeros((_stage_values(params), n), dtype=dtype, device="cuda")


def _stage_values(params):
    if params.flags & (L.FLAG_ATTEN | L.FLAG_FARADAY):
        return L.STAGE_RK45X
    return L.STAGE_TSIT5 if params.method == L.METHOD_TSIT5 else L.STAGE_RK45


def propagate_window(field, params, state, record, w_lo, w_hi, grid_range, *, idx=None, rf=None, jf=None, channels=(),
                     stats=None, stages=None):
    """One call of ``sp_propagate_window``: advance the rays ``idx`` (int32 CUDA tensor of indices, None = all) of the
    (9, N) CUDA float64 ``state`` in place, each until it finishes or parks at the window [w_lo, w_hi] of the probing
    axis (``grid_range``: the whole grid's extent along it).  With a channel flag in ``params`` (attenuation / Faraday, RK45
    only) this is ``sp_propagate_window_channels``: amp and pol (rows 6, 8) are integrated too, and ``field`` needs the
    grids (``attach_channels``).  ``record`` from ``controller_record``; ``rf`` (4, N) / ``jf`` (2, N) complex128 receive the rays that finish;
    ``stats`` an int64 (6,) CUDA tensor accumulated into.  With ``stages`` (from ``stage_store``) this is
    ``sp_propagate_window_staged``: rays park between stage evaluations and keep their attempt in progress there.  No sync."""
    require_cuda()
    if not (isinstance(state, torch.Tensor) and state.is_cuda and state.dtype == torch.float64 and state.is_contiguous()
            and state.ndim == 2 and state.shape[0] == 9):
        raise TypeError("state must be a contiguous (9, N) CUDA float64 tensor")
    n = state.shape[1]
    if idx is not None and not (idx.is_cuda and idx.dtype == torch.int32 and idx.is_contiguous()):
        raise TypeError("idx must be a contiguous CUDA int32 tensor")
    keep, structs = [], []
    for ops, image, wl in channels:
        if image is not None:
            image.touched()
        ch, k = make_channel(ops, image, wl)
        structs.append(ch)
        keep.append(k)
    ch_arr = (L.Channel * max(1, len(structs)))(*structs)
    if stages is not None:
        dtype = torch.float32 if params.flags & L.FLAG_FP32 else torch.float64
        if not (isinstance(stages, torch.Tensor) and stages.is_cuda and stages.dtype == dtype and stages.is_contiguous()
                and tuple(stages.shape) == (_stage_values(params), n)):
            raise TypeError("stages must be the contiguous CUDA tensor of stage_store(n, params) for this state")
        L.check(L.lib.sp_propagate_window_staged(field._h, C.byref(params), workspace(), _ptr(state), n, _ptr(idx),
                                                 0 if idx is None else idx.numel(), _ptr(record["ctl"]), _ptr(record["flags"]),
                                                 _ptr(record["steps"]), _ptr(stages), float(w_lo), float(w_hi),
                                                 float(grid_range[0]), float(grid_range[1]), _ptr(rf), _ptr(jf), ch_arr,
                                                 len(structs), _ptr(stats), _stream()))
        return
    fn = L.lib.sp_propagate_window_channels if params.flags & (L.FLAG_ATTEN | L.FLAG_FARADAY) else L.lib.sp_propagate_window
    L.check(fn(field._h, C.byref(params), workspace(), _ptr(state), n, _ptr(idx),
                                      0 if idx is None else idx.numel(), _ptr(record["ctl"]), _ptr(record["flags"]),
                                      _ptr(record["steps"]), float(w_lo), float(w_hi), float(grid_range[0]),
                                      float(grid_range[1]), _ptr(rf), _ptr(jf), ch_arr,
                                      len(structs), _ptr(stats), _stream()))


STAT_NAMES = ("ray_steps", "ray_steps_acc", "rays_capped", "rays_binned", "rays_rejected", "rhs_evals")


def stats_dict(stats_dev):
    return dict(zip(STAT_NAMES, [int(v) for v in stats_dev.cpu().tolist()]))


def rhs(field, params, s):
    """d(state)/dt for a (9,N) CUDA float64 tensor (parity level L0)."""
    require_cuda()
    out = torch.empty_like(s)
    L.check(L.lib.sp_rhs(field._h, C.byref(params), _ptr(s), s.shape[1], _ptr(out), _stream()))
    return out


def exit_plane(sf, probing_axis, out_axes, extent, *, keep_current_plane=False, want_rf=True, want_jf=False, want_state=False):
    """sp_exit_plane on a (9,N) CUDA float64 state: returns (rf, jf, back-propagated state), None where not asked."""
    require_cuda()
    n = sf.shape[1]
    rf = torch.empty((4, n), dtype=torch.float64, device="cuda") if want_rf else None
    jf = torch.empty((2, n), dtype=torch.complex128, device="cuda") if want_jf else None
    sb = torch.empty((9, n), dtype=torch.float64, device="cuda") if want_state else None
    L.check(L.lib.sp_exit_plane(_ptr(sf), n, int(probing_axis), int(out_axes[0]), int(out_axes[1]), float(extent),
                                int(bool(keep_current_plane)), _ptr(rf), _ptr(jf), _ptr(sb), _stream()))
    return rf, jf, sb


def beam_generate(beam, n, ray_offset=0):
    require_cuda()
    s0 = torch.empty((9, int(n)), dtype=torch.float64, device="cuda")
    L.check(L.lib.sp_beam_generate(C.byref(beam), int(ray_offset), int(n), _ptr(s0), _stream()))
    return s0


def noise_spectrum(S, shape, seed):
    """sp_noise_spectrum: the Hermitian half spectrum sqrt(S) (Z + conj Z(-k)) / 2 of Philox complex white noise for a
    ``shape`` = (n0, n1, n2) grid.  S: contiguous float32 CUDA tensor (n0, n1, n2 // 2 + 1); returns complex128 of the
    same shape on S's device, ready for ``torch.fft.irfftn(H, s=shape)``."""
    require_cuda()
    n0, n1, n2 = (int(n) for n in shape)
    if not (S.is_cuda and S.dtype == torch.float32 and S.is_contiguous() and tuple(S.shape) == (n0, n1, n2 // 2 + 1)):
        raise ValueError(f"S must be a contiguous float32 CUDA tensor of shape {(n0, n1, n2 // 2 + 1)}")
    if not 0 <= int(seed) < 2 ** 64:
        raise ValueError("seed must be in [0, 2**64)")
    with torch.cuda.device(S.device):
        H = torch.empty(S.shape, dtype=torch.complex128, device=S.device)
        L.check(L.lib.sp_noise_spectrum(_ptr(S), n0, n1, n2, int(seed), _ptr(H), _stream()))
    return H


def noise_spectrum_box(S, shape, order, lo, cnt, seed, out=None):
    """sp_noise_spectrum_box: ``noise_spectrum``'s H on the box [lo, lo + cnt) (per grid axis) of the full ``shape`` grid,
    stored with box axis t along grid axis order[t].  S: contiguous float32 CUDA tensor of the box shape
    (cnt[order[0]], cnt[order[1]], cnt[order[2]]); ``out``: a contiguous complex128 tensor (or view) of that shape on S's
    device to write into, else a new one.  Returns the written tensor."""
    require_cuda()
    n = tuple(int(v) for v in shape)
    order, lo, cnt = (tuple(int(v) for v in a) for a in (order, lo, cnt))
    if len(n) != 3 or len(order) != 3 or len(lo) != 3 or len(cnt) != 3:
        raise ValueError("shape, order, lo and cnt need three entries each")
    if sorted(order) != [0, 1, 2]:
        raise ValueError(f"order {order} is not a permutation of 0, 1, 2")
    if any(a < 0 or c < 1 or a + c > m for a, c, m in zip(lo, cnt, n)):
        raise ValueError(f"box lo={lo} cnt={cnt} is not inside the grid {n}")
    box = tuple(cnt[o] for o in order)
    if not (S.is_cuda and S.dtype == torch.float32 and S.is_contiguous() and tuple(S.shape) == box):
        raise ValueError(f"S must be a contiguous float32 CUDA tensor of shape {box}")
    if not 0 <= int(seed) < 2 ** 64:
        raise ValueError("seed must be in [0, 2**64)")
    if out is not None and not (out.device == S.device and out.dtype == torch.complex128 and out.is_contiguous()
                                and tuple(out.shape) == box):
        raise ValueError(f"out must be a contiguous complex128 tensor of shape {box} on {S.device}")
    ints = lambda v: (C.c_int * 3)(*v)
    with torch.cuda.device(S.device):
        H = torch.empty(box, dtype=torch.complex128, device=S.device) if out is None else out
        L.check(L.lib.sp_noise_spectrum_box(_ptr(S), *n, ints(order), ints(lo), ints(cnt), int(seed), _ptr(H), _stream()))
    return H


def optics_image(rf, ops, *, jf=None, image=None, wavelength=0.0, input_mm=False, want_rays=True):
    """Optical train (+ optional binning) on existing rays.  rf: (4,N) CUDA float64; jf: (2,N) complex128.
    Returns (rf_out, jf_out) at the detector plane (mm; NaN columns = rejected), or (None, None)."""
    require_cuda()
    n = rf.shape[1]
    rf_out = torch.empty_like(rf) if want_rays else None
    jf_out = torch.empty_like(jf) if (want_rays and jf is not None) else None
    ch, keep = make_channel(ops, image, wavelength, input_mm)
    L.check(L.lib.sp_optics_image(_ptr(rf), _ptr(jf), n, C.byref(ch), _ptr(rf_out), _ptr(jf_out), _stream()))
    return rf_out, jf_out
