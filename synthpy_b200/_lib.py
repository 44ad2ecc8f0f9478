"""ctypes binding of include/synthpy_b200.h.

There is no CPU fallback: importing this module without the built CUDA library raises, and every call
checks the return code and raises with ``sp_last_error()``.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SYNTHPY_B200_LIB") or os.path.join(_HERE, "csrc", "libsynthpy_b200.so")   # override: A/B builds

# ---- constants (mirror the header) ---------------------------------------------------------------
FIELD_PHASE, FIELD_PHASE_F64 = 1, 2
BEAM_CIRCULAR_FOLD, BEAM_CIRCULAR_POW2, BEAM_SQUARE, BEAM_RECTANGULAR, BEAM_LINEAR = range(5)
OP_TRAVEL, OP_TRAVEL_NOE, OP_LENS, OP_CIRC_AP, OP_CIRC_STOP, OP_RECT_AP, OP_KNIFE, OP_REF_BEAM = range(8)
IMG_HISTOGRAM, IMG_INTERFEROGRAM, IMG_STOKES = 0, 1, 2
PLANE_FRAC_BITS = 40          # SP_PLANE_FRAC_BITS: interferogram planes are int64 in units of 2^-40
STOKES_FRAC_BITS = 32         # SP_STOKES_FRAC_BITS: Stokes I, Q, U planes are int64 in units of 2^-32
METHOD_RK4, METHOD_RK45, METHOD_RK45_JOINT, METHOD_TSIT5 = 0, 1, 2, 6
FLAG_PHASE, FLAG_EARLY_EXIT, FLAG_FP32, FLAG_PHASE_F64, FLAG_NO_SORT, FLAG_ATTEN, FLAG_FARADAY, FLAG_BUNDLE_STEP = 1, 2, 4, 8, 16, 32, 64, 128


class Beam(C.Structure):
    _fields_ = [("beam_type", C.c_int32), ("probing_axis", C.c_int32), ("size_a", C.c_double),
                ("size_b", C.c_double), ("divergence", C.c_double), ("start", C.c_double), ("seed", C.c_uint64)]


class OpticOp(C.Structure):
    _fields_ = [("kind", C.c_int32), ("_pad", C.c_int32), ("p0", C.c_double), ("p1", C.c_double), ("p2", C.c_double)]


class Image(C.Structure):
    _fields_ = [("kind", C.c_int32), ("nx", C.c_int32), ("ny", C.c_int32), ("_pad", C.c_int32),
                ("x_lo", C.c_double), ("x_hi", C.c_double), ("y_lo", C.c_double), ("y_hi", C.c_double),
                ("counts_dev", C.c_void_p), ("planes_dev", C.c_void_p)]


class Channel(C.Structure):
    _fields_ = [("ops_host", C.POINTER(OpticOp)), ("n_ops", C.c_int32), ("input_mm", C.c_int32),
                ("wavelength", C.c_double), ("image", Image)]


class Params(C.Structure):
    _fields_ = [("method", C.c_int32), ("flags", C.c_int32), ("n_steps", C.c_int32), ("n_state", C.c_int32),
                ("h", C.c_double), ("t_end", C.c_double), ("rtol", C.c_double), ("atol", C.c_double),
                ("omega", C.c_double), ("extent", C.c_double), ("probing_axis", C.c_int32),
                ("out_axis_a", C.c_int32), ("out_axis_b", C.c_int32), ("_pad", C.c_int32), ("verdet", C.c_double)]


class Stats(C.Structure):
    _fields_ = [("ray_steps", C.c_uint64), ("ray_steps_acc", C.c_uint64), ("rays_capped", C.c_uint64),
                ("rays_binned", C.c_uint64), ("rays_rejected", C.c_uint64), ("rhs_evals", C.c_uint64)]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


EXPORTS = {
    # name: (restype, argtypes)
    "sp_version": (C.c_int, []),
    "sp_last_error": (C.c_char_p, []),
    "sp_launch_count": (C.c_uint64, []),
    "sp_field_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, C.c_void_p]),
    "sp_field_create_from_gradients": (C.c_int, [C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p, C.c_void_p,
                                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                 C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "sp_field_attach_channels": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sp_field_destroy": (C.c_int, [C.c_void_p]),
    "sp_field_export_gradients": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sp_field_bytes": (C.c_uint64, [C.c_void_p]),
    "sp_beam_generate": (C.c_int, [C.POINTER(Beam), C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p]),
    "sp_optics_image": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(Channel), C.c_void_p, C.c_void_p,
                                  C.c_void_p]),
    "sp_image_finalize": (C.c_int, [C.POINTER(Image), C.c_void_p, C.c_void_p]),
    "sp_workspace_create": (C.c_int, [C.POINTER(C.c_void_p)]),
    "sp_workspace_destroy": (C.c_int, [C.c_void_p]),
    "sp_workspace_joint_log": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int)]),
    "sp_workspace_propagate_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    "sp_propagate": (C.c_int, [C.c_void_p, C.POINTER(Params), C.c_void_p, C.c_void_p, C.POINTER(Beam), C.c_uint64,
                               C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Channel),
                               C.c_int, C.c_void_p, C.c_void_p]),
    "sp_exit_plane": (C.c_int, [C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_void_p]),
    "sp_scatter_to_grid": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p,
                                     C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sp_fresnel_prepare": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_void_p]),
    "sp_fresnel_transfer": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double,
                                      C.c_void_p]),
    "sp_fresnel_finish": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_void_p, C.c_void_p]),
    "sp_rhs": (C.c_int, [C.c_void_p, C.POINTER(Params), C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "sp_fp64_peak": (C.c_int, [C.c_int, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.c_void_p]),
}


class SynthpyB200Error(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C synthpy_b200/csrc`).  synthpy_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)          # AttributeError here = header and library out of sync
        fn.restype, fn.argtypes = res, args
    return lib


lib = _load()


def check(rc):
    if rc != 0:
        raise SynthpyB200Error(f"synthpy_b200 error {rc}: {lib.sp_last_error().decode()}")


def launch_count():
    return int(lib.sp_launch_count())
