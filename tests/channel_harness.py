"""ctypes loader of tests/channel_harness.cpp: tests/host_harness.cpp plus out-of-core tracing with the attenuation /
Faraday channels (ray_core.h dp5x_window, RK4 with the channels and its steps per ray, deriv9 through one walked cell
cache), built with the same flags into its own library."""
import ctypes as C
import os
import subprocess

import numpy as np

import harness

SO = os.path.join(harness.HERE, "_build", "libchannel_harness.so")
SRC = os.path.join(harness.HERE, "channel_harness.cpp")
DEPS = [SRC] + harness.DEPS


def build():
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    if os.path.exists(SO) and all(os.path.getmtime(SO) >= os.path.getmtime(d) for d in DEPS):
        return SO
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", SRC, "-o", SO], check=True)
    return SO


class ChannelHarness(harness.Harness):
    """``harness.Harness`` over this library: the same host fields (``attach`` their channel grids), plus ``window_ext``,
    ``rk4_ext_steps`` and ``rhs_ext_walk``."""

    def __init__(self):
        self.lib = C.CDLL(build())
        self.lib.hh_field_create.restype = C.c_void_p

    def window_ext(self, field, s, rec, w_lo, w_hi, grid_range=(-np.inf, np.inf), *, t_end, verdet, rtol=1e-3, atol=1e-6, cap=0,
                   early=False, atten=True, faraday=True):
        """One launch of the windowed nine-row RK45 (``dp5x_window``) on every ray of ``s`` (advanced in place, amp and pol
        included) through ``field`` with its ``attach``ed grids; ``rec`` from ``window_harness.window_record``."""
        assert s.flags.c_contiguous and s.dtype == np.float64
        p = harness._p
        self.lib.hh_slab_window_ext(field.h, p(s), C.c_uint64(s.shape[1]), p(rec["ctl"]), p(rec["flags"]), p(rec["steps"]),
                                    C.c_double(w_lo), C.c_double(w_hi), C.c_double(grid_range[0]), C.c_double(grid_range[1]),
                                    C.c_double(t_end), C.c_double(rtol), C.c_double(atol), C.c_double(field.omega),
                                    C.c_double(verdet), C.c_int(int(atten)), C.c_int(int(faraday)), C.c_int(cap),
                                    C.c_int(int(early)), p(rec["evals"]))

    def rhs_ext_walk(self, field, s, verdet):
        """deriv9 at the points of ``s`` in order through one cell cache (``field.rhs_ext`` looks each one up afresh)."""
        s = np.ascontiguousarray(s, dtype=np.float64)
        out = np.empty_like(s)
        self.lib.hh_rhs_ext_walk(field.h, harness._p(s), C.c_uint64(s.shape[1]), harness._p(out), C.c_double(field.omega),
                                 C.c_double(verdet))
        return out

    def rk4_ext_steps(self, field, s0, n_steps, h, verdet, early=True):
        """``field.rk4_ext`` (the same loop) plus the steps taken per ray."""
        s0 = np.ascontiguousarray(s0, dtype=np.float64)
        sf = np.empty_like(s0)
        steps = np.empty(s0.shape[1], dtype=np.uint32)
        self.lib.hh_rk4_ext_steps(field.h, harness._p(s0), C.c_uint64(s0.shape[1]), C.c_int(n_steps), C.c_double(h),
                                  C.c_double(field.omega), C.c_double(verdet), C.c_int(int(early)), harness._p(sf),
                                  harness._p(steps))
        return sf, steps
