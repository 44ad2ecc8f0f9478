"""ctypes loader of tests/window_harness.cpp: tests/host_harness.cpp plus the windowed per-ray adaptive solves of
out-of-core tracing (ray_core.h dp5_window / tsit5_window), built with the same flags into its own library."""
import ctypes as C
import os
import subprocess

import numpy as np

import harness

SO = os.path.join(harness.HERE, "_build", "libwindow_harness.so")
SRC = os.path.join(harness.HERE, "window_harness.cpp")
DEPS = [SRC] + harness.DEPS


def build():
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    if os.path.exists(SO) and all(os.path.getmtime(SO) >= os.path.getmtime(d) for d in DEPS):
        return SO
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", SRC, "-o", SO], check=True)
    return SO


class WindowHarness(harness.Harness):
    """``harness.Harness`` over this library: the same host fields, plus ``window``."""

    def __init__(self):
        self.lib = C.CDLL(build())
        self.lib.hh_field_create.restype = C.c_void_p

    def window(self, field, s, rec, w_lo, w_hi, grid_range=(-np.inf, np.inf), *, method, t_end, dt0=0.0, rtol=1e-3,
               atol=1e-6, n_state=9, cap=0, early=False, aux64=None):
        """One launch of the windowed RK45 ('rk45') / Tsit5 ('tsit5') solve on every ray of ``s`` (advanced in place) through
        ``field`` (from ``self.field``); ``rec`` from ``window_record`` (updated in place)."""
        assert s.flags.c_contiguous and s.dtype == np.float64
        p = harness._p
        self.lib.hh_slab_window(field.h, C.c_int(int(method == "tsit5")), p(s), C.c_uint64(s.shape[1]), p(rec["ctl"]),
                                p(rec["flags"]), p(rec["steps"]), C.c_double(w_lo), C.c_double(w_hi),
                                C.c_double(grid_range[0]), C.c_double(grid_range[1]), C.c_double(t_end), C.c_double(dt0),
                                C.c_double(rtol), C.c_double(atol), C.c_double(field.omega), C.c_int(int(field.phase)),
                                C.c_int(int(field.f64 if aux64 is None else aux64)), C.c_int(n_state), C.c_int(cap),
                                C.c_int(int(early)), p(rec["evals"]))


def window_record(n):
    """Zeroed controller record of ``WindowHarness.window`` (the layout of engine.controller_record, w_park at +inf) plus
    the per-ray evaluation counts."""
    ctl = np.zeros((3, n))
    ctl[2] = np.inf
    return dict(ctl=ctl, flags=np.zeros(n, dtype=np.uint32), steps=np.zeros(n, dtype=np.uint32),
                evals=np.zeros(n, dtype=np.uint32))
