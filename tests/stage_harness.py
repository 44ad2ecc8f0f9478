"""ctypes loader of tests/stage_harness.cpp: tests/host_harness.cpp plus the windowed adaptive solves with stage parking
(ray_core.h dp5_window / tsit5_window / dp5x_window with STAGED), built with the same flags into its own library."""
import ctypes as C
import os
import subprocess

import numpy as np

import harness

SO = os.path.join(harness.HERE, "_build", "libstage_harness.so")
SRC = os.path.join(harness.HERE, "stage_harness.cpp")
DEPS = [SRC] + harness.DEPS
STAGE_VALUES = {"rk45": 23, "tsit5": 42, "rk45x": 54}         # SP_STAGE_RK45 / SP_STAGE_TSIT5 / SP_STAGE_RK45X
CTL_STAGED, ROW_SHIFT = 16, 8                                 # SP_CTL_STAGED, SP_CTL_ROW_SHIFT


def build():
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    if os.path.exists(SO) and all(os.path.getmtime(SO) >= os.path.getmtime(d) for d in DEPS):
        return SO
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", SRC, "-o", SO], check=True)
    return SO


class StageHarness(harness.Harness):
    """``harness.Harness`` over this library: the same host fields (``attach`` their channel grids), plus ``staged``."""

    def __init__(self):
        self.lib = C.CDLL(build())
        self.lib.hh_field_create.restype = C.c_void_p

    def staged(self, field, s, rec, w_lo, w_hi, grid_range=(-np.inf, np.inf), *, method, t_end, dt0=0.0, rtol=1e-3, atol=1e-6,
               verdet=0.0, atten=False, faraday=False, n_state=9, cap=0, early=False, aux64=None):
        """One launch of the windowed RK45 ('rk45'), Tsit5 ('tsit5') or nine-row RK45 with the channels ('rk45x') solve with
        stage parking on every ray of ``s`` (advanced in place) through ``field``; ``rec`` from ``stage_record`` (updated in
        place, stage store included)."""
        assert s.flags.c_contiguous and s.dtype == np.float64 and rec["stage"].shape == (STAGE_VALUES[method], s.shape[1])
        p = harness._p
        self.lib.hh_slab_window_staged(field.h, C.c_int(["rk45", "tsit5", "rk45x"].index(method)), p(s), C.c_uint64(s.shape[1]),
                                       p(rec["ctl"]), p(rec["flags"]), p(rec["steps"]), p(rec["stage"]), C.c_double(w_lo),
                                       C.c_double(w_hi), C.c_double(grid_range[0]), C.c_double(grid_range[1]), C.c_double(t_end),
                                       C.c_double(dt0), C.c_double(rtol), C.c_double(atol), C.c_double(field.omega),
                                       C.c_double(verdet), C.c_int(int(atten)), C.c_int(int(faraday)), C.c_int(int(field.phase)),
                                       C.c_int(int(field.f64 if aux64 is None else aux64)), C.c_int(n_state), C.c_int(cap),
                                       C.c_int(int(early)), p(rec["evals"]))


def stage_record(n, method):
    """Zeroed controller record (``window_harness.window_record``'s layout, w_park at +inf), the per-ray evaluation counts
    and the zeroed stage store of ``method``."""
    ctl = np.zeros((3, n))
    ctl[2] = np.inf
    return dict(ctl=ctl, flags=np.zeros(n, dtype=np.uint32), steps=np.zeros(n, dtype=np.uint32),
                evals=np.zeros(n, dtype=np.uint32), stage=np.zeros((STAGE_VALUES[method], n)))
