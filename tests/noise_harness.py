"""ctypes loader of tests/noise_harness.cpp (CPU self-test build of the turbulent-field noise, noise_core.h)."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "_build", "libnoise_harness.so")
SRC = os.path.join(HERE, "noise_harness.cpp")
DEPS = [SRC, os.path.join(HERE, "..", "synthpy_b200", "csrc", "ray_core.h"),
        os.path.join(HERE, "..", "synthpy_b200", "csrc", "noise_core.h")]


def build():
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    if os.path.exists(SO) and all(os.path.getmtime(SO) >= os.path.getmtime(d) for d in DEPS):
        return SO
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", SRC, "-o", SO], check=True)
    return SO


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class NoiseHarness:
    def __init__(self):
        self.lib = C.CDLL(build())

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
