"""ctypes loader of tests/noise_box_harness.cpp (CPU self-test build of the box noise, noise_core.h: noise_box)."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "_build", "libnoise_box_harness.so")
SRC = os.path.join(HERE, "noise_box_harness.cpp")
DEPS = [SRC, os.path.join(HERE, "..", "synthpy_b200", "csrc", "ray_core.h"),
        os.path.join(HERE, "..", "synthpy_b200", "csrc", "noise_core.h")]


def build():
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    if os.path.exists(SO) and all(os.path.getmtime(SO) >= os.path.getmtime(d) for d in DEPS):
        return SO
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", SRC, "-o", SO], check=True)
    return SO


class NoiseBoxHarness:
    def __init__(self):
        self.lib = C.CDLL(build())

    def noise_box(self, S, shape, order, lo, cnt, seed):
        """The box k_noise_spectrum_box writes: complex128 of shape (cnt[order[0]], cnt[order[1]], cnt[order[2]]) from
        float32 S of that shape; lo, cnt per grid axis."""
        S = np.ascontiguousarray(S, dtype=np.float32)
        assert S.shape == tuple(cnt[o] for o in order)
        ints = lambda v: (C.c_int * 3)(*(int(x) for x in v))
        out = np.empty(S.shape, dtype=np.complex128)
        self.lib.hh_noise_box(S.ctypes.data_as(C.c_void_p), *(C.c_int(n) for n in shape), ints(order), ints(lo),
                              ints(cnt), C.c_uint64(seed), out.ctypes.data_as(C.c_void_p))
        return out
