// CPU self-test build of the turbulent-field noise (synthpy_b200/csrc/noise_core.h): the very source that is inlined
// into k_noise_spectrum, compiled by g++ so that the CPU test-suite can check it.  It is TEST code: nothing in
// synthpy_b200/ loads it, and it is not a fallback.
#include <stdint.h>

#include "../synthpy_b200/csrc/noise_core.h"

using namespace sp;

// Z at every full-grid index, complex128 interleaved [n0][n1][n2]
extern "C" void hh_noise_full(int n0, int n1, int n2, uint64_t seed, double* out) {
    const uint64_t n = (uint64_t)n0 * n1 * n2;
    for (uint64_t f = 0; f < n; ++f) noise_z(seed, f, out[2 * f], out[2 * f + 1]);
}

// the half spectrum H that k_noise_spectrum writes, from S float32 [n0][n1][n2/2+1]
extern "C" void hh_noise_half(const float* S, int n0, int n1, int n2, uint64_t seed, double* out) {
    const int nh = n2 / 2 + 1;
    for (int i = 0; i < n0; ++i)
        for (int j = 0; j < n1; ++j)
            for (int l = 0; l < nh; ++l) {
                const uint64_t h = ((uint64_t)i * n1 + j) * nh + l;
                const d2 v = noise_half(S[h], n0, n1, n2, seed, i, j, l);
                out[2 * h] = v.x; out[2 * h + 1] = v.y;
            }
}
