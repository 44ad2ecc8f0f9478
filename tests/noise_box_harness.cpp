// CPU self-test build of the box noise (synthpy_b200/csrc/noise_core.h: noise_box): the very source that is inlined into
// k_noise_spectrum_box, compiled by g++ so that the CPU test-suite can check it.  It is TEST code: nothing in
// synthpy_b200/ loads it, and it is not a fallback.
#include <stdint.h>

#include "../synthpy_b200/csrc/noise_core.h"

using namespace sp;

// the box k_noise_spectrum_box writes: grid box [lo, lo + cnt) (per grid axis) in axis order `order`, from S float32 in the
// same box layout
extern "C" void hh_noise_box(const float* S, int n0, int n1, int n2, const int* order, const int* lo, const int* cnt,
                             uint64_t seed, double* out) {
    NoiseBox B;
    for (int t = 0; t < 3; ++t) { B.order[t] = order[t]; B.lo[t] = lo[t]; B.dim[t] = cnt[order[t]]; }
    for (int a = 0; a < B.dim[0]; ++a)
        for (int b = 0; b < B.dim[1]; ++b)
            for (int c = 0; c < B.dim[2]; ++c) {
                const uint64_t h = ((uint64_t)a * B.dim[1] + b) * B.dim[2] + c;
                const d2 v = noise_box(S[h], n0, n1, n2, seed, B, a, b, c);
                out[2 * h] = v.x; out[2 * h + 1] = v.y;
            }
}
