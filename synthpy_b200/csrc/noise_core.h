// Per-element math of the turbulent-field noise (k_noise_spectrum): complex white noise drawn from a counter, folded
// into the Hermitian half spectrum that torch.fft.irfftn / cuFFT C2R take.
//
// The reference (src/field_generator/gaussian3D.py:215-271) returns Re ifftn(Z sqrt(S)) for complex white noise Z and a
// power spectrum S(|k|).  The real part of an inverse FFT is the inverse FFT of the Hermitian part of its input, so the
// same field is irfftn(H) with H(k) = sqrt(S(k)) (Z(k) + conj Z(-k)) / 2 on the half grid kz in [0, n2/2]
// (S(-k) == S(k) bit for bit: fftfreq gives exact negatives).  A counter-based generator evaluates Z(-k) where it is
// needed, so H is written in one pass and nothing of grid size exists before it.
//
// SP_HD like ray_core.h: the same source is inlined into the sm_100a kernels and compiled by g++ into
// tests/host_harness.cpp.
#pragma once
#include "ray_core.h"

namespace sp {

// Philox counter word 3 of the field noise; the beam uses 0x5eed, so one seed drives unrelated beam and field streams
#define SP_NOISE_TAG 0xf1e1du

SP_HD float sp_sqrtf(float x) {
#if defined(__CUDA_ARCH__)
    return __fsqrt_rn(x);
#else
    return sqrtf(x);
#endif
}

// Z at full-grid flat index `flat`: one Philox4x32-10 block (key = seed, counter = (flat lo, flat hi, 0, tag)), two
// 53-bit uniforms, Box-Muller.  Re and Im are independent N(0, 1).
SP_HD void noise_z(uint64_t seed, uint64_t flat, double& re, double& im) {
    const double PI = 3.14159265358979323846;
    Philox ph; ph.k0 = (uint32_t)seed; ph.k1 = (uint32_t)(seed >> 32);
    uint32_t r[4];
    ph.block((uint32_t)flat, (uint32_t)(flat >> 32), 0u, SP_NOISE_TAG, r);
    const double U0 = u53(r[0], r[1]), U1 = u53(r[2], r[3]);
    const double rad = sqrt(-2.0 * log(1.0 - U0));
    double s, c; sp_sincos(2.0 * PI * U1, &s, &c);
    re = rad * c; im = rad * s;
}

// H at half-grid element (i, j, l) of a (n0, n1, n2) grid; s32 = S at that element (float32, 0 outside the band).
// At a self-conjugate point the mirror is the point itself and Im H is exactly +0.
SP_HD d2 noise_half(float s32, int n0, int n1, int n2, uint64_t seed, int i, int j, int l) {
    const int mi = i ? n0 - i : 0, mj = j ? n1 - j : 0, ml = l ? n2 - l : 0;
    double are, aim, bre, bim;
    noise_z(seed, ((uint64_t)i * n1 + j) * n2 + l, are, aim);
    noise_z(seed, ((uint64_t)mi * n1 + mj) * n2 + ml, bre, bim);
    const double s = (double)sp_sqrtf(s32);
    d2 h;
    h.x = s * (0.5 * (are + bre));
    h.y = s * (0.5 * (aim - bim));
    return h;
}

// A box of the full grid stored in axis order `order` (a permutation of 0, 1, 2): element (a, b, c) of the box is grid
// index lo[order[t]] + (a, b, c)[t] along grid axis order[t].  lo is per grid axis, dim per box axis.
struct NoiseBox {
    int order[3], lo[3], dim[3];
};

// the box coordinate that runs along grid axis `axis` (selects, no indexed access: the kernel keeps it in registers)
SP_HD int box_coord(const NoiseBox& B, int axis, int a, int b, int c) {
    return B.order[0] == axis ? a : B.order[1] == axis ? b : c;
}

// H at box element (a, b, c).  Inside the half grid (l <= n2/2) this is noise_half at the element, the value
// k_noise_spectrum writes.  Above it, it is conj H(-k) with H(-k) from noise_half at the mirrored half-grid element: the
// formula would give the same value at k itself, but a device build may fuse the sum of the two draws' real parts into
// an FMA in either order, so only the mirror makes the box the Hermitian extension of k_noise_spectrum's half spectrum
// bit for bit.  s32 is S at k, which equals S(-k) bit for bit.
SP_HD d2 noise_box(float s32, int n0, int n1, int n2, uint64_t seed, const NoiseBox& B, int a, int b, int c) {
    int i = B.lo[0] + box_coord(B, 0, a, b, c), j = B.lo[1] + box_coord(B, 1, a, b, c);
    int l = B.lo[2] + box_coord(B, 2, a, b, c);
    const bool upper = 2 * l > n2;
    if (upper) {
        i = i ? n0 - i : 0;
        j = j ? n1 - j : 0;
        l = n2 - l;
    }
    d2 h = noise_half(s32, n0, n1, n2, seed, i, j, l);
    if (upper) h.y = -h.y;
    return h;
}

}  // namespace sp
