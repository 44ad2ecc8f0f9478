// CPU self-test build of out-of-core tracing with the attenuation / Faraday channels: the windowed nine-row RK45
// (synthpy_b200/csrc/ray_core.h dp5x_window, which the SP_METHOD_RK45XW kernels of sp_propagate_window_channels inline),
// RK4 with the channels counting its steps, and the channel derivative through one walked cell cache -- on the host field
// of tests/host_harness.cpp with hh_attach's grids.  TEST code, like that harness.
#include "host_harness.cpp"

// The windowed per-ray solve over all nine rows (attenuation / Faraday channels: ray_core.h dp5x_window, the loop of the
// SP_METHOD_RK45XW kernel of sp_propagate_window_channels) over the host field with hh_attach's grids; the phase lane and
// the float64 aux grid compiled in, as hh_rk45_ext.  s (9 x n) is advanced in place, amp and pol included.
extern "C" void hh_slab_window_ext(void* h, double* s, uint64_t n, double* ctl, uint32_t* flags, uint32_t* att, double w_lo,
                                   double w_hi, double g_lo, double g_hi, double t_end, double rtol, double atol, double omega,
                                   double verdet, int atten, int faraday, int cap, int early, uint32_t* evals) {
    const HostField* f = (const HostField*)h;
    FieldView<double> F = f->view64();
    const ExtView X = f->ext_view(verdet, atten != 0, faraday != 0);
    Window W; W.lo = w_lo; W.hi = w_hi; W.g_lo = g_lo; W.g_hi = g_hi;
    for (uint64_t i = 0; i < n; ++i) {
        double y[9];
        for (int k = 0; k < 3; ++k) { y[k] = s[(uint64_t)f->perm[k] * n + i]; y[3 + k] = s[(uint64_t)(3 + f->perm[k]) * n + i]; }
        for (int k = 6; k < 9; ++k) y[k] = s[(uint64_t)k * n + i];
        WinCtl c;
        c.t = ctl[i]; c.h = ctl[n + i]; c.w_park = ctl[2 * n + i]; c.n_att = att[i]; c.flags = flags[i];
        unsigned acc = 0, capped = 0;
        const int t = dp5x_window<true, true>(F, X, W, omega, true, t_end, rtol, atol, cap > 0 ? (unsigned)cap : (1u << 30),
                                              early != 0, 0u, y, c, acc, capped);
        for (int k = 0; k < 3; ++k) { s[(uint64_t)f->perm[k] * n + i] = y[k]; s[(uint64_t)(3 + f->perm[k]) * n + i] = y[3 + k]; }
        for (int k = 6; k < 9; ++k) s[(uint64_t)k * n + i] = y[k];
        ctl[i] = c.t; ctl[n + i] = c.h; ctl[2 * n + i] = c.w_park; att[i] = c.n_att; flags[i] = c.flags;
        evals[i] += (uint32_t)t;
    }
}

// deriv9 at every point of s in order through ONE cell cache (the adaptive steppers' direct search), in hh_rhs_ext's
// layout: what dp5x_window evaluates after a walk, to hold against fresh lookups (a resumed ray starts a fresh cache).
extern "C" void hh_rhs_ext_walk(void* h, const double* s, uint64_t n, double* out, double omega, double verdet) {
    const HostField* f = (const HostField*)h;
    FieldView<double> F = f->view64();
    const ExtView X = f->ext_view(verdet, true, true);
    CellCache<double, true> cc;
    for (uint64_t i = 0; i < n; ++i) {
        double y[9], d[9];
        for (int k = 0; k < 3; ++k) { y[k] = s[(uint64_t)f->perm[k] * n + i]; y[3 + k] = s[(uint64_t)(3 + f->perm[k]) * n + i]; }
        for (int k = 6; k < 9; ++k) y[k] = s[(uint64_t)k * n + i];
        deriv9<true, true>(F, X, cc, omega, true, y, d);
        for (int k = 0; k < 3; ++k) { out[(uint64_t)f->perm[k] * n + i] = d[k]; out[(uint64_t)(3 + f->perm[k]) * n + i] = d[3 + k]; }
        for (int k = 6; k < 9; ++k) out[(uint64_t)k * n + i] = d[k];
    }
}

// hh_rk4_ext (tests/host_harness.cpp) with the steps taken per ray, for the slab driver of out-of-core RK4 with the channels.
extern "C" void hh_rk4_ext_steps(void* hnd, const double* s0, uint64_t n, int n_steps, double h, double omega, double verdet,
                                 int early, double* sf, uint32_t* steps) {
    const HostField* f = (const HostField*)hnd;
    FieldView<double> F = f->view64();
    const ExtView X = f->ext_view(verdet, true, true);
    for (uint64_t i = 0; i < n; ++i) {
        Ray<double> r; load(f, s0, n, i, r);
        ExtState e; e.amp = s0[6 * n + i]; e.pol = s0[8 * n + i];
        CellCache<double, true> cc;
        int it = 0;
        for (; it < n_steps; ++it)
            if (rk4_step_ext<true, true>(F, X, cc, h, omega, true, r, e, early != 0) < 0) break;
        for (int k = 0; k < 3; ++k) { sf[(uint64_t)f->perm[k] * n + i] = r.p[k]; sf[(uint64_t)(3 + f->perm[k]) * n + i] = r.v[k]; }
        sf[6 * n + i] = e.amp; sf[7 * n + i] = r.ph; sf[8 * n + i] = e.pol;
        steps[i] = (uint32_t)it;
    }
}
