// CPU self-test build of stage parking (out-of-core park='stage'): the windowed loops dp5_window / tsit5_window /
// dp5x_window of synthpy_b200/csrc/ray_core.h with STAGED on, which the staged kernels of sp_propagate_window_staged inline,
// on the host field of tests/host_harness.cpp (hh_attach's grids for the channel variant).  TEST code, like that harness.
#include "host_harness.cpp"

// One launch on every ray of s (9 x n, advanced in place).  ctl (3 x n), flags and attempts are the controller record and
// stage (values x n) the stage store, all in / out; evals[i] accumulates ray i's field evaluations.
// method: 0 = RK45, 1 = Tsit5, 2 = RK45 over the nine rows with the channels (phase lane and float64 aux grid compiled in,
// as hh_rk45_ext).
template <bool PH, bool A64>
static void staged_t(const HostField* f, int method, double* s, uint64_t n, double* ctl, uint32_t* flags, uint32_t* att,
                     double* stage, const Window& W, double t_end, double dt0, double rtol, double atol, double omega, double verdet,
                     int atten, int faraday, int n_state, int cap_in, int early, uint32_t* evals) {
    FieldView<double> F = f->view64();
    const ExtView X = f->ext_view(verdet, atten != 0, faraday != 0);
    for (uint64_t i = 0; i < n; ++i) {
        WinCtl c;
        c.t = ctl[i]; c.h = ctl[n + i]; c.w_park = ctl[2 * n + i]; c.n_att = att[i]; c.flags = flags[i];
        StageStore<double> G; G.p = stage + i; G.stride = n;
        unsigned acc = 0, capped = 0;
        int t;
        if (method == 2) {
            double y[9];
            for (int k = 0; k < 3; ++k) { y[k] = s[(uint64_t)f->perm[k] * n + i]; y[3 + k] = s[(uint64_t)(3 + f->perm[k]) * n + i]; }
            for (int k = 6; k < 9; ++k) y[k] = s[(uint64_t)k * n + i];
            t = dp5x_window<true, true, true>(F, X, W, omega, true, t_end, rtol, atol, cap_in > 0 ? (unsigned)cap_in : (1u << 30),
                                              early != 0, 0u, y, c, acc, capped, G);
            for (int k = 0; k < 3; ++k) { s[(uint64_t)f->perm[k] * n + i] = y[k]; s[(uint64_t)(3 + f->perm[k]) * n + i] = y[3 + k]; }
            for (int k = 6; k < 9; ++k) s[(uint64_t)k * n + i] = y[k];
        } else {
            Ray<double> r; load(f, s, n, i, r);
            if (method == 1) {
                t = tsit5_window<double, PH, A64, true>(F, W, omega, t_end, dt0, rtol, atol, n_state,
                                                        cap_in > 0 ? (unsigned)cap_in : 10000u, 0u, r, c, acc, capped, G);
            } else {
                StageRegs<double> S;
                memset(&S, 0, sizeof(S));
                t = dp5_window<double, PH, A64, StageRegs<double>, true>(F, W, omega, t_end, rtol, atol, n_state, s[6 * n + i],
                                                                         s[8 * n + i], cap_in > 0 ? (unsigned)cap_in : (1u << 30),
                                                                         early != 0, 0u, r, c, S, acc, capped, G);
            }
            store(f, s, s, n, i, r);
        }
        ctl[i] = c.t; ctl[n + i] = c.h; ctl[2 * n + i] = c.w_park; att[i] = c.n_att; flags[i] = c.flags;
        evals[i] += (uint32_t)t;
    }
}

extern "C" void hh_slab_window_staged(void* h, int method, double* s, uint64_t n, double* ctl, uint32_t* flags, uint32_t* att,
                                      double* stage, double w_lo, double w_hi, double g_lo, double g_hi, double t_end, double dt0,
                                      double rtol, double atol, double omega, double verdet, int atten, int faraday, int phase,
                                      int aux64, int n_state, int cap, int early, uint32_t* evals) {
    const HostField* f = (const HostField*)h;
    Window W; W.lo = w_lo; W.hi = w_hi; W.g_lo = g_lo; W.g_hi = g_hi;
#define SP_S(PH, A64) staged_t<PH, A64>(f, method, s, n, ctl, flags, att, stage, W, t_end, dt0, rtol, atol, omega, verdet, atten, \
                                        faraday, n_state, cap, early, evals)
    if (!phase) SP_S(false, false);
    else if (!aux64) SP_S(true, false);
    else SP_S(true, true);
#undef SP_S
}
