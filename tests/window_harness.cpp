// CPU self-test build of the windowed per-ray adaptive solves (out-of-core tracing): the controller loops dp5_window /
// tsit5_window of synthpy_b200/csrc/ray_core.h, which the SP_METHOD_RK45W / SP_METHOD_TSIT5W kernels of
// sp_propagate_window inline, on the host field of tests/host_harness.cpp.  TEST code, like that harness.
#include "host_harness.cpp"

// One launch on every ray of s (9 x n, advanced in place).  ctl (3 x n), flags and attempts are the controller record
// (in / out); evals[i] accumulates ray i's field evaluations.
template <bool PH, bool A64, bool TSIT>
static void window_t(const HostField* f, double* s, uint64_t n, double* ctl, uint32_t* flags, uint32_t* att, double w_lo,
                     double w_hi, double g_lo, double g_hi, double t_end, double dt0, double rtol, double atol, double omega,
                     int n_state, int cap_in, int early, uint32_t* evals) {
    FieldView<double> F = f->view64();
    Window W; W.lo = w_lo; W.hi = w_hi; W.g_lo = g_lo; W.g_hi = g_hi;
    for (uint64_t i = 0; i < n; ++i) {
        Ray<double> r; load(f, s, n, i, r);
        WinCtl c;
        c.t = ctl[i]; c.h = ctl[n + i]; c.w_park = ctl[2 * n + i]; c.n_att = att[i]; c.flags = flags[i];
        unsigned acc = 0, capped = 0;
        int t;
        if (TSIT) {
            t = tsit5_window<double, PH, A64>(F, W, omega, t_end, dt0, rtol, atol, n_state, cap_in > 0 ? (unsigned)cap_in : 10000u,
                                              0u, r, c, acc, capped);
        } else {
            StageRegs<double> S;
            memset(&S, 0, sizeof(S));
            t = dp5_window<double, PH, A64, StageRegs<double> >(F, W, omega, t_end, rtol, atol, n_state, s[6 * n + i], s[8 * n + i],
                                                               cap_in > 0 ? (unsigned)cap_in : (1u << 30), early != 0, 0u, r, c, S,
                                                               acc, capped);
        }
        store(f, s, s, n, i, r);
        ctl[i] = c.t; ctl[n + i] = c.h; ctl[2 * n + i] = c.w_park; att[i] = c.n_att; flags[i] = c.flags;
        evals[i] += (uint32_t)t;
    }
}

extern "C" void hh_slab_window(void* h, int tsit, double* s, uint64_t n, double* ctl, uint32_t* flags, uint32_t* att, double w_lo,
                               double w_hi, double g_lo, double g_hi, double t_end, double dt0, double rtol, double atol,
                               double omega, int phase, int aux64, int n_state, int cap, int early, uint32_t* evals) {
    const HostField* f = (const HostField*)h;
#define SP_W(PH, A64) (tsit ? window_t<PH, A64, true>(f, s, n, ctl, flags, att, w_lo, w_hi, g_lo, g_hi, t_end, dt0, rtol, atol, omega, n_state, cap, early, evals) \
                            : window_t<PH, A64, false>(f, s, n, ctl, flags, att, w_lo, w_hi, g_lo, g_hi, t_end, dt0, rtol, atol, omega, n_state, cap, early, evals))
    if (!phase) SP_W(false, false);
    else if (!aux64) SP_W(true, false);
    else SP_W(true, true);
#undef SP_W
}
