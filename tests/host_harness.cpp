// CPU self-test build of the product's per-ray math (synthpy_b200/csrc/ray_core.h, field_prep.h), wave optics
// (fresnel_core.h) and turbulent-field noise (noise_core.h).
// The build container has no GPU; this harness lets the CPU test-suite run the very same source that is
// inlined into the sm_100a kernels against the golden vectors.  It is TEST code: nothing in synthpy_b200/
// loads it, and it is not a fallback.
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "../synthpy_b200/csrc/field_prep.h"
#include "../synthpy_b200/csrc/ray_core.h"

using namespace sp;

struct HostField {
    int n[3], perm[3], nk[3];
    std::vector<f4> data;
    std::vector<double> aux64;
    std::vector<double> ext[5];          // kappa, ne, B_u, B_v, B_w (kernel frame)
    AxisTables tabs[3];
    ExtView ext_view(double verdet, bool atten, bool faraday) const {
        ExtView X; X.verdet = verdet;
        X.ch[0] = (atten && !ext[0].empty()) ? ext[0].data() : nullptr;
        for (int c = 1; c < 5; ++c) X.ch[c] = (faraday && !ext[c].empty()) ? ext[c].data() : nullptr;
        return X;
    }
    FieldView<double> view64() const {
        FieldView<double> V;
        V.data = data.data(); V.aux64 = aux64.empty() ? nullptr : aux64.data();
        for (int k = 0; k < 3; ++k) {
            V.ax[k].tab = tabs[k].t64.data(); V.ax[k].g0 = tabs[k].g0; V.ax[k].inv_d = tabs[k].inv_d;
            V.ax[k].lo = tabs[k].lo; V.ax[k].hi = tabs[k].hi; V.ax[k].n = nk[k];
        }
        V.su = (long long)nk[1] * nk[2]; V.sv = nk[2];
        return V;
    }
    FieldView<float> view32() const {
        FieldView<float> V;
        V.data = data.data(); V.aux64 = aux64.empty() ? nullptr : aux64.data();
        for (int k = 0; k < 3; ++k) {
            V.ax[k].tab = tabs[k].t32.data(); V.ax[k].g0 = (float)tabs[k].g0; V.ax[k].inv_d = (float)tabs[k].inv_d;
            V.ax[k].lo = (float)tabs[k].lo; V.ax[k].hi = (float)tabs[k].hi; V.ax[k].n = nk[k];
        }
        V.su = (long long)nk[1] * nk[2]; V.sv = nk[2];
        return V;
    }
};

// Same arithmetic as sp_field_create: returns an opaque host field.
extern "C" void* hh_field_create(const double* ne, const float* ax, const float* ay, const float* az, int nx, int ny, int nz,
                      double omega, int march_axis, int flags) {
    HostField* f = new HostField();
    f->n[0] = nx; f->n[1] = ny; f->n[2] = nz;
    f->perm[0] = (march_axis + 1) % 3; f->perm[1] = (march_axis + 2) % 3; f->perm[2] = march_axis;
    const float* axh[3] = {ax, ay, az};
    for (int k = 0; k < 3; ++k) {
        f->nk[k] = f->n[f->perm[k]];
        if (!build_axis_tables(axh[f->perm[k]], f->nk[k], f->tabs[k])) { delete f; return nullptr; }
    }
    const long long cells = (long long)nx * ny * nz;
    const double nc = 3.14207787e-4 * omega * omega;
    std::vector<float> ne_nc(cells);
    for (long long i = 0; i < cells; ++i) ne_nc[i] = normalise_ne(ne[i], nc);
    AxisCoef C[3];
    PackArgs P; memset(&P, 0, sizeof(P));
    for (int a = 0; a < 3; ++a) {
        C[a] = axis_coef(axh[a], f->n[a]);
        P.n[a] = f->n[a]; P.perm[a] = f->perm[a]; P.nk[a] = f->nk[a];
        P.st[a].a = C[a].a.data(); P.st[a].b = C[a].b.data(); P.st[a].c = C[a].c.data();
        P.st[a].two_dx = C[a].two_dx; P.st[a].dx0 = C[a].dx0; P.st[a].dxn = C[a].dxn;
        P.st[a].uniform = C[a].uniform; P.st[a].n = f->n[a];
    }
    const double c = 299792458.0;
    P.k32 = (float)(-0.5 * c * c); P.omega = omega; P.flags = flags;
    f->data.resize(cells);
    if (flags & 2) f->aux64.resize(cells);
    for (long long t = 0; t < cells; ++t) {
        double nm1;
        f->data[t] = pack_cell<double>(t, ne_nc.data(), ne, P, nm1);
        if (flags & 2) f->aux64[t] = nm1;
    }
    return f;
}

extern "C" void hh_field_destroy(void* h) { delete (HostField*)h; }

// gradients back in caller order [x][y][z]
extern "C" void hh_field_export(void* h, float* gx, float* gy, float* gz, float* aux) {
    HostField* f = (HostField*)h;
    PackArgs P; memset(&P, 0, sizeof(P));
    for (int a = 0; a < 3; ++a) { P.n[a] = f->n[a]; P.perm[a] = f->perm[a]; P.nk[a] = f->nk[a]; }
    const long long cells = (long long)f->n[0] * f->n[1] * f->n[2];
    for (long long t = 0; t < cells; ++t) {
        int ic[3];
        const long long idx = unpack_index(t, P, ic);
        float g[3];
        g[P.perm[0]] = f->data[t].x; g[P.perm[1]] = f->data[t].y; g[P.perm[2]] = f->data[t].z;
        gx[idx] = g[0]; gy[idx] = g[1]; gz[idx] = g[2]; aux[idx] = f->data[t].w;
    }
}

static void load(const HostField* f, const double* s, uint64_t n, uint64_t i, Ray<double>& r) {
    for (int k = 0; k < 3; ++k) { r.p[k] = s[(uint64_t)f->perm[k] * n + i]; r.v[k] = s[(uint64_t)(3 + f->perm[k]) * n + i]; }
    r.ph = s[7 * n + i];
}
static void store(const HostField* f, double* s, const double* s0, uint64_t n, uint64_t i, const Ray<double>& r) {
    for (int k = 0; k < 3; ++k) { s[(uint64_t)f->perm[k] * n + i] = r.p[k]; s[(uint64_t)(3 + f->perm[k]) * n + i] = r.v[k]; }
    s[6 * n + i] = s0[6 * n + i]; s[7 * n + i] = r.ph; s[8 * n + i] = s0[8 * n + i];
}

template <bool PH, bool A64>
static void rhs_t(const HostField* f, const double* s, uint64_t n, double* out, double omega) {
    FieldView<double> F = f->view64();
    for (uint64_t i = 0; i < n; ++i) {
        Ray<double> r; load(f, s, n, i, r);
        Deriv<double> d;
        CellCache<double, PH> cc;
        deriv<double, PH, A64>(F, cc, omega, r.p, r.v, d);
        for (int k = 0; k < 3; ++k) { out[(uint64_t)f->perm[k] * n + i] = d.dp[k]; out[(uint64_t)(3 + f->perm[k]) * n + i] = d.dv[k]; }
        out[6 * n + i] = 0; out[7 * n + i] = d.dph; out[8 * n + i] = 0;
    }
}
extern "C" void hh_rhs(void* h, const double* s, uint64_t n, double* out, double omega, int phase, int aux64) {
    const HostField* f = (const HostField*)h;
    if (!phase) rhs_t<false, false>(f, s, n, out, omega);
    else if (!aux64) rhs_t<true, false>(f, s, n, out, omega);
    else rhs_t<true, true>(f, s, n, out, omega);
}

// The cache-free evaluation of the adaptive integrators (rhs_direct): same interface as hh_rhs.
template <bool PH, bool A64>
static void rhs_direct_t(const HostField* f, const double* s, uint64_t n, double* out, double omega) {
    FieldView<double> F = f->view64();
    for (uint64_t i = 0; i < n; ++i) {
        Ray<double> r; load(f, s, n, i, r);
        Deriv<double> d;
        deriv_direct<double, PH, A64>(F, omega, r.p, r.v, d);
        for (int k = 0; k < 3; ++k) { out[(uint64_t)f->perm[k] * n + i] = d.dp[k]; out[(uint64_t)(3 + f->perm[k]) * n + i] = d.dv[k]; }
        out[6 * n + i] = 0; out[7 * n + i] = d.dph; out[8 * n + i] = 0;
    }
}
extern "C" void hh_rhs_direct(void* h, const double* s, uint64_t n, double* out, double omega, int phase, int aux64) {
    const HostField* f = (const HostField*)h;
    if (!phase) rhs_direct_t<false, false>(f, s, n, out, omega);
    else if (!aux64) rhs_direct_t<true, false>(f, s, n, out, omega);
    else rhs_direct_t<true, true>(f, s, n, out, omega);
}

// One persistent cell cache walked through the points in order (near = the fixed-step neighbour relocation, else the
// direct search of the adaptive steppers): must give what a fresh cache gives at every point.
template <bool NEARP>
static void rhs_walk_t(const HostField* f, const double* s, uint64_t n, double* out) {
    FieldView<double> F = f->view64();
    CellCache<double, false> cc;
    for (uint64_t i = 0; i < n; ++i) {
        Ray<double> r; load(f, s, n, i, r);
        double a[3], nm1;
        const bool in = rhs<double, false, false, NEARP>(F, cc, r.p[0], r.p[1], r.p[2], a[0], a[1], a[2], nm1);
        for (int k = 0; k < 3; ++k) { out[(uint64_t)f->perm[k] * n + i] = r.v[k]; out[(uint64_t)(3 + f->perm[k]) * n + i] = in ? a[k] : 0.0; }
        out[6 * n + i] = 0; out[7 * n + i] = 0; out[8 * n + i] = 0;
    }
}
extern "C" void hh_rhs_walk(void* h, const double* s, uint64_t n, double* out, int near_) {
    if (near_) rhs_walk_t<true>((const HostField*)h, s, n, out);
    else rhs_walk_t<false>((const HostField*)h, s, n, out);
}

template <typename T, bool PH, bool A64>
static void rk4_t(const HostField* f, const FieldView<T>& F, const double* s0, uint64_t n, int n_steps, double h,
                  double omega, int early, double* sf, uint32_t* steps) {
    for (uint64_t i = 0; i < n; ++i) {
        Ray<double> rd; load(f, s0, n, i, rd);
        Ray<T> r;
        for (int k = 0; k < 3; ++k) { r.p[k] = (T)rd.p[k]; r.v[k] = (T)rd.v[k]; }
        r.ph = (T)rd.ph;
        uint32_t it = 0;
        CellCache<T, PH> cc;
        for (; it < (uint32_t)n_steps; ++it)
            if (rk4_step<T, PH, A64>(F, cc, (T)h, (T)omega, r, early != 0) < 0) break;
        for (int k = 0; k < 3; ++k) { rd.p[k] = r.p[k]; rd.v[k] = r.v[k]; }
        rd.ph = r.ph;
        store(f, sf, s0, n, i, rd);
        if (steps) steps[i] = it;
    }
}
extern "C" void hh_rk4(void* h, const double* s0, uint64_t n, int n_steps, double hstep, double omega, int phase, int aux64,
            int early, int fp32, double* sf, uint32_t* steps) {
    const HostField* f = (const HostField*)h;
    if (fp32) {
        FieldView<float> F = f->view32();
        if (!phase) rk4_t<float, false, false>(f, F, s0, n, n_steps, hstep, omega, early, sf, steps);
        else rk4_t<float, true, false>(f, F, s0, n, n_steps, hstep, omega, early, sf, steps);
        return;
    }
    FieldView<double> F = f->view64();
    if (!phase) rk4_t<double, false, false>(f, F, s0, n, n_steps, hstep, omega, early, sf, steps);
    else if (!aux64) rk4_t<double, true, false>(f, F, s0, n, n_steps, hstep, omega, early, sf, steps);
    else rk4_t<double, true, true>(f, F, s0, n, n_steps, hstep, omega, early, sf, steps);
}

// per-ray adaptive driver: same control flow as k_propagate<.., SP_METHOD_RK45, ..>
template <bool PH, bool A64>
static void rk45_t(const HostField* f, const double* s0, uint64_t n, double t_end, double rtol, double atol, double omega,
                   int n_state, int cap_in, double* sf, uint32_t* attempts, uint32_t* nfev) {
    FieldView<double> F = f->view64();
    for (uint64_t i = 0; i < n; ++i) {
        Ray<double> r; load(f, s0, n, i, r);
        const double amp = s0[6 * n + i], pol = s0[8 * n + i];
        Deriv<double> fd; int touched = 0; uint32_t evals = 1;
        deriv_direct<double, PH, A64>(F, omega, r.p, r.v, fd);
        double h_abs = dp5_initial_step<double, PH, A64>(F, omega, t_end, rtol, atol, n_state, amp, pol, r, fd, touched);
        evals += 1;
        double t = 0; uint32_t n_att = 0;
        const uint32_t cap = cap_in > 0 ? (uint32_t)cap_in : (1u << 30);
        bool failed = false;
        while (t < t_end && !failed) {
            const double min_step = 10 * (nextafter(t, INFINITY) - t);
            if (h_abs < min_step) h_abs = min_step;
            bool rejected = false;
            for (;;) {
                if (n_att >= cap || h_abs < min_step) { failed = true; break; }
                double t_new = t + h_abs;
                if (t_new - t_end > 0) t_new = t_end;
                const double h = t_new - t;
                h_abs = fabs(h);
                Ray<double> rn; Deriv<double> fn; double esq;
                dp5_attempt<double, PH, A64>(F, omega, h, rtol, atol, r, fd, rn, fn, esq);
                ++n_att; evals += 6;
                const double en = sqrt(esq / n_state);
                if (en < 1) { h_abs *= dp5_factor<double>(en, true, rejected); t = t_new; r = rn; fd = fn; break; }
                h_abs *= dp5_factor<double>(en, false, rejected);
                rejected = true;
            }
        }
        store(f, sf, s0, n, i, r);
        if (attempts) attempts[i] = n_att;
        if (nfev) nfev[i] = evals;
    }
}
extern "C" void hh_rk45(void* h, const double* s0, uint64_t n, double t_end, double rtol, double atol, double omega, int phase,
             int aux64, int n_state, int cap, double* sf, uint32_t* attempts, uint32_t* nfev) {
    const HostField* f = (const HostField*)h;
    if (!phase) rk45_t<false, false>(f, s0, n, t_end, rtol, atol, omega, n_state, cap, sf, attempts, nfev);
    else if (!aux64) rk45_t<true, false>(f, s0, n, t_end, rtol, atol, omega, n_state, cap, sf, attempts, nfev);
    else rk45_t<true, true>(f, s0, n, t_end, rtol, atol, omega, n_state, cap, sf, attempts, nfev);
}

// per-ray Tsit5 + PID controller: the loop of the SP_METHOD_TSIT5 branch of k_propagate
template <bool PH, bool A64>
static void tsit5_t(const HostField* f, const double* s0, uint64_t n, double T_norm, double dt0, double rtol, double atol, double omega,
                    int n_state, int cap_in, double* sf, uint32_t* attempts, uint32_t* accepted) {
    FieldView<double> F = f->view64();
    for (uint64_t i = 0; i < n; ++i) {
        Ray<double> r; load(f, s0, n, i, r);
        double y[7], fy[7], yn[7], fn[7];
        for (int k = 0; k < 3; ++k) { y[k] = r.p[k]; y[3 + k] = r.v[k]; }
        y[6] = r.ph;
        tsit5_f<double, PH, A64>(F, omega, y, fy);
        double tau = 0.0, dt = dt0;
        uint32_t n_att = 0, n_acc = 0;
        const uint32_t cap = cap_in > 0 ? (uint32_t)cap_in : 10000u;
        while (tau < 1.0 && n_att < cap) {
            const bool last = tau + dt >= 1.0;
            const double d = last ? 1.0 - tau : dt;
            double esq;
            tsit5_attempt<double, PH, A64>(F, omega, d * T_norm, rtol, atol, y, fy, yn, fn, esq);
            ++n_att;
            const double en = sqrt(esq / (double)n_state);
            if (!(en == en)) break;
            const bool keep = en < 1.0;
            dt = d * pid_factor<double>(en, keep);
            if (keep) { tau = last ? 1.0 : tau + d; ++n_acc; for (int k = 0; k < 7; ++k) { y[k] = yn[k]; fy[k] = fn[k]; } }
        }
        for (int k = 0; k < 3; ++k) { r.p[k] = y[k]; r.v[k] = y[3 + k]; }
        r.ph = y[6];
        store(f, sf, s0, n, i, r);
        attempts[i] = n_att; accepted[i] = n_acc;
    }
}

extern "C" void hh_tsit5(void* h, const double* s0, uint64_t n, double T_norm, double dt0, double rtol, double atol, double omega, int phase,
                         int aux64, int n_state, int cap, double* sf, uint32_t* attempts, uint32_t* accepted) {
    const HostField* f = (const HostField*)h;
    if (!phase) tsit5_t<false, false>(f, s0, n, T_norm, dt0, rtol, atol, omega, n_state, cap, sf, attempts, accepted);
    else if (!aux64) tsit5_t<true, false>(f, s0, n, T_norm, dt0, rtol, atol, omega, n_state, cap, sf, attempts, accepted);
    else tsit5_t<true, true>(f, s0, n, T_norm, dt0, rtol, atol, omega, n_state, cap, sf, attempts, accepted);
}

// exit projection in the caller frame: kp/ka/kb are caller axes
extern "C" void hh_exit(void* h, const double* sf, uint64_t n, int p, int a, int b, double extent, double* rf) {
    const HostField* f = (const HostField*)h;
    int inv[3];
    for (int k = 0; k < 3; ++k) inv[f->perm[k]] = k;
    for (uint64_t i = 0; i < n; ++i) {
        Ray<double> r; load(f, sf, n, i, r);
        exit_project<double>(r, inv[p], inv[a], inv[b], extent, rf[i], rf[n + i], rf[2 * n + i], rf[3 * n + i]);
    }
}

struct HOp { int32_t kind, pad; double p0, p1, p2; };

extern "C" void hh_optics(const double* rf, const double* jf, uint64_t n, const HOp* ops, int n_ops, double wavelength, int input_mm,
               double* rf_out, double* jf_out) {
    std::vector<OpticOp> o(n_ops > 0 ? n_ops : 1);
    for (int i = 0; i < n_ops; ++i) { o[i].kind = ops[i].kind; o[i].p0 = ops[i].p0; o[i].p1 = ops[i].p1; o[i].p2 = ops[i].p2; }
    const double kw = wavelength > 0 ? 2.0 * 3.14159265358979323846 / wavelength : 0.0;
    const double nanv = NAN;
    for (uint64_t i = 0; i < n; ++i) {
        DetRay d; d.alive = true;
        const double unit = input_mm ? 1.0 : 1e3;
        d.x = rf[i] * unit; d.th = rf[n + i]; d.y = rf[2 * n + i] * unit; d.ph = rf[3 * n + i];
        d.ex_re = d.ex_im = d.ey_re = d.ey_im = 0;
        if (jf) { d.ex_re = jf[2 * i]; d.ex_im = jf[2 * i + 1]; d.ey_re = jf[2 * (n + i)]; d.ey_im = jf[2 * (n + i) + 1]; }
        run_optics(d, rf[i], rf[2 * n + i], o.data(), n_ops, jf != nullptr, kw);
        rf_out[i] = d.alive ? d.x : nanv; rf_out[n + i] = d.alive ? d.th : nanv;
        rf_out[2 * n + i] = d.alive ? d.y : nanv; rf_out[3 * n + i] = d.alive ? d.ph : nanv;
        if (jf_out) {
            jf_out[2 * i] = d.alive ? d.ex_re : nanv; jf_out[2 * i + 1] = d.alive ? d.ex_im : nanv;
            jf_out[2 * (n + i)] = d.alive ? d.ey_re : nanv; jf_out[2 * (n + i) + 1] = d.alive ? d.ey_im : nanv;
        }
    }
}

extern "C" void hh_bin(const double* v, uint64_t n, double lo, double hi, int nb, int right_inclusive, int32_t* out) {
    for (uint64_t i = 0; i < n; ++i) out[i] = bin_index(v[i], lo, hi, nb, right_inclusive != 0);
}

extern "C" void hh_beam(int beam_type, int probing_axis, double size_a, double size_b, double divergence, double start,
             uint64_t seed, uint64_t off, uint64_t n, double* s0) {
    BeamSpec B; B.beam_type = beam_type; B.probing_axis = probing_axis; B.size_a = size_a; B.size_b = size_b;
    B.divergence = divergence; B.start = start; B.seed = seed;
    for (uint64_t i = 0; i < n; ++i) {
        double s[6]; beam_ray(B, off + i, s);
        for (int k = 0; k < 6; ++k) s0[(uint64_t)k * n + i] = s[k];
        s0[6 * n + i] = 1.0; s0[7 * n + i] = 0.0; s0[8 * n + i] = 0.0;
    }
}

extern "C" void hh_philox(uint32_t k0, uint32_t k1, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t* out) {
    Philox p; p.k0 = k0; p.k1 = k1; p.block(c0, c1, c2, c3, out);
}

// debug/test helper: RHS evaluated with the float32 code path (state rounded to float32 first)
extern "C" void hh_rhs_fp32(void* hnd, const double* s, uint64_t n, double* out) {
    const HostField* f = (const HostField*)hnd;
    FieldView<float> F = f->view32();
    for (uint64_t i = 0; i < n; ++i) {
        float p[3], v[3];
        for (int k = 0; k < 3; ++k) { p[k] = (float)s[(uint64_t)f->perm[k] * n + i]; v[k] = (float)s[(uint64_t)(3 + f->perm[k]) * n + i]; }
        Deriv<float> d;
        CellCache<float, false> cc;
        deriv<float, false, false>(F, cc, 0.f, p, v, d);
        for (int k = 0; k < 3; ++k) { out[(uint64_t)f->perm[k] * n + i] = d.dp[k]; out[(uint64_t)(3 + f->perm[k]) * n + i] = d.dv[k]; }
        out[6 * n + i] = out[7 * n + i] = out[8 * n + i] = 0;
    }
}

// attenuation / Faraday channels: same repacking as sp_field_attach_channels (inputs [x][y][z], B as 3 grids)
extern "C" void hh_attach(void* hnd, const double* kappa, const double* ne, const double* bx, const double* by, const double* bz) {
    HostField* f = (HostField*)hnd;
    PackArgs P; memset(&P, 0, sizeof(P));
    for (int a = 0; a < 3; ++a) { P.n[a] = f->n[a]; P.perm[a] = f->perm[a]; P.nk[a] = f->nk[a]; }
    const double* b[3] = {bx, by, bz};
    const double* src[5] = {kappa, ne, b[f->perm[0]], b[f->perm[1]], b[f->perm[2]]};
    const long long cells = (long long)f->n[0] * f->n[1] * f->n[2];
    for (int c = 0; c < 5; ++c) {
        f->ext[c].clear();
        if (!src[c]) continue;
        f->ext[c].resize(cells);
        for (long long t = 0; t < cells; ++t) { int ic[3]; f->ext[c][t] = src[c][unpack_index(t, P, ic)]; }
    }
}

extern "C" void hh_rhs_ext(void* hnd, const double* s, uint64_t n, double* out, double omega, double verdet) {
    const HostField* f = (const HostField*)hnd;
    FieldView<double> F = f->view64();
    const ExtView X = f->ext_view(verdet, true, true);
    for (uint64_t i = 0; i < n; ++i) {
        Ray<double> r; load(f, s, n, i, r);
        Deriv<double> d; CellCache<double, true> cc;
        const int inside = deriv<double, true, true>(F, cc, omega, r.p, r.v, d);
        for (int k = 0; k < 3; ++k) { out[(uint64_t)f->perm[k] * n + i] = d.dp[k]; out[(uint64_t)(3 + f->perm[k]) * n + i] = d.dv[k]; }
        double x[5];
        ext_eval<true>(F, X, cc, inside != 0, r.p, x);
        out[6 * n + i] = x[0] * s[6 * n + i];
        out[7 * n + i] = d.dph;
        out[8 * n + i] = verdet * x[1] * (x[2] * r.v[0] + x[3] * r.v[1] + x[4] * r.v[2]);
    }
}

extern "C" void hh_rk4_ext(void* hnd, const double* s0, uint64_t n, int n_steps, double h, double omega, double verdet,
                           int early, double* sf) {
    const HostField* f = (const HostField*)hnd;
    FieldView<double> F = f->view64();
    const ExtView X = f->ext_view(verdet, true, true);
    for (uint64_t i = 0; i < n; ++i) {
        Ray<double> r; load(f, s0, n, i, r);
        ExtState e; e.amp = s0[6 * n + i]; e.pol = s0[8 * n + i];
        CellCache<double, true> cc;
        for (int it = 0; it < n_steps; ++it)
            if (rk4_step_ext<true, true>(F, X, cc, h, omega, true, r, e, early != 0) < 0) break;
        for (int k = 0; k < 3; ++k) { sf[(uint64_t)f->perm[k] * n + i] = r.p[k]; sf[(uint64_t)(3 + f->perm[k]) * n + i] = r.v[k]; }
        sf[6 * n + i] = e.amp; sf[7 * n + i] = r.ph; sf[8 * n + i] = e.pol;
    }
}

// per-ray adaptive solve over all nine rows (channels on): the loop of rk45x_integrate in synthpy_b200.cu
extern "C" void hh_rk45_ext(void* hnd, const double* s0, uint64_t n, double t_end, double rtol, double atol, double omega,
                            double verdet, double* sf, uint32_t* nfev) {
    const HostField* f = (const HostField*)hnd;
    FieldView<double> F = f->view64();
    const ExtView X = f->ext_view(verdet, true, true);
    for (uint64_t i = 0; i < n; ++i) {
        double y[9], fy[9], yn[9], fn[9];
        for (int k = 0; k < 3; ++k) { y[k] = s0[(uint64_t)f->perm[k] * n + i]; y[3 + k] = s0[(uint64_t)(3 + f->perm[k]) * n + i]; }
        for (int k = 6; k < 9; ++k) y[k] = s0[(uint64_t)k * n + i];
        CellCache<double, true> cc;
        int touched = 0; uint32_t evals = 2;
        deriv9<true, true>(F, X, cc, omega, true, y, fy);
        double h_abs = dp5_initial_step9<true, true>(F, X, cc, omega, true, t_end, rtol, atol, y, fy, touched);
        double t = 0;
        while (t < t_end) {
            const double min_step = 10 * (nextafter(t, INFINITY) - t);
            if (h_abs < min_step) h_abs = min_step;
            bool rejected = false, failed = false;
            for (;;) {
                if (h_abs < min_step) { failed = true; break; }
                double t_new = t + h_abs;
                if (t_new - t_end > 0) t_new = t_end;
                const double h = t_new - t;
                h_abs = fabs(h);
                double esq;
                dp5_attempt9<true, true>(F, X, cc, omega, true, h, rtol, atol, y, fy, yn, fn, esq);
                evals += 6;
                const double en = sqrt(esq / 9.0);
                if (en < 1) { h_abs *= dp5_factor<double>(en, true, rejected); t = t_new; for (int k = 0; k < 9; ++k) { y[k] = yn[k]; fy[k] = fn[k]; } break; }
                h_abs *= dp5_factor<double>(en, false, rejected);
                rejected = true;
            }
            if (failed) break;
        }
        for (int k = 0; k < 3; ++k) { sf[(uint64_t)f->perm[k] * n + i] = y[k]; sf[(uint64_t)(3 + f->perm[k]) * n + i] = y[3 + k]; }
        for (int k = 6; k < 9; ++k) sf[(uint64_t)k * n + i] = y[k];
        if (nfev) nfev[i] = evals;
    }
}

// ---- wave-optics step (fresnel_core.h): the loops below are the kernels of synthpy_b200.cu run serially ------------
#include <limits.h>

#include "../synthpy_b200/csrc/fresnel_core.h"

extern "C" void hh_scatter_to_grid(const double* px, const double* py, const double* val, int n_val, uint64_t n_pts,
                                   const int32_t* tri, uint64_t n_tri, const double* gx, const double* gy, int nx, int ny,
                                   double fill, double* out) {
    const size_t npix = (size_t)nx * ny;
    std::vector<int32_t> owner(npix, INT32_MAX);
    for (uint64_t t = 0; t < n_tri; ++t) {                                 // k_tri_owner
        const int32_t ia = tri[3 * t], ib = tri[3 * t + 1], ic = tri[3 * t + 2];
        const double ax = px[ia], ay = py[ia], bx = px[ib], by = py[ib], cx = px[ic], cy = py[ic];
        const double x0 = fmin(ax, fmin(bx, cx)), x1 = fmax(ax, fmax(bx, cx));
        const double y0 = fmin(ay, fmin(by, cy)), y1 = fmax(ay, fmax(by, cy));
        const double sx = (x1 - x0) * 1e-12, sy = (y1 - y0) * 1e-12;
        const int i0 = lower_bound_d(gx, nx, x0 - sx), j0 = lower_bound_d(gy, ny, y0 - sy);
        for (int j = j0; j < ny && gy[j] <= y1 + sy; ++j)
            for (int i = i0; i < nx && gx[i] <= x1 + sx; ++i) {
                double l0, l1, l2;
                if (bary2(ax, ay, bx, by, cx, cy, gx[i], gy[j], l0, l1, l2) && tri_inside(l0, l1, l2)) {
                    int32_t& o = owner[(size_t)j * nx + i];
                    if ((int32_t)t < o) o = (int32_t)t;
                }
            }
    }
    for (size_t p = 0; p < npix; ++p) {                                    // k_tri_interp
        const int32_t t = owner[p];
        if (t == INT32_MAX) {
            for (int v = 0; v < n_val; ++v) out[v * npix + p] = fill;
            continue;
        }
        const int32_t ia = tri[3 * (size_t)t], ib = tri[3 * (size_t)t + 1], ic = tri[3 * (size_t)t + 2];
        double l0, l1, l2;
        bary2(px[ia], py[ia], px[ib], py[ib], px[ic], py[ic], gx[p % nx], gy[p / nx], l0, l1, l2);
        for (int v = 0; v < n_val; ++v) {
            const double* w = val + (size_t)v * n_pts;
            out[v * npix + p] = l0 * w[ia] + l1 * w[ib] + l2 * w[ic];
        }
    }
}

extern "C" void hh_fresnel_prepare(const double* a, const double* b, int mode, int n0, int n1, int pad, double alpha, double* out) {
    const long long m0 = (2LL * pad + 1) * n0, m1 = (2LL * pad + 1) * n1;
    for (long long p = 0; p < m0 * m1; ++p) prepare_sample(a, b, mode, n0, n1, pad, alpha, p / m1, p % m1, out[2 * p], out[2 * p + 1]);
}

extern "C" void hh_fresnel_transfer(double* spec, int m0, int m1, double d0, double d1, double wavelength, double z, double sigma) {
    for (long long p = 0; p < (long long)m0 * m1; ++p)
        transfer_sample(spec[2 * p], spec[2 * p + 1], p / m1, p % m1, m0, m1, d0, d1, wavelength, z, sigma);
}

extern "C" void hh_window(int M, double alpha, double* w) {
    for (int i = 0; i < M; ++i) w[i] = tukey_w(i, M, alpha);
}

extern "C" void hh_reflect(int n, int lo, int hi, int32_t* out) {
    for (int i = lo; i < hi; ++i) out[i - lo] = (int32_t)reflect_idx(i, n);
}

// ---- turbulent-field noise (noise_core.h): the loops of k_noise_spectrum / k_noise_spectrum_box run serially -------
#include "../synthpy_b200/csrc/noise_core.h"

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
