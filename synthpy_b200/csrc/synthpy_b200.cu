// synthpy_b200 -- sm_100a kernels and the C ABI of include/synthpy_b200.h.
//
// Kernels (all hand-written for sm_100a; no library calls on the data path):
//   k_normalise_ne / k_pack_from_ne / k_pack_from_grads : field preparation (float32 stencil == np.gradient)
//   k_sort_keys / k_scan_* / k_sort_scatter             : counting sort of rays into coherent bundles
//   k_propagate<T, METHOD, PHASE, AUX64>                 : persistent ray integrator + fused optics/binning
//   k_joint_*                                           : the reference's joint-step RK45 (one h for all rays)
//   k_optics_image / k_finalize / k_rhs / k_beam        : stand-alone entry points
//
// Per-ray arithmetic lives in ray_core.h (shared with the CPU self-test build).
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <string>
#include <vector>

#include "../../include/synthpy_b200.h"
#include "ray_core.h"
#include "field_prep.h"

using namespace sp;

// ------------------------------------------------------------------------------------------------ errors
static thread_local std::string g_err;
static std::atomic<uint64_t> g_launches{0};

static int fail(int code, const std::string& msg) { g_err = msg; return code; }
#define CU(x)                                                                                            \
    do {                                                                                                 \
        cudaError_t e_ = (x);                                                                            \
        if (e_ != cudaSuccess)                                                                           \
            return fail(SP_ECUDA, std::string(#x) + ": " + cudaGetErrorString(e_));                      \
    } while (0)
#define LAUNCH_CHECK()                                                                                   \
    do {                                                                                                 \
        g_launches.fetch_add(1);                                                                         \
        CU(cudaGetLastError());                                                                          \
    } while (0)

extern "C" int sp_version(void) { return SP_ABI_VERSION; }
extern "C" const char* sp_last_error(void) { return g_err.c_str(); }
extern "C" uint64_t sp_launch_count(void) { return g_launches.load(); }

// ------------------------------------------------------------------------------------------------- field
struct sp_field {
    int n[3];          // caller-frame dims nx, ny, nz
    int perm[3];       // kernel axis k -> caller axis
    int nk[3];         // kernel-frame dims nu, nv, nw
    f4* data = nullptr;
    double* aux64 = nullptr;
    double* ext[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};   // kappa, ne, B_u, B_v, B_w (kernel frame)
    d2* tab64[3] = {nullptr, nullptr, nullptr};   // kernel-frame axis tables
    f2* tab32[3] = {nullptr, nullptr, nullptr};
    double g0[3], inv_d[3], lo[3], hi[3];         // kernel frame
    int device = 0;
    uint64_t bytes = 0;
};

template <typename T> static FieldView<T> make_view(const sp_field* f);
template <> FieldView<double> make_view<double>(const sp_field* f) {
    FieldView<double> V;
    V.data = f->data; V.aux64 = f->aux64;
    for (int k = 0; k < 3; ++k) {
        V.ax[k].tab = f->tab64[k]; V.ax[k].g0 = f->g0[k]; V.ax[k].inv_d = f->inv_d[k];
        V.ax[k].lo = f->lo[k]; V.ax[k].hi = f->hi[k]; V.ax[k].n = f->nk[k];
    }
    V.su = (long long)f->nk[1] * f->nk[2]; V.sv = f->nk[2];
#ifdef SP_BRICK
    V.bsv = (long long)((f->nk[2] + 7) >> 3) * 512; V.bsu = (long long)((f->nk[1] + 7) >> 3) * V.bsv;
#endif
    return V;
}
template <> FieldView<float> make_view<float>(const sp_field* f) {
    FieldView<float> V;
    V.data = f->data; V.aux64 = f->aux64;
    for (int k = 0; k < 3; ++k) {
        V.ax[k].tab = f->tab32[k]; V.ax[k].g0 = (float)f->g0[k]; V.ax[k].inv_d = (float)f->inv_d[k];
        V.ax[k].lo = (float)f->lo[k]; V.ax[k].hi = (float)f->hi[k]; V.ax[k].n = f->nk[k];
    }
    V.su = (long long)f->nk[1] * f->nk[2]; V.sv = f->nk[2];
#ifdef SP_BRICK
    V.bsv = (long long)((f->nk[2] + 7) >> 3) * 512; V.bsu = (long long)((f->nk[1] + 7) >> 3) * V.bsv;
#endif
    return V;
}

template <typename NE>
__global__ void k_normalise_ne(const NE* __restrict__ ne, float* __restrict__ out, long long total, double nc) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < total; i += stride) out[i] = normalise_ne(ne[i], nc);
}

// One thread per packed cell; neighbouring threads are neighbours along w (coalesced float4 stores).
template <typename NE>
__global__ void k_pack_from_ne(const float* __restrict__ ne_nc, const NE* __restrict__ ne, f4* __restrict__ out,
                               double* __restrict__ aux64, PackArgs P) {
    const long long total = (long long)P.nk[0] * P.nk[1] * P.nk[2];
    long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long gstride = (long long)gridDim.x * blockDim.x;
    for (; t < total; t += gstride) {
        double nm1;
        out[packed_slot(t, P)] = pack_cell(t, ne_nc, ne, P, nm1);
        if (aux64) aux64[t] = nm1;
    }
}

__global__ void k_pack_from_grads(const float* __restrict__ gx, const float* __restrict__ gy,
                                  const float* __restrict__ gz, const float* __restrict__ aux32,
                                  const double* __restrict__ aux64_in, f4* __restrict__ out,
                                  double* __restrict__ aux64, PackArgs P) {
    const long long total = (long long)P.nk[0] * P.nk[1] * P.nk[2];
    long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long gstride = (long long)gridDim.x * blockDim.x;
    for (; t < total; t += gstride) {
        int ic[3];
        const long long idx = unpack_index(t, P, ic);
        const float g[3] = {gx[idx], gy[idx], gz[idx]};
        f4 v; v.x = g[P.perm[0]]; v.y = g[P.perm[1]]; v.z = g[P.perm[2]];
        v.w = aux32 ? aux32[idx] : (aux64_in ? (float)aux64_in[idx] : 0.f);
        if (aux64 && aux64_in) aux64[t] = aux64_in[idx];
        out[packed_slot(t, P)] = v;
    }
}

__global__ void k_export_grads(const f4* __restrict__ in, float* gx, float* gy, float* gz, float* aux, PackArgs P) {
    const long long total = (long long)P.nk[0] * P.nk[1] * P.nk[2];
    long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long gstride = (long long)gridDim.x * blockDim.x;
    for (; t < total; t += gstride) {
        int ic[3];
        const long long idx = unpack_index(t, P, ic);
        const f4 v = in[packed_slot(t, P)];
        float g[3];
        g[P.perm[0]] = v.x; g[P.perm[1]] = v.y; g[P.perm[2]] = v.z;
        if (gx) gx[idx] = g[0];
        if (gy) gy[idx] = g[1];
        if (gz) gz[idx] = g[2];
        if (aux) aux[idx] = v.w;
    }
}

static int field_common(sp_field* f, const float* axh[3], int nx, int ny, int nz, int march_axis, cudaStream_t st) {
    if (nx < 2 || ny < 2 || nz < 2) return fail(SP_EINVAL, "grid needs at least 2 nodes per axis");
    if (march_axis < 0 || march_axis > 2) return fail(SP_EINVAL, "march_axis must be 0, 1 or 2");
    f->n[0] = nx; f->n[1] = ny; f->n[2] = nz;
    f->perm[0] = (march_axis + 1) % 3; f->perm[1] = (march_axis + 2) % 3; f->perm[2] = march_axis;
    CU(cudaGetDevice(&f->device));
    for (int k = 0; k < 3; ++k) {
        const int ca = f->perm[k], n = f->n[ca];
        AxisTables T;
        if (!build_axis_tables(axh[ca], n, T)) return fail(SP_EINVAL, "axes must be strictly ascending");
        f->nk[k] = n;
        std::vector<d2>& t64 = T.t64; std::vector<f2>& t32 = T.t32;
        f->g0[k] = T.g0; f->lo[k] = T.lo; f->hi[k] = T.hi; f->inv_d[k] = T.inv_d;
        CU(cudaMalloc(&f->tab64[k], n * sizeof(d2)));
        CU(cudaMalloc(&f->tab32[k], n * sizeof(f2)));
        CU(cudaMemcpyAsync(f->tab64[k], t64.data(), n * sizeof(d2), cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(f->tab32[k], t32.data(), n * sizeof(f2), cudaMemcpyHostToDevice, st));
        CU(cudaStreamSynchronize(st));   // host vectors go out of scope
        f->bytes += n * (sizeof(d2) + sizeof(f2));
    }
#ifdef SP_BRICK
    const size_t cells = (size_t)((f->nk[0] + 7) >> 3) * ((f->nk[1] + 7) >> 3) * ((f->nk[2] + 7) >> 3) * 512;    // padded to whole bricks
#else
    const size_t cells = (size_t)nx * ny * nz;
#endif
    CU(cudaMalloc(&f->data, cells * sizeof(f4)));
    CU(cudaMemsetAsync(f->data, 0, cells * sizeof(f4), st));
    f->bytes += cells * sizeof(f4);
    return SP_OK;
}

static PackArgs pack_args(const sp_field* f) {
    PackArgs P; memset(&P, 0, sizeof(P));
    for (int k = 0; k < 3; ++k) { P.n[k] = f->n[k]; P.perm[k] = f->perm[k]; P.nk[k] = f->nk[k]; }
    return P;
}

static int pack_grid(long long total) {
    long long b = (total + 255) / 256;
    return (int)(b > 148 * 32 ? 148 * 32 : (b < 1 ? 1 : b));
}

__global__ void k_repack_f64(const double* __restrict__ in, double* __restrict__ out, PackArgs P) {
    const long long total = (long long)P.nk[0] * P.nk[1] * P.nk[2];
    long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long gstride = (long long)gridDim.x * blockDim.x;
    for (; t < total; t += gstride) {
        int ic[3];
        out[t] = in[unpack_index(t, P, ic)];
    }
}

extern "C" int sp_field_attach_channels(sp_field* f, const double* kappa_dev, const double* ne_dev, const double* bx_dev,
                                        const double* by_dev, const double* bz_dev, void* stream) {
    if (!f) return fail(SP_EINVAL, "null field");
    const long long cells = (long long)f->n[0] * f->n[1] * f->n[2];
    const double* b_caller[3] = {bx_dev, by_dev, bz_dev};
    const double* src[5] = {kappa_dev, ne_dev, b_caller[f->perm[0]], b_caller[f->perm[1]], b_caller[f->perm[2]]};
    PackArgs P = pack_args(f);
    for (int c = 0; c < 5; ++c) {
        cudaFree(f->ext[c]); f->ext[c] = nullptr;
        if (!src[c]) continue;
        CU(cudaMalloc(&f->ext[c], cells * sizeof(double)));
        f->bytes += cells * sizeof(double);
        k_repack_f64<<<pack_grid(cells), 256, 0, (cudaStream_t)stream>>>(src[c], f->ext[c], P);
        LAUNCH_CHECK();
    }
    return SP_OK;
}

static ExtView make_ext(const sp_field* f, double verdet, int flags) {
    ExtView X;
    X.verdet = verdet;
    X.ch[0] = (flags & SP_FLAG_ATTEN) ? f->ext[0] : nullptr;
    for (int c = 1; c < 5; ++c) X.ch[c] = (flags & SP_FLAG_FARADAY) ? f->ext[c] : nullptr;
    return X;
}

extern "C" int sp_field_destroy(sp_field* f) {
    if (!f) return SP_OK;
    cudaFree(f->data); cudaFree(f->aux64);
    for (int c = 0; c < 5; ++c) cudaFree(f->ext[c]);
    for (int k = 0; k < 3; ++k) { cudaFree(f->tab64[k]); cudaFree(f->tab32[k]); }
    delete f;
    return SP_OK;
}

extern "C" uint64_t sp_field_bytes(const sp_field* f) { return f ? f->bytes : 0; }

extern "C" int sp_field_create(sp_field** out, const void* ne_dev, int ne_is_f64, const float* ax_x_host,
                               const float* ax_y_host, const float* ax_z_host, int nx, int ny, int nz,
                               double omega, int march_axis, int flags, void* stream) {
    if (!out || !ne_dev || !ax_x_host || !ax_y_host || !ax_z_host) return fail(SP_EINVAL, "null argument");
    cudaStream_t st = (cudaStream_t)stream;
    sp_field* f = new sp_field();
    const float* axh[3] = {ax_x_host, ax_y_host, ax_z_host};
    int rc = field_common(f, axh, nx, ny, nz, march_axis, st);
    if (rc) { sp_field_destroy(f); return rc; }
    const long long cells = (long long)nx * ny * nz;
    float* ne_nc = nullptr;
    float* coef = nullptr;
    auto cleanup = [&]() { cudaFree(ne_nc); cudaFree(coef); };
    PackArgs P = pack_args(f);
    // coefficient tables
    size_t ncoef = 3 * (size_t)(nx + ny + nz);
    std::vector<float> hc(ncoef);
    size_t off = 0;
    AxisCoef C[3];
    size_t offs[3];
    for (int a = 0; a < 3; ++a) {
        C[a] = axis_coef(axh[a], f->n[a]);
        offs[a] = off;
        for (int i = 0; i < f->n[a]; ++i) { hc[off + i] = C[a].a[i]; hc[off + f->n[a] + i] = C[a].b[i]; hc[off + 2 * f->n[a] + i] = C[a].c[i]; }
        off += 3 * (size_t)f->n[a];
    }
#define CUF(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { cleanup(); sp_field_destroy(f); return fail(SP_ECUDA, std::string(#x) + ": " + cudaGetErrorString(e_)); } } while (0)
    CUF(cudaMalloc(&ne_nc, cells * sizeof(float)));
    CUF(cudaMalloc(&coef, ncoef * sizeof(float)));
    CUF(cudaMemcpyAsync(coef, hc.data(), ncoef * sizeof(float), cudaMemcpyHostToDevice, st));
    for (int a = 0; a < 3; ++a) {
        P.st[a].a = coef + offs[a]; P.st[a].b = coef + offs[a] + f->n[a]; P.st[a].c = coef + offs[a] + 2 * f->n[a];
        P.st[a].two_dx = C[a].two_dx; P.st[a].dx0 = C[a].dx0; P.st[a].dxn = C[a].dxn;
        P.st[a].uniform = C[a].uniform; P.st[a].n = f->n[a];
    }
    const double c = 299792458.0;
    P.k32 = (float)(-0.5 * c * c);
    P.omega = omega; P.flags = flags;
    const double nc = 3.14207787e-4 * omega * omega;
    if (flags & SP_FIELD_PHASE_F64) {
        CUF(cudaMalloc(&f->aux64, cells * sizeof(double)));
        f->bytes += cells * sizeof(double);
    }
    const int grid = pack_grid(cells);
    if (ne_is_f64) {
        k_normalise_ne<double><<<grid, 256, 0, st>>>((const double*)ne_dev, ne_nc, cells, nc);
        g_launches++; CUF(cudaGetLastError());
        k_pack_from_ne<double><<<grid, 256, 0, st>>>(ne_nc, (const double*)ne_dev, f->data, f->aux64, P);
    } else {
        k_normalise_ne<float><<<grid, 256, 0, st>>>((const float*)ne_dev, ne_nc, cells, nc);
        g_launches++; CUF(cudaGetLastError());
        k_pack_from_ne<float><<<grid, 256, 0, st>>>(ne_nc, (const float*)ne_dev, f->data, f->aux64, P);
    }
    g_launches++; CUF(cudaGetLastError());
    CUF(cudaStreamSynchronize(st));   // temporaries are freed below; creation is a one-off
#undef CUF
    cleanup();
    *out = f;
    return SP_OK;
}

extern "C" int sp_field_create_from_gradients(sp_field** out, const float* gx_dev, const float* gy_dev,
                                              const float* gz_dev, const float* aux_f32_dev,
                                              const double* aux_f64_dev, const float* ax_x_host,
                                              const float* ax_y_host, const float* ax_z_host, int nx, int ny,
                                              int nz, int march_axis, void* stream) {
    if (!out || !gx_dev || !gy_dev || !gz_dev || !ax_x_host || !ax_y_host || !ax_z_host)
        return fail(SP_EINVAL, "null argument");
    cudaStream_t st = (cudaStream_t)stream;
    sp_field* f = new sp_field();
    const float* axh[3] = {ax_x_host, ax_y_host, ax_z_host};
    int rc = field_common(f, axh, nx, ny, nz, march_axis, st);
    if (rc) { sp_field_destroy(f); return rc; }
    const long long cells = (long long)nx * ny * nz;
    if (aux_f64_dev) {
        if (cudaMalloc(&f->aux64, cells * sizeof(double)) != cudaSuccess) { sp_field_destroy(f); return fail(SP_ENOMEM, "aux64"); }
        f->bytes += cells * sizeof(double);
    }
    PackArgs P = pack_args(f);
    k_pack_from_grads<<<pack_grid(cells), 256, 0, st>>>(gx_dev, gy_dev, gz_dev, aux_f32_dev, aux_f64_dev, f->data,
                                                        f->aux64, P);
    g_launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { sp_field_destroy(f); return fail(SP_ECUDA, cudaGetErrorString(e)); }
    *out = f;
    return SP_OK;
}

extern "C" int sp_field_export_gradients(const sp_field* f, float* gx_dev, float* gy_dev, float* gz_dev,
                                         float* aux_dev, void* stream) {
    if (!f) return fail(SP_EINVAL, "null field");
    PackArgs P = pack_args(f);
    const long long cells = (long long)f->n[0] * f->n[1] * f->n[2];
    k_export_grads<<<pack_grid(cells), 256, 0, (cudaStream_t)stream>>>(f->data, gx_dev, gy_dev, gz_dev, aux_dev, P);
    LAUNCH_CHECK();
    return SP_OK;
}

// -------------------------------------------------------------------------------------- detector channels
#ifndef SP_RK4F_MIN_BLOCKS
#define SP_RK4F_MIN_BLOCKS 1
#endif
#ifndef SP_RK45_MIN_BLOCKS
#define SP_RK45_MIN_BLOCKS 4
#endif
#ifndef SP_RK4_MIN_BLOCKS
#define SP_RK4_MIN_BLOCKS 4
#endif
#define SP_METHOD_RK4X 3      // internal: RK4 with the attenuation / Faraday channels (float64)
#define SP_METHOD_RK45X 4     // internal: per-ray Dormand-Prince over all nine rows (channels on, float64)
#define SP_METHOD_RK45B 5     // internal: Dormand-Prince with one step size per 32-ray bundle (SP_FLAG_BUNDLE_STEP)
#define SP_MAX_OPS 16
#define SP_MAX_CHANNELS 4

struct ChannelDev {
    OpticOp ops[SP_MAX_OPS];
    int n_ops, kind, nx, ny, with_E, input_mm;
    double kwave, x_lo, x_hi, y_lo, y_hi;
    unsigned long long* counts;
    long long* planes;
};

static int channel_to_dev(const sp_channel* c, ChannelDev& d) {
    if (c->n_ops < 0 || c->n_ops > SP_MAX_OPS) return fail(SP_EINVAL, "too many optic ops (max 16)");
    memset(&d, 0, sizeof(d));
    for (int i = 0; i < c->n_ops; ++i) {
        d.ops[i].kind = c->ops_host[i].kind;
        d.ops[i].p0 = c->ops_host[i].p0; d.ops[i].p1 = c->ops_host[i].p1; d.ops[i].p2 = c->ops_host[i].p2;
        if (d.ops[i].kind < 0 || d.ops[i].kind > SP_OP_REF_BEAM) return fail(SP_EINVAL, "unknown optic op");
    }
    d.n_ops = c->n_ops; d.input_mm = c->input_mm;
    d.kind = c->image.kind; d.nx = c->image.nx; d.ny = c->image.ny;
    d.x_lo = c->image.x_lo; d.x_hi = c->image.x_hi; d.y_lo = c->image.y_lo; d.y_hi = c->image.y_hi;
    d.counts = (unsigned long long*)c->image.counts_dev; d.planes = (long long*)c->image.planes_dev;
    d.with_E = (c->image.kind == SP_IMG_INTERFEROGRAM);
    d.kwave = c->wavelength > 0 ? 2.0 * 3.14159265358979323846 / c->wavelength : 0.0;
    if (d.kind < SP_IMG_HISTOGRAM || d.kind > SP_IMG_STOKES) return fail(SP_EINVAL, "unknown image kind");
    if (d.kind == SP_IMG_HISTOGRAM && !d.counts && d.nx > 0) return fail(SP_EINVAL, "histogram channel without counts buffer");
    if (d.kind == SP_IMG_INTERFEROGRAM && !d.planes && d.nx > 0) return fail(SP_EINVAL, "interferogram channel without planes buffer");
    if (d.kind == SP_IMG_STOKES && !d.planes && d.nx > 0) return fail(SP_EINVAL, "Stokes channel without planes buffer");
    if (d.kind == SP_IMG_STOKES)
        for (int i = 0; i < d.n_ops; ++i)     // a reference beam added to Ey would be counted as a polarisation change
            if (d.ops[i].kind == SP_OP_REF_BEAM) return fail(SP_EINVAL, "Stokes channel cannot contain a reference beam (ref_beam)");
    return SP_OK;
}

// Detector binning of one ray.  Lanes that hit the same pixel are aggregated in the warp: __match_any_sync groups
// them, every lane of a group sums the group's contributions in lane order over shuffles, and the group's lowest lane
// issues the atomics (rays are bundled coherently, so neighbouring lanes land in neighbouring pixels).
// Histogram: one 64-bit count.  Interferogram: the four sums of complex E are accumulated in FIXED POINT (int64,
// SP_PLANE_FRAC_BITS fractional bits): integer addition is associative, so an image does not depend on the order in
// which warps, kernels, chunks or GPUs contribute -- run-to-run and partition-to-partition identical, like the
// counts -- at a quantisation of 2^-40 per contribution (|E| <= amp + 1 ~ 2; range +-2^23 per pixel).
// Stokes: one 64-bit count and I, Q, U of the ray's Jones vector at the detector, fixed point with SP_STOKES_FRAC_BITS
// fractional bits (a pixel holds +-2^31: 2^31 contributions of unit intensity).  The
// optics are ray-transfer matrices and the E-phase advance multiplies both Jones components by the same unit factor,
// so the Stokes parameters do not depend on it: Stokes channels run with with_E = 0.
// Returns 1 if binned.
// (a NaN amplitude contributes nothing -- the reference would poison the pixel with NaN -- and values beyond the
// per-contribution range (+-2^22 for interferogram planes, +-2^20 for Stokes planes) saturate instead of wrapping)
template <int FRAC_BITS>
__device__ __forceinline__ long long to_fixed(double v, double lim) {
    v = (v == v) ? fmin(fmax(v, -lim), lim) : 0.0;
    return __double2ll_rn(v * (double)(1ll << FRAC_BITS));
}
__device__ __forceinline__ long long to_plane_fixed(double v) { return to_fixed<SP_PLANE_FRAC_BITS>(v, 4194304.0); }
__device__ __forceinline__ long long to_stokes_fixed(double v) { return to_fixed<SP_STOKES_FRAC_BITS>(v, 1048576.0); }

__device__ __forceinline__ int bin_ray(const ChannelDev& ch, const DetRay& d, bool active) {
    int pix = -1;
    if (active && d.alive && ch.nx > 0) {
        const bool hist = (ch.kind != SP_IMG_INTERFEROGRAM);        // histogram edges for counts and Stokes images
        const int ix = bin_index(d.x, ch.x_lo, ch.x_hi, ch.nx, hist);
        const int iy = bin_index(d.y, ch.y_lo, ch.y_hi, ch.ny, hist);
        if (ix >= 0 && iy >= 0) pix = iy * ch.nx + ix;
        SP_ASSERT(pix < ch.nx * ch.ny && ix < ch.nx && iy < ch.ny);
    }
    const unsigned peers = __match_any_sync(__activemask(), pix);
    const bool leader = pix >= 0 && (__ffs(peers) - 1) == (int)(threadIdx.x & 31);
    if (ch.kind == SP_IMG_HISTOGRAM) {
        if (leader) atomicAdd(ch.counts + pix, (unsigned long long)__popc(peers));
    } else {
        long long v0 = 0, v1 = 0, v2 = 0, v3 = 0;
        if (pix >= 0) {
            if (ch.kind == SP_IMG_STOKES) {         // count, I = |Ex|^2 + |Ey|^2, Q = |Ex|^2 - |Ey|^2, U = 2 Re(Ex conj(Ey))
                const double xx = d.ex_re * d.ex_re + d.ex_im * d.ex_im, yy = d.ey_re * d.ey_re + d.ey_im * d.ey_im;
                const double u = 2.0 * (d.ex_re * d.ey_re + d.ex_im * d.ey_im);
                v0 = 1; v1 = to_stokes_fixed(xx + yy); v2 = to_stokes_fixed(xx - yy); v3 = to_stokes_fixed(u);
            } else {
                v0 = to_plane_fixed(d.ex_re); v1 = to_plane_fixed(d.ex_im); v2 = to_plane_fixed(d.ey_re); v3 = to_plane_fixed(d.ey_im);
            }
        }
        if (peers & (peers - 1)) {                       // more than one lane on this pixel (coarse images): sum the group
            long long s0 = 0, s1 = 0, s2 = 0, s3 = 0;
            for (unsigned m = peers; m; m &= m - 1) {
                const int src = __ffs(m) - 1;
                s0 += __shfl_sync(peers, v0, src); s1 += __shfl_sync(peers, v1, src);
                s2 += __shfl_sync(peers, v2, src); s3 += __shfl_sync(peers, v3, src);
            }
            v0 = s0; v1 = s1; v2 = s2; v3 = s3;
        }
        if (leader) {
            const size_t plane = (size_t)ch.nx * ch.ny;
            unsigned long long* p = (unsigned long long*)ch.planes + pix;
            atomicAdd(p, (unsigned long long)v0);
            atomicAdd(p + plane, (unsigned long long)v1);
            atomicAdd(p + 2 * plane, (unsigned long long)v2);
            atomicAdd(p + 3 * plane, (unsigned long long)v3);
        }
    }
    return pix >= 0;
}

struct Epilogue {
    double* sf; double* rf; double* jf; uint32_t* steps;
    int n_channels;
    ChannelDev ch[SP_MAX_CHANNELS];
};

// --------------------------------------------------------------------------------------------- ray sorting
struct SortArgs {
    const double* s0; uint64_t n_total;        // caller arrays hold n_total rays (row stride)
    uint64_t chunk_off; uint32_t chunk_n;      // this chunk = rays [chunk_off, chunk_off + chunk_n)
    BeamSpec beam; int use_beam; uint64_t ray_offset;
    int perm[3];
    double g0u, inv_du, g0v, inv_dv; int nu, nv;
    int key_shift; uint32_t n_keys;
};

__device__ __forceinline__ uint32_t part1by1(uint32_t x) {
    x &= 0x0000ffffu; x = (x | (x << 8)) & 0x00ff00ffu; x = (x | (x << 4)) & 0x0f0f0f0fu;
    x = (x | (x << 2)) & 0x33333333u; x = (x | (x << 1)) & 0x55555555u;
    return x;
}

__device__ __forceinline__ void load_ray_caller(const double* s0, uint64_t n_total, uint64_t gi, const BeamSpec& B,
                                                int use_beam, uint64_t ray_offset, double s[6]) {
    if (use_beam) beam_ray(B, ray_offset + gi, s);
    else {
#pragma unroll
        for (int k = 0; k < 6; ++k) s[k] = s0[(uint64_t)k * n_total + gi];
    }
}

// Key = Morton code of the (u, v) cell column the ray starts in: rays of one warp then walk the same few
// 128-byte lines of the field for their whole flight.
__global__ void k_sort_keys(SortArgs A, uint32_t* __restrict__ keys, uint32_t* __restrict__ hist) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= A.chunk_n) return;
    double s[6];
    load_ray_caller(A.s0, A.n_total, A.chunk_off + i, A.beam, A.use_beam, A.ray_offset, s);
    const double pu = s[A.perm[0]], pv = s[A.perm[1]];
    int iu = floor_to_int((pu - A.g0u) * A.inv_du), iv = floor_to_int((pv - A.g0v) * A.inv_dv);
    iu = min(max(iu, 0), A.nu - 1); iv = min(max(iv, 0), A.nv - 1);
    uint32_t key = (part1by1((uint32_t)iu) | (part1by1((uint32_t)iv) << 1)) >> A.key_shift;
    key = min(key, A.n_keys - 1);
    keys[i] = key;
    atomicAdd(hist + key, 1u);
}

// Exclusive scan of the key histogram (n_keys <= 4 Mi) in three coalesced passes: every 1024-thread block scans a
// tile of 4096 counts in place (16 bytes per thread, warp shuffles + one shared-memory hop) and publishes the tile
// total; one block scans the <= 1024 totals; the tiles add their offset.  (Round 1 used one block whose threads each
// walked a private 4096-element slice -- uncoalesced -- and a serial pass over 1024 partial sums in thread 0.)
#define SP_SCAN_TILE 4096
__device__ __forceinline__ uint32_t block_exclusive_scan_1024(uint32_t v, uint32_t* total) {
    __shared__ uint32_t warp_sum[32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
    if (lane == 31) warp_sum[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        uint32_t w = warp_sum[lane], wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, wi, o); if (lane >= o) wi += t; }
        warp_sum[lane] = wi - w;                           // exclusive prefix of the warp totals
        if (lane == 31 && total) *total = wi;
    }
    __syncthreads();
    return inc - v + warp_sum[wid];
}

__global__ void __launch_bounds__(1024) k_scan_tiles(uint32_t* __restrict__ data, uint32_t n, uint32_t* __restrict__ tile_sums) {
    const uint32_t i0 = blockIdx.x * SP_SCAN_TILE + threadIdx.x * 4;
    uint32_t a[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) a[k] = (i0 + k < n) ? data[i0 + k] : 0u;
    const uint32_t mine = a[0] + a[1] + a[2] + a[3];
    __shared__ uint32_t tot;
    uint32_t run = block_exclusive_scan_1024(mine, &tot);
#pragma unroll
    for (int k = 0; k < 4; ++k) { if (i0 + k < n) data[i0 + k] = run; run += a[k]; }
    if (threadIdx.x == 0) tile_sums[blockIdx.x] = tot;
}

__global__ void __launch_bounds__(1024) k_scan_tops(uint32_t* __restrict__ tile_sums, uint32_t n_tiles) {
    const uint32_t v = threadIdx.x < n_tiles ? tile_sums[threadIdx.x] : 0u;
    const uint32_t ex = block_exclusive_scan_1024(v, nullptr);
    if (threadIdx.x < n_tiles) tile_sums[threadIdx.x] = ex;
}

__global__ void __launch_bounds__(1024) k_scan_add(uint32_t* __restrict__ data, uint32_t n, const uint32_t* __restrict__ tile_sums) {
    const uint32_t off = tile_sums[blockIdx.x];
    const uint32_t i0 = blockIdx.x * SP_SCAN_TILE + threadIdx.x * 4;
#pragma unroll
    for (int k = 0; k < 4; ++k) if (i0 + k < n) data[i0 + k] += off;
}

__global__ void k_sort_scatter(const uint32_t* __restrict__ keys, uint32_t* __restrict__ cursor,
                               uint32_t* __restrict__ order, uint32_t n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t pos = atomicAdd(cursor + keys[i], 1u);
    SP_ASSERT(pos < n);
    order[pos] = i;
}

// The scatter above fills each key's segment in atomic (i.e. arbitrary) order; sorting every segment by ray index
// makes the bundle order -- and with it the membership of the bundles of the bundle-step mode -- reproducible from run
// to run.  Segments are normally short (rays per cell column): one thread each, insertion sort.  Segments longer than
// SP_LONG_SEGMENT (a pencil beam inside one column, or many rays on a coarse grid) are listed and sorted by
// k_sort_fix_long below.
#define SP_LONG_SEGMENT 2048u
__global__ void k_sort_fix(const uint32_t* __restrict__ seg_end, uint32_t* __restrict__ order, uint32_t n_keys,
                           uint32_t* __restrict__ long_list, uint32_t* __restrict__ long_count) {
    const uint32_t key = blockIdx.x * blockDim.x + threadIdx.x;
    if (key >= n_keys) return;
    const uint32_t b = key ? seg_end[key - 1] : 0u, e = seg_end[key];
    if (e - b > SP_LONG_SEGMENT) {
        const uint32_t slot = atomicAdd(long_count, 1u);
        SP_ASSERT((uint64_t)slot * SP_LONG_SEGMENT < (uint64_t)seg_end[n_keys - 1] + SP_LONG_SEGMENT);
        long_list[slot] = key;
        return;
    }
    for (uint32_t i = b + 1; i < e; ++i) {
        const uint32_t v = order[i];
        uint32_t j = i;
        while (j > b && order[j - 1] > v) { order[j] = order[j - 1]; --j; }
        order[j] = v;
    }
}

// Long segments: one 256-thread block per listed segment runs a stable LSD radix sort of the ray indices (8-bit digits,
// tiles of 256 elements taken in order; ranks inside a tile from __match_any_sync per warp + an 8 x 256 table of warp
// counts), ping-ponging between `order` and the same range of `scratch` (the key array, free once the scatter has run).
// Four passes cover 32-bit indices and leave the result in `order`.  Not a throughput path: it exists so that results
// that depend on bundle membership are reproducible for degenerate beams too.
__global__ void __launch_bounds__(256) k_sort_fix_long(const uint32_t* __restrict__ seg_end, uint32_t* __restrict__ order,
                                                       uint32_t* __restrict__ scratch, const uint32_t* __restrict__ long_list,
                                                       const uint32_t* __restrict__ long_count) {
    __shared__ uint32_t base[256];
    __shared__ uint32_t wcnt[8][256];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (uint32_t j = blockIdx.x; j < *long_count; j += gridDim.x) {
        const uint32_t key = long_list[j];
        const uint32_t b = key ? seg_end[key - 1] : 0u, L = seg_end[key] - b;
        uint32_t* src = order + b;
        uint32_t* dst = scratch + b;
        for (int pass = 0; pass < 4; ++pass) {
            const int shift = 8 * pass;
            base[threadIdx.x] = 0u;
            __syncthreads();
            for (uint32_t i = threadIdx.x; i < L; i += 256) atomicAdd(&base[(src[i] >> shift) & 255u], 1u);
            __syncthreads();
            if (threadIdx.x == 0) {                                   // exclusive scan of 256 counts
                uint32_t run = 0;
                for (int d = 0; d < 256; ++d) { const uint32_t c = base[d]; base[d] = run; run += c; }
            }
            __syncthreads();
            for (uint32_t t0 = 0; t0 < L; t0 += 256) {
                const uint32_t i = t0 + threadIdx.x;
                const bool have = i < L;
                const uint32_t v = have ? src[i] : 0u;
                const uint32_t d = have ? ((v >> shift) & 255u) : 256u;
#pragma unroll
                for (int w = 0; w < 8; ++w) wcnt[w][threadIdx.x] = 0u;
                __syncthreads();
                const unsigned peers = __match_any_sync(0xffffffffu, d);
                const uint32_t rank = __popc(peers & ((1u << lane) - 1u));
                if (have && rank == 0) wcnt[warp][d] = __popc(peers);
                __syncthreads();
                if (have) {
                    uint32_t off = base[d] + rank;
                    for (int w = 0; w < warp; ++w) off += wcnt[w][d];
                    SP_ASSERT(off < L);
                    dst[off] = v;
                }
                __syncthreads();
                uint32_t add = 0;
#pragma unroll
                for (int w = 0; w < 8; ++w) add += wcnt[w][threadIdx.x];
                base[threadIdx.x] += add;
                __syncthreads();
            }
            uint32_t* t = src; src = dst; dst = t;
        }
    }
}

// ---------------------------------------------------------------------------------------------- propagate
template <typename T> struct PropArgs {
    FieldView<T> F;
    const double* s0; uint64_t n_total;
    uint64_t chunk_off; uint32_t chunk_n;
    const uint32_t* order;                    // sorted slot -> ray index within the chunk, or nullptr
    unsigned long long* cursor;               // bundle dispenser
    BeamSpec beam; int use_beam; uint64_t ray_offset;
    int perm[3];                              // kernel axis -> caller axis
    int kp, ka, kb;                           // kernel-frame indices: probing axis, rf rows (0,1), rf rows (2,3)
    int method, flags, n_steps, n_state;
    T h, t_end, rtol, atol, omega, extent;
    RK4Step<T> rk;                            // constants of the fixed step (host-computed, constant-bank operands)
    sp_stats* stats;
    ExtView X;                                // attenuation / Faraday channels (METHOD == SP_METHOD_RK4X only)
};

struct LaneStats { unsigned long long steps, acc, capped, binned, rejected, evals; };

__device__ __forceinline__ unsigned long long warp_sum(unsigned long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Dormand-Prince with ONE step size per 32-ray bundle: the reference's shipped algorithm (joint RK45 over the
// flattened state, full_solver.py:391) applied to the rays of a warp -- exactly what ScalarDomain.solve does
// when called with a 32-ray chunk, as the reference's own drivers chunk their rays.  All lanes share t and h,
// so the bundle marches in lock-step like the fixed-step kernel (coherent gathers, uniform accept/reject).
// The RMS error norm runs over the n_state components of the valid lanes (butterfly sum: deterministic).
template <typename T, bool PHASE, bool AUX64>
__device__ __forceinline__ void rk45_bundle_integrate(const PropArgs<T>& A, Ray<T>& r, StageSmem<T>& S, bool valid, bool early,
                                                      double amp0, double pol0, unsigned& n_att, LaneStats& ls) {
    const unsigned vmask = __ballot_sync(0xffffffffu, valid);
    const double size = (double)A.n_state * (double)__popc(vmask);        // x.size of the flattened bundle state
    Deriv<T> f; int touched = 0;
    f.dp[0] = f.dp[1] = f.dp[2] = f.dv[0] = f.dv[1] = f.dv[2] = f.dph = (T)0;
    const T rtol = A.rtol, atol = A.atol;
    double s_a = 0.0, s_b = 0.0;
    T sc_p[3], sc_v[3], sc_ph = atol;
    if (valid) {
        touched += deriv_direct<T, PHASE, AUX64>(A.F, A.omega, r.p, r.v, f);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            sc_p[k] = atol + fabs(r.p[k]) * rtol; sc_v[k] = atol + fabs(r.v[k]) * rtol;
            double q = r.p[k] / sc_p[k]; s_a += q * q; q = r.v[k] / sc_v[k]; s_a += q * q;
            q = f.dp[k] / sc_p[k]; s_b += q * q; q = f.dv[k] / sc_v[k]; s_b += q * q;
        }
        sc_ph = atol + fabs(r.ph) * rtol;
        double q = r.ph / sc_ph; s_a += q * q; q = f.dph / sc_ph; s_b += q * q;
        if (A.n_state > 6) {
            q = amp0 / (atol + fabs(amp0) * rtol); s_a += q * q;
            q = pol0 / (atol + fabs(pol0) * rtol); s_a += q * q;
        }
    }
    // select_initial_step (scipy/integrate/_ivp/common.py) on the bundle
    const double d0 = sqrt(warp_sum_f64(s_a)) / sqrt(size), d1 = sqrt(warp_sum_f64(s_b)) / sqrt(size);
    const double t_end = (double)A.t_end;
    double h0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * d0 / d1;
    h0 = fmin(h0, t_end);
    double s_c = 0.0;
    if (valid) {
        T p1[3], v1[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) { p1[k] = r.p[k] + (T)h0 * f.dp[k]; v1[k] = r.v[k] + (T)h0 * f.dv[k]; }
        Deriv<T> f1;
        touched += deriv_direct<T, PHASE, AUX64>(A.F, A.omega, p1, v1, f1);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            double q = (f1.dp[k] - f.dp[k]) / sc_p[k]; s_c += q * q;
            q = (f1.dv[k] - f.dv[k]) / sc_v[k]; s_c += q * q;
        }
        const double q = (f1.dph - f.dph) / sc_ph; s_c += q * q;
    }
    const double d2 = sqrt(warp_sum_f64(s_c)) / sqrt(size) / h0;
    const double h1 = (d1 <= 1e-15 && d2 <= 1e-15) ? fmax(1e-6, h0 * 1e-3) : pow(0.01 / fmax(d1, d2), 0.2);
    double h_abs = fmin(fmin(100 * h0, h1), t_end);
    double t = 0.0;
    const unsigned cap = A.n_steps > 0 ? (unsigned)A.n_steps : (1u << 30);
    bool failed = false;
    while (t < t_end && !failed) {
        if (early && __all_sync(0xffffffffu, !valid || escaped(A.F, r))) break;
        const double min_step = 10.0 * (nextafter(t, (double)INFINITY) - t);
        if (h_abs < min_step) h_abs = min_step;
        bool rejected = false;
        for (;;) {
            if (n_att >= cap || h_abs < min_step) { failed = true; ls.capped += valid ? 1 : 0; break; }
            double t_new = t + h_abs;
            if (t_new - t_end > 0.0) t_new = t_end;
            const double h = t_new - t;
            h_abs = fabs(h);
            Ray<T> rn = r; Deriv<T> fn = f; T esq = (T)0;
            if (valid) touched += dp5_attempt<T, PHASE, AUX64, StageSmem<T> >(A.F, A.omega, (T)h, rtol, atol, r, f, rn, fn, esq, S);
            ++n_att;
            const double en = sqrt(warp_sum_f64((double)esq)) / sqrt(size);
            if (!(en == en)) { failed = true; ls.capped += valid ? 1 : 0; break; }   // NaN state: solve_ivp would never return
            if (en < 1.0) {
                h_abs *= dp5_factor<double>(en, true, rejected);
                t = t_new; r = rn; f = fn; ls.acc += valid ? 1 : 0;
                break;
            }
            h_abs *= dp5_factor<double>(en, false, rejected);
            rejected = true;
        }
    }
    ls.evals += touched;
}

// RK4 over the full 9-component state (attenuation and Faraday rotation on): float64 only.
template <bool PHASE, bool AUX64, typename T>
__device__ __forceinline__ void rk4x_integrate(const PropArgs<T>& A, Ray<T>& r, CellCache<T, PHASE>& cc, bool early, uint64_t gi,
                                               unsigned& n_att, LaneStats& ls, double& amp, double& pol) {}
template <bool PHASE, bool AUX64>
__device__ __forceinline__ void rk4x_integrate(const PropArgs<double>& A, Ray<double>& r, CellCache<double, PHASE>& cc, bool early,
                                               uint64_t gi, unsigned& n_att, LaneStats& ls, double& amp, double& pol) {
    ExtState e;
    e.amp = A.use_beam ? 1.0 : A.s0[6 * A.n_total + gi];
    e.pol = A.use_beam ? 0.0 : A.s0[8 * A.n_total + gi];
    for (int it = 0; it < A.n_steps; ++it) {
        const int t = rk4_step_ext<PHASE, AUX64>(A.F, A.X, cc, A.h, A.omega, (A.flags & SP_FLAG_PHASE) != 0, r, e, early);
        if (t < 0) break;
        ls.evals += t;
        ++n_att;
    }
    ls.acc += n_att;
    amp = e.amp; pol = e.pol;
}

// Per-ray adaptive solve over the full 9-component state (same controller as the RK45 branch of k_propagate).
template <bool PHASE, bool AUX64, typename T>
__device__ __forceinline__ void rk45x_integrate(const PropArgs<T>& A, Ray<T>& r, CellCache<T, PHASE>& cc, bool early, unsigned lanes, uint64_t gi,
                                                unsigned& n_att, LaneStats& ls, double& amp, double& pol) {}
template <bool PHASE, bool AUX64>
__device__ __noinline__ void rk45x_integrate(const PropArgs<double>& A, Ray<double>& r, CellCache<double, PHASE>& cc, bool early,
                                             unsigned lanes, uint64_t gi, unsigned& n_att, LaneStats& ls, double& amp, double& pol) {
    const bool with_phase = (A.flags & SP_FLAG_PHASE) != 0;
    double y[9], f[9], yn[9], fn[9];
    for (int k = 0; k < 3; ++k) { y[k] = r.p[k]; y[3 + k] = r.v[k]; }
    y[6] = A.use_beam ? 1.0 : A.s0[6 * A.n_total + gi];
    y[7] = r.ph;
    y[8] = A.use_beam ? 0.0 : A.s0[8 * A.n_total + gi];
    int touched = deriv9<PHASE, AUX64>(A.F, A.X, cc, A.omega, with_phase, y, f);
    double h_abs = dp5_initial_step9<PHASE, AUX64>(A.F, A.X, cc, A.omega, with_phase, A.t_end, A.rtol, A.atol, y, f, touched);
    double t = 0.0;
    const unsigned cap = A.n_steps > 0 ? (unsigned)A.n_steps : (1u << 30);
    // one attempt per iteration and lane (new step or retry), warp-voted loop condition: see k_propagate
    bool failed = false, rejected = false, fresh = true;
    double min_step = 0.0;
    for (;;) {
        bool go = (t < A.t_end) && !failed;
        if (go && fresh) {
            bool out = false;
            if (early) {
                Ray<double> q;
                for (int k = 0; k < 3; ++k) { q.p[k] = y[k]; q.v[k] = y[3 + k]; }
                out = escaped(A.F, q);
            }
            if (out) go = false;
            else {
                min_step = 10.0 * (nextafter(t, (double)INFINITY) - t);
                if (h_abs < min_step) h_abs = min_step;
                rejected = false; fresh = false;
            }
        }
        if (go && (n_att >= cap || h_abs < min_step)) { failed = true; ls.capped += 1; go = false; }
        if (!__any_sync(lanes, go)) break;
        if (go) {
            double t_new = t + h_abs;
            if (t_new - A.t_end > 0.0) t_new = A.t_end;
            const double h = t_new - t;
            h_abs = fabs(h);
            double esq;
            touched += dp5_attempt9<PHASE, AUX64>(A.F, A.X, cc, A.omega, with_phase, h, A.rtol, A.atol, y, f, yn, fn, esq);
            ++n_att;
            const double en = sqrt(esq / 9.0);
            if (!(en == en)) { failed = true; ls.capped += 1; }                      // NaN state: solve_ivp would never return
            else if (en < 1.0) {
                h_abs *= dp5_factor<double>(en, true, rejected);
                t = t_new; ls.acc += 1;
                for (int i = 0; i < 9; ++i) { y[i] = yn[i]; f[i] = fn[i]; }
                fresh = true;
            } else {
                h_abs *= dp5_factor<double>(en, false, rejected);
                rejected = true;
            }
        }
    }
    ls.evals += touched;
    for (int k = 0; k < 3; ++k) { r.p[k] = y[k]; r.v[k] = y[3 + k]; }
    r.ph = y[7]; amp = y[6]; pol = y[8];
}

template <typename T, int METHOD, bool PHASE, bool AUX64>
__global__ void __launch_bounds__(128, (METHOD == SP_METHOD_RK4 && sizeof(T) == 8) ? SP_RK4_MIN_BLOCKS : (((METHOD == SP_METHOD_RK45 || METHOD == SP_METHOD_RK45B) && sizeof(T) == 8) ? SP_RK45_MIN_BLOCKS : ((METHOD == SP_METHOD_RK4 && sizeof(T) == 4) ? SP_RK4F_MIN_BLOCKS : 1))) k_propagate(const PropArgs<T> A, const Epilogue E) {
    const int lane = threadIdx.x & 31;
    const bool early = (A.flags & SP_FLAG_EARLY_EXIT) != 0;
    extern __shared__ double sp_dyn_smem[];     // adaptive methods only: SP_STAGE_DOUBLES values per thread (see StageSmem)
    StageSmem<T> S;
    S.base = reinterpret_cast<T*>(sp_dyn_smem) + threadIdx.x; S.stride = blockDim.x;
    for (;;) {
        LaneStats ls = {0, 0, 0, 0, 0, 0};      // per bundle: nothing but the ray itself is live across the integration
        unsigned long long slot0 = 0;
        if (lane == 0) slot0 = atomicAdd(A.cursor, 32ull);
        slot0 = __shfl_sync(0xffffffffu, slot0, 0);
        if (slot0 >= A.chunk_n) break;
        const unsigned long long slot = slot0 + lane;
        const bool valid = slot < A.chunk_n;
        const unsigned vmask = __ballot_sync(0xffffffffu, valid);      // the lanes that integrate a ray (warp converged here)
        const uint64_t li = valid ? (A.order ? (uint64_t)A.order[slot] : slot) : 0;
        const uint64_t gi = A.chunk_off + li;         // index into the caller's arrays
        double s[6];
        double ph0 = 0.0;
        if (valid) {
            load_ray_caller(A.s0, A.n_total, gi, A.beam, A.use_beam, A.ray_offset, s);
            if (!A.use_beam) ph0 = A.s0[7 * A.n_total + gi];
        } else {
#pragma unroll
            for (int k = 0; k < 6; ++k) s[k] = 0.0;
        }
        Ray<T> r;
#pragma unroll
        for (int k = 0; k < 3; ++k) { r.p[k] = (T)s[A.perm[k]]; r.v[k] = (T)s[3 + A.perm[k]]; }
        r.ph = (T)ph0;
        unsigned n_att = 0;
        CellCache<T, PHASE> cc;
        double amp_x = 1.0, pol_x = 0.0;
        if (METHOD == SP_METHOD_RK45B) {
            const double amp0 = (valid && !A.use_beam) ? A.s0[6 * A.n_total + gi] : 1.0;
            const double pol0 = (valid && !A.use_beam) ? A.s0[8 * A.n_total + gi] : 0.0;
            rk45_bundle_integrate<T, PHASE, AUX64>(A, r, S, valid, early, amp0, pol0, n_att, ls);
            if (valid) ls.steps += n_att; else n_att = 0;
        } else if (valid) {
            if (METHOD == SP_METHOD_RK4X) {
                rk4x_integrate<PHASE, AUX64>(A, r, cc, early, gi, n_att, ls, amp_x, pol_x);
            } else if (METHOD == SP_METHOD_RK45X) {
                rk45x_integrate<PHASE, AUX64>(A, r, cc, early, vmask, gi, n_att, ls, amp_x, pol_x);
            } else if (METHOD == SP_METHOD_TSIT5) {
                // diffrax.diffeqsolve(Tsit5, PIDController) per ray in normalised time tau in [0, 1]: A.t_end = T, A.h = dt0
                T y[7], f[7], yn[7], fn[7];
#pragma unroll
                for (int k = 0; k < 3; ++k) { y[k] = r.p[k]; y[3 + k] = r.v[k]; }
                y[6] = r.ph;
                int touched = tsit5_f<T, PHASE, AUX64>(A.F, A.omega, y, f);
                T tau = (T)0, dt = A.h;
                const unsigned cap = A.n_steps > 0 ? (unsigned)A.n_steps : 10000u;
                const T inv_n = (T)1 / (T)A.n_state;
                bool failed = false;
                const unsigned lanes = vmask;
                for (;;) {
                    bool go = (tau < (T)1) && !failed;
                    if (go && n_att >= cap) { failed = true; ls.capped += 1; go = false; }
                    if (!__any_sync(lanes, go)) break;
                    if (go) {
                        const bool last = tau + dt >= (T)1;
                        const T d = last ? (T)1 - tau : dt;
                        T esq;
                        touched += tsit5_attempt<T, PHASE, AUX64>(A.F, A.omega, d * A.t_end, A.rtol, A.atol, y, f, yn, fn, esq);
                        ++n_att;
                        const T en = sqrt(esq * inv_n);
                        if (!(en == en)) { failed = true; ls.capped += 1; }
                        else {
                            const bool keep = en < (T)1;
                            dt = d * pid_factor<T>(en, keep);
                            if (keep) {
                                tau = last ? (T)1 : tau + d; ls.acc += 1;
#pragma unroll
                                for (int i = 0; i < 7; ++i) { y[i] = yn[i]; f[i] = fn[i]; }
                            }
                        }
                    }
                }
                ls.evals += touched;
#pragma unroll
                for (int k = 0; k < 3; ++k) { r.p[k] = y[k]; r.v[k] = y[3 + k]; }
                r.ph = y[6];
            } else if (METHOD == SP_METHOD_RK45B) {
                // handled above (whole-warp path)
            } else if (METHOD == SP_METHOD_RK4) {
                for (int it = 0; it < A.n_steps; ++it) {
                    const int t = rk4_step<T, PHASE, AUX64>(A.F, cc, A.rk, A.omega, r, early);
                    if (t < 0) break;
                    ls.evals += t;
                    ++n_att;
                }
                ls.acc += n_att;
            } else {
                // SciPy RK45 driven as solve_ivp does (rk.py:_step_impl), one controller per ray
                Deriv<T> f; int touched = 0;
                touched += deriv_direct<T, PHASE, AUX64>(A.F, A.omega, r.p, r.v, f);
                const double amp0 = A.use_beam ? 1.0 : A.s0[6 * A.n_total + gi], pol0 = A.use_beam ? 0.0 : A.s0[8 * A.n_total + gi];
                T h_abs = dp5_initial_step<T, PHASE, AUX64>(A.F, A.omega, A.t_end, A.rtol, A.atol, A.n_state, (T)amp0,
                                                            (T)pol0, r, f, touched);
                T t = (T)0;
                const unsigned cap = A.n_steps > 0 ? (unsigned)A.n_steps : (1u << 30);
                const T inv_n = (T)1 / (T)A.n_state;
                // One attempt per loop iteration and per lane, whether it opens a new step or retries a rejected one:
                // with solve_ivp's nested "retry until accepted" loop, the lanes that accepted idled while the few that
                // rejected repeated the whole attempt (ncu: 10 of 32 lanes active on average).  The loop condition is a
                // warp vote, so the lanes reconverge every iteration; per-lane arithmetic and order are unchanged.
                bool failed = false, rejected = false, fresh = true;
                T min_step = (T)0;
                const unsigned lanes = vmask;
                for (;;) {
                    bool go = (t < A.t_end) && !failed;
                    if (go && fresh) {
                        if (early && escaped(A.F, r)) go = false;
                        else {
                            min_step = (T)10 * (nextafter(t, (T)INFINITY) - t);
                            if (h_abs < min_step) h_abs = min_step;
                            rejected = false; fresh = false;
                        }
                    }
                    if (go && (n_att >= cap || h_abs < min_step)) { failed = true; ls.capped += 1; go = false; }
                    if (!__any_sync(lanes, go)) break;
                    if (go) {
                        T t_new = t + h_abs;
                        if (t_new - A.t_end > (T)0) t_new = A.t_end;
                        const T h = t_new - t;
                        h_abs = fabs(h);
                        Ray<T> rn; Deriv<T> fn; T esq;
                        touched += dp5_attempt<T, PHASE, AUX64, StageSmem<T> >(A.F, A.omega, h, A.rtol, A.atol, r, f, rn, fn, esq, S);
                        ++n_att;
                        const T en = sqrt(esq * inv_n);
                        if (!(en == en)) { failed = true; ls.capped += 1; }          // NaN state: solve_ivp would never return
                        else {
                            const bool acc_ = en < (T)1;
                            h_abs *= dp5_factor<T>(en, acc_, rejected);         // one call: the lanes stay converged through pow()
                            if (acc_) { t = t_new; r = rn; f = fn; ls.acc += 1; fresh = true; }
                            else rejected = true;
                        }
                    }
                }
                ls.evals += touched;
            }
            ls.steps += n_att;
        }
        // ---- epilogue: exit plane, outputs, fused optics + binning ----
        T xa = 0, tha = 0, xb = 0, thb = 0;
        if (valid) exit_project<T>(r, A.kp, A.ka, A.kb, A.extent, xa, tha, xb, thb);
        const uint64_t N = A.n_total;
        double amp = 1.0, pol = 0.0;              // constant along the ray (zero derivative): re-read instead of kept live
        if (valid && !A.use_beam) { amp = A.s0[6 * N + gi]; pol = A.s0[8 * N + gi]; }
        if (METHOD == SP_METHOD_RK4X || METHOD == SP_METHOD_RK45X) { amp = amp_x; pol = pol_x; }
        if (valid) {
            if (E.sf) {
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    E.sf[(uint64_t)A.perm[k] * N + gi] = (double)r.p[k];
                    E.sf[(uint64_t)(3 + A.perm[k]) * N + gi] = (double)r.v[k];
                }
                E.sf[6 * N + gi] = amp; E.sf[7 * N + gi] = (double)r.ph; E.sf[8 * N + gi] = pol;
            }
            if (E.rf) {
                E.rf[gi] = (double)xa; E.rf[N + gi] = (double)tha; E.rf[2 * N + gi] = (double)xb; E.rf[3 * N + gi] = (double)thb;
            }
            if (E.steps) E.steps[gi] = n_att;
        }
        if (E.jf || E.n_channels > 0) {
            // Jones vector (full_solver.py:883-890): amp e^{i phase} R(pol) (0, 1)^T
            double sp_, cp_, ss, cs;
            sp_sincos((double)r.ph, &sp_, &cp_);
            sp_sincos(pol, &ss, &cs);
            const double rr = amp * cp_, ri = amp * sp_;
            const double ex_re = rr * (-ss), ex_im = ri * (-ss), ey_re = rr * cs, ey_im = ri * cs;
            if (valid && E.jf) {
                E.jf[2 * gi] = ex_re; E.jf[2 * gi + 1] = ex_im;
                E.jf[2 * (N + gi)] = ey_re; E.jf[2 * (N + gi) + 1] = ey_im;
            }
            for (int c = 0; c < E.n_channels; ++c) {
                const ChannelDev& ch = E.ch[c];
                DetRay d;
                d.x = (double)xa * 1e3; d.th = (double)tha; d.y = (double)xb * 1e3; d.ph = (double)thb;   // m_to_mm
                d.ex_re = ex_re; d.ex_im = ex_im; d.ey_re = ey_re; d.ey_im = ey_im; d.alive = valid;
                if (valid) run_optics(d, (double)xa, (double)xb, ch.ops, ch.n_ops, ch.with_E != 0, ch.kwave);
                const int b = bin_ray(ch, d, valid);
                ls.binned += b;
                ls.rejected += (valid && !d.alive) ? 1 : 0;
            }
        }
        if (A.stats) {
        const unsigned long long a = warp_sum(ls.steps), b = warp_sum(ls.acc), c = warp_sum(ls.capped),
                                 d = warp_sum(ls.binned), e = warp_sum(ls.rejected), f = warp_sum(ls.evals);
        if (lane == 0) {
            if (a) atomicAdd((unsigned long long*)&A.stats->ray_steps, a);
            if (b) atomicAdd((unsigned long long*)&A.stats->ray_steps_acc, b);
            if (c) atomicAdd((unsigned long long*)&A.stats->rays_capped, c);
            if (d) atomicAdd((unsigned long long*)&A.stats->rays_binned, d);
            if (e) atomicAdd((unsigned long long*)&A.stats->rays_rejected, e);
            if (f) atomicAdd((unsigned long long*)&A.stats->rhs_evals, f);
        }
        }
    }
}

// ------------------------------------------------------------------------------------------- joint RK45
// The reference as shipped integrates ALL rays as one 9N-dimensional system: one step size, accepted or
// rejected from the RMS error norm over every component of every ray (full_solver.py:391 -> scipy RK45).
// State lives in HBM between attempts; the controller runs on the host exactly like SciPy's Python loop.
struct JointBuf {               // SoA over rays, kernel frame
    double *p[3], *v[3], *ph;   // current state
    double *fv[3], *fph;        // f = derivative at current state (dv and dphase; dp = v)
    double *pn[3], *vn[3], *phn, *fvn[3], *fphn;   // candidate
    double* amp; double* pol;
    double* partial;            // per-block partial sums
};

template <bool PHASE, bool AUX64>
__global__ void k_joint_init(FieldView<double> F, JointBuf B, const double* s0, uint64_t n, int p0, int p1, int p2,
                             double omega, double rtol, double atol, int pass, double h0) {
    // pass 0: load state, f0 = f(y0); partial sums of (y0/scale)^2 and (f0/scale)^2
    // pass 1: f1 = f(y0 + h0 f0); partial sums of ((f1 - f0)/scale)^2
    __shared__ double sh0[128], sh1[128];
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double s_a = 0.0, s_b = 0.0;
    if (i < n) {
        const int perm[3] = {p0, p1, p2};
        Ray<double> r; Deriv<double> f;
        CellCache<double, PHASE> cc;
        if (pass == 0) {
            for (int k = 0; k < 3; ++k) { r.p[k] = s0[(uint64_t)perm[k] * n + i]; r.v[k] = s0[(uint64_t)(3 + perm[k]) * n + i]; }
            r.ph = s0[7 * n + i];
            B.amp[i] = s0[6 * n + i]; B.pol[i] = s0[8 * n + i];
            deriv_direct<double, PHASE, AUX64>(F, omega, r.p, r.v, f);
            for (int k = 0; k < 3; ++k) { B.p[k][i] = r.p[k]; B.v[k][i] = r.v[k]; B.fv[k][i] = f.dv[k]; }
            B.ph[i] = r.ph; B.fph[i] = f.dph;
            for (int k = 0; k < 3; ++k) {
                const double sp_ = atol + fabs(r.p[k]) * rtol, sv_ = atol + fabs(r.v[k]) * rtol;
                double q = r.p[k] / sp_; s_a += q * q; q = r.v[k] / sv_; s_a += q * q;
                q = f.dp[k] / sp_; s_b += q * q; q = f.dv[k] / sv_; s_b += q * q;
            }
            const double sph = atol + fabs(r.ph) * rtol;
            double q = r.ph / sph; s_a += q * q; q = f.dph / sph; s_b += q * q;
            q = B.amp[i] / (atol + fabs(B.amp[i]) * rtol); s_a += q * q;
            q = B.pol[i] / (atol + fabs(B.pol[i]) * rtol); s_a += q * q;
        } else {
            double p1_[3], v1_[3];
            for (int k = 0; k < 3; ++k) {
                r.p[k] = B.p[k][i]; r.v[k] = B.v[k][i];
                p1_[k] = r.p[k] + h0 * r.v[k]; v1_[k] = r.v[k] + h0 * B.fv[k][i];
            }
            deriv_direct<double, PHASE, AUX64>(F, omega, p1_, v1_, f);
            for (int k = 0; k < 3; ++k) {
                const double sp_ = atol + fabs(r.p[k]) * rtol, sv_ = atol + fabs(r.v[k]) * rtol;
                double q = (f.dp[k] - r.v[k]) / sp_; s_a += q * q;
                q = (f.dv[k] - B.fv[k][i]) / sv_; s_a += q * q;
            }
            const double sph = atol + fabs(B.ph[i]) * rtol;
            const double q = (f.dph - B.fph[i]) / sph; s_a += q * q;
        }
    }
    sh0[threadIdx.x] = s_a; sh1[threadIdx.x] = s_b;
    __syncthreads();
    for (int o = 64; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) { sh0[threadIdx.x] += sh0[threadIdx.x + o]; sh1[threadIdx.x] += sh1[threadIdx.x + o]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { B.partial[2 * blockIdx.x] = sh0[0]; B.partial[2 * blockIdx.x + 1] = sh1[0]; }
}

template <bool PHASE, bool AUX64>
__global__ void k_joint_attempt(FieldView<double> F, JointBuf B, uint64_t n, double omega, double h, double rtol,
                                double atol) {
    __shared__ double sh0[128];
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double esq = 0.0;
    if (i < n) {
        Ray<double> r, rn; Deriv<double> f, fn;
        CellCache<double, PHASE> cc;
        for (int k = 0; k < 3; ++k) { r.p[k] = B.p[k][i]; r.v[k] = B.v[k][i]; f.dp[k] = r.v[k]; f.dv[k] = B.fv[k][i]; }
        r.ph = B.ph[i]; f.dph = B.fph[i];
        dp5_attempt<double, PHASE, AUX64>(F, omega, h, rtol, atol, r, f, rn, fn, esq);
        for (int k = 0; k < 3; ++k) { B.pn[k][i] = rn.p[k]; B.vn[k][i] = rn.v[k]; B.fvn[k][i] = fn.dv[k]; }
        B.phn[i] = rn.ph; B.fphn[i] = fn.dph;
    }
    sh0[threadIdx.x] = esq;
    __syncthreads();
    for (int o = 64; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh0[threadIdx.x] += sh0[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) B.partial[2 * blockIdx.x] = sh0[0];
}

// Joint solve with the attenuation / Faraday channels: all nine rows, state as a [9][n] SoA (kernel-frame rows
// p, v, amp, phase, pol).  pass 0 / 1 as in k_joint_init.
template <bool PHASE, bool AUX64>
__global__ void k_jointx_init(FieldView<double> F, ExtView X, double* __restrict__ Y, double* __restrict__ Fy,
                              double* __restrict__ partial, const double* __restrict__ s0, uint64_t n, int p0, int p1, int p2,
                              double omega, int with_phase, double rtol, double atol, int pass, double h0) {
    __shared__ double sh0[128], sh1[128];
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double s_a = 0.0, s_b = 0.0;
    if (i < n) {
        const int perm[3] = {p0, p1, p2};
        double y[9], f[9];
        CellCache<double, PHASE> cc;
        if (pass == 0) {
            for (int k = 0; k < 3; ++k) { y[k] = s0[(uint64_t)perm[k] * n + i]; y[3 + k] = s0[(uint64_t)(3 + perm[k]) * n + i]; }
            for (int k = 6; k < 9; ++k) y[k] = s0[(uint64_t)k * n + i];
            deriv9<PHASE, AUX64>(F, X, cc, omega, with_phase != 0, y, f);
            for (int k = 0; k < 9; ++k) {
                Y[(uint64_t)k * n + i] = y[k]; Fy[(uint64_t)k * n + i] = f[k];
                const double sc = atol + fabs(y[k]) * rtol;
                double q = y[k] / sc; s_a += q * q; q = f[k] / sc; s_b += q * q;
            }
        } else {
            double y1[9], f1[9];
            for (int k = 0; k < 9; ++k) { y[k] = Y[(uint64_t)k * n + i]; f[k] = Fy[(uint64_t)k * n + i]; y1[k] = y[k] + h0 * f[k]; }
            deriv9<PHASE, AUX64>(F, X, cc, omega, with_phase != 0, y1, f1);
            for (int k = 0; k < 9; ++k) { const double q = (f1[k] - f[k]) / (atol + fabs(y[k]) * rtol); s_a += q * q; }
        }
    }
    sh0[threadIdx.x] = s_a; sh1[threadIdx.x] = s_b;
    __syncthreads();
    for (int o = 64; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) { sh0[threadIdx.x] += sh0[threadIdx.x + o]; sh1[threadIdx.x] += sh1[threadIdx.x + o]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { partial[2 * blockIdx.x] = sh0[0]; partial[2 * blockIdx.x + 1] = sh1[0]; }
}

template <bool PHASE, bool AUX64>
__global__ void k_jointx_attempt(FieldView<double> F, ExtView X, const double* __restrict__ Y, const double* __restrict__ Fy,
                                 double* __restrict__ Yn, double* __restrict__ Fn, double* __restrict__ partial, uint64_t n,
                                 double omega, int with_phase, double h, double rtol, double atol) {
    __shared__ double sh0[128];
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double esq = 0.0;
    if (i < n) {
        double y[9], f[9], yn[9], fn[9];
        CellCache<double, PHASE> cc;
        for (int k = 0; k < 9; ++k) { y[k] = Y[(uint64_t)k * n + i]; f[k] = Fy[(uint64_t)k * n + i]; }
        dp5_attempt9<PHASE, AUX64>(F, X, cc, omega, with_phase != 0, h, rtol, atol, y, f, yn, fn, esq);
        for (int k = 0; k < 9; ++k) { Yn[(uint64_t)k * n + i] = yn[k]; Fn[(uint64_t)k * n + i] = fn[k]; }
    }
    sh0[threadIdx.x] = esq;
    __syncthreads();
    for (int o = 64; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh0[threadIdx.x] += sh0[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[2 * blockIdx.x] = sh0[0];
}

// Deterministic (fixed-order) final reduction of the per-block partials -> out[0], out[1] (mapped host memory).
__global__ void k_joint_reduce(const double* __restrict__ partial, int nblocks, double* __restrict__ out) {
    __shared__ double sh0[256], sh1[256];
    double a = 0.0, b = 0.0;
    for (int i = threadIdx.x; i < nblocks; i += blockDim.x) { a += partial[2 * i]; b += partial[2 * i + 1]; }
    sh0[threadIdx.x] = a; sh1[threadIdx.x] = b;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) { sh0[threadIdx.x] += sh0[threadIdx.x + o]; sh1[threadIdx.x] += sh1[threadIdx.x + o]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { out[0] = sh0[0]; out[1] = sh1[0]; }
}

// Exit projection + outputs + optics/binning for rays whose state sits in a JointBuf (used after the joint solve).
__global__ void k_joint_finish(JointBuf B, uint64_t n, int use_new, int p0, int p1, int p2, int kp, int ka, int kb,
                               double extent, const Epilogue E, sp_stats* stats) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = i < n;
    const int perm[3] = {p0, p1, p2};
    Ray<double> r; double amp = 1.0, pol = 0.0;
    for (int k = 0; k < 3; ++k) { r.p[k] = 0; r.v[k] = 1; }
    r.ph = 0;
    if (valid) {
        for (int k = 0; k < 3; ++k) { r.p[k] = (use_new ? B.pn : B.p)[k][i]; r.v[k] = (use_new ? B.vn : B.v)[k][i]; }
        r.ph = (use_new ? B.phn : B.ph)[i]; amp = B.amp[i]; pol = B.pol[i];
    }
    double xa = 0, tha = 0, xb = 0, thb = 0;
    if (valid) exit_project<double>(r, kp, ka, kb, extent, xa, tha, xb, thb);
    if (valid) {
        if (E.sf) {
            for (int k = 0; k < 3; ++k) { E.sf[(uint64_t)perm[k] * n + i] = r.p[k]; E.sf[(uint64_t)(3 + perm[k]) * n + i] = r.v[k]; }
            E.sf[6 * n + i] = amp; E.sf[7 * n + i] = r.ph; E.sf[8 * n + i] = pol;
        }
        if (E.rf) { E.rf[i] = xa; E.rf[n + i] = tha; E.rf[2 * n + i] = xb; E.rf[3 * n + i] = thb; }
    }
    unsigned long long binned = 0, rejected = 0;
    if (E.jf || E.n_channels > 0) {
        double sp_, cp_, ss, cs;
        sp_sincos(r.ph, &sp_, &cp_); sp_sincos(pol, &ss, &cs);
        const double rr = amp * cp_, ri = amp * sp_;
        const double ex_re = rr * (-ss), ex_im = ri * (-ss), ey_re = rr * cs, ey_im = ri * cs;
        if (valid && E.jf) {
            E.jf[2 * i] = ex_re; E.jf[2 * i + 1] = ex_im; E.jf[2 * (n + i)] = ey_re; E.jf[2 * (n + i) + 1] = ey_im;
        }
        for (int c = 0; c < E.n_channels; ++c) {
            const ChannelDev& ch = E.ch[c];
            DetRay d;
            d.x = xa * 1e3; d.th = tha; d.y = xb * 1e3; d.ph = thb;
            d.ex_re = ex_re; d.ex_im = ex_im; d.ey_re = ey_re; d.ey_im = ey_im; d.alive = valid;
            if (valid) run_optics(d, xa, xb, ch.ops, ch.n_ops, ch.with_E != 0, ch.kwave);
            binned += bin_ray(ch, d, valid);
            rejected += (valid && !d.alive) ? 1 : 0;
        }
    }
    if (stats) {
        binned = warp_sum(binned); rejected = warp_sum(rejected);
        if ((threadIdx.x & 31) == 0) {
            if (binned) atomicAdd((unsigned long long*)&stats->rays_binned, binned);
            if (rejected) atomicAdd((unsigned long long*)&stats->rays_rejected, rejected);
        }
    }
}

// ------------------------------------------------------------------------------------ stand-alone kernels
// SMEM_HIST: the image is small enough (<= 12 Ki bins) for a CTA-private uint32 histogram in shared memory:
// lanes that hit the same pixel are aggregated in the warp (__match_any_sync), one shared-memory atomic per
// distinct pixel, and each CTA flushes its non-zero bins to the global uint64 image once at the end.
template <bool SMEM_HIST>
__global__ void k_optics_image(const double* __restrict__ rf, const double* __restrict__ jf, uint64_t n,
                               const ChannelDev ch, double* __restrict__ rf_out, double* __restrict__ jf_out) {
    extern __shared__ unsigned int s_hist[];
    const int nbins = ch.nx * ch.ny;
    if (SMEM_HIST) {
        for (int i = threadIdx.x; i < nbins; i += blockDim.x) s_hist[i] = 0u;
        __syncthreads();
    }
    const uint64_t i0 = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const uint64_t n_round = (n + 31) / 32 * 32;      // keep warps converged for __match_any_sync
    for (uint64_t i = i0; i < n_round; i += stride) {
        const bool valid = i < n;
        DetRay d;
        d.alive = valid; d.x = d.th = d.y = d.ph = 0.0;
        d.ex_re = d.ex_im = d.ey_re = d.ey_im = 0.0;
        double xm = 0.0, ym = 0.0;
        if (valid) {
            xm = rf[i]; ym = rf[2 * n + i];
            const double unit = ch.input_mm ? 1.0 : 1e3;      // m_to_mm (diagnostics.py:122-127)
            d.x = xm * unit; d.th = rf[n + i]; d.y = ym * unit; d.ph = rf[3 * n + i];
            if (jf) { d.ex_re = jf[2 * i]; d.ex_im = jf[2 * i + 1]; d.ey_re = jf[2 * (n + i)]; d.ey_im = jf[2 * (n + i) + 1]; }
            // a Stokes image does not need the E-phase advance (see bin_ray); the Jones vectors handed back do
            run_optics(d, xm, ym, ch.ops, ch.n_ops, jf != nullptr && (ch.kind != SP_IMG_STOKES || jf_out != nullptr), ch.kwave);
        }
        if (valid && rf_out) {
            const double nanv = __longlong_as_double(0x7ff8000000000000ULL);
            rf_out[i] = d.alive ? d.x : nanv; rf_out[n + i] = d.alive ? d.th : nanv;
            rf_out[2 * n + i] = d.alive ? d.y : nanv; rf_out[3 * n + i] = d.alive ? d.ph : nanv;
            if (jf_out) {
                jf_out[2 * i] = d.alive ? d.ex_re : nanv; jf_out[2 * i + 1] = d.alive ? d.ex_im : nanv;
                jf_out[2 * (n + i)] = d.alive ? d.ey_re : nanv; jf_out[2 * (n + i) + 1] = d.alive ? d.ey_im : nanv;
            }
        }
        if (ch.nx > 0) {
            if (SMEM_HIST) {
                int pix = -1;
                if (valid && d.alive) {
                    const int ix = bin_index(d.x, ch.x_lo, ch.x_hi, ch.nx, true), iy = bin_index(d.y, ch.y_lo, ch.y_hi, ch.ny, true);
                    if (ix >= 0 && iy >= 0) pix = iy * ch.nx + ix;
                }
                const unsigned peers = __match_any_sync(__activemask(), pix);
                if (pix >= 0 && (__ffs(peers) - 1) == (int)(threadIdx.x & 31)) atomicAdd(s_hist + pix, (unsigned)__popc(peers));
            } else {
                bin_ray(ch, d, valid);
            }
        }
    }
    if (SMEM_HIST) {
        __syncthreads();
        for (int i = threadIdx.x; i < nbins; i += blockDim.x) {
            const unsigned c = s_hist[i];
            if (c) atomicAdd(ch.counts + i, (unsigned long long)c);
        }
    }
}

__global__ void k_exit_plane(const double* __restrict__ sf, uint64_t n, int kp, int ka, int kb, double extent, int keep,
                             double* __restrict__ rf, double* __restrict__ jf, double* __restrict__ sback) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Ray<double> r;                                   // caller frame here: kernel index == caller axis
    for (int k = 0; k < 3; ++k) { r.p[k] = sf[(uint64_t)k * n + i]; r.v[k] = sf[(uint64_t)(3 + k) * n + i]; }
    double xa, tha, xb, thb;
    exit_project<double>(r, kp, ka, kb, extent, xa, tha, xb, thb);
    if (rf) {
        rf[i] = keep ? pick3(r.p, ka) : xa; rf[n + i] = tha;
        rf[2 * n + i] = keep ? pick3(r.p, kb) : xb; rf[3 * n + i] = thb;
    }
    if (jf) {
        const double amp = sf[6 * n + i], ph = sf[7 * n + i], pol = sf[8 * n + i];
        double sp_, cp_, ss, cs;
        sp_sincos(ph, &sp_, &cp_); sp_sincos(pol, &ss, &cs);
        const double rr = amp * cp_, ri = amp * sp_;
        jf[2 * i] = rr * (-ss); jf[2 * i + 1] = ri * (-ss); jf[2 * (n + i)] = rr * cs; jf[2 * (n + i) + 1] = ri * cs;
    }
    if (sback) {
        const double tbp = (pick3(r.p, kp) - extent) / pick3(r.v, kp);
        for (int k = 0; k < 3; ++k) {
            sback[(uint64_t)k * n + i] = (k == kp) ? extent : r.p[k] - r.v[k] * tbp;
            sback[(uint64_t)(3 + k) * n + i] = r.v[k];
        }
        for (int k = 6; k < 9; ++k) sback[(uint64_t)k * n + i] = sf[(uint64_t)k * n + i];
    }
}

__global__ void k_finalize(const long long* __restrict__ planes, double* __restrict__ H, size_t npix) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npix) return;
    const double q = 1.0 / (double)(1ll << SP_PLANE_FRAC_BITS);
    const double a = (double)planes[i] * q, b = (double)planes[2 * npix + i] * q;     // Re(sum Ex), Re(sum Ey)
    H[i] = sqrt(a * a + b * b);
}

__global__ void k_finalize_stokes(const long long* __restrict__ planes, double* __restrict__ H, size_t npix) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npix) return;
    const double q = 1.0 / (double)(1ll << SP_STOKES_FRAC_BITS);
    H[i] = (double)planes[i];                                                          // N
    for (int k = 1; k < 4; ++k) H[k * npix + i] = (double)planes[k * npix + i] * q;    // I, Q, U
}

template <bool PHASE, bool AUX64>
__global__ void k_rhs(FieldView<double> F, ExtView X, const double* __restrict__ s, uint64_t n, double* __restrict__ out,
                      int p0, int p1, int p2, double omega) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int perm[3] = {p0, p1, p2};
    double p[3], v[3];
    for (int k = 0; k < 3; ++k) { p[k] = s[(uint64_t)perm[k] * n + i]; v[k] = s[(uint64_t)(3 + perm[k]) * n + i]; }
    Deriv<double> f;
    CellCache<double, PHASE> cc;
    const int inside = deriv<double, PHASE, AUX64>(F, cc, omega, p, v, f);
    for (int k = 0; k < 3; ++k) { out[(uint64_t)perm[k] * n + i] = f.dp[k]; out[(uint64_t)(3 + perm[k]) * n + i] = f.dv[k]; }
    double x[5];
    ext_eval<PHASE>(F, X, cc, inside != 0, p, x);
    out[6 * n + i] = X.ch[0] ? x[0] * s[6 * n + i] : 0.0;
    out[7 * n + i] = f.dph;
    out[8 * n + i] = X.ch[1] ? X.verdet * x[1] * (x[2] * v[0] + x[3] * v[1] + x[4] * v[2]) : 0.0;
}

__global__ void k_beam(BeamSpec B, uint64_t off, uint64_t n, double* __restrict__ s0) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double s[6];
    beam_ray(B, off + i, s);
    for (int k = 0; k < 6; ++k) s0[(uint64_t)k * n + i] = s[k];
    s0[6 * n + i] = 1.0; s0[7 * n + i] = 0.0; s0[8 * n + i] = 0.0;
}

// ---------------------------------------------------------------------------------------------- workspace
struct sp_workspace {
    uint32_t *keys = nullptr, *order = nullptr, *hist = nullptr, *tile_sums = nullptr, *long_list = nullptr, *long_count = nullptr;
    size_t cap_rays = 0, cap_keys = 0;
    unsigned long long* cursor = nullptr;
    double* joint = nullptr; size_t joint_cap = 0;
    double* host_pair = nullptr;     // pinned, 2 doubles
    int sm_count = 0;
    std::vector<cudaEvent_t> ev;     // start/stop pairs around k_propagate launches
    size_t ev_used = 0;
    double ev_ms = 0.0; uint64_t ev_n = 0;   // launches already folded out of the event list
    std::vector<double> jlog_h, jlog_en;   // attempts of the last joint solve
};

extern "C" int sp_workspace_joint_log(const sp_workspace* w, double* h_out, double* en_out, int cap, int* n_out) {
    if (!w || !n_out) return fail(SP_EINVAL, "null argument");
    const int n = (int)w->jlog_h.size();
    for (int i = 0; i < n && i < cap; ++i) { if (h_out) h_out[i] = w->jlog_h[i]; if (en_out) en_out[i] = w->jlog_en[i]; }
    *n_out = n;
    return SP_OK;
}

// Start/stop events around every k_propagate launch.  The log is bounded without ever dropping a launch: when it
// reaches EV_FOLD events, the pairs that have already completed are folded into a running total and their events
// recycled (no wait: cudaEventQuery); only pairs still in flight stay in the list.
static const size_t EV_FOLD = 1024;
static int ws_fold(sp_workspace* w, bool wait) {
    size_t keep = 0;
    for (size_t i = 0; i + 1 < w->ev_used; i += 2) {
        bool done = true;
        if (wait) CU(cudaEventSynchronize(w->ev[i + 1]));
        else {
            const cudaError_t q = cudaEventQuery(w->ev[i + 1]);
            if (q == cudaErrorNotReady) done = false;
            else if (q != cudaSuccess) return fail(SP_ECUDA, std::string("cudaEventQuery: ") + cudaGetErrorString(q));
        }
        if (done) {
            float ms = 0.f;
            CU(cudaEventElapsedTime(&ms, w->ev[i], w->ev[i + 1]));
            w->ev_ms += ms; w->ev_n += 1;
        } else {
            std::swap(w->ev[keep], w->ev[i]); std::swap(w->ev[keep + 1], w->ev[i + 1]);
            keep += 2;
        }
    }
    if (w->ev_used & 1) { std::swap(w->ev[keep], w->ev[w->ev_used - 1]); keep += 1; }     // a start without its stop yet
    w->ev_used = keep;
    return SP_OK;
}

static int ws_event(sp_workspace* w, cudaStream_t st) {
    if (w->ev_used >= EV_FOLD && !(w->ev_used & 1)) {
        const int rc = ws_fold(w, false);
        if (rc) return rc;
    }
    if (w->ev_used == w->ev.size()) {
        cudaEvent_t e;
        CU(cudaEventCreate(&e));
        w->ev.push_back(e);
    }
    CU(cudaEventRecord(w->ev[w->ev_used++], st));
    return SP_OK;
}

extern "C" int sp_workspace_propagate_ms(sp_workspace* w, double* total_ms, int* n_launches) {
    if (!w || !total_ms || !n_launches) return fail(SP_EINVAL, "null argument");
    const int rc = ws_fold(w, true);
    if (rc) return rc;
    *total_ms = w->ev_ms; *n_launches = (int)w->ev_n;
    w->ev_ms = 0.0; w->ev_n = 0; w->ev_used = 0;
    return SP_OK;
}

extern "C" int sp_workspace_create(sp_workspace** out) {
    if (!out) return fail(SP_EINVAL, "null argument");
    sp_workspace* w = new sp_workspace();
    int dev = 0;
    CU(cudaGetDevice(&dev));
    CU(cudaDeviceGetAttribute(&w->sm_count, cudaDevAttrMultiProcessorCount, dev));
    CU(cudaMalloc(&w->cursor, sizeof(unsigned long long)));
    CU(cudaMalloc(&w->tile_sums, 1024 * sizeof(uint32_t)));
    CU(cudaMalloc(&w->long_count, sizeof(uint32_t)));
    CU(cudaMallocHost(&w->host_pair, 2 * sizeof(double)));
    *out = w;
    return SP_OK;
}
extern "C" int sp_workspace_destroy(sp_workspace* w) {
    if (!w) return SP_OK;
    cudaFree(w->keys); cudaFree(w->order); cudaFree(w->hist); cudaFree(w->tile_sums); cudaFree(w->long_list); cudaFree(w->long_count);
    cudaFree(w->cursor); cudaFree(w->joint);
    cudaFreeHost(w->host_pair);
    for (cudaEvent_t e : w->ev) cudaEventDestroy(e);
    delete w;
    return SP_OK;
}

static int ws_reserve_sort(sp_workspace* w, size_t rays, size_t keys) {
    if (rays > w->cap_rays) {
        cudaFree(w->keys); cudaFree(w->order); cudaFree(w->long_list); w->keys = w->order = w->long_list = nullptr; w->cap_rays = 0;
        CU(cudaMalloc(&w->keys, rays * sizeof(uint32_t)));
        CU(cudaMalloc(&w->order, rays * sizeof(uint32_t)));
        CU(cudaMalloc(&w->long_list, (rays / SP_LONG_SEGMENT + 2) * sizeof(uint32_t)));
        w->cap_rays = rays;
    }
    if (keys > w->cap_keys) {
        cudaFree(w->hist); w->hist = nullptr; w->cap_keys = 0;
        CU(cudaMalloc(&w->hist, keys * sizeof(uint32_t)));
        w->cap_keys = keys;
    }
    return SP_OK;
}

static BeamSpec beam_to_spec(const sp_beam* b) {
    BeamSpec B; memset(&B, 0, sizeof(B));
    if (b) {
        B.beam_type = b->beam_type; B.probing_axis = b->probing_axis; B.size_a = b->size_a; B.size_b = b->size_b;
        B.divergence = b->divergence; B.start = b->start; B.seed = b->seed;
    }
    return B;
}

static int kernel_index_of(const sp_field* f, int caller_axis) {
    for (int k = 0; k < 3; ++k) if (f->perm[k] == caller_axis) return k;
    return 0;
}

template <typename T, int METHOD> static constexpr size_t stage_smem_bytes() {
    return (METHOD == SP_METHOD_RK45 || METHOD == SP_METHOD_RK45B) ? (size_t)SP_STAGE_DOUBLES * 128 * sizeof(T) : 0;
}

template <typename T, int METHOD>
static int launch_propagate(const PropArgs<T>& A, const Epilogue& E, int grid, cudaStream_t st) {
    const bool phase = (A.flags & SP_FLAG_PHASE) != 0, aux64 = phase && (A.flags & SP_FLAG_PHASE_F64) != 0;
    const size_t sm = stage_smem_bytes<T, METHOD>();
    if (!phase) k_propagate<T, METHOD, false, false><<<grid, 128, sm, st>>>(A, E);
    else if (!aux64) k_propagate<T, METHOD, true, false><<<grid, 128, sm, st>>>(A, E);
    else k_propagate<T, METHOD, true, true><<<grid, 128, sm, st>>>(A, E);
    LAUNCH_CHECK();
    return SP_OK;
}

template <typename T, int METHOD> static int occupancy_grid(int sm_count, int flags, int& grid) {
    int per_sm = 0;
    const bool phase = (flags & SP_FLAG_PHASE) != 0, aux64 = phase && (flags & SP_FLAG_PHASE_F64) != 0;
    const size_t sm = stage_smem_bytes<T, METHOD>();
    if (!phase) CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_propagate<T, METHOD, false, false>, 128, sm));
    else if (!aux64) CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_propagate<T, METHOD, true, false>, 128, sm));
    else CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_propagate<T, METHOD, true, true>, 128, sm));
    if (per_sm < 1) per_sm = 1;
    grid = sm_count * per_sm;
    return SP_OK;
}

static int joint_solve(const sp_field* field, const sp_params* P, sp_workspace* ws, const double* s0_dev, uint64_t n,
                       const Epilogue& E, sp_stats* stats_dev, cudaStream_t st);

// attenuation / Faraday variant: float64, PHASE lane always compiled in (its integration is a run-time flag)
static int ext_grid(int sm_count, bool adaptive, bool aux64, int& grid) {
    int per_sm = 0;
    if (adaptive) {
        if (aux64) CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_propagate<double, SP_METHOD_RK45X, true, true>, 128, 0));
        else CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_propagate<double, SP_METHOD_RK45X, true, false>, 128, 0));
    } else {
        if (aux64) CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_propagate<double, SP_METHOD_RK4X, true, true>, 128, 0));
        else CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_propagate<double, SP_METHOD_RK4X, true, false>, 128, 0));
    }
    grid = sm_count * (per_sm < 1 ? 1 : per_sm);
    return SP_OK;
}
static int launch_ext(const PropArgs<double>& A, const Epilogue& E, bool adaptive, bool aux64, int grid, cudaStream_t st) {
    if (adaptive) {
        if (aux64) k_propagate<double, SP_METHOD_RK45X, true, true><<<grid, 128, 0, st>>>(A, E);
        else k_propagate<double, SP_METHOD_RK45X, true, false><<<grid, 128, 0, st>>>(A, E);
    } else {
        if (aux64) k_propagate<double, SP_METHOD_RK4X, true, true><<<grid, 128, 0, st>>>(A, E);
        else k_propagate<double, SP_METHOD_RK4X, true, false><<<grid, 128, 0, st>>>(A, E);
    }
    LAUNCH_CHECK();
    return SP_OK;
}

extern "C" int sp_propagate(const sp_field* field, const sp_params* P, sp_workspace* ws, const double* s0_dev,
                            const sp_beam* beam, uint64_t n, uint64_t ray_offset, double* sf_dev, double* rf_dev,
                            double* jf_dev, uint32_t* steps_dev, const sp_channel* channels_host, int n_channels,
                            sp_stats* stats_dev, void* stream) {
    if (!field || !P || !ws) return fail(SP_EINVAL, "null field / params / workspace");
    if (!s0_dev && !beam) return fail(SP_EINVAL, "need either s0_dev or a beam spec");
    if (n_channels < 0 || n_channels > SP_MAX_CHANNELS) return fail(SP_EINVAL, "at most 4 detector channels");
    if (P->probing_axis < 0 || P->probing_axis > 2 || P->out_axis_a < 0 || P->out_axis_a > 2 || P->out_axis_b < 0 ||
        P->out_axis_b > 2)
        return fail(SP_EINVAL, "axis index out of range");
    if (P->method == SP_METHOD_RK4 && (P->n_steps < 0 || !(P->h > 0))) return fail(SP_EINVAL, "RK4 needs n_steps >= 0 and h > 0");
    if ((P->flags & SP_FLAG_PHASE_F64) && !field->aux64) return fail(SP_ESTATE, "field was built without SP_FIELD_PHASE_F64");
    if (n == 0) return SP_OK;
    cudaStream_t st = (cudaStream_t)stream;
    Epilogue E; memset(&E, 0, sizeof(E));
    E.sf = sf_dev; E.rf = rf_dev; E.jf = jf_dev; E.steps = steps_dev; E.n_channels = n_channels;
    for (int c = 0; c < n_channels; ++c) {
        int rc = channel_to_dev(channels_host + c, E.ch[c]);
        if (rc) return rc;
    }
    const bool ext = (P->flags & (SP_FLAG_ATTEN | SP_FLAG_FARADAY)) != 0;
    if (ext) {
        if (P->flags & SP_FLAG_FP32) return fail(SP_EINVAL, "attenuation / Faraday channels are float64 only");
        if ((P->flags & SP_FLAG_ATTEN) && !field->ext[0]) return fail(SP_ESTATE, "SP_FLAG_ATTEN without a kappa grid (sp_field_attach_channels)");
        if ((P->flags & SP_FLAG_FARADAY) && !(field->ext[1] && field->ext[2] && field->ext[3] && field->ext[4]))
            return fail(SP_ESTATE, "SP_FLAG_FARADAY without ne and B grids (sp_field_attach_channels)");
    }
    if (P->method == SP_METHOD_RK45_JOINT) {
        if (!s0_dev) return fail(SP_EINVAL, "joint RK45 needs explicit s0");
        if (P->flags & SP_FLAG_FP32) return fail(SP_EINVAL, "joint RK45 is float64 only");
        return joint_solve(field, P, ws, s0_dev, n, E, stats_dev, st);
    }
    if (P->method == SP_METHOD_TSIT5) {
        if (ext) return fail(SP_EINVAL, "tsit5 does not integrate the attenuation / Faraday channels");
        if (!(P->h > 0) || !(P->t_end > 0)) return fail(SP_EINVAL, "tsit5 needs h = dt0 > 0 (units of t_end) and t_end > 0");
    } else if (P->method != SP_METHOD_RK4 && P->method != SP_METHOD_RK45) return fail(SP_EINVAL, "unknown method");
    if (ext && (P->flags & SP_FLAG_BUNDLE_STEP)) return fail(SP_EINVAL, "bundle-step RK45 does not integrate the attenuation / Faraday channels");
    const bool ext_aux64 = ext && (P->flags & SP_FLAG_PHASE) && (P->flags & SP_FLAG_PHASE_F64);

    const bool fp32 = (P->flags & SP_FLAG_FP32) != 0;
    const bool sort = !(P->flags & SP_FLAG_NO_SORT);
    const uint64_t CHUNK = 1ull << 25;
    // sort key geometry: Morton code over (u, v) cell columns, coarsened to at most 2^22 keys
    int bits = 1;
    while ((1 << bits) < (field->nk[0] > field->nk[1] ? field->nk[0] : field->nk[1])) ++bits;
    int key_shift = 2 * bits > 22 ? 2 * bits - 22 : 0;
    const uint32_t n_keys = 1u << (2 * bits - key_shift);

    int grid = 0, rc = 0;
    const bool bundle_step = P->method == SP_METHOD_RK45 && (P->flags & SP_FLAG_BUNDLE_STEP);
    const bool tsit = P->method == SP_METHOD_TSIT5;
    if (tsit) rc = fp32 ? occupancy_grid<float, SP_METHOD_TSIT5>(ws->sm_count, P->flags, grid) : occupancy_grid<double, SP_METHOD_TSIT5>(ws->sm_count, P->flags, grid);
    else if (ext) rc = ext_grid(ws->sm_count, P->method == SP_METHOD_RK45, ext_aux64, grid);
    else if (fp32) rc = (P->method == SP_METHOD_RK4) ? occupancy_grid<float, SP_METHOD_RK4>(ws->sm_count, P->flags, grid)
                        : (bundle_step ? occupancy_grid<float, SP_METHOD_RK45B>(ws->sm_count, P->flags, grid)
                                       : occupancy_grid<float, SP_METHOD_RK45>(ws->sm_count, P->flags, grid));
    else rc = (P->method == SP_METHOD_RK4) ? occupancy_grid<double, SP_METHOD_RK4>(ws->sm_count, P->flags, grid)
              : (bundle_step ? occupancy_grid<double, SP_METHOD_RK45B>(ws->sm_count, P->flags, grid)
                             : occupancy_grid<double, SP_METHOD_RK45>(ws->sm_count, P->flags, grid));
    if (rc) return rc;

    for (uint64_t off = 0; off < n; off += CHUNK) {
        const uint32_t cn = (uint32_t)((n - off) < CHUNK ? (n - off) : CHUNK);
        const uint32_t* order = nullptr;
        if (sort && cn > 64) {
            rc = ws_reserve_sort(ws, cn, n_keys);
            if (rc) return rc;
            SortArgs S; memset(&S, 0, sizeof(S));
            S.s0 = s0_dev; S.n_total = n; S.chunk_off = off; S.chunk_n = cn;
            S.beam = beam_to_spec(beam); S.use_beam = s0_dev ? 0 : 1; S.ray_offset = ray_offset;
            for (int k = 0; k < 3; ++k) S.perm[k] = field->perm[k];
            S.g0u = field->g0[0]; S.inv_du = field->inv_d[0]; S.g0v = field->g0[1]; S.inv_dv = field->inv_d[1];
            S.nu = field->nk[0]; S.nv = field->nk[1]; S.key_shift = key_shift; S.n_keys = n_keys;
            CU(cudaMemsetAsync(ws->hist, 0, n_keys * sizeof(uint32_t), st));
            k_sort_keys<<<(cn + 255) / 256, 256, 0, st>>>(S, ws->keys, ws->hist);
            LAUNCH_CHECK();
            const uint32_t n_tiles = (n_keys + SP_SCAN_TILE - 1) / SP_SCAN_TILE;       // <= 1024 (n_keys <= 2^22)
            k_scan_tiles<<<n_tiles, 1024, 0, st>>>(ws->hist, n_keys, ws->tile_sums);
            LAUNCH_CHECK();
            if (n_tiles > 1) {
                k_scan_tops<<<1, 1024, 0, st>>>(ws->tile_sums, n_tiles);
                LAUNCH_CHECK();
                k_scan_add<<<n_tiles, 1024, 0, st>>>(ws->hist, n_keys, ws->tile_sums);
                LAUNCH_CHECK();
            }
            k_sort_scatter<<<(cn + 255) / 256, 256, 0, st>>>(ws->keys, ws->hist, ws->order, cn);
            LAUNCH_CHECK();
            CU(cudaMemsetAsync(ws->long_count, 0, sizeof(uint32_t), st));
            k_sort_fix<<<(n_keys + 255) / 256, 256, 0, st>>>(ws->hist, ws->order, n_keys, ws->long_list, ws->long_count);   // hist now holds segment ends
            LAUNCH_CHECK();
            k_sort_fix_long<<<ws->sm_count, 256, 0, st>>>(ws->hist, ws->order, ws->keys, ws->long_list, ws->long_count);
            LAUNCH_CHECK();
            order = ws->order;
        }
        CU(cudaMemsetAsync(ws->cursor, 0, sizeof(unsigned long long), st));
        const uint64_t bundles = (cn + 31) / 32;
        int g = grid;
        if ((uint64_t)g * 4 > bundles) g = (int)((bundles + 3) / 4);
        if (g < 1) g = 1;
#define FILL(T)                                                                                          \
        PropArgs<T> A; memset(&A, 0, sizeof(A));                                                         \
        A.F = make_view<T>(field); A.s0 = s0_dev; A.n_total = n; A.chunk_off = off; A.chunk_n = cn;      \
        A.order = order; A.cursor = ws->cursor; A.beam = beam_to_spec(beam); A.use_beam = s0_dev ? 0 : 1; \
        A.ray_offset = ray_offset;                                                                       \
        for (int k = 0; k < 3; ++k) A.perm[k] = field->perm[k];                                          \
        A.kp = kernel_index_of(field, P->probing_axis); A.ka = kernel_index_of(field, P->out_axis_a);    \
        A.kb = kernel_index_of(field, P->out_axis_b);                                                    \
        A.method = P->method; A.flags = P->flags; A.n_steps = P->n_steps; A.n_state = P->n_state > 0 ? P->n_state : 9; \
        A.h = (T)P->h; A.t_end = (T)P->t_end; A.rtol = (T)P->rtol; A.atol = (T)P->atol; A.omega = (T)P->omega; \
        A.extent = (T)P->extent; A.stats = stats_dev; A.rk = RK4Step<T>((T)P->h);
        rc = ws_event(ws, st);
        if (rc) return rc;
        if (tsit && fp32) {
            FILL(float)
            rc = launch_propagate<float, SP_METHOD_TSIT5>(A, E, g, st);
        } else if (tsit) {
            FILL(double)
            rc = launch_propagate<double, SP_METHOD_TSIT5>(A, E, g, st);
        } else if (fp32) {
            FILL(float)
            rc = (P->method == SP_METHOD_RK4) ? launch_propagate<float, SP_METHOD_RK4>(A, E, g, st)
                 : (bundle_step ? launch_propagate<float, SP_METHOD_RK45B>(A, E, g, st) : launch_propagate<float, SP_METHOD_RK45>(A, E, g, st));
        } else if (ext) {
            FILL(double)
            A.X = make_ext(field, P->verdet, P->flags);
            rc = launch_ext(A, E, P->method == SP_METHOD_RK45, ext_aux64, g, st);
        } else {
            FILL(double)
            rc = (P->method == SP_METHOD_RK4) ? launch_propagate<double, SP_METHOD_RK4>(A, E, g, st)
                 : (bundle_step ? launch_propagate<double, SP_METHOD_RK45B>(A, E, g, st) : launch_propagate<double, SP_METHOD_RK45>(A, E, g, st));
        }
#undef FILL
        if (rc) return rc;
        rc = ws_event(ws, st);
        if (rc) return rc;
    }
    return SP_OK;
}

// Host controller of the joint solve: a line-for-line counterpart of scipy's RK45._step_impl loop, with the
// vector norms evaluated on the device (deterministic two-level reduction).
static int joint_solve(const sp_field* field, const sp_params* P, sp_workspace* ws, const double* s0_dev, uint64_t n,
                       const Epilogue& E, sp_stats* stats_dev, cudaStream_t st) {
    const int threads = 128;
    const int nblocks = (int)((n + threads - 1) / threads);
    const size_t per = n;
    const size_t need = (size_t)(7 + 4 + 7 + 4 + 2) * per + 2 * (size_t)nblocks;
    if (need > ws->joint_cap) {
        cudaFree(ws->joint); ws->joint = nullptr; ws->joint_cap = 0;
        CU(cudaMalloc(&ws->joint, need * sizeof(double)));
        ws->joint_cap = need;
    }
    JointBuf B; double* q = ws->joint;
    for (int k = 0; k < 3; ++k) { B.p[k] = q; q += per; }
    for (int k = 0; k < 3; ++k) { B.v[k] = q; q += per; }
    B.ph = q; q += per;
    for (int k = 0; k < 3; ++k) { B.fv[k] = q; q += per; }
    B.fph = q; q += per;
    for (int k = 0; k < 3; ++k) { B.pn[k] = q; q += per; }
    for (int k = 0; k < 3; ++k) { B.vn[k] = q; q += per; }
    B.phn = q; q += per;
    for (int k = 0; k < 3; ++k) { B.fvn[k] = q; q += per; }
    B.fphn = q; q += per;
    B.amp = q; q += per; B.pol = q; q += per;
    B.partial = q;

    FieldView<double> F = make_view<double>(field);
    const bool phase = (P->flags & SP_FLAG_PHASE) != 0, aux64 = phase && (P->flags & SP_FLAG_PHASE_F64) != 0;
    const int p0 = field->perm[0], p1 = field->perm[1], p2 = field->perm[2];
    const double rtol = P->rtol, atol = P->atol, omega = P->omega, t_end = P->t_end;
    const int n_state = P->n_state > 0 ? P->n_state : 9;
    const double size = (double)n_state * (double)n;     // x.size of the flattened state
    uint64_t evals = 0;

    // attenuation / Faraday channels on: nine-row kernels over a second set of buffers (Y, F, Yn, Fn: [9][n] each)
    const bool ext = (P->flags & (SP_FLAG_ATTEN | SP_FLAG_FARADAY)) != 0;
    const ExtView X = make_ext(field, P->verdet, P->flags);
    double *Yc = nullptr, *Fc = nullptr, *Yn = nullptr, *Fn = nullptr;
    if (ext) {
        const size_t need_x = need + 36 * per;
        if (need_x > ws->joint_cap) {
            cudaFree(ws->joint); ws->joint = nullptr; ws->joint_cap = 0;
            CU(cudaMalloc(&ws->joint, need_x * sizeof(double)));
            ws->joint_cap = need_x;
        }
        B.partial = ws->joint;                               // 2 * nblocks doubles, then the four state blocks
        Yc = ws->joint + 2 * (size_t)nblocks; Fc = Yc + 9 * per; Yn = Fc + 9 * per; Fn = Yn + 9 * per;
    }
    const bool ext_aux64 = ext && aux64;

    auto init_pass = [&](int pass, double h0) -> int {
        if (ext) {
            if (ext_aux64) k_jointx_init<true, true><<<nblocks, threads, 0, st>>>(F, X, Yc, Fc, B.partial, s0_dev, n, p0, p1, p2, omega, phase, rtol, atol, pass, h0);
            else k_jointx_init<true, false><<<nblocks, threads, 0, st>>>(F, X, Yc, Fc, B.partial, s0_dev, n, p0, p1, p2, omega, phase, rtol, atol, pass, h0);
        } else if (!phase) k_joint_init<false, false><<<nblocks, threads, 0, st>>>(F, B, s0_dev, n, p0, p1, p2, omega, rtol, atol, pass, h0);
        else if (!aux64) k_joint_init<true, false><<<nblocks, threads, 0, st>>>(F, B, s0_dev, n, p0, p1, p2, omega, rtol, atol, pass, h0);
        else k_joint_init<true, true><<<nblocks, threads, 0, st>>>(F, B, s0_dev, n, p0, p1, p2, omega, rtol, atol, pass, h0);
        LAUNCH_CHECK();
        k_joint_reduce<<<1, 256, 0, st>>>(B.partial, nblocks, ws->host_pair);
        LAUNCH_CHECK();
        CU(cudaStreamSynchronize(st));
        evals += n;
        return SP_OK;
    };
    // select_initial_step (scipy/integrate/_ivp/common.py)
    int rc = init_pass(0, 0.0);
    if (rc) return rc;
    const double d0 = sqrt(ws->host_pair[0]) / sqrt(size), d1 = sqrt(ws->host_pair[1]) / sqrt(size);
    double h0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * d0 / d1;
    h0 = h0 < t_end ? h0 : t_end;
    rc = init_pass(1, h0);
    if (rc) return rc;
    const double d2 = sqrt(ws->host_pair[0]) / sqrt(size) / h0;
    double h1;
    if (d1 <= 1e-15 && d2 <= 1e-15) h1 = (1e-6 > h0 * 1e-3) ? 1e-6 : h0 * 1e-3;
    else h1 = pow(0.01 / (d1 > d2 ? d1 : d2), 0.2);
    double h_abs = 100 * h0 < h1 ? 100 * h0 : h1;
    h_abs = h_abs < t_end ? h_abs : t_end;

    double t = 0.0;
    uint64_t attempts = 0, accepted = 0;
    ws->jlog_h.clear(); ws->jlog_en.clear();
    const uint64_t cap = P->n_steps > 0 ? (uint64_t)P->n_steps : (1ull << 30);
    bool failed = false;
    while (t < t_end && !failed) {
        const double min_step = 10 * fabs(nextafter(t, INFINITY) - t);
        if (h_abs < min_step) h_abs = min_step;
        bool rejected = false;
        for (;;) {
            if (attempts >= cap || h_abs < min_step) { failed = true; break; }
            double t_new = t + h_abs;
            if (t_new - t_end > 0) t_new = t_end;
            const double h = t_new - t;
            h_abs = fabs(h);
            if (ext) {
                if (ext_aux64) k_jointx_attempt<true, true><<<nblocks, threads, 0, st>>>(F, X, Yc, Fc, Yn, Fn, B.partial, n, omega, phase, h, rtol, atol);
                else k_jointx_attempt<true, false><<<nblocks, threads, 0, st>>>(F, X, Yc, Fc, Yn, Fn, B.partial, n, omega, phase, h, rtol, atol);
            } else if (!phase) k_joint_attempt<false, false><<<nblocks, threads, 0, st>>>(F, B, n, omega, h, rtol, atol);
            else if (!aux64) k_joint_attempt<true, false><<<nblocks, threads, 0, st>>>(F, B, n, omega, h, rtol, atol);
            else k_joint_attempt<true, true><<<nblocks, threads, 0, st>>>(F, B, n, omega, h, rtol, atol);
            LAUNCH_CHECK();
            k_joint_reduce<<<1, 256, 0, st>>>(B.partial, nblocks, ws->host_pair);
            LAUNCH_CHECK();
            CU(cudaStreamSynchronize(st));
            ++attempts; evals += 6 * n;
            const double en = sqrt(ws->host_pair[0]) / sqrt(size);
            ws->jlog_h.push_back(h); ws->jlog_en.push_back(en);
            if (!(en == en)) { failed = true; break; }                               // NaN state: solve_ivp would never return
            if (en < 1) {
                double f = (en == 0) ? DP::MAX_FACTOR : fmin(DP::MAX_FACTOR, DP::SAFETY * pow(en, -0.2));
                if (rejected) f = fmin(1.0, f);
                h_abs *= f;
                t = t_new; ++accepted;
                // accept: candidate becomes current (pointer swap)
                for (int k = 0; k < 3; ++k) { std::swap(B.p[k], B.pn[k]); std::swap(B.v[k], B.vn[k]); std::swap(B.fv[k], B.fvn[k]); }
                std::swap(B.ph, B.phn); std::swap(B.fph, B.fphn);
                std::swap(Yc, Yn); std::swap(Fc, Fn);
                break;
            }
            h_abs *= fmax(DP::MIN_FACTOR, DP::SAFETY * pow(en, -0.2));
            rejected = true;
        }
    }
    if (ext) {                                               // present the nine-row state through the JointBuf view
        for (int k = 0; k < 3; ++k) { B.p[k] = Yc + (size_t)k * per; B.v[k] = Yc + (size_t)(3 + k) * per; }
        B.amp = Yc + 6 * per; B.ph = Yc + 7 * per; B.pol = Yc + 8 * per;
    }
    k_joint_finish<<<nblocks, threads, 0, st>>>(B, n, 0, p0, p1, p2, kernel_index_of(field, P->probing_axis),
                                                kernel_index_of(field, P->out_axis_a), kernel_index_of(field, P->out_axis_b),
                                                P->extent, E, stats_dev);
    LAUNCH_CHECK();
    if (stats_dev) {
        sp_stats hs; memset(&hs, 0, sizeof(hs));
        sp_stats cur;
        CU(cudaMemcpyAsync(&cur, stats_dev, sizeof(cur), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        cur.ray_steps += attempts * n; cur.ray_steps_acc += accepted * n; cur.rhs_evals += evals;
        cur.rays_capped += failed ? n : 0;
        CU(cudaMemcpyAsync(stats_dev, &cur, sizeof(cur), cudaMemcpyHostToDevice, st));
        CU(cudaStreamSynchronize(st));
    }
    if (E.steps) {
        // every ray took the same number of attempts
        std::vector<uint32_t> hsteps(n, (uint32_t)attempts);
        CU(cudaMemcpyAsync(E.steps, hsteps.data(), n * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        CU(cudaStreamSynchronize(st));
    }
    return SP_OK;
}

extern "C" int sp_rhs(const sp_field* field, const sp_params* P, const double* s_dev, uint64_t n, double* dsdt_dev,
                      void* stream) {
    if (!field || !P || !s_dev || !dsdt_dev) return fail(SP_EINVAL, "null argument");
    if ((P->flags & SP_FLAG_PHASE_F64) && !field->aux64) return fail(SP_ESTATE, "field was built without SP_FIELD_PHASE_F64");
    if (n == 0) return SP_OK;
    FieldView<double> F = make_view<double>(field);
    const bool phase = (P->flags & SP_FLAG_PHASE) != 0, aux64 = phase && (P->flags & SP_FLAG_PHASE_F64) != 0;
    const int blocks = (int)((n + 127) / 128);
    cudaStream_t st = (cudaStream_t)stream;
    const int p0 = field->perm[0], p1 = field->perm[1], p2 = field->perm[2];
    const ExtView X = make_ext(field, P->verdet, P->flags);
    if (!phase) k_rhs<false, false><<<blocks, 128, 0, st>>>(F, X, s_dev, n, dsdt_dev, p0, p1, p2, P->omega);
    else if (!aux64) k_rhs<true, false><<<blocks, 128, 0, st>>>(F, X, s_dev, n, dsdt_dev, p0, p1, p2, P->omega);
    else k_rhs<true, true><<<blocks, 128, 0, st>>>(F, X, s_dev, n, dsdt_dev, p0, p1, p2, P->omega);
    LAUNCH_CHECK();
    return SP_OK;
}

extern "C" int sp_beam_generate(const sp_beam* beam, uint64_t ray_offset, uint64_t n, double* s0_dev, void* stream) {
    if (!beam || !s0_dev) return fail(SP_EINVAL, "null argument");
    if (n == 0) return SP_OK;
    k_beam<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(beam_to_spec(beam), ray_offset, n, s0_dev);
    LAUNCH_CHECK();
    return SP_OK;
}

extern "C" int sp_optics_image(const double* rf_dev, const double* jf_dev, uint64_t n, const sp_channel* chan,
                               double* rf_out_dev, double* jf_out_dev, void* stream) {
    if (!rf_dev || !chan) return fail(SP_EINVAL, "null argument");
    if (n == 0) return SP_OK;
    ChannelDev ch;
    int rc = channel_to_dev(chan, ch);
    if (rc) return rc;
    if (ch.kind == SP_IMG_INTERFEROGRAM && ch.nx > 0 && !jf_dev) return fail(SP_EINVAL, "interferogram needs Jones vectors");
    if (ch.kind == SP_IMG_STOKES && ch.nx > 0 && !jf_dev) return fail(SP_EINVAL, "Stokes image needs Jones vectors");
    uint64_t blocks = (n + 255) / 256;
    const size_t nbins = (size_t)ch.nx * ch.ny;
    if (ch.kind == SP_IMG_HISTOGRAM && nbins > 0 && nbins <= 12288) {
        if (blocks > 148 * 4) blocks = 148 * 4;           // few, fat CTAs: each flushes its private image once
        k_optics_image<true><<<(unsigned)blocks, 256, nbins * sizeof(unsigned), (cudaStream_t)stream>>>(rf_dev, jf_dev, n, ch,
                                                                                                     rf_out_dev, jf_out_dev);
    } else {
        if (blocks > 148 * 16) blocks = 148 * 16;
        k_optics_image<false><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(rf_dev, jf_dev, n, ch, rf_out_dev, jf_out_dev);
    }
    LAUNCH_CHECK();
    return SP_OK;
}

extern "C" int sp_exit_plane(const double* sf_dev, uint64_t n, int probing_axis, int out_axis_a, int out_axis_b, double extent,
                             int keep_current_plane, double* rf_dev, double* jf_dev, double* sback_dev, void* stream) {
    if (!sf_dev) return fail(SP_EINVAL, "null argument");
    if (probing_axis < 0 || probing_axis > 2 || out_axis_a < 0 || out_axis_a > 2 || out_axis_b < 0 || out_axis_b > 2)
        return fail(SP_EINVAL, "axis index out of range");
    if (n == 0) return SP_OK;
    k_exit_plane<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(sf_dev, n, probing_axis, out_axis_a, out_axis_b,
                                                                               extent, keep_current_plane, rf_dev, jf_dev, sback_dev);
    LAUNCH_CHECK();
    return SP_OK;
}

extern "C" int sp_image_finalize(const sp_image* img, double* H_dev, void* stream) {
    if (!img || !H_dev || !img->planes_dev) return fail(SP_EINVAL, "null argument");
    const size_t npix = (size_t)img->nx * img->ny;
    if (npix == 0) return SP_OK;
    if (img->kind == SP_IMG_STOKES)
        k_finalize_stokes<<<(unsigned)((npix + 255) / 256), 256, 0, (cudaStream_t)stream>>>((const long long*)img->planes_dev, H_dev, npix);
    else
        k_finalize<<<(unsigned)((npix + 255) / 256), 256, 0, (cudaStream_t)stream>>>((const long long*)img->planes_dev, H_dev, npix);
    LAUNCH_CHECK();
    return SP_OK;
}

// ------------------------------------------------------------------------------- FP64 pipe peak (measurement aid)
// The ray integrator is bound by the FP64 pipe and its issue slots, not by HBM (ncu: DRAM < 1 % of peak), so
// bench.py's roofline needs an FP64 denominator measured on the same GPU in the same run.  Every thread runs 8
// independent DFMA chains (no memory traffic, full occupancy): the launch sustains the pipe's issue rate.
__global__ void __launch_bounds__(256) k_fp64_peak(int iters, double seed, double* __restrict__ out, uint64_t out_len) {
    double a0 = seed, a1 = seed + 1.0, a2 = seed + 2.0, a3 = seed + 3.0, a4 = seed + 4.0, a5 = seed + 5.0, a6 = seed + 6.0, a7 = seed + 7.0;
    const double m = 1.0 - 1e-9 * (double)(threadIdx.x & 7), c = 1e-12;
#pragma unroll 4
    for (int i = 0; i < iters; ++i) {
        a0 = __fma_rn(a0, m, c); a1 = __fma_rn(a1, m, c); a2 = __fma_rn(a2, m, c); a3 = __fma_rn(a3, m, c);
        a4 = __fma_rn(a4, m, c); a5 = __fma_rn(a5, m, c); a6 = __fma_rn(a6, m, c); a7 = __fma_rn(a7, m, c);
    }
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < out_len) out[t] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

extern "C" int sp_fp64_peak(int iters, double* out_dev, uint64_t out_len, uint64_t* n_dfma_out, void* stream) {
    if (iters < 1 || !out_dev || !n_dfma_out) return fail(SP_EINVAL, "need iters >= 1, an output buffer and n_dfma_out");
    int dev = 0, sms = 0;
    CU(cudaGetDevice(&dev));
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int grid = sms * 8;                                  // 8 x 256 threads = 2048 resident threads per SM
    k_fp64_peak<<<grid, 256, 0, (cudaStream_t)stream>>>(iters, 1.0, out_dev, out_len);
    LAUNCH_CHECK();
    *n_dfma_out = (uint64_t)grid * 256ull * (uint64_t)iters * 8ull;
    return SP_OK;
}

// ------------------------------------------------------------------------------- wave-optics step (SURVEY 8f-2)
// Scattered rays -> detector grid on a triangulation, then the Fresnel step around the library FFT.  All four
// kernels are streaming passes (HBM-bound: 16-32 B per sample); per-sample math is fresnel_core.h.
#include "fresnel_core.h"

static unsigned stream_grid(unsigned long long n) {                    // grid-stride launches: a few waves of 148 SMs
    unsigned long long b = (n + 255) / 256;
    return (unsigned)(b < 148ull * 16 ? (b ? b : 1) : 148ull * 16);
}

// pass 1: every triangle claims the grid nodes it contains; ties (nodes on shared edges) go to the lowest index,
// so the result does not depend on scheduling
__global__ void k_tri_owner(const double* __restrict__ px, const double* __restrict__ py, const int32_t* __restrict__ tri,
                            unsigned long long n_tri, const double* __restrict__ gx, const double* __restrict__ gy, int nx,
                            int ny, int32_t* __restrict__ owner) {
    for (unsigned long long t = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; t < n_tri;
         t += (unsigned long long)gridDim.x * blockDim.x) {
        const int32_t ia = tri[3 * t], ib = tri[3 * t + 1], ic = tri[3 * t + 2];
        const double ax = px[ia], ay = py[ia], bx = px[ib], by = py[ib], cx = px[ic], cy = py[ic];
        const double x0 = fmin(ax, fmin(bx, cx)), x1 = fmax(ax, fmax(bx, cx));
        const double y0 = fmin(ay, fmin(by, cy)), y1 = fmax(ay, fmax(by, cy));
        const double sx = (x1 - x0) * 1e-12, sy = (y1 - y0) * 1e-12;
        const int i0 = lower_bound_d(gx, nx, x0 - sx), j0 = lower_bound_d(gy, ny, y0 - sy);
        for (int j = j0; j < ny && gy[j] <= y1 + sy; ++j)
            for (int i = i0; i < nx && gx[i] <= x1 + sx; ++i) {
                double l0, l1, l2;
                if (bary2(ax, ay, bx, by, cx, cy, gx[i], gy[j], l0, l1, l2) && tri_inside(l0, l1, l2))
                    atomicMin(owner + (size_t)j * nx + i, (int32_t)t);
            }
    }
}

// pass 2: one thread per grid node interpolates every value array inside its owning triangle
__global__ void k_tri_interp(const double* __restrict__ px, const double* __restrict__ py, const double* __restrict__ val,
                             int n_val, unsigned long long n_pts, const int32_t* __restrict__ tri,
                             const double* __restrict__ gx, const double* __restrict__ gy, int nx, int ny,
                             const int32_t* __restrict__ owner, double fill, double* __restrict__ out) {
    const size_t npix = (size_t)nx * ny;
    for (size_t p = blockIdx.x * (size_t)blockDim.x + threadIdx.x; p < npix; p += (size_t)gridDim.x * blockDim.x) {
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

__global__ void k_fill_i32(int32_t* __restrict__ a, size_t n, int32_t v) {
    for (size_t p = blockIdx.x * (size_t)blockDim.x + threadIdx.x; p < n; p += (size_t)gridDim.x * blockDim.x) a[p] = v;
}

extern "C" int sp_scatter_to_grid(const double* px_dev, const double* py_dev, const double* val_dev, int n_val,
                                  uint64_t n_pts, const int32_t* tri_dev, uint64_t n_tri, const double* gx_dev,
                                  const double* gy_dev, int nx, int ny, double fill_value, int32_t* owner_dev,
                                  double* out_dev, void* stream) {
    if (!px_dev || !py_dev || !val_dev || !gx_dev || !gy_dev || !owner_dev || !out_dev) return fail(SP_EINVAL, "null argument");
    if (n_val < 1 || nx < 1 || ny < 1) return fail(SP_EINVAL, "need n_val, nx, ny >= 1");
    if (n_tri && !tri_dev) return fail(SP_EINVAL, "null triangulation");
    if (n_pts > (uint64_t)INT32_MAX || n_tri >= (uint64_t)INT32_MAX) return fail(SP_EINVAL, "more than 2^31 - 1 points / triangles");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t npix = (size_t)nx * ny;
    k_fill_i32<<<stream_grid(npix), 256, 0, st>>>(owner_dev, npix, INT32_MAX);
    LAUNCH_CHECK();
    if (n_tri) {
        k_tri_owner<<<stream_grid(n_tri), 256, 0, st>>>(px_dev, py_dev, tri_dev, n_tri, gx_dev, gy_dev, nx, ny, owner_dev);
        LAUNCH_CHECK();
    }
    k_tri_interp<<<stream_grid(npix), 256, 0, st>>>(px_dev, py_dev, val_dev, n_val, n_pts, tri_dev, gx_dev, gy_dev, nx, ny,
                                                    owner_dev, fill_value, out_dev);
    LAUNCH_CHECK();
    return SP_OK;
}

// U0 = amp exp(-i phase) on the source grid: one sincos per source sample instead of one per padded sample (x25 at pad 2)
__global__ void k_fresnel_u0(const double* __restrict__ amp, const double* __restrict__ phase, long long n, d2* __restrict__ u0) {
    for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < n; p += (long long)gridDim.x * blockDim.x) {
        d2 u;
        u0_from_amp_phase(amp[p], phase[p], u.x, u.y);
        u0[p] = u;
    }
}

// Reflect padding + separable Tukey window.  A CTA writes a tile of FR_ROWS rows x 256 columns: every thread keeps its
// column's source index and window factor, the first FR_ROWS threads compute the rows', so a padded sample costs one
// 16-byte gather (the source grid is 1/25 of the output and stays in L2), two multiplies and one coalesced 16-byte store.
#define FR_ROWS 16
__global__ void __launch_bounds__(256) k_fresnel_pad(const d2* __restrict__ u0, int n0, int n1, int pad, double alpha,
                                                     d2* __restrict__ out) {
    __shared__ double w0s[FR_ROWS];
    __shared__ int s0s[FR_ROWS];
    const long long m0 = (2LL * pad + 1) * n0, m1 = (2LL * pad + 1) * n1;
    const long long c = blockIdx.x * 256LL + threadIdx.x, r0 = blockIdx.y * (long long)FR_ROWS;
    if (threadIdx.x < FR_ROWS && r0 + threadIdx.x < m0) {
        w0s[threadIdx.x] = tukey_w(r0 + threadIdx.x, m0, alpha);
        s0s[threadIdx.x] = (int)reflect_idx(r0 + threadIdx.x - (long long)pad * n0, n0);
    }
    __syncthreads();
    if (c >= m1) return;
    const double w1 = tukey_w(c, m1, alpha);
    const long long s1 = reflect_idx(c - (long long)pad * n1, n1);
    const int rows = (int)((m0 - r0) < FR_ROWS ? (m0 - r0) : FR_ROWS);
#pragma unroll 4
    for (int k = 0; k < rows; ++k) {
        const d2 u = u0[(long long)s0s[k] * n1 + s1];
        const double w = w0s[k] * w1;
        d2 o;
        o.x = u.x * w;
        o.y = u.y * w;
        out[(r0 + k) * m1 + c] = o;
    }
}

// Transfer function in place, same tiling: the column frequency once per thread, the row frequency once per row.
__global__ void __launch_bounds__(256) k_fresnel_transfer(d2* __restrict__ spec, int m0, int m1, double d0, double d1,
                                                          double wavelength, double z, double sigma) {
    const long long c = blockIdx.x * 256LL + threadIdx.x, r0 = blockIdx.y * (long long)FR_ROWS;
    if (c >= m1) return;
    const double f1 = fft_freq(c, m1, d1);
    const int rows = (int)((m0 - r0) < FR_ROWS ? (m0 - r0) : FR_ROWS);
#pragma unroll 2
    for (int k = 0; k < rows; ++k) {
        d2 u = spec[(r0 + k) * m1 + c];
        transfer_apply(u.x, u.y, fft_freq(r0 + k, m0, d0), f1, wavelength, z, sigma);
        spec[(r0 + k) * m1 + c] = u;
    }
}

__global__ void k_fresnel_finish(const d2* __restrict__ u_pad, long long n0, long long n1, long long pad, double cr,
                                 double ci, d2* __restrict__ out) {
    const long long m1 = (2 * pad + 1) * n1, total = n0 * n1;
    for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < total; p += (long long)gridDim.x * blockDim.x) {
        const d2 u = u_pad[(p / n1 + pad * n0) * m1 + (p % n1 + pad * n1)];
        d2 o;
        o.x = u.x * cr - u.y * ci;
        o.y = u.x * ci + u.y * cr;
        out[p] = o;
    }
}

extern "C" int sp_fresnel_prepare(const double* a_dev, const double* b_dev, int mode, int n0, int n1, int pad_factor,
                                  double alpha, double* u_pad_dev, void* stream) {
    if (!a_dev || !u_pad_dev || (mode == 1 && !b_dev)) return fail(SP_EINVAL, "null argument");
    if (mode != 0 && mode != 1) return fail(SP_EINVAL, "mode must be 0 (complex field) or 1 (amplitude, phase)");
    if (n0 < 1 || n1 < 1 || pad_factor < 0) return fail(SP_EINVAL, "need n0, n1 >= 1 and pad_factor >= 0");
    const long long m0 = (2LL * pad_factor + 1) * n0, m1 = (2LL * pad_factor + 1) * n1;
    if ((m0 + FR_ROWS - 1) / FR_ROWS > 65535 || m1 > INT32_MAX) return fail(SP_EINVAL, "padded grid too large");
    cudaStream_t st = (cudaStream_t)stream;
    const d2* u0 = (const d2*)a_dev;
    d2* scratch = nullptr;
    if (mode == 1) {                    // stream-ordered scratch for U0, released after the padding pass has read it
        CU(cudaMallocAsync((void**)&scratch, (size_t)n0 * n1 * sizeof(d2), st));
        k_fresnel_u0<<<stream_grid((unsigned long long)n0 * n1), 256, 0, st>>>(a_dev, b_dev, (long long)n0 * n1, scratch);
        LAUNCH_CHECK();
        u0 = scratch;
    }
    const dim3 grid((unsigned)((m1 + 255) / 256), (unsigned)((m0 + FR_ROWS - 1) / FR_ROWS));
    k_fresnel_pad<<<grid, 256, 0, st>>>(u0, n0, n1, pad_factor, alpha, (d2*)u_pad_dev);
    LAUNCH_CHECK();
    if (scratch) CU(cudaFreeAsync(scratch, st));
    return SP_OK;
}

extern "C" int sp_fresnel_transfer(double* spec_dev, int m0, int m1, double d0, double d1, double wavelength, double z,
                                   double psf_sigma, void* stream) {
    if (!spec_dev) return fail(SP_EINVAL, "null argument");
    if (m0 < 1 || m1 < 1 || !(d0 > 0) || !(d1 > 0)) return fail(SP_EINVAL, "need m0, m1 >= 1 and positive sample spacings");
    if ((m0 + FR_ROWS - 1) / FR_ROWS > 65535) return fail(SP_EINVAL, "grid too large");
    const dim3 grid((unsigned)((m1 + 255) / 256), (unsigned)((m0 + FR_ROWS - 1) / FR_ROWS));
    k_fresnel_transfer<<<grid, 256, 0, (cudaStream_t)stream>>>((d2*)spec_dev, m0, m1, d0, d1, wavelength, z, psf_sigma);
    LAUNCH_CHECK();
    return SP_OK;
}

extern "C" int sp_fresnel_finish(const double* u_pad_dev, int n0, int n1, int pad_factor, double scale_re, double scale_im,
                                 double* out_dev, void* stream) {
    if (!u_pad_dev || !out_dev) return fail(SP_EINVAL, "null argument");
    if (n0 < 1 || n1 < 1 || pad_factor < 0) return fail(SP_EINVAL, "need n0, n1 >= 1 and pad_factor >= 0");
    k_fresnel_finish<<<stream_grid((unsigned long long)n0 * n1), 256, 0, (cudaStream_t)stream>>>((const d2*)u_pad_dev, n0, n1,
                                                                                                pad_factor, scale_re, scale_im,
                                                                                                (d2*)out_dev);
    LAUNCH_CHECK();
    return SP_OK;
}
