/*
 * synthpy_b200 -- C ABI of the B200-native ray-propagation hot path.
 *
 * The reference (MAGPIE-ICL/synthPy) is pure Python and has no FFI layer: its boundary for this path is
 * the Python call surface  ScalarDomain / Beam / propagator.solve / diagnostics.*  (SURVEY.md 8b).  This
 * header is what a binding for that surface calls; `synthpy_b200/_lib.py` is the ctypes binding and
 * INTEGRATION.md shows the stub a reference maintainer would add.  Each entry point cites the reference
 * interface it replaces (paths relative to the reference repo root).
 *
 * Conventions
 *   - every function returns 0 on success or a negative SP_E* code; sp_last_error() gives the text
 *     (thread-local).  Nothing throws across the boundary.
 *   - all `*_dev` pointers are CUDA device pointers owned by the caller (the Python host side owns them
 *     as torch tensors); `*_host` pointers are ordinary host memory.  The library keeps no device memory
 *     besides what hangs off an sp_field / sp_workspace handle.
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*; NULL = legacy default stream).  Calls
 *     do not synchronise, with these documented exceptions (all one-off or parity-mode paths, none on the
 *     fixed-step / per-ray adaptive hot path):
 *       sp_field_create / sp_field_create_from_gradients  wait for `stream` before returning (host-side axis and
 *                                 stencil tables, and for sp_field_create the float32 ne/nc scratch, are released);
 *       sp_propagate with SP_METHOD_RK45_JOINT  waits once per attempted step (its step-size controller is a
 *                                 host loop over device-side norms, as the reference's is a Python loop), and twice
 *                                 more when stats_dev / steps_dev are given;
 *       sp_workspace_propagate_ms waits for the last recorded launch (that is its purpose).
 *   - ray state layout is the reference's: 9 x N row-major float64
 *       [x, y, z, vx, vy, vz, amp, phase, pol]   (src/simulator/beam.py:63, src/solvers-legacy/full_solver.py:563)
 *     exit rays: 4 x N row-major float64 [x, theta, y, phi] (full_solver.py:849-881); Jones: 2 x N complex128.
 */
#ifndef SYNTHPY_B200_H
#define SYNTHPY_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SP_ABI_VERSION 4

/* error codes */
#define SP_OK 0
#define SP_EINVAL (-1)
#define SP_ECUDA (-2)
#define SP_ENOMEM (-3)
#define SP_ESTATE (-4)

/* ---------------------------------------------------------------------------------------------- field */

typedef struct sp_field sp_field; /* opaque: packed float4 {g_u, g_v, g_w, aux} grid + axis tables in HBM */

/* sp_field_create flags */
#define SP_FIELD_PHASE 1     /* aux lane = float32(n - 1), n = sqrt(1 - (5.64e4 sqrt(ne 1e-6)/omega)^2)           */
#define SP_FIELD_PHASE_F64 2 /* additionally keep n - 1 as a separate float64 grid (exact phase parity, +64 B/eval) */

/*
 * Builds the device field from an electron-density grid.  Replaces ScalarDomain.calc_dndr
 * (src/solvers-legacy/full_solver.py:211-234; recomputed per RHS call in src/simulator/propagator.py:66-91)
 * and the n_refrac grid of full_solver.py:270-274,344.  The arithmetic is the reference's, bit for bit:
 * ne_nc = float32(ne / nc); g_a = float32(-0.5 c^2) * np.gradient(ne_nc, axis_a) evaluated in float32 with
 * NumPy's second-order non-uniform-spacing stencil (uniform stencil when all float32 spacings are equal).
 *
 *   ne_dev      nx*ny*nz values, C order [x][y][z], float64 (ne_is_f64=1) or float32 (0)
 *   ax_*_host   the float32-rounded coordinate axes (full_solver.py:119, src/simulator/domain.py:230-232)
 *   omega       2 pi c / lambda
 *   march_axis  0|1|2: the probing axis; it becomes the fastest-varying axis of the packed layout
 */
int sp_field_create(sp_field** out, const void* ne_dev, int ne_is_f64, const float* ax_x_host,
                    const float* ax_y_host, const float* ax_z_host, int nx, int ny, int nz, double omega,
                    int march_axis, int flags, void* stream);

/*
 * Same, from gradients the caller already computed (e.g. with NumPy exactly as the reference does):
 * three float32 grids [x][y][z] on the device, optional aux grids (may be NULL).
 */
int sp_field_create_from_gradients(sp_field** out, const float* gx_dev, const float* gy_dev,
                                   const float* gz_dev, const float* aux_f32_dev, const double* aux_f64_dev,
                                   const float* ax_x_host, const float* ax_y_host, const float* ax_z_host,
                                   int nx, int ny, int nz, int march_axis, void* stream);

/*
 * Optional attenuation / Faraday channels (state rows 6 and 8): float64 grids [x][y][z] on the device, any may
 * be NULL.  kappa = inverse-bremsstrahlung rate (ScalarDomain.kappa, full_solver.py:243-268), ne and B for
 * pol' = V ne (B.v) (full_solver.py:356-374).  The grids are copied (re-ordered to the packed layout).
 * Used by sp_propagate when SP_FLAG_ATTEN / SP_FLAG_FARADAY are set (SP_METHOD_RK4, float64 only) and by sp_rhs.
 */
int sp_field_attach_channels(sp_field* f, const double* kappa_dev, const double* ne_dev, const double* bx_dev,
                             const double* by_dev, const double* bz_dev, void* stream);

int sp_field_destroy(sp_field* f);

/* Copies the three gradient grids back out in [x][y][z] order (tests: bit-equality with np.gradient). */
int sp_field_export_gradients(const sp_field* f, float* gx_dev, float* gy_dev, float* gz_dev,
                              float* aux_dev, void* stream);

/* Bytes of HBM held by the handle. */
uint64_t sp_field_bytes(const sp_field* f);

/* ------------------------------------------------------------------------------------------------ beam */

/* On-device ray generation (counter-based Philox4x32-10; ray i depends on (seed, i) only, so results do
 * not depend on how rays are partitioned over GPUs).  Replaces Beam.init_beam (src/simulator/beam.py:35-303)
 * / init_beam (src/solvers-legacy/full_solver.py:547-835) for bundles too large to draw on the host. */
#define SP_BEAM_CIRCULAR_FOLD 0 /* legacy radial law  u = fold(U+U)           full_solver.py:567-569 */
#define SP_BEAM_CIRCULAR_POW2 1 /* current radial law u = power(2)            beam.py:66-74          */
#define SP_BEAM_SQUARE 2        /*                                             full_solver.py:612-618 */
#define SP_BEAM_RECTANGULAR 3   /*                                             full_solver.py:658-667 */
#define SP_BEAM_LINEAR 4        /*                                             full_solver.py:707-720 */

typedef struct sp_beam {
    int32_t beam_type;
    int32_t probing_axis; /* 0|1|2 */
    double size_a;        /* beam_size (radius / half-width), m */
    double size_b;        /* second half-width (rectangular only) */
    double divergence;    /* rad */
    double start;         /* start coordinate along the probing axis = -ne_extent */
    uint64_t seed;
} sp_beam;

/* Materialise rays [ray_offset, ray_offset + n) as a 9 x n state (tests / small runs). */
int sp_beam_generate(const sp_beam* beam, uint64_t ray_offset, uint64_t n, double* s0_dev, void* stream);

/* -------------------------------------------------------------------------------------------- detector */

#define SP_OP_TRAVEL 0     /* p0 = d            rtm_solver.py:73-82   diagnostics.py:167-180 (advances E)   */
#define SP_OP_TRAVEL_NOE 1 /* p0 = d            travel that does not advance E (rtm_solver.py:308-314 quirk) */
#define SP_OP_LENS 2       /* p0 = f1, p1 = f2  rtm_solver.py:53-65   diagnostics.py:141-165                */
#define SP_OP_CIRC_AP 3    /* p0 = R            rtm_solver.py:84-90   diagnostics.py:182-199                */
#define SP_OP_CIRC_STOP 4  /* p0 = R            rtm_solver.py:92-98   diagnostics.py:201-209                */
#define SP_OP_RECT_AP 5    /* p0 = Lx, p1 = Ly  rtm_solver.py:110-118 (rejects only if outside BOTH)        */
#define SP_OP_KNIFE 6      /* p0 = offset, p1 = row (0|2), p2 = direction   rtm_solver.py:120-136           */
#define SP_OP_REF_BEAM 7   /* p0 = n_fringes, p1 = deg  diagnostics.py:559-581; must be first, uses metres  */

typedef struct sp_optic_op {
    int32_t kind;
    int32_t _pad;
    double p0, p1, p2;
} sp_optic_op;

#define SP_IMG_HISTOGRAM 0    /* np.histogram2d semantics (rtm_solver.py:156-174, diagnostics.py:323-353):
                                 nb+1 linspace edges, right-most edge inclusive, counts uint64               */
#define SP_IMG_INTERFEROGRAM 1 /* np.digitize-1 on nb linspace edges -> nb-1 bins, sums of complex E
                                 (rtm_solver.py:424-453, diagnostics.py:358-379); planes int64 fixed point  */
#define SP_PLANE_FRAC_BITS 40  /* interferogram planes hold round(value * 2^40): integer sums are exact and
                                 order-independent (run-to-run and GPU-count invariant images), quantisation
                                 9e-13 per contribution, range +-8.4e6 per pixel (|E| per ray is <= ~2)       */
#define SP_IMG_STOKES 2        /* polarimetry: histogram bins (np.histogram2d semantics, as SP_IMG_HISTOGRAM) of the
                                 ray count and of Stokes I, Q, U of the Jones vector E at the detector, summed
                                 incoherently over the rays of a pixel:  I = |Ex|^2 + |Ey|^2,  Q = |Ex|^2 - |Ey|^2,
                                 U = 2 Re(Ex conj(Ey)).  For the reference's E = amp e^{i phase} (-sin pol, cos pol)
                                 (full_solver.py:883-890): I = amp^2, Q = -amp^2 cos 2pol, U = -amp^2 sin 2pol.
                                 Stokes V = 2 Im(Ex conj(Ey)) is identically 0 for that Jones form: not stored.
                                 planes_dev [4][ny][nx] int64: count, then I, Q, U in fixed point
                                 (SP_STOKES_FRAC_BITS).  Channels must not contain SP_OP_REF_BEAM.            */
#define SP_STOKES_FRAC_BITS 32 /* Stokes planes hold round(value * 2^32): quantisation 2.3e-10 per contribution,
                                 range +-2^31 per pixel (2^31 unit contributions: every ray of a 1e9 bundle in
                                 one pixel); a contribution beyond +-2^20 saturates                           */

typedef struct sp_image {
    int32_t kind;
    int32_t nx, ny;           /* number of BINS along detector x / y */
    int32_t _pad;
    double x_lo, x_hi;        /* edges = np.linspace(lo, hi, nx+1) in both modes (digitize: nx = n_edges - 1)  */
    double y_lo, y_hi;
    uint64_t* counts_dev;     /* [ny][nx], histogram only (caller zeroes; calls accumulate)                  */
    int64_t* planes_dev;      /* [4][ny][nx], caller zeroes; calls accumulate.  Interferogram: Re Ex, Im Ex, Re Ey,
                                 Im Ey (SP_PLANE_FRAC_BITS); Stokes: count, I, Q, U (SP_STOKES_FRAC_BITS)         */
} sp_image;

/* One detector channel: an optical train ending in an image.  Several channels can share one bundle of
 * rays (e.g. shadowgraphy + schlieren of the same propagation). */
typedef struct sp_channel {
    const sp_optic_op* ops_host;
    int32_t n_ops;
    int32_t input_mm;         /* sp_optics_image only: 1 = rf_dev positions are already in mm (skip m_to_mm)  */
    double wavelength;        /* for E-field phase advance k = 2 pi / wavelength (diagnostics.py:315-321)    */
    sp_image image;
} sp_channel;

/* Optics + binning on exit rays that already exist in HBM: Diagnostic.*_solve() + histogram()/interferogram()
 * (diagnostics.py:388-640, rtm_solver.py:191-453).  rf_dev is 4 x n in METRES as returned by the solver
 * (m_to_mm is applied inside, diagnostics.py:313).  jf_dev (2 x n complex128 interleaved) may be NULL, except for an
 * interferogram or Stokes image.
 * rf_out_dev / jf_out_dev (may be NULL) receive the rays at the detector plane (NaN = rejected). */
int sp_optics_image(const double* rf_dev, const double* jf_dev, uint64_t n, const sp_channel* chan,
                    double* rf_out_dev, double* jf_out_dev, void* stream);

/* SP_IMG_INTERFEROGRAM: H_dev [ny][nx] = sqrt(Re(sum Ex)^2 + Re(sum Ey)^2)  (rtm_solver.py:450-453).
 * SP_IMG_STOKES:        H_dev [4][ny][nx] float64 = N, I, Q, U (the fixed-point format stays inside the library). */
int sp_image_finalize(const sp_image* img, double* H_dev, void* stream);

/* ------------------------------------------------------------------------------------------- propagate */

#define SP_METHOD_RK4 0        /* fixed step, classical RK4                                                  */
#define SP_METHOD_RK45 1       /* Dormand-Prince 5(4), SciPy's controller, step size chosen PER RAY           */
#define SP_METHOD_RK45_JOINT 2 /* the reference as shipped: ONE step size for the whole bundle from the RMS
                                  error norm over all 9N components (full_solver.py:391)                     */
#define SP_METHOD_TSIT5 6      /* the current generation's solver: Tsitouras 5(4) per ray under diffrax's PID
                                  controller in normalised time (src/simulator/propagator.py:533-599).  params: h =
                                  dt0 in units of t_end, t_end = the normalisation T, rtol / atol, n_steps =
                                  max_steps.  PARITY UNPINNED (jax / diffrax absent here): published method +
                                  documented controller defaults.  (3-5 are internal variants.)              */

#define SP_FLAG_PHASE 1      /* integrate d(phase)/dt = omega (n - 1)   (full_solver.py:342-345)             */
#define SP_FLAG_EARLY_EXIT 2 /* stop a ray once it is outside the grid and moving away (RHS == 0 for good)   */
#define SP_FLAG_FP32 4       /* float32 state and arithmetic (the JAX generation's default, config.py:127)   */
#define SP_FLAG_PHASE_F64 8  /* interpolate n-1 from the float64 aux grid                                    */
#define SP_FLAG_NO_SORT 16   /* do not reorder rays into coherent bundles                                    */
#define SP_FLAG_ATTEN 32     /* integrate amp' = kappa(r) amp            (full_solver.py:540)                */
#define SP_FLAG_FARADAY 64   /* integrate pol' = verdet ne(r) (B(r).v)   (full_solver.py:542)                */
#define SP_FLAG_BUNDLE_STEP 128 /* SP_METHOD_RK45: one step size per 32-ray bundle (the shipped joint solver applied to
                                   32-ray chunks; lanes stay in lock-step).  Results depend on bundle membership.  */

typedef struct sp_params {
    int32_t method;
    int32_t flags;
    int32_t n_steps;       /* RK4: steps to take; RK45*: cap on attempted steps per ray (0 = 1<<30)          */
    int32_t n_state;       /* components in the RMS error norm: 9 (full_solver) or 6 (minimal_solver)       */
    double h;              /* RK4 step, seconds                                                              */
    double t_end;          /* RK45: integrate t in [0, t_end];  reference: sqrt(8) extent / c               */
    double rtol, atol;     /* RK45 (SciPy defaults 1e-3 / 1e-6)                                              */
    double omega;          /* 2 pi c / lambda                                                                */
    double extent;         /* exit-plane coordinate along the probing axis (ray_to_Jonesvector)             */
    int32_t probing_axis;  /* 0|1|2                                                                          */
    int32_t out_axis_a;    /* which spatial axis lands in rf rows 0,1 ...                                    */
    int32_t out_axis_b;    /* ... and rows 2,3  (legacy 'y': a=x,b=z; current API 'y': a=z,b=x)              */
    int32_t _pad;
    double verdet;         /* Verdet constant 2.62e-13 lambda^2 (full_solver.py:223); SP_FLAG_FARADAY only  */
} sp_params;

typedef struct sp_stats {
    uint64_t ray_steps;      /* attempted integrator steps summed over rays (the rays.steps metric)          */
    uint64_t ray_steps_acc;  /* accepted steps (== ray_steps for RK4)                                        */
    uint64_t rays_capped;    /* rays that hit the n_steps cap before t_end (RK45)                            */
    uint64_t rays_binned;    /* rays that landed inside an image, summed over channels                       */
    uint64_t rays_rejected;  /* rays removed by an aperture/stop, summed over channels                       */
    uint64_t rhs_evals;      /* right-hand-side evaluations (RK4: 4 per step; RK45: those that touched the field) */
} sp_stats;

/* Opaque scratch reused across calls: bundle dispenser, sort keys / order / histogram, joint-mode stage buffers, the
 * pinned pair the joint controller reads, and the timing events.  ONE STREAM PER WORKSPACE: everything sp_propagate
 * enqueues through a workspace assumes the launches before it on that workspace have been ordered by the same
 * stream (the dispenser is reset with a memset, scratch may be re-allocated).  Callers that propagate on several
 * streams or threads of one device create one workspace per stream (synthpy_b200/engine.py keys them by
 * (device, stream)). */
typedef struct sp_workspace sp_workspace;
int sp_workspace_create(sp_workspace** out);
int sp_workspace_destroy(sp_workspace* ws);

/*
 * The hot path.  Replaces propagator.solve (src/simulator/propagator.py:351-702) /
 * ScalarDomain.solve (src/solvers-legacy/full_solver.py:376-403) + ray_to_Jonesvector
 * (full_solver.py:838-894), and -- when channels are given -- fuses Diagnostic.*_solve + histogram /
 * interferogram into the kernel epilogue so exit rays never touch HBM.
 *
 *   rays:   s0_dev (9 x n float64) if non-NULL, else generated on device from `beam` for global ray indices
 *           [ray_offset, ray_offset + n)
 *   sf_dev  (9 x n)  final ODE state, or NULL
 *   rf_dev  (4 x n)  exit rays [x, theta, y, phi] in m / rad, or NULL
 *   jf_dev  (2 x n complex128) Jones vectors, or NULL
 *   steps_dev (n uint32) attempted steps per ray, or NULL
 *   channels_host / n_channels: fused detector channels (may be 0)
 *   stats_dev: device sp_stats accumulated into (caller zeroes), or NULL
 */
int sp_propagate(const sp_field* field, const sp_params* params, sp_workspace* ws, const double* s0_dev,
                 const sp_beam* beam, uint64_t n, uint64_t ray_offset, double* sf_dev, double* rf_dev,
                 double* jf_dev, uint32_t* steps_dev, const sp_channel* channels_host, int n_channels,
                 sp_stats* stats_dev, void* stream);

/* Device time of the k_propagate launches issued through `ws` since the last call (CUDA events recorded
 * around each launch on its stream; this call waits for the last one).  bench.py's roofline figure. */
int sp_workspace_propagate_ms(sp_workspace* ws, double* total_ms, int* n_launches);

/* (h, error_norm) of every attempted step of the last SP_METHOD_RK45_JOINT solve issued through `ws`
 * (the counterpart of instrumenting scipy's RK45._estimate_error_norm).  Copies min(cap, n) entries. */
int sp_workspace_joint_log(const sp_workspace* ws, double* h_out, double* en_out, int cap, int* n_out);

/*
 * Exit-plane projection of ODE states that already exist in HBM: ray_to_Jonesvector
 * (src/solvers-legacy/full_solver.py:838-894; src/simulator/propagator.py:178-298 with keep_current_plane) and
 * back_propogate (propagator.py:300-349).  sf_dev is 9 x n; any output may be NULL.
 *   rf_dev  4 x n  [x, theta, y, phi]           jf_dev  2 x n complex128 Jones vectors
 *   sback_dev 9 x n: the state moved along its straight line onto the plane coord[probing_axis] = extent
 */
int sp_exit_plane(const double* sf_dev, uint64_t n, int probing_axis, int out_axis_a, int out_axis_b, double extent,
                  int keep_current_plane, double* rf_dev, double* jf_dev, double* sback_dev, void* stream);

/* Right-hand side only: d(state)/dt for arbitrary states (parity level L0; full_solver.py:516-544). */
int sp_rhs(const sp_field* field, const sp_params* params, const double* s_dev, uint64_t n, double* dsdt_dev,
           void* stream);

/* ------------------------------------------------------------------------------------- wave-optics step */
/* The step that follows the ray path in the reference's coherent refractometer (SURVEY.md 8f-2):
 * src/simulator/fresnel_integral.py, called from Refractometry.fresnel_solve (src/simulator/diagnostics.py:529-552).
 * The 2-D FFT between sp_fresnel_transfer's two neighbours is the caller's (cuFFT via torch.fft), as np.fft.fft2 is
 * the reference's. */

/*
 * Piecewise-linear interpolation of scattered samples on a triangulation, evaluated on the nodes of a rectilinear
 * grid: scipy.interpolate.LinearNDInterpolator((px, py), v, fill_value)(np.meshgrid(gx, gy)) of
 * fresnel_integral.py:71-77.  The triangulation is the caller's (the host side builds it with scipy.spatial.Delaunay,
 * i.e. the same Qhull call LinearNDInterpolator makes).
 *   px_dev, py_dev  n_pts sample positions           val_dev  [n_val][n_pts] sample values (interpolated in one pass)
 *   tri_dev         [n_tri][3] vertex indices        gx_dev (nx), gy_dev (ny) ascending grid coordinates
 *   owner_dev       ny*nx int32 scratch              out_dev  [n_val][ny][nx]; fill_value outside the hull
 */
int sp_scatter_to_grid(const double* px_dev, const double* py_dev, const double* val_dev, int n_val, uint64_t n_pts,
                       const int32_t* tri_dev, uint64_t n_tri, const double* gx_dev, const double* gy_dev, int nx, int ny,
                       double fill_value, int32_t* owner_dev, double* out_dev, void* stream);

/*
 * prepare_field_for_propagation (fresnel_integral.py:7-24) fused with the construction of U0 (:79-84):
 * np.pad(U0, pad_factor * shape, mode='reflect') times the outer product of two Tukey(alpha) windows.
 *   mode 0: a_dev = U0 as interleaved complex128 [n0][n1], b_dev unused
 *   mode 1: a_dev = amplitude grid, b_dev = phase grid, U0 = a exp(-i b)
 *   u_pad_dev: complex128 [(2 pad_factor + 1) n0][(2 pad_factor + 1) n1]
 */
int sp_fresnel_prepare(const double* a_dev, const double* b_dev, int mode, int n0, int n1, int pad_factor, double alpha,
                       double* u_pad_dev, void* stream);

/* In place: spectrum[k0][k1] *= exp(-i pi lambda z (f0^2 + f1^2)) [* exp(-2 (pi sigma)^2 (f0^2 + f1^2)) if
 * psf_sigma > 0], f = np.fft.fftfreq(m, d)  (fresnel_integral.py:36-49). */
int sp_fresnel_transfer(double* spec_dev, int m0, int m1, double d0, double d1, double wavelength, double z,
                        double psf_sigma, void* stream);

/* Crop the centre [n0][n1] window of the padded field and multiply by the complex constant
 * exp(i k z) / (i lambda z) given as (scale_re, scale_im)  (fresnel_integral.py:51-59). */
int sp_fresnel_finish(const double* u_pad_dev, int n0, int n1, int pad_factor, double scale_re, double scale_im,
                      double* out_dev, void* stream);

/* Measurement aid for bench.py's roofline (no reference counterpart: the reference has no device code).  Enqueues
 * one launch in which every resident thread of every SM runs 8 independent DFMA chains of `iters` links and writes
 * one double to out_dev[thread] (thread < out_len); *n_dfma_out = DFMA thread-instructions of the launch.  The caller
 * times it with CUDA events on `stream`: 2 * n_dfma / seconds is the FP64 FMA peak the integrator is held against. */
int sp_fp64_peak(int iters, double* out_dev, uint64_t out_len, uint64_t* n_dfma_out, void* stream);

/* Number of kernels this library has launched in the calling process (bench.py's gpu_launches). */
uint64_t sp_launch_count(void);

int sp_version(void);
const char* sp_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* SYNTHPY_B200_H */
