// Per-ray math of the synthpy_b200 hot path: trilinear field lookup, RHS, RK4 / Dormand-Prince steps,
// exit-plane projection, ray-transfer-matrix optics and detector bin search.
//
// Everything here is `SP_HD` (host + device) and free of CUDA runtime calls so that the very same source
// is (a) inlined into the sm_100a kernels in synthpy_b200.cu and (b) compiled by g++ into the CPU-side
// self-test harness (tests/host_harness.cpp) -- the build container has no GPU, so (b) is how the
// arithmetic is exercised before a gpurun call.  (b) is a test build, not a product path.
//
// Reference semantics restated here (paths relative to the reference repo root):
//   locate()/trilinear : scipy RegularGridInterpolator linear, bounds_error=False, fill 0
//                        (src/solvers-legacy/full_solver.py:232-234,317-332; JAX copy src/simulator/utils.py:124-214)
//   rhs()              : dsdt, full_solver.py:516-544 (propagator.py:94-175)
//   dp5_*              : scipy.integrate RK45 as driven by solve_ivp at full_solver.py:391
//   exit_project()     : ray_to_Jonesvector, full_solver.py:838-894 (propagator.py:178-298)
//   optic ops / bins   : src/solvers-legacy/rtm_solver.py:48-178,424-453 (src/simulator/diagnostics.py:122-379)
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define SP_HD __host__ __device__ __forceinline__
#else
#define SP_HD inline
#endif

// -DSP_BOUNDS_CHECK: device-side asserts on every index that feeds a global load (compute-sanitizer is not
// available on the GPU pool; the test-suite is run once against a library built this way).
#if defined(SP_BOUNDS_CHECK) && defined(__CUDA_ARCH__)
#include <assert.h>
#define SP_ASSERT(c) assert(c)
#else
#define SP_ASSERT(c) ((void)0)
#endif

namespace sp {

struct alignas(16) f4 { float x, y, z, w; };
struct alignas(16) d2 { double x, y; };
struct alignas(8) f2 { float x, y; };

template <typename T> struct Pair;
template <> struct Pair<double> { typedef d2 type; };
template <> struct Pair<float> { typedef f2 type; };

// ---- small portability layer -------------------------------------------------------------------------
SP_HD double sp_fma(double a, double b, double c) {
#if defined(__CUDA_ARCH__)
    return __fma_rn(a, b, c);
#else
    return a * b + c;
#endif
}
SP_HD float sp_fma(float a, float b, float c) {
#if defined(__CUDA_ARCH__)
    return __fmaf_rn(a, b, c);
#else
    return a * b + c;
#endif
}
// exactly-rounded, never-contracted multiply/add: used where the reference's value feeds an index decision
SP_HD double mul_rn(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    volatile double r = a * b; return r;
#endif
}
SP_HD double add_rn(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    volatile double r = a + b; return r;
#endif
}
SP_HD int floor_to_int(double x) {
#if defined(__CUDA_ARCH__)
    return __double2int_rd(x);
#else
    if (!(x == x)) return 0;
    if (x >= 2147483000.0) return 2147483000;
    if (x <= -2147483000.0) return -2147483000;
    return (int)floor(x);
#endif
}
SP_HD int floor_to_int(float x) {
#if defined(__CUDA_ARCH__)
    return __float2int_rd(x);
#else
    return floor_to_int((double)x);
#endif
}
SP_HD double ldg(const double* p) {
#if defined(__CUDA_ARCH__)
    return __ldg(p);
#else
    return *p;
#endif
}
// Load that the compiler may not sink into a later branch (asm volatile): used to put two independent
// requests in flight before the first comparison that would otherwise serialise them.
SP_HD double ldg_now(const double* p) {
#if defined(__CUDA_ARCH__)
    double v; asm volatile("ld.global.nc.f64 %0, [%1];" : "=d"(v) : "l"(p)); return v;
#else
    return *p;
#endif
}
SP_HD float ldg_now(const float* p) {
#if defined(__CUDA_ARCH__)
    float v; asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(v) : "l"(p)); return v;
#else
    return *p;
#endif
}
SP_HD f4 ldg(const f4* p) {
#if defined(__CUDA_ARCH__)
    const float4 v = __ldg(reinterpret_cast<const float4*>(p));
    f4 r; r.x = v.x; r.y = v.y; r.z = v.z; r.w = v.w; return r;
#else
    return *p;
#endif
}
SP_HD d2 ldg(const d2* p) {
#if defined(__CUDA_ARCH__)
    const double2 v = __ldg(reinterpret_cast<const double2*>(p));
    d2 r; r.x = v.x; r.y = v.y; return r;
#else
    return *p;
#endif
}
SP_HD f2 ldg(const f2* p) {
#if defined(__CUDA_ARCH__)
    const float2 v = __ldg(reinterpret_cast<const float2*>(p));
    f2 r; r.x = v.x; r.y = v.y; return r;
#else
    return *p;
#endif
}

// 0 <= w < 1 decided on the bit pattern (one integer compare on the ALU pipe instead of two FP64 compares on the
// FP64 pipe, whose latency the dependent branch would expose).  -0.0, negatives, w >= 1, inf and NaN all fail.
SP_HD bool unit_interval(double w) {
#if defined(__CUDA_ARCH__)
    return (unsigned)__double2hiint(w) < 0x3FF00000u;
#else
    uint64_t b; memcpy(&b, &w, 8); return (uint32_t)(b >> 32) < 0x3FF00000u;
#endif
}
SP_HD bool unit_interval(float w) {
#if defined(__CUDA_ARCH__)
    return (unsigned)__float_as_int(w) < 0x3F800000u;
#else
    uint32_t b; memcpy(&b, &w, 4); return b < 0x3F800000u;
#endif
}

// float32 -> T.  For T = double the default is the hardware conversion (F2F on the quarter-rate XU pipe);
// -DSP_INT_CVT re-biases the exponent with integer ops on the ALU pipe instead (exact for normal numbers;
// zero / denormal / inf / nan take the hardware path).
template <typename T> SP_HD T cvt(float f);
template <> SP_HD float cvt<float>(float f) { return f; }
template <> SP_HD double cvt<double>(float f) {
#if defined(__CUDA_ARCH__) && defined(SP_INT_CVT)
    const unsigned b = __float_as_uint(f);
    const unsigned m = b & 0x7fffffffu;
    if (m - 0x00800000u < 0x7f000000u)
        return __hiloint2double((int)((b & 0x80000000u) | ((m >> 3) + 0x38000000u)), (int)(b << 29));
    return (double)f;
#else
    return (double)f;
#endif
}

// all three weights in [0, 1): one 3-input unsigned max + one compare
SP_HD bool unit_interval3(double a, double b, double c) {
#if defined(__CUDA_ARCH__)
    const unsigned x = (unsigned)__double2hiint(a), y = (unsigned)__double2hiint(b), z = (unsigned)__double2hiint(c);
    return max(max(x, y), z) < 0x3FF00000u;
#else
    return unit_interval(a) && unit_interval(b) && unit_interval(c);
#endif
}
SP_HD bool unit_interval3(float a, float b, float c) {
#if defined(__CUDA_ARCH__)
    const unsigned x = (unsigned)__float_as_int(a), y = (unsigned)__float_as_int(b), z = (unsigned)__float_as_int(c);
    return max(max(x, y), z) < 0x3F800000u;
#else
    return unit_interval(a) && unit_interval(b) && unit_interval(c);
#endif
}

// ---- field view --------------------------------------------------------------------------------------
// Kernel frame: axes (u, v, w) = (m+1, m+2, m) mod 3 of the caller's (x, y, z), m = march (probing) axis;
// w is the fastest-varying axis of the packed grid, so the two corners a ray needs along its direction of
// travel are one 32-byte read and a 128-byte line holds 8 consecutive cells of one (u, v) column.
template <typename T> struct AxisTab {
    const typename Pair<T>::type* tab;  // [n] {g[i], 1/(g[i+1]-g[i])}; entry n-1 = {g[n-1], 0}
    T g0, inv_d;                        // uniform first guess  i ~ floor((x - g0) * inv_d)
    T lo, hi;                           // g[0], g[n-1]: the reference's out-of-bounds test
    int n;
};

template <typename T> struct FieldView {
    const f4* data;       // [nu][nv][nw] {g_u, g_v, g_w, aux}
    const double* aux64;  // [nu][nv][nw] n-1 in float64, or nullptr
    AxisTab<T> ax[3];
    long long su;         // element stride of u  (= nv*nw)
    int sv;               // element stride of v  (= nw)
#ifdef SP_BRICK
    long long bsu;        // A/B layout (-DSP_BRICK): `data` in 8 x 8 x 8 bricks of float4 (8 KB, w fastest inside a brick);
    long long bsv;        // element strides between bricks along u and v (bricks along w are 512 elements apart)
#endif
};

// Element offsets of grid index i along u / v / w inside `data`: the offset of node (iu, iv, iw) is their sum in both
// layouts, so the eight corners of a cell are the sums of two offsets per axis.
#ifdef SP_BRICK
template <typename T> SP_HD long long off_u(const FieldView<T>& F, int i) { return (long long)(i >> 3) * F.bsu + ((i & 7) << 6); }
template <typename T> SP_HD long long off_v(const FieldView<T>& F, int i) { return (long long)(i >> 3) * F.bsv + ((i & 7) << 3); }
template <typename T> SP_HD long long off_w(const FieldView<T>&, int i) { return ((long long)(i >> 3) << 9) + (i & 7); }
#else
template <typename T> SP_HD long long off_u(const FieldView<T>& F, int i) { return (long long)i * F.su; }
template <typename T> SP_HD long long off_v(const FieldView<T>& F, int i) { return (long long)i * F.sv; }
template <typename T> SP_HD long long off_w(const FieldView<T>&, int i) { return i; }
#endif

// Cell index i with g[i] <= x < g[i+1] (clipped to [0, n-2]; x == g[n-1] -> n-2); false when x is outside
// [g[0], g[n-1]] (the fill value applies).  NaN is "in bounds" (cell 0, NaN weight later), as in scipy
// (_rgi.py: find_indices + _find_out_of_bounds).  The decision is made against the real (float32-rounded)
// coordinate table, not an ideal uniform grid: uniform first guess, then an exact walk if needed.
template <typename T> SP_HD bool locate(const AxisTab<T>& A, T x, int& i) {
    if (x < A.lo || x > A.hi) return false;
    int k = floor_to_int((x - A.g0) * A.inv_d);
    k = k < 0 ? 0 : (k > A.n - 2 ? A.n - 2 : k);
    SP_ASSERT(A.n >= 2);
    if (x == x) {
        while (k > 0 && x < ldg(A.tab + k).x) --k;
        while (k < A.n - 2 && x >= ldg(A.tab + k + 1).x) ++k;
    }
    i = k;
    return true;
}

// Uniform first guess of the cell index (clipped to [0, n-2]); right on float32-rounded linspace axes except within
// rounding of a node, and always checked against the table entries it points at.
template <typename T> SP_HD int guess_cell(const AxisTab<T>& A, T x) {
    const int k = floor_to_int((x - A.g0) * A.inv_d);
    return k < 0 ? 0 : (k > A.n - 2 ? A.n - 2 : k);
}
// locate()'s acceptance of cell k given its table entry: g[k] <= x < g[k+1], with x == hi belonging to the last cell.
// Points outside [lo, hi] and NaNs fail here (k is clipped to [0, n-2], so g[0] = lo and g[n-1] = hi bound the test) and
// are sorted out by the exact search.
template <typename T> SP_HD bool cell_holds(const AxisTab<T>& A, T x, int k, T g_k, T g_k1) {
    (void)k;
    return x >= g_k && (x < g_k1 || x == A.hi);
}

// Per-ray register cache of the cell the ray is in.  A ray takes ~8 RHS evaluations per cell (two RK4 steps
// of four stages), so the 8 corner reads, the float32->float64 conversions and the axis-table lookups are
// done once per cell instead of once per evaluation; ncu on the uncached kernel showed the L1 data pipe
// (l1tex__data_pipe_lsu_wavefronts) at 88 % of peak and DRAM at 0.2 %, i.e. the gathers, not HBM, were the
// bound.  The cell is held as the trilinear polynomial
//     f = a0 + ww a1 + wv (a2 + ww a3) + wu (a4 + ww a5 + wv (a6 + ww a7))
// (7 fused multiply-adds per component), whose coefficients are corner differences.
template <typename T, bool PHASE> struct CellCache {
    T lo[3], rinv[3];                   // g[i] and 1/(g[i+1]-g[i]) of the cached cell, per axis
    T a[PHASE ? 4 : 3][8];
    float af[PHASE ? 8 : 1];            // n - 1 polynomial in float32 when the aux lane itself is float32 (see rhs())
    int idx[3];
    // "no cell cached" is encoded as rinv[2] = NaN: the w-weight is then NaN and fails the unit-interval test,
    // so the hot path needs no separate flag
    SP_HD bool valid() const { return rinv[2] == rinv[2]; }
    SP_HD void invalidate() { rinv[2] = (T)NAN; }
    SP_HD CellCache() {
        for (int k = 0; k < 3; ++k) { lo[k] = rinv[k] = (T)0; idx[k] = 0; }
        invalidate();
        for (int c = 0; c < (PHASE ? 4 : 3); ++c)
            for (int k = 0; k < 8; ++k) a[c][k] = (T)0;
        for (int k = 0; k < (PHASE ? 8 : 1); ++k) af[k] = 0.f;
    }
};

// locate() plus the cell's (g[i], 1/(g[i+1]-g[i])): the table entry of the uniform first guess and the next node are
// requested together and, when the guess is right (the rule on float32-rounded linspace axes), nothing else is read.
template <typename T> SP_HD bool locate_cell(const AxisTab<T>& A, T x, int& i, T& lo, T& rinv) {
    if (x < A.lo || x > A.hi) return false;
    int k = floor_to_int((x - A.g0) * A.inv_d);
    k = k < 0 ? 0 : (k > A.n - 2 ? A.n - 2 : k);
    SP_ASSERT(A.n >= 2);
    typename Pair<T>::type e = ldg(A.tab + k);
    const T up = ldg_now(&(A.tab + k + 1)->x);
    if (x == x && ((k > 0 && x < e.x) || (k < A.n - 2 && x >= up))) {       // exact walk, as locate()
        while (k > 0 && x < ldg(A.tab + k).x) --k;
        while (k < A.n - 2 && x >= ldg(A.tab + k + 1).x) ++k;
        e = ldg(A.tab + k);
    }
    i = k; lo = e.x; rinv = e.y;
    return true;
}

// Move the cached interval of one axis to the cell containing x.  `w_ok` = the weight test already placed x
// in the cached cell.  NEAR (fixed-step marching: a miss is almost always the neighbouring cell): two table reads
// and exact comparisons, anything else falls back to the exact search.  !NEAR (adaptive steps jump several cells
// and the lanes of a warp disagree on how far): straight to the search, one code path for every lane.
// False = x is outside the grid.
template <bool NEAR, typename T> SP_HD bool relocate_axis(const AxisTab<T>& A, T x, bool w_ok, bool valid, int& i, T& lo, T& rinv) {
    if (valid) {
        if (w_ok) return true;
        if (NEAR) {
            if (x >= lo) {
                if (i + 2 < A.n) {
                    const typename Pair<T>::type e1 = ldg(A.tab + i + 1);
                    const T e2x = ldg_now(&(A.tab + i + 2)->x);          // requested together with e1: one round trip
                    if (x < e1.x) return true;                       // weight rounded up to 1: still this cell
                    if (x < e2x) { ++i; lo = e1.x; rinv = e1.y; return true; }
                }
            } else if (x < lo && i > 0) {
                const typename Pair<T>::type e0 = ldg(A.tab + i - 1);
                if (x >= e0.x) { --i; lo = e0.x; rinv = e0.y; return true; }
            }
        }
    }
    return locate_cell(A, x, i, lo, rinv);
}

template <typename T> SP_HD void tri_coef(T c000, T c001, T c010, T c011, T c100, T c101, T c110, T c111, T* a) {
    a[0] = c000;
    a[1] = c001 - c000;
    a[2] = c010 - c000;
    a[3] = (c011 - c010) - (c001 - c000);
    a[4] = c100 - c000;
    a[5] = (c101 - c100) - (c001 - c000);
    a[6] = (c110 - c100) - (c010 - c000);
    a[7] = ((c111 - c110) - (c101 - c100)) - ((c011 - c010) - (c001 - c000));
}

template <typename T> SP_HD T tri_eval(const T* a, T wu, T wv, T ww) {
    const T t0 = sp_fma(ww, a[1], a[0]);
    const T t1 = sp_fma(ww, a[3], a[2]);
    const T t2 = sp_fma(ww, a[5], a[4]);
    const T t3 = sp_fma(ww, a[7], a[6]);
    return sp_fma(wu, sp_fma(wv, t3, t2), sp_fma(wv, t1, t0));
}

// Acceleration a = interp(grad) and, optionally, n-1 at (pu, pv, pw).  Returns false (and zeros) when the
// point is outside the grid: no memory is touched then.  Trilinear weights are the reference's normalised
// distances (x - g[i]) / (g[i+1] - g[i]) (reciprocal multiply: <= 1 ulp from the division).
// Fast path: the point is still in the cached cell iff all three weights are in [0, 1) -- decided from the
// weights (needed anyway) with integer compares.  (A point within one ulp above a cell face can thus still be
// evaluated with the previous cell's polynomial; the trilinear interpolant is continuous across faces, so
// the value is the same to rounding.  Every decision taken on a miss is exact against the axis tables.)
template <typename T, bool PHASE, bool AUX64, bool NEAR = true>
SP_HD bool rhs(const FieldView<T>& F, CellCache<T, PHASE>& cc, T pu, T pv, T pw, T& au, T& av, T& aw, T& nm1) {
    T wu = (pu - cc.lo[0]) * cc.rinv[0], wv = (pv - cc.lo[1]) * cc.rinv[1], ww = (pw - cc.lo[2]) * cc.rinv[2];
    if (!unit_interval3(wu, wv, ww)) {
        au = av = aw = nm1 = (T)0;
        const bool oku = unit_interval(wu), okv = unit_interval(wv), okw = unit_interval(ww);
        const bool v = cc.valid();
        if (!relocate_axis<NEAR>(F.ax[0], pu, oku, v, cc.idx[0], cc.lo[0], cc.rinv[0])) { cc.invalidate(); return false; }
        if (!relocate_axis<NEAR>(F.ax[1], pv, okv, v, cc.idx[1], cc.lo[1], cc.rinv[1])) { cc.invalidate(); return false; }
        if (!relocate_axis<NEAR>(F.ax[2], pw, okw, v, cc.idx[2], cc.lo[2], cc.rinv[2])) { cc.invalidate(); return false; }
        SP_ASSERT(cc.idx[0] >= 0 && cc.idx[0] <= F.ax[0].n - 2 && cc.idx[1] >= 0 && cc.idx[1] <= F.ax[1].n - 2 &&
                  cc.idx[2] >= 0 && cc.idx[2] <= F.ax[2].n - 2);
        const long long base = (long long)cc.idx[0] * F.su + (long long)cc.idx[1] * F.sv + cc.idx[2];
#ifdef SP_BRICK
        const long long u0 = off_u(F, cc.idx[0]), u1 = off_u(F, cc.idx[0] + 1), v0 = off_v(F, cc.idx[1]), v1 = off_v(F, cc.idx[1] + 1);
        const long long w0 = off_w(F, cc.idx[2]), w1 = off_w(F, cc.idx[2] + 1);
        const f4* p = F.data;
        const f4 c000 = ldg(p + u0 + v0 + w0), c001 = ldg(p + u0 + v0 + w1);
        const f4 c010 = ldg(p + u0 + v1 + w0), c011 = ldg(p + u0 + v1 + w1);
        const f4 c100 = ldg(p + u1 + v0 + w0), c101 = ldg(p + u1 + v0 + w1);
        const f4 c110 = ldg(p + u1 + v1 + w0), c111 = ldg(p + u1 + v1 + w1);
#else
        const f4* p = F.data + base;
        const f4 c000 = ldg(p), c001 = ldg(p + 1);
        const f4 c010 = ldg(p + F.sv), c011 = ldg(p + F.sv + 1);
        const f4 c100 = ldg(p + F.su), c101 = ldg(p + F.su + 1);
        const f4 c110 = ldg(p + F.su + F.sv), c111 = ldg(p + F.su + F.sv + 1);
#endif
        tri_coef<T>(cvt<T>(c000.x), cvt<T>(c001.x), cvt<T>(c010.x), cvt<T>(c011.x), cvt<T>(c100.x), cvt<T>(c101.x), cvt<T>(c110.x), cvt<T>(c111.x), cc.a[0]);
        tri_coef<T>(cvt<T>(c000.y), cvt<T>(c001.y), cvt<T>(c010.y), cvt<T>(c011.y), cvt<T>(c100.y), cvt<T>(c101.y), cvt<T>(c110.y), cvt<T>(c111.y), cc.a[1]);
        tri_coef<T>(cvt<T>(c000.z), cvt<T>(c001.z), cvt<T>(c010.z), cvt<T>(c011.z), cvt<T>(c100.z), cvt<T>(c101.z), cvt<T>(c110.z), cvt<T>(c111.z), cc.a[2]);
        if (PHASE) {
            if (AUX64) {
                const double* q = F.aux64 + base;
                tri_coef<T>((T)ldg(q), (T)ldg(q + 1), (T)ldg(q + F.sv), (T)ldg(q + F.sv + 1), (T)ldg(q + F.su),
                            (T)ldg(q + F.su + 1), (T)ldg(q + F.su + F.sv), (T)ldg(q + F.su + F.sv + 1), cc.a[PHASE ? 3 : 0]);
            } else if (sizeof(T) == 8) {
                // float32 aux lane: n - 1 is stored as float32 (6e-8 relative), so its polynomial is kept and evaluated in
                // float32 as well: 8 registers instead of 16, no conversions on reload, and the 7 FMAs per evaluation
                // leave the FP64 pipe (the bound of this kernel).  SP_FLAG_PHASE_F64 keeps everything in float64.
                tri_coef<float>(c000.w, c001.w, c010.w, c011.w, c100.w, c101.w, c110.w, c111.w, cc.af);
            } else {
                tri_coef<T>(cvt<T>(c000.w), cvt<T>(c001.w), cvt<T>(c010.w), cvt<T>(c011.w), cvt<T>(c100.w), cvt<T>(c101.w), cvt<T>(c110.w), cvt<T>(c111.w),
                            cc.a[PHASE ? 3 : 0]);
            }
        }
        wu = (pu - cc.lo[0]) * cc.rinv[0]; wv = (pv - cc.lo[1]) * cc.rinv[1]; ww = (pw - cc.lo[2]) * cc.rinv[2];
    }
    au = tri_eval<T>(cc.a[0], wu, wv, ww);
    av = tri_eval<T>(cc.a[1], wu, wv, ww);
    aw = tri_eval<T>(cc.a[2], wu, wv, ww);
    if (PHASE && !AUX64 && sizeof(T) == 8) nm1 = (T)tri_eval<float>(cc.af, (float)wu, (float)wv, (float)ww);
    else nm1 = PHASE ? tri_eval<T>(cc.a[PHASE ? 3 : 0], wu, wv, ww) : (T)0;
    return true;
}

// The same interpolation WITHOUT a cell cache, for the adaptive integrators: a Dormand-Prince step at SciPy's default
// tolerances spans ~1.7 cells of the benchmarked grids, so consecutive evaluations land in different cells, the cache
// misses on nearly every call and its upkeep (hit test, neighbour probe, face bookkeeping, ~50 live registers) is pure
// overhead -- round 1's adaptive kernel spent ~3600 warp-instructions per attempted step at 18 of 32 lanes, with 900
// bytes of spills.  Here every evaluation runs the identical straight-line sequence (bounds test, exact cell search on
// the axis tables, eight 16-byte corner reads, the reference's sum over corners of value x weight product), so the
// lanes of a warp stay converged whatever cells they are in.
template <typename T, bool PHASE, bool AUX64>
SP_HD bool rhs_direct(const FieldView<T>& F, T pu, T pv, T pw, T& au, T& av, T& aw, T& nm1) {
    au = av = aw = nm1 = (T)0;
    // The three table entries AND the eight corners of the guessed cell are requested together -- one memory round trip
    // per evaluation instead of two dependent ones (table -> index -> corners); the guess is then verified exactly and,
    // in the rare cases it is a node off, the point is outside the grid (fill value 0) or NaN, the exact search decides
    // and its cell goes through the same (single) copy of the loads once more.  No separate bounds test on the fast path.
    int iu = guess_cell(F.ax[0], pu), iv = guess_cell(F.ax[1], pv), iw = guess_cell(F.ax[2], pw);
    typename Pair<T>::type eu, ev, ew;
    f4 c000, c001, c010, c011, c100, c101, c110, c111;
    long long base = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int pass = 0;; ++pass) {
        SP_ASSERT(iu >= 0 && iu <= F.ax[0].n - 2 && iv >= 0 && iv <= F.ax[1].n - 2 && iw >= 0 && iw <= F.ax[2].n - 2);
        eu = ldg(F.ax[0].tab + iu); ev = ldg(F.ax[1].tab + iv); ew = ldg(F.ax[2].tab + iw);
        const T gu1 = ldg_now(&(F.ax[0].tab + iu + 1)->x), gv1 = ldg_now(&(F.ax[1].tab + iv + 1)->x), gw1 = ldg_now(&(F.ax[2].tab + iw + 1)->x);
        base = (long long)iu * F.su + (long long)iv * F.sv + iw;
#ifdef SP_BRICK
        const long long u0 = off_u(F, iu), u1 = off_u(F, iu + 1), v0 = off_v(F, iv), v1 = off_v(F, iv + 1), w0 = off_w(F, iw), w1 = off_w(F, iw + 1);
        const f4* p = F.data;
        c000 = ldg(p + u0 + v0 + w0); c001 = ldg(p + u0 + v0 + w1); c010 = ldg(p + u0 + v1 + w0); c011 = ldg(p + u0 + v1 + w1);
        c100 = ldg(p + u1 + v0 + w0); c101 = ldg(p + u1 + v0 + w1); c110 = ldg(p + u1 + v1 + w0); c111 = ldg(p + u1 + v1 + w1);
#else
        const f4* p = F.data + base;
        c000 = ldg(p); c001 = ldg(p + 1); c010 = ldg(p + F.sv); c011 = ldg(p + F.sv + 1);
        c100 = ldg(p + F.su); c101 = ldg(p + F.su + 1); c110 = ldg(p + F.su + F.sv); c111 = ldg(p + F.su + F.sv + 1);
#endif
        if (pass || (cell_holds(F.ax[0], pu, iu, eu.x, gu1) && cell_holds(F.ax[1], pv, iv, ev.x, gv1) && cell_holds(F.ax[2], pw, iw, ew.x, gw1)))
            break;
        T l, r;                                              // exact search; its answer is final
        if (!locate_cell(F.ax[0], pu, iu, l, r) || !locate_cell(F.ax[1], pv, iv, l, r) || !locate_cell(F.ax[2], pw, iw, l, r)) return false;
    }
    const T lu = eu.x, ru = eu.y, lv = ev.x, rv = ev.y, lw = ew.x, rw = ew.y;
    const T wu = (pu - lu) * ru, wv = (pv - lv) * rv, ww = (pw - lw) * rw;
    const T mu = (T)1 - wu, mv = (T)1 - wv, mw = (T)1 - ww;
    const T k00 = mu * mv, k01 = mu * wv, k10 = wu * mv, k11 = wu * wv;
    const T k000 = k00 * mw, k001 = k00 * ww, k010 = k01 * mw, k011 = k01 * ww;
    const T k100 = k10 * mw, k101 = k10 * ww, k110 = k11 * mw, k111 = k11 * ww;
#define SP_TRI(m) sp_fma(cvt<T>(c111.m), k111, sp_fma(cvt<T>(c110.m), k110, sp_fma(cvt<T>(c101.m), k101, sp_fma(cvt<T>(c100.m), k100, \
                  sp_fma(cvt<T>(c011.m), k011, sp_fma(cvt<T>(c010.m), k010, sp_fma(cvt<T>(c001.m), k001, cvt<T>(c000.m) * k000)))))))
    au = SP_TRI(x); av = SP_TRI(y); aw = SP_TRI(z);
    if (PHASE) {
        if (AUX64) {
            const double* q = F.aux64 + base;
            nm1 = sp_fma((T)ldg(q + F.su + F.sv + 1), k111, sp_fma((T)ldg(q + F.su + F.sv), k110, sp_fma((T)ldg(q + F.su + 1), k101,
                  sp_fma((T)ldg(q + F.su), k100, sp_fma((T)ldg(q + F.sv + 1), k011, sp_fma((T)ldg(q + F.sv), k010,
                  sp_fma((T)ldg(q + 1), k001, (T)ldg(q) * k000)))))));
        } else {
            nm1 = SP_TRI(w);
        }
    }
#undef SP_TRI
    return true;
}

// ---- ray state ---------------------------------------------------------------------------------------
template <typename T> struct Ray {
    T p[3];   // position, kernel frame
    T v[3];   // velocity
    T ph;     // accumulated phase (state row 7)
};

// True when the ray is outside the grid on some axis and not moving back towards it: its RHS is zero for
// ever, so integration can stop (exit_project puts it on the same straight line).
template <typename T> SP_HD bool escaped(const FieldView<T>& F, const Ray<T>& r) {
    bool e = false;
#pragma unroll
    for (int k = 0; k < 3; ++k)
        e = e || (r.p[k] > F.ax[k].hi && r.v[k] >= (T)0) || (r.p[k] < F.ax[k].lo && r.v[k] <= (T)0);
    return e;
}

// Classical RK4 step of  p' = v, v' = a(p), ph' = omega (n(p) - 1).  Because p' = v is linear, the four
// velocity stages can be eliminated algebraically (Nystrom form of the same method):
//     p2 = p + h/2 v            p3 = p2 + h^2/4 a1          p4 = (p + h v) + h^2/2 a2
//     p' = (p + h v) + h^2/6 (a1 + a2 + a3)                 v' = v + h/6 (((a1 + 2 a2) + 2 a3) + a4)
// This is classical RK4 exactly (same stage points, same weights); only the floating-point association of
// the position update differs from y + h/6 (k1 + 2 k2 + 2 k3 + k4), at the 1e-16 level per step.
// Returns the number of RHS evaluations (4), or -1 (state untouched) when `early` is set and the ray has
// escaped: that test is only evaluated when the first stage is out of bounds, which is necessary for "escaped"
// and costs nothing on the in-grid path.
// Step-size constants of the Nystrom form.  The kernel takes them as launch parameters (constant bank operands of the
// FP64 instructions) instead of recomputing them every step: the compiler rematerialised them inside the step loop
// (6 DMUL + 3 LDC per step) rather than hold ten more registers.
template <typename T> struct RK4Step {
    T h, hh, h6, hh2, h2_2, h2_6;
    SP_HD RK4Step() : h(0), hh(0), h6(0), hh2(0), h2_2(0), h2_6(0) {}
    SP_HD explicit RK4Step(T h_) : h(h_), hh((T)0.5 * h_), h6(h_ / (T)6) { hh2 = hh * hh; h2_2 = h * hh; h2_6 = h * h6; }
};

template <typename T, bool PHASE, bool AUX64>
SP_HD int rk4_step(const FieldView<T>& F, CellCache<T, PHASE>& cc, const RK4Step<T>& K, T omega, Ray<T>& r, bool early = false) {
    const T h = K.h, hh = K.hh, h6 = K.h6, hh2 = K.hh2, h2_2 = K.h2_2, h2_6 = K.h2_6;
    T a[3], n, sa[3], sv[3], q[3], ph_[3], sn = (T)0;
    const bool in1 = rhs<T, PHASE, AUX64>(F, cc, r.p[0], r.p[1], r.p[2], a[0], a[1], a[2], n);
    if (early && !in1 && escaped(F, r)) return -1;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        sa[k] = a[k]; sv[k] = a[k];
        q[k] = sp_fma(hh, r.v[k], r.p[k]);            // p2
        ph_[k] = sp_fma(h, r.v[k], r.p[k]);           // p + h v
    }
    if (PHASE) sn = n;
    rhs<T, PHASE, AUX64>(F, cc, q[0], q[1], q[2], a[0], a[1], a[2], n);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        q[k] = sp_fma(hh2, sa[k], q[k]);              // p3 = p2 + h^2/4 a1
        sa[k] = sa[k] + a[k]; sv[k] = sp_fma((T)2, a[k], sv[k]);
    }
    if (PHASE) sn = sp_fma((T)2, n, sn);
    const T a2u = a[0], a2v = a[1], a2w = a[2];
    rhs<T, PHASE, AUX64>(F, cc, q[0], q[1], q[2], a[0], a[1], a[2], n);
    q[0] = sp_fma(h2_2, a2u, ph_[0]); q[1] = sp_fma(h2_2, a2v, ph_[1]); q[2] = sp_fma(h2_2, a2w, ph_[2]);   // p4
#pragma unroll
    for (int k = 0; k < 3; ++k) { sa[k] = sa[k] + a[k]; sv[k] = sp_fma((T)2, a[k], sv[k]); }
    if (PHASE) sn = sp_fma((T)2, n, sn);
    rhs<T, PHASE, AUX64>(F, cc, q[0], q[1], q[2], a[0], a[1], a[2], n);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        r.p[k] = sp_fma(h2_6, sa[k], ph_[k]);
        r.v[k] = sp_fma(h6, sv[k] + a[k], r.v[k]);
    }
    if (PHASE) r.ph = sp_fma(h6, omega * (sn + n), r.ph);
    return 4;
}

template <typename T, bool PHASE, bool AUX64>
SP_HD int rk4_step(const FieldView<T>& F, CellCache<T, PHASE>& cc, T h, T omega, Ray<T>& r, bool early = false) {
    return rk4_step<T, PHASE, AUX64>(F, cc, RK4Step<T>(h), omega, r, early);
}

// ---- attenuation and Faraday-rotation channels (slow path, float64, RK4 only) ---------------------------------
// Reference: dsdt rows 6 and 8 (src/solvers-legacy/full_solver.py:540-542):
//     amp' = kappa(r) amp          kappa_interp, fill 0     (full_solver.py:243-268,286,335-339)
//     pol' = V ne(r) (B(r) . v)    ne_interp / B*_interp, fill 0, V = 2.62e-13 lambda^2  (full_solver.py:223,356-374)
// The five grids stay float64 (the reference does not round them to float32) and are interpolated directly from
// HBM with the weights of the cached cell; these channels are rare and not on the throughput path.
struct ExtView {
    const double* ch[5];   // kappa, ne, B_u, B_v, B_w in the kernel frame ([nu][nv][nw]); nullptr = channel off
    double verdet;
};

template <bool PHASE>
SP_HD void ext_eval(const FieldView<double>& F, const ExtView& X, const CellCache<double, PHASE>& cc, bool inside,
                    const double* p, double out[5]) {
#pragma unroll
    for (int c = 0; c < 5; ++c) out[c] = 0.0;
    if (!inside) return;
    const double wu = (p[0] - cc.lo[0]) * cc.rinv[0], wv = (p[1] - cc.lo[1]) * cc.rinv[1], ww = (p[2] - cc.lo[2]) * cc.rinv[2];
    const double mu = 1.0 - wu, mv = 1.0 - wv, mw = 1.0 - ww;
    const double k[8] = {mu * mv * mw, mu * mv * ww, mu * wv * mw, mu * wv * ww, wu * mv * mw, wu * mv * ww, wu * wv * mw, wu * wv * ww};
    SP_ASSERT(cc.valid() && cc.idx[0] >= 0 && cc.idx[0] <= F.ax[0].n - 2 && cc.idx[1] >= 0 && cc.idx[1] <= F.ax[1].n - 2 &&
              cc.idx[2] >= 0 && cc.idx[2] <= F.ax[2].n - 2);
    const long long base = (long long)cc.idx[0] * F.su + (long long)cc.idx[1] * F.sv + cc.idx[2];
    const long long off[8] = {0, 1, F.sv, F.sv + 1, F.su, F.su + 1, F.su + F.sv, F.su + F.sv + 1};
#pragma unroll
    for (int c = 0; c < 5; ++c) {
        if (!X.ch[c]) continue;
        const double* q = X.ch[c] + base;
        double acc = ldg(q) * k[0];
#pragma unroll
        for (int j = 1; j < 8; ++j) acc = sp_fma(ldg(q + off[j]), k[j], acc);
        out[c] = acc;
    }
}

struct ExtState { double amp, pol; };

// Classical RK4 on the full 9-component state (explicit stage velocities: pol' depends on them).
template <bool PHASE, bool AUX64>
SP_HD int rk4_step_ext(const FieldView<double>& F, const ExtView& X, CellCache<double, PHASE>& cc, double h, double omega,
                       bool with_phase, Ray<double>& r, ExtState& e, bool early = false) {
    const double hh = 0.5 * h, h6 = h / 6.0;
    double p[3], v[3], a[3], n, x[5];
    double sp[3] = {0, 0, 0}, sv[3] = {0, 0, 0}, sn = 0, sA = 0, sR = 0;
    double A = e.amp, kA = 0;
    int touched = 0;
    const double wgt[4] = {1.0, 2.0, 2.0, 1.0}, adv[4] = {0.0, hh, hh, h};
    double kv_prev[3] = {0, 0, 0}, kp_prev[3] = {0, 0, 0};
#pragma unroll
    for (int s = 0; s < 4; ++s) {
#pragma unroll
        for (int k = 0; k < 3; ++k) { p[k] = sp_fma(adv[s], kp_prev[k], r.p[k]); v[k] = sp_fma(adv[s], kv_prev[k], r.v[k]); }
        A = sp_fma(adv[s], kA, e.amp);
        const bool in = rhs<double, PHASE, AUX64>(F, cc, p[0], p[1], p[2], a[0], a[1], a[2], n);
        if (s == 0 && early && !in && escaped(F, r)) return -1;
        touched += in;
        ext_eval<PHASE>(F, X, cc, in, p, x);
        kA = x[0] * A;                                                        // kappa(r) * amp
        const double kR = X.verdet * x[1] * (x[2] * v[0] + x[3] * v[1] + x[4] * v[2]);   // V ne (B . v)
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            sp[k] = (s == 0) ? v[k] : sp_fma(wgt[s], v[k], sp[k]);
            sv[k] = (s == 0) ? a[k] : sp_fma(wgt[s], a[k], sv[k]);
            kp_prev[k] = v[k]; kv_prev[k] = a[k];
        }
        sn = (s == 0) ? n : sp_fma(wgt[s], n, sn);
        sA = (s == 0) ? kA : sp_fma(wgt[s], kA, sA);
        sR = (s == 0) ? kR : sp_fma(wgt[s], kR, sR);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) { r.p[k] = sp_fma(h6, sp[k], r.p[k]); r.v[k] = sp_fma(h6, sv[k], r.v[k]); }
    if (PHASE && with_phase) r.ph = sp_fma(h6, omega * sn, r.ph);
    e.amp = sp_fma(h6, sA, e.amp);
    e.pol = sp_fma(h6, sR, e.pol);
    return touched;
}

// ---- Dormand-Prince 5(4) with SciPy's controller -------------------------------------------------------
// Tableau of scipy/integrate/_ivp/rk.py::RK45 (Dormand & Prince 1980).
struct DP {
    static constexpr double c2 = 1.0 / 5, c3 = 3.0 / 10, c4 = 4.0 / 5, c5 = 8.0 / 9;
    static constexpr double a21 = 1.0 / 5;
    static constexpr double a31 = 3.0 / 40, a32 = 9.0 / 40;
    static constexpr double a41 = 44.0 / 45, a42 = -56.0 / 15, a43 = 32.0 / 9;
    static constexpr double a51 = 19372.0 / 6561, a52 = -25360.0 / 2187, a53 = 64448.0 / 6561, a54 = -212.0 / 729;
    static constexpr double a61 = 9017.0 / 3168, a62 = -355.0 / 33, a63 = 46732.0 / 5247, a64 = 49.0 / 176,
                            a65 = -5103.0 / 18656;
    static constexpr double b1 = 35.0 / 384, b3 = 500.0 / 1113, b4 = 125.0 / 192, b5 = -2187.0 / 6784, b6 = 11.0 / 84;
    static constexpr double e1 = -71.0 / 57600, e3 = 71.0 / 16695, e4 = -71.0 / 1920, e5 = 17253.0 / 339200,
                            e6 = -22.0 / 525, e7 = 1.0 / 40;
    static constexpr double SAFETY = 0.9, MIN_FACTOR = 0.2, MAX_FACTOR = 10.0;
};

// Derivative of the 7 live components (p, v, ph) at a state; amp and pol have zero derivative.
template <typename T> struct Deriv { T dp[3]; T dv[3]; T dph; };

template <typename T, bool PHASE, bool AUX64>
SP_HD int deriv(const FieldView<T>& F, CellCache<T, PHASE>& cc, T omega, const T* p, const T* v, Deriv<T>& k) {
    T nm1;
    int t = rhs<T, PHASE, AUX64>(F, cc, p[0], p[1], p[2], k.dv[0], k.dv[1], k.dv[2], nm1);
    k.dp[0] = v[0]; k.dp[1] = v[1]; k.dp[2] = v[2];
    k.dph = PHASE ? omega * nm1 : (T)0;
    return t;
}

template <typename T, bool PHASE, bool AUX64>
SP_HD int deriv_direct(const FieldView<T>& F, T omega, const T* p, const T* v, Deriv<T>& k) {
    T nm1;
    int t = rhs_direct<T, PHASE, AUX64>(F, p[0], p[1], p[2], k.dv[0], k.dv[1], k.dv[2], nm1);
    k.dp[0] = v[0]; k.dp[1] = v[1]; k.dp[2] = v[2];
    k.dph = PHASE ? omega * nm1 : (T)0;
    return t;
}

// One attempted DP5 step of size h from (r, k1 = f(r)).  Outputs the 5th-order state, f(new state) (FSAL)
// and sum over the live components of (err_i / scale_i)^2 with scale = atol + rtol max(|y|, |y_new|)
// (rk.py:_step_impl).  amp (|y| = amp0) and pol contribute zero error.
//
// Because p' = v is linear, the position rows of the stage matrix K are the stage velocities
// v_s = v + h sum_j a_sj Kv_j; substituting them (Nystrom form of the same tableau) leaves only the velocity rows
// Kv and the phase row to keep:   p_s = p + c_s h v + h^2 sum_j Abar_sj Kv_j,  Abar_sj = sum_i a_si a_ij,
//                                 p'  = p + h v + h^2 sum_j Bbar_j Kv_j,       err_p = h^2 sum_j Ebar_j Kv_j
// (sum_s E_s = 0, so the h v term drops out of the error).  Same method, same stage points; 21 fewer live
// doubles per ray than carrying the position rows.
struct DPN {
    static constexpr double A31 = DP::a32 * DP::a21;
    static constexpr double A41 = DP::a42 * DP::a21 + DP::a43 * DP::a31, A42 = DP::a43 * DP::a32;
    static constexpr double A51 = DP::a52 * DP::a21 + DP::a53 * DP::a31 + DP::a54 * DP::a41,
                            A52 = DP::a53 * DP::a32 + DP::a54 * DP::a42, A53 = DP::a54 * DP::a43;
    static constexpr double A61 = DP::a62 * DP::a21 + DP::a63 * DP::a31 + DP::a64 * DP::a41 + DP::a65 * DP::a51,
                            A62 = DP::a63 * DP::a32 + DP::a64 * DP::a42 + DP::a65 * DP::a52,
                            A63 = DP::a64 * DP::a43 + DP::a65 * DP::a53, A64 = DP::a65 * DP::a54;
    static constexpr double B1 = DP::b3 * DP::a31 + DP::b4 * DP::a41 + DP::b5 * DP::a51 + DP::b6 * DP::a61,
                            B2 = DP::b3 * DP::a32 + DP::b4 * DP::a42 + DP::b5 * DP::a52 + DP::b6 * DP::a62,
                            B3 = DP::b4 * DP::a43 + DP::b5 * DP::a53 + DP::b6 * DP::a63,
                            B4 = DP::b5 * DP::a54 + DP::b6 * DP::a64, B5 = DP::b6 * DP::a65;
    static constexpr double E1 = DP::e3 * DP::a31 + DP::e4 * DP::a41 + DP::e5 * DP::a51 + DP::e6 * DP::a61 + DP::e7 * DP::b1,
                            E2 = DP::e3 * DP::a32 + DP::e4 * DP::a42 + DP::e5 * DP::a52 + DP::e6 * DP::a62,
                            E3 = DP::e4 * DP::a43 + DP::e5 * DP::a53 + DP::e6 * DP::a63 + DP::e7 * DP::b3,
                            E4 = DP::e5 * DP::a54 + DP::e6 * DP::a64 + DP::e7 * DP::b4,
                            E5 = DP::e6 * DP::a65 + DP::e7 * DP::b5, E6 = DP::e7 * DP::b6;
};

// Where the stage derivatives K2..K6 (velocity rows) and the stage values n3..n6 wait between the six evaluations of an
// attempt.  StageRegs: local arrays that the compiler keeps in registers (every index is a compile-time constant) -- the
// joint kernels and the CPU self-test.  StageSmem: a per-thread column of shared memory; the per-ray / per-bundle
// adaptive kernels are latency-bound at 3 resident CTAs per SM (168 registers, ncu: issue active 38 %), and these 19
// doubles are the largest block of state that is only touched between evaluations.
template <typename T> struct StageRegs {
    T k[5][3], n[4];
    SP_HD T K(int j, int c) const { return k[j][c]; }
    SP_HD void setK(int j, int c, T v) { k[j][c] = v; }
    SP_HD T N(int j) const { return n[j]; }
    SP_HD void setN(int j, T v) { n[j] = v; }
};
template <typename T> struct StageSmem {
    T* base; int stride;                                   // element (j, c) at base[(3 j + c) * stride]: conflict-free across a warp
    SP_HD T K(int j, int c) const { return base[(3 * j + c) * stride]; }
    SP_HD void setK(int j, int c, T v) { base[(3 * j + c) * stride] = v; }
    SP_HD T N(int j) const { return base[(15 + j) * stride]; }
    SP_HD void setN(int j, T v) { base[(15 + j) * stride] = v; }
};
#define SP_STAGE_DOUBLES 19

// ---- windowed integration (out-of-core tracing) ------------------------------------------------------------------
// [lo, hi] along kernel axis w (the probing axis) is where the resident slab's field equals the whole grid's; so does every
// point outside the whole grid (w outside [g_lo, g_hi], the grid's w range, or u / v outside the axes the slab shares with
// the grid), where both give the fill value 0.  An attempt with a point anywhere else is abandoned before that point is
// evaluated (WIN instantiations only): *out is set to the point's w and the caller discards the attempt.  NaN is never
// outside, so a NaN ray fails as it does in core.
struct Window { double lo, hi, g_lo, g_hi; };
template <typename T> SP_HD bool outside(const Window& W, const FieldView<T>& F, const T* p) {
    const double w = (double)p[2];
    if (!(w < W.lo || w > W.hi)) return false;
    if (w < W.g_lo || w > W.g_hi) return false;
    return !(p[0] < F.ax[0].lo || p[0] > F.ax[0].hi || p[1] < F.ax[1].lo || p[1] > F.ax[1].hi);
}

// STAGED (stage parking): the attempt starts at stage `s_first` (2 .. 7) with the stage values of the stages before it
// already in S, and a park reports its stage in *s_park; the stage points are the same instructions on both paths.
template <typename T, bool PHASE, bool AUX64, typename Store, bool WIN = false, bool STAGED = false>
SP_HD int dp5_attempt(const FieldView<T>& F, T omega, T h, T rtol, T atol, const Ray<T>& r, const Deriv<T>& k1,
                      Ray<T>& rn, Deriv<T>& k7, T& err_sq, Store& S, const Window* W = nullptr, double* out = nullptr,
                      int s_first = 2, int* s_park = nullptr) {
    T n7 = (T)0;
    const T* K1 = k1.dv;
    const T h2 = h * h;
    int touched = 0;
    // The six evaluations go through ONE copy of rhs_direct() (a rolled loop with the stage-specific algebra in switch
    // arms): with the evaluation inlined six times the step loop was ~80 KB of SASS against a 32 KB instruction cache,
    // and ncu showed `no_instruction` as the top stall (5 per issue).  Every index below is a compile-time constant,
    // so the stage vectors stay in registers; the arithmetic is unchanged.
#define SP_POS(cs, expr) (r.p[c] + (T)(cs) * h * r.v[c] + h2 * (expr))
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int s = STAGED ? s_first : 2; s <= 7; ++s) {
        T p[3] = {0, 0, 0};
        switch (s) {
        case 2:
#pragma unroll
            for (int c = 0; c < 3; ++c) p[c] = r.p[c] + (T)DP::c2 * h * r.v[c];
            break;
        case 3:
#pragma unroll
            for (int c = 0; c < 3; ++c) p[c] = SP_POS(DP::c3, (T)DPN::A31 * K1[c]);
            break;
        case 4:
#pragma unroll
            for (int c = 0; c < 3; ++c) p[c] = SP_POS(DP::c4, (T)DPN::A41 * K1[c] + (T)DPN::A42 * S.K(0, c));
            break;
        case 5:
#pragma unroll
            for (int c = 0; c < 3; ++c) p[c] = SP_POS(DP::c5, (T)DPN::A51 * K1[c] + (T)DPN::A52 * S.K(0, c) + (T)DPN::A53 * S.K(1, c));
            break;
        case 6:
#pragma unroll
            for (int c = 0; c < 3; ++c)
                p[c] = SP_POS(1.0, (T)DPN::A61 * K1[c] + (T)DPN::A62 * S.K(0, c) + (T)DPN::A63 * S.K(1, c) + (T)DPN::A64 * S.K(2, c));
            break;
        default:   // 7: y_new = y + h * (K[:-1].T @ B), then f(y_new) (FSAL)
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                rn.p[c] = r.p[c] + h * r.v[c] + h2 * ((T)DPN::B1 * K1[c] + (T)DPN::B2 * S.K(0, c) + (T)DPN::B3 * S.K(1, c) + (T)DPN::B4 * S.K(2, c) +
                                                      (T)DPN::B5 * S.K(3, c));
                rn.v[c] = r.v[c] + h * ((T)DP::b1 * K1[c] + (T)DP::b3 * S.K(1, c) + (T)DP::b4 * S.K(2, c) + (T)DP::b5 * S.K(3, c) + (T)DP::b6 * S.K(4, c));
                p[c] = rn.p[c];
            }
            rn.ph = r.ph;
            if (PHASE)
                rn.ph = r.ph + h * ((T)DP::b1 * k1.dph + omega * ((T)DP::b3 * S.N(0) + (T)DP::b4 * S.N(1) + (T)DP::b5 * S.N(2) + (T)DP::b6 * S.N(3)));
            break;
        }
        if (WIN && outside(*W, F, p)) {
            *out = (double)p[2];
            if constexpr (STAGED) *s_park = s;
            return touched;
        }
        T a0, a1, a2, nn;
        touched += rhs_direct<T, PHASE, AUX64>(F, p[0], p[1], p[2], a0, a1, a2, nn);
        switch (s) {
        case 2: S.setK(0, 0, a0); S.setK(0, 1, a1); S.setK(0, 2, a2); break;
        case 3: S.setK(1, 0, a0); S.setK(1, 1, a1); S.setK(1, 2, a2); if (PHASE) S.setN(0, nn); break;
        case 4: S.setK(2, 0, a0); S.setK(2, 1, a1); S.setK(2, 2, a2); if (PHASE) S.setN(1, nn); break;
        case 5: S.setK(3, 0, a0); S.setK(3, 1, a1); S.setK(3, 2, a2); if (PHASE) S.setN(2, nn); break;
        case 6: S.setK(4, 0, a0); S.setK(4, 1, a1); S.setK(4, 2, a2); if (PHASE) S.setN(3, nn); break;
        default: k7.dv[0] = a0; k7.dv[1] = a1; k7.dv[2] = a2; n7 = nn; break;
        }
    }
#undef SP_POS
#pragma unroll
    for (int c = 0; c < 3; ++c) k7.dp[c] = rn.v[c];
    k7.dph = PHASE ? omega * n7 : (T)0;
    // error estimate  (K.T @ E) * h / scale
    T acc = (T)0;
#define SP_SCALE(y0, y1) (atol + (fabs(y0) > fabs(y1) ? fabs(y0) : fabs(y1)) * rtol)
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const T ep = h2 * ((T)DPN::E1 * K1[c] + (T)DPN::E2 * S.K(0, c) + (T)DPN::E3 * S.K(1, c) + (T)DPN::E4 * S.K(2, c) + (T)DPN::E5 * S.K(3, c) +
                           (T)DPN::E6 * S.K(4, c));
        const T ev = h * ((T)DP::e1 * K1[c] + (T)DP::e3 * S.K(1, c) + (T)DP::e4 * S.K(2, c) + (T)DP::e5 * S.K(3, c) + (T)DP::e6 * S.K(4, c) +
                          (T)DP::e7 * k7.dv[c]);
        const T qp = ep / SP_SCALE(r.p[c], rn.p[c]), qv = ev / SP_SCALE(r.v[c], rn.v[c]);
        acc += qp * qp + qv * qv;
    }
    if (PHASE) {
        const T e = h * ((T)DP::e1 * k1.dph + omega * ((T)DP::e3 * S.N(0) + (T)DP::e4 * S.N(1) + (T)DP::e5 * S.N(2) + (T)DP::e6 * S.N(3) + (T)DP::e7 * n7));
        const T q = e / SP_SCALE(r.ph, rn.ph);
        acc += q * q;
    }
#undef SP_SCALE
    err_sq = acc;
    return touched;
}

// the register-resident form (joint kernels, CPU self-test)
template <typename T, bool PHASE, bool AUX64>
SP_HD int dp5_attempt(const FieldView<T>& F, T omega, T h, T rtol, T atol, const Ray<T>& r, const Deriv<T>& k1,
                      Ray<T>& rn, Deriv<T>& k7, T& err_sq) {
    StageRegs<T> S;
#pragma unroll
    for (int j = 0; j < 5; ++j)
#pragma unroll
        for (int c = 0; c < 3; ++c) S.k[j][c] = (T)0;
#pragma unroll
    for (int j = 0; j < 4; ++j) S.n[j] = (T)0;
    return dp5_attempt<T, PHASE, AUX64, StageRegs<T> >(F, omega, h, rtol, atol, r, k1, rn, k7, err_sq, S);
}

// Step-size factor after an attempt with RMS error norm `en` (rk.py:_step_impl).  One pow() for both outcomes: the
// accepting and the rejecting lanes of a warp would otherwise each run their own copy of it (ncu: pow() executed 1.9x
// per attempt at 13 of 32 lanes, 12 % of the adaptive kernel's instructions).
template <typename T> SP_HD T dp5_factor(T en, bool accepted, bool rejected_before) {
    const T g = (en == (T)0) ? (T)DP::MAX_FACTOR : (T)DP::SAFETY * pow(en, (T)-0.2);
    if (accepted) {
        T f = fmin((T)DP::MAX_FACTOR, g);
        if (rejected_before) f = fmin((T)1, f);
        return f;
    }
    return fmax((T)DP::MIN_FACTOR, g);
}

// Hairer's initial step as coded in scipy/integrate/_ivp/common.py::select_initial_step (order = 4), with
// the RMS norms taken over the ray's own n_state components (amp contributes (amp/scale)^2 to d0 only).
template <typename T, bool PHASE, bool AUX64, bool WIN = false>
SP_HD T dp5_initial_step(const FieldView<T>& F, T omega, T t_end, T rtol, T atol, int n_state, T amp, T pol,
                         const Ray<T>& r, const Deriv<T>& f0, int& touched, const Window* W = nullptr, double* out = nullptr) {
    if (t_end == (T)0) return (T)0;
    const T inv_n = (T)1 / (T)n_state;
    T s0 = (T)0, s1 = (T)0;
    T sc_p[3], sc_v[3], sc_ph;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        sc_p[c] = atol + fabs(r.p[c]) * rtol;
        sc_v[c] = atol + fabs(r.v[c]) * rtol;
        T q = r.p[c] / sc_p[c]; s0 += q * q;
        q = r.v[c] / sc_v[c]; s0 += q * q;
        q = f0.dp[c] / sc_p[c]; s1 += q * q;
        q = f0.dv[c] / sc_v[c]; s1 += q * q;
    }
    sc_ph = atol + fabs(r.ph) * rtol;
    { T q = r.ph / sc_ph; s0 += q * q; q = f0.dph / sc_ph; s1 += q * q; }
    if (n_state > 6) {
        T q = amp / (atol + fabs(amp) * rtol); s0 += q * q;
        q = pol / (atol + fabs(pol) * rtol); s0 += q * q;
    }
    const T d0 = sqrt(s0 * inv_n), d1 = sqrt(s1 * inv_n);
    T h0 = (d0 < (T)1e-5 || d1 < (T)1e-5) ? (T)1e-6 : (T)0.01 * d0 / d1;
    h0 = fmin(h0, t_end);
    T p1[3], v1[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) { p1[c] = r.p[c] + h0 * f0.dp[c]; v1[c] = r.v[c] + h0 * f0.dv[c]; }
    if (WIN && outside(*W, F, p1)) { *out = (double)p1[2]; return (T)0; }
    Deriv<T> f1;
    touched += deriv_direct<T, PHASE, AUX64>(F, omega, p1, v1, f1);
    T s2 = (T)0;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        T q = (f1.dp[c] - f0.dp[c]) / sc_p[c]; s2 += q * q;
        q = (f1.dv[c] - f0.dv[c]) / sc_v[c]; s2 += q * q;
    }
    { T q = (f1.dph - f0.dph) / sc_ph; s2 += q * q; }
    const T d2 = sqrt(s2 * inv_n) / h0;
    T h1;
    if (d1 <= (T)1e-15 && d2 <= (T)1e-15) h1 = fmax((T)1e-6, h0 * (T)1e-3);
    else h1 = pow((T)0.01 / fmax(d1, d2), (T)0.2);
    return fmin(fmin((T)100 * h0, h1), t_end);
}

// ---- Tsitouras 5(4) with diffrax's PID step-size controller (the current generation's solver) -----------------------
// src/simulator/propagator.py:533-599 integrates every ray with diffrax.Tsit5 under PIDController(rtol, atol) in
// normalised time tau = t / T, T = sqrt(8) depth / c, dt0 = T / save_steps (in tau units, as written upstream),
// max_steps = 10000.  PARITY UNPINNED: jax / diffrax cannot be installed here, so this follows the published method
// (Tsitouras 2011; the tableau below satisfies every order condition up to 5, b - btilde up to 4, to 1e-16 -- checked in
// tests/test_host_misc.py) and diffrax's documented controller defaults: pcoeff = 0, icoeff = 1, dcoeff = 0, i.e.
//     factor = clip(safety * err^(-1/5), factormin, factormax),  safety 0.9, factormax 10,
//     factormin = 0.2 after a rejected step and 1 after an accepted one,  accept iff err < 1,
//     err = rms_i( y_error_i / (atol + rtol max(|y0_i|, |y1_i|)) ) over the 9 state components.
// State here: y = {p[3], v[3], phase}; amp and pol have zero derivative (zero error) and only count in the mean.
template <typename T, bool PHASE, bool AUX64>
SP_HD int tsit5_f(const FieldView<T>& F, T omega, const T* y, T* f) {
    T nm1;
    const int t = rhs_direct<T, PHASE, AUX64>(F, y[0], y[1], y[2], f[3], f[4], f[5], nm1);
    f[0] = y[3]; f[1] = y[4]; f[2] = y[5];
    f[6] = PHASE ? omega * nm1 : (T)0;
    return t;
}

// STAGED: the stage matrix is the caller's Ks ([7][7], rows 1 .. s_first - 1 filled), the attempt starts with the evaluation
// that fills row s_first (1 .. 6; 6 = the one at yn), and a park reports the row it was about to fill in *s_park.
template <typename T, bool PHASE, bool AUX64, bool WIN = false, bool STAGED = false>
SP_HD int tsit5_attempt(const FieldView<T>& F, T omega, T h, T rtol, T atol, const T* y, const T* k1, T* yn, T* k7, T& err_sq,
                        const Window* W = nullptr, double* out = nullptr, int s_first = 1, int* s_park = nullptr, T* Ks = nullptr) {
    const double A[5][5] = {{0.161, 0, 0, 0, 0},
                            {-0.008480655492356989, 0.335480655492357, 0, 0, 0},
                            {2.8971530571054935, -6.359448489975075, 4.3622954328695815, 0, 0},
                            {5.325864828439257, -11.748883564062828, 7.4955393428898365, -0.09249506636175525, 0},
                            {5.86145544294642, -12.92096931784711, 8.159367898576159, -0.071584973281401, -0.028269050394068383}};
    const double B[6] = {0.09646076681806523, 0.01, 0.4798896504144996, 1.379008574103742, -3.290069515436081, 2.324710524099774};
    const double Bt[7] = {-0.00178001105222577714, -0.0008164344596567469, 0.007880878010261995, -0.1447110071732629,
                          0.5823571654525552, -0.45808210592918697, 0.015151515151515152};
    T Kl[STAGED ? 1 : 7][7], ys[7];
    T (*K)[7] = STAGED ? reinterpret_cast<T (*)[7]>(Ks) : Kl;
    int touched = 0;
    for (int i = 0; i < 7; ++i) K[0][i] = k1[i];
    for (int s = 1; s < 6; ++s) {
        if (STAGED && s < s_first) continue;           // the same loop as in core, so the compiler contracts it alike
        for (int i = 0; i < 7; ++i) {
            T acc = (T)A[s - 1][0] * K[0][i];
            for (int j = 1; j < s; ++j) acc += (T)A[s - 1][j] * K[j][i];
            ys[i] = y[i] + acc * h;
        }
        if (WIN && outside(*W, F, ys)) {
            *out = (double)ys[2];
            if constexpr (STAGED) *s_park = s;
            return touched;
        }
        touched += tsit5_f<T, PHASE, AUX64>(F, omega, ys, K[s]);
    }
    for (int i = 0; i < 7; ++i) {
        T acc = (T)B[0] * K[0][i];
        for (int j = 1; j < 6; ++j) acc += (T)B[j] * K[j][i];
        yn[i] = y[i] + h * acc;
    }
    if (WIN && outside(*W, F, yn)) {
        *out = (double)yn[2];
        if constexpr (STAGED) *s_park = 6;
        return touched;
    }
    touched += tsit5_f<T, PHASE, AUX64>(F, omega, yn, K[6]);
    T tot = (T)0;
    for (int i = 0; i < 7; ++i) {
        k7[i] = K[6][i];
        T e = (T)Bt[0] * K[0][i];
        for (int j = 1; j < 7; ++j) e += (T)Bt[j] * K[j][i];
        e *= h;
        const T a0 = fabs(y[i]), a1 = fabs(yn[i]);
        const T q = e / (atol + (a0 > a1 ? a0 : a1) * rtol);
        tot += q * q;
    }
    err_sq = tot;
    return touched;
}

// diffrax PIDController.adapt_step_size with the default (integral-only) coefficients
template <typename T> SP_HD T pid_factor(T err, bool keep) {
    const T fmin_ = keep ? (T)1 : (T)0.2;
    if (err == (T)0) return (T)10;
    const T f = (T)0.9 * pow(err, (T)-0.2);
    return f < fmin_ ? fmin_ : (f > (T)10 ? (T)10 : f);
}

// ---- the per-ray adaptive solves restricted to a window (out-of-core tracing, sp_propagate_window) -----------------
// The controller loops of k_propagate's SP_METHOD_RK45 and SP_METHOD_TSIT5 branches, resumable: a ray PARKS when its
// next attempt (or RK45's initial-step probe p + h0 f0) would evaluate the field outside the window W.  The attempt is
// dropped -- no attempt counted, no state committed -- and the record is left exactly as it was at the top of that loop
// iteration (h before the clip to t_end: storing the clipped one would move the final step by an ulp on resume; the
// min_step clamp is idempotent).  The next launch, over a slab that holds the point, resumes from the record: the FSAL
// derivative is recomputed at the committed state (rhs_direct has no cache, so it is the same bits) and min_step from t.
// Every committed attempt therefore does exactly the in-core arithmetic.  One code for the kernels and the CPU test
// build; the warp vote only keeps the lanes converged.
#define SP_CTL_STARTED 1u     // RK45: initial step chosen / Tsit5: dt holds the controller's step
#define SP_CTL_PENDING 2u     // RK45: a rejected attempt is pending (the retry keeps min_step and the rejected flag)
#define SP_CTL_FINISHED 4u    // t == t_end, escaped (early exit) or failed: the epilogue has run
#define SP_CTL_FAILED 8u      // attempt cap, step below min_step, or NaN error norm
struct WinCtl {
    double t, h;              // RK45: t, h_abs / Tsit5: tau, dt
    double w_park;            // w of the point that parked the ray (the next window must hold it)
    unsigned n_att, flags;
};

// ---- stage parking (sp_propagate_window_staged, out_of_core park='stage') ----------------------------------------------
// The loops above park a ray a whole attempt at a time, so a window must hold the ray's position and every stage point of
// its next attempt.  With STAGED they park between stage evaluations instead: a ray parks right before the first point of
// its attempt (or of RK45's initial-step probe) that lies outside the window, and the per-ray STAGE STORE in HBM keeps
//   * K1, the FSAL derivative at the committed state (for the probe: f0),
//   * the stage values evaluated so far in this attempt,
// while the record flags get SP_CTL_STAGED and, in bits SP_CTL_ROW_SHIFT.., the row of the stage matrix the next evaluation
// fills (1 .. 6; 0 = RK45's initial-step probe).  The record's t / h / PENDING are as at the top of the loop iteration, as
// for an attempt park, so the resumed attempt recomputes its h with the same instructions.  On resume nothing is evaluated
// at the ray's own position: the next evaluation is the stage point, in whichever slab holds it.  Every stage derivative is
// a pure function of its point (rhs_direct has no cache; deriv9's fresh cell lookup is the cached one), so the committed
// arithmetic and the evaluation count are the in-core ones.  Store layout: value j of ray i at stg[j * stride + i]
// (stride = the rays of the state), in the solve's precision (float32 for float32 instantiations):
//   RK45  (SP_STAGE_RK45,  23 values, 184 B per ray in float64): K1 dv[3], K1 dph, StageSmem's 19 values (K2..K6 dv, n3..n6)
//   Tsit5 (SP_STAGE_TSIT5, 42 values, 336 B): the stage matrix rows K[0..5][7]
//   RK45X (SP_STAGE_RK45X, 54 values, 432 B): the stage matrix rows K[0..5][9]
#define SP_CTL_STAGED 16u
#define SP_CTL_ROW_SHIFT 8
#define SP_STAGE_RK45 23
#define SP_STAGE_TSIT5 42
#define SP_STAGE_RK45X 54
template <typename T> struct StageStore {
    T* p; unsigned long long stride;
    SP_HD T get(int j) const { return p[(unsigned long long)j * stride]; }
    SP_HD void set(int j, T v) const { p[(unsigned long long)j * stride] = v; }
};
SP_HD int staged_row(unsigned flags) { return (int)((flags >> SP_CTL_ROW_SHIFT) & 15u); }

// escaped() for stage parking.  A resumed ray's position may lie outside the slab (only its next point has to be inside the
// window), so along w the test takes the whole grid's bounds, not the slab's: the slab's own where the window reaches a
// grid edge (w_lo / w_hi infinite: the slab starts / ends with the grid), [g_lo, g_hi] elsewhere.  Both are the grid's
// float32-rounded end planes, so the decision is the in-core one.
template <typename T> SP_HD bool escaped_grid(const FieldView<T>& F, const Window& W, const Ray<T>& r) {
    const double lo = W.lo == -(double)INFINITY ? (double)F.ax[2].lo : W.g_lo;
    const double hi = W.hi == (double)INFINITY ? (double)F.ax[2].hi : W.g_hi;
    const double w = (double)r.p[2];
    bool e = (w > hi && r.v[2] >= (T)0) || (w < lo && r.v[2] <= (T)0);
#pragma unroll
    for (int k = 0; k < 2; ++k)
        e = e || (r.p[k] > F.ax[k].hi && r.v[k] >= (T)0) || (r.p[k] < F.ax[k].lo && r.v[k] <= (T)0);
    return e;
}

#if defined(__CUDA_ARCH__)
#define SP_WIN_VOTE(lanes, go) __any_sync(lanes, go)
#else
#define SP_WIN_VOTE(lanes, go) (go)
#endif

template <typename T, bool PHASE, bool AUX64, typename Store, bool STAGED = false>
SP_HD int dp5_window(const FieldView<T>& F, const Window& W, T omega, T t_end, T rtol, T atol, int n_state, T amp, T pol,
                     unsigned cap, bool early, unsigned lanes, Ray<T>& r, WinCtl& c, Store& S, unsigned& acc, unsigned& capped,
                     StageStore<T> G = StageStore<T>()) {
    int touched = 0;
    const bool skip = (c.flags & SP_CTL_FINISHED) != 0;   // finished in an earlier launch: takes part in the votes only
    const bool held = STAGED && !skip && (c.flags & SP_CTL_STAGED) != 0;   // K1 and the first stages are in the stage store
    const int row = held ? staged_row(c.flags) : 0;
    int s_first = row >= 1 ? row + 1 : 2, s_park = 0, park_row = -1;
    double pw = NAN;                                       // set (not NaN) once the ray parks
    if (skip) pw = 0.0;
    else if (!held && outside(W, F, r.p)) pw = (double)r.p[2];   // before the escape test: the slab's w bounds are not the grid's
    T t = (T)c.t, h_abs = (T)c.h;
    unsigned n_att = c.n_att;
    bool failed = false, rejected = (c.flags & SP_CTL_PENDING) != 0, fresh = !rejected, started = (c.flags & SP_CTL_STARTED) != 0;
    T min_step = (T)10 * (nextafter(t, (T)INFINITY) - t);
    const T inv_n = (T)1 / (T)n_state;
    Deriv<T> f;
    f.dp[0] = f.dp[1] = f.dp[2] = f.dv[0] = f.dv[1] = f.dv[2] = f.dph = (T)0;
    if (pw != pw) {
        if constexpr (STAGED) {
            if (held) {
#pragma unroll
                for (int k = 0; k < 3; ++k) { f.dp[k] = r.v[k]; f.dv[k] = G.get(k); }
                f.dph = G.get(3);
                for (int j = 0; j < row - 1; ++j)              // K2 .. K(row): S.K(j) is stage j + 2, S.N(j) stage j + 3
                    for (int k = 0; k < 3; ++k) S.setK(j, k, G.get(4 + 3 * j + k));
                for (int j = 0; j < row - 2; ++j) S.setN(j, G.get(19 + j));
            } else {
                touched += deriv_direct<T, PHASE, AUX64>(F, omega, r.p, r.v, f);
            }
        } else {
            touched += deriv_direct<T, PHASE, AUX64>(F, omega, r.p, r.v, f);
        }
        if (!started) {
            const T h0 = dp5_initial_step<T, PHASE, AUX64, true>(F, omega, t_end, rtol, atol, n_state, amp, pol, r, f, touched, &W, &pw);
            if (pw != pw) { h_abs = h0; started = true; }
            if constexpr (STAGED) if (pw == pw) park_row = 0;
        }
    }
    for (;;) {
        bool go = (pw != pw) && (t < t_end) && !failed;
        const T h_top = h_abs;
        const bool fresh_top = fresh;
        if (go && fresh) {
            if (early && (STAGED ? escaped_grid(F, W, r) : escaped(F, r))) go = false;
            else {
                min_step = (T)10 * (nextafter(t, (T)INFINITY) - t);
                if (h_abs < min_step) h_abs = min_step;
                rejected = false; fresh = false;
            }
        }
        if (go && (n_att >= cap || h_abs < min_step)) { failed = true; capped += 1; go = false; }
        if (!SP_WIN_VOTE(lanes, go)) break;
        if (go) {
            T t_new = t + h_abs;
            if (t_new - t_end > (T)0) t_new = t_end;
            const T h = t_new - t;
            h_abs = fabs(h);
            Ray<T> rn; Deriv<T> fn; T esq;
            if constexpr (STAGED) {
                touched += dp5_attempt<T, PHASE, AUX64, Store, true, true>(F, omega, h, rtol, atol, r, f, rn, fn, esq, S, &W, &pw,
                                                                           s_first, &s_park);
                s_first = 2;
                if (pw == pw) park_row = s_park - 1;
            } else {
                touched += dp5_attempt<T, PHASE, AUX64, Store, true>(F, omega, h, rtol, atol, r, f, rn, fn, esq, S, &W, &pw);
            }
            if (pw == pw) { h_abs = h_top; fresh = fresh_top; }          // parked: the record as at the top of this iteration
            else {
                ++n_att;
                const T en = sqrt(esq * inv_n);
                if (!(en == en)) { failed = true; capped += 1; }
                else {
                    const bool acc_ = en < (T)1;
                    h_abs *= dp5_factor<T>(en, acc_, rejected);
                    if (acc_) { t = t_new; r = rn; f = fn; acc += 1; fresh = true; }
                    else rejected = true;
                }
            }
        }
    }
    if (skip) return touched;
    c.t = (double)t; c.h = (double)h_abs; c.n_att = n_att; c.w_park = pw;
    c.flags = (started ? SP_CTL_STARTED : 0u) | (fresh ? 0u : SP_CTL_PENDING) | (pw != pw ? SP_CTL_FINISHED : 0u) | (failed ? SP_CTL_FAILED : 0u);
    if constexpr (STAGED) if (pw == pw && park_row >= 0) {
        c.flags |= SP_CTL_STAGED | ((unsigned)park_row << SP_CTL_ROW_SHIFT);
#pragma unroll
        for (int k = 0; k < 3; ++k) G.set(k, f.dv[k]);
        G.set(3, f.dph);
        for (int j = 0; j < park_row - 1; ++j)
            for (int k = 0; k < 3; ++k) G.set(4 + 3 * j + k, S.K(j, k));
        for (int j = 0; j < park_row - 2; ++j) G.set(19 + j, S.N(j));
    }
    return touched;
}

// Tsit5 + PID per ray (k_propagate's SP_METHOD_TSIT5 branch), resumable in the same way; dt0 is taken when !STARTED.
template <typename T, bool PHASE, bool AUX64, bool STAGED = false>
SP_HD int tsit5_window(const FieldView<T>& F, const Window& W, T omega, T t_end, T dt0, T rtol, T atol, int n_state,
                       unsigned cap, unsigned lanes, Ray<T>& r, WinCtl& c, unsigned& acc, unsigned& capped,
                       StageStore<T> G = StageStore<T>()) {
    int touched = 0;
    const bool skip = (c.flags & SP_CTL_FINISHED) != 0;
    const bool held = STAGED && !skip && (c.flags & SP_CTL_STAGED) != 0;
    const int row = held ? staged_row(c.flags) : 0;
    int s_first = row >= 1 ? row : 1, s_park = 0, park_row = -1;
    double pw = NAN;
    if (skip) pw = 0.0;
    else if (!held && outside(W, F, r.p)) pw = (double)r.p[2];
    T y[7], f[7], yn[7], fn[7];
    T K[STAGED ? 7 : 1][7];                                // STAGED: the attempt's stage matrix, saved at a park
#pragma unroll
    for (int k = 0; k < 3; ++k) { y[k] = r.p[k]; y[3 + k] = r.v[k]; }
    y[6] = r.ph;
#pragma unroll
    for (int k = 0; k < 7; ++k) f[k] = (T)0;
    if constexpr (STAGED) {
        if (held) {
            for (int j = 0; j < row; ++j)
                for (int i = 0; i < 7; ++i) K[j][i] = G.get(7 * j + i);
            for (int i = 0; i < 7; ++i) f[i] = K[0][i];
        } else if (pw != pw) {
            touched += tsit5_f<T, PHASE, AUX64>(F, omega, y, f);
        }
    } else {
        if (pw != pw) touched += tsit5_f<T, PHASE, AUX64>(F, omega, y, f);
    }
    T tau = (T)c.t, dt = (c.flags & SP_CTL_STARTED) ? (T)c.h : dt0;
    unsigned n_att = c.n_att;
    const T inv_n = (T)1 / (T)n_state;
    bool failed = false;
    for (;;) {
        bool go = (pw != pw) && (tau < (T)1) && !failed;
        if (go && n_att >= cap) { failed = true; capped += 1; go = false; }
        if (!SP_WIN_VOTE(lanes, go)) break;
        if (go) {
            const bool last = tau + dt >= (T)1;
            const T d = last ? (T)1 - tau : dt;
            T esq;
            if constexpr (STAGED) {
                touched += tsit5_attempt<T, PHASE, AUX64, true, true>(F, omega, d * t_end, rtol, atol, y, f, yn, fn, esq, &W, &pw,
                                                                      s_first, &s_park, &K[0][0]);
                s_first = 1;
                if (pw == pw) park_row = s_park;
            } else {
                touched += tsit5_attempt<T, PHASE, AUX64, true>(F, omega, d * t_end, rtol, atol, y, f, yn, fn, esq, &W, &pw);
            }
            if (pw != pw) {
                ++n_att;
                const T en = sqrt(esq * inv_n);
                if (!(en == en)) { failed = true; capped += 1; }
                else {
                    const bool keep = en < (T)1;
                    dt = d * pid_factor<T>(en, keep);
                    if (keep) {
                        tau = last ? (T)1 : tau + d; acc += 1;
#pragma unroll
                        for (int i = 0; i < 7; ++i) { y[i] = yn[i]; f[i] = fn[i]; }
                    }
                }
            }
        }
    }
    if (skip) return touched;
#pragma unroll
    for (int k = 0; k < 3; ++k) { r.p[k] = y[k]; r.v[k] = y[3 + k]; }
    r.ph = y[6];
    c.t = (double)tau; c.h = (double)dt; c.n_att = n_att; c.w_park = pw;
    c.flags = SP_CTL_STARTED | (pw != pw ? SP_CTL_FINISHED : 0u) | (failed ? SP_CTL_FAILED : 0u);
    if constexpr (STAGED) if (pw == pw && park_row >= 1) {
        c.flags |= SP_CTL_STAGED | ((unsigned)park_row << SP_CTL_ROW_SHIFT);
        for (int j = 0; j < park_row; ++j)
            for (int i = 0; i < 7; ++i) G.set(7 * j + i, K[j][i]);
    }
    return touched;
}

// ---- Dormand-Prince on the full 9-component state (attenuation / Faraday channels on; slow path) ----------------
// State y = {p[3], v[3], amp, phase, pol} in the kernel frame; the same controller arithmetic as above, written
// generically over the nine rows exactly as scipy does (rk.py: rk_step, _estimate_error_norm).
template <bool PHASE, bool AUX64>
SP_HD int deriv9(const FieldView<double>& F, const ExtView& X, CellCache<double, PHASE>& cc, double omega, bool with_phase,
                 const double* y, double* f) {
    double a[3], n, x[5];
    const bool in = rhs<double, PHASE, AUX64>(F, cc, y[0], y[1], y[2], a[0], a[1], a[2], n);
    ext_eval<PHASE>(F, X, cc, in, y, x);
    f[0] = y[3]; f[1] = y[4]; f[2] = y[5];
    f[3] = a[0]; f[4] = a[1]; f[5] = a[2];
    f[6] = x[0] * y[6];
    f[7] = (PHASE && with_phase) ? omega * n : 0.0;
    f[8] = X.verdet * x[1] * (x[2] * y[3] + x[3] * y[4] + x[4] * y[5]);
    return in;
}

// STAGED: as tsit5_attempt, with the caller's [7][9] stage matrix Ks.
template <bool PHASE, bool AUX64, bool WIN = false, bool STAGED = false>
SP_HD int dp5_attempt9(const FieldView<double>& F, const ExtView& X, CellCache<double, PHASE>& cc, double omega, bool with_phase,
                       double h, double rtol, double atol, const double* y, const double* k1, double* yn, double* k7,
                       double& err_sq, const Window* W = nullptr, double* out = nullptr, int s_first = 1, int* s_park = nullptr,
                       double* Ks = nullptr) {
    const double A[5][5] = {{DP::a21, 0, 0, 0, 0}, {DP::a31, DP::a32, 0, 0, 0}, {DP::a41, DP::a42, DP::a43, 0, 0},
                            {DP::a51, DP::a52, DP::a53, DP::a54, 0}, {DP::a61, DP::a62, DP::a63, DP::a64, DP::a65}};
    const double Bc[6] = {DP::b1, 0.0, DP::b3, DP::b4, DP::b5, DP::b6};
    const double Ec[7] = {DP::e1, 0.0, DP::e3, DP::e4, DP::e5, DP::e6, DP::e7};
    double Kl[STAGED ? 1 : 7][9], ys[9];
    double (*K)[9] = STAGED ? reinterpret_cast<double (*)[9]>(Ks) : Kl;
    int touched = 0;
    for (int i = 0; i < 9; ++i) K[0][i] = k1[i];
    for (int s = 1; s < 6; ++s) {
        if (STAGED && s < s_first) continue;           // the same loop as in core, so the compiler contracts it alike
        for (int i = 0; i < 9; ++i) {
            double acc = A[s - 1][0] * K[0][i];
            for (int j = 1; j < s; ++j) acc += A[s - 1][j] * K[j][i];
            ys[i] = y[i] + acc * h;
        }
        if (WIN && outside(*W, F, ys)) {
            *out = ys[2];
            if constexpr (STAGED) *s_park = s;
            return touched;
        }
        touched += deriv9<PHASE, AUX64>(F, X, cc, omega, with_phase, ys, K[s]);
    }
    for (int i = 0; i < 9; ++i) {
        double acc = Bc[0] * K[0][i];
        for (int j = 2; j < 6; ++j) acc += Bc[j] * K[j][i];
        yn[i] = y[i] + h * acc;
    }
    if (WIN && outside(*W, F, yn)) {
        *out = yn[2];
        if constexpr (STAGED) *s_park = 6;
        return touched;
    }
    touched += deriv9<PHASE, AUX64>(F, X, cc, omega, with_phase, yn, K[6]);
    double tot = 0.0;
    for (int i = 0; i < 9; ++i) {
        k7[i] = K[6][i];
        double e = Ec[0] * K[0][i];
        for (int j = 2; j < 7; ++j) e += Ec[j] * K[j][i];
        e *= h;
        const double a0 = fabs(y[i]), a1 = fabs(yn[i]);
        const double q = e / (atol + (a0 > a1 ? a0 : a1) * rtol);
        tot += q * q;
    }
    err_sq = tot;
    return touched;
}

template <bool PHASE, bool AUX64, bool WIN = false>
SP_HD double dp5_initial_step9(const FieldView<double>& F, const ExtView& X, CellCache<double, PHASE>& cc, double omega,
                               bool with_phase, double t_end, double rtol, double atol, const double* y, const double* f0,
                               int& touched, const Window* W = nullptr, double* out = nullptr) {
    if (t_end == 0.0) return 0.0;
    double s0 = 0, s1 = 0, sc[9], y1[9], f1[9];
    for (int i = 0; i < 9; ++i) {
        sc[i] = atol + fabs(y[i]) * rtol;
        double q = y[i] / sc[i]; s0 += q * q;
        q = f0[i] / sc[i]; s1 += q * q;
    }
    const double d0 = sqrt(s0 / 9.0), d1 = sqrt(s1 / 9.0);
    double h0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * d0 / d1;
    h0 = fmin(h0, t_end);
    for (int i = 0; i < 9; ++i) y1[i] = y[i] + h0 * f0[i];
    if (WIN && outside(*W, F, y1)) { *out = y1[2]; return 0.0; }
    touched += deriv9<PHASE, AUX64>(F, X, cc, omega, with_phase, y1, f1);
    double s2 = 0;
    for (int i = 0; i < 9; ++i) { const double q = (f1[i] - f0[i]) / sc[i]; s2 += q * q; }
    const double d2 = sqrt(s2 / 9.0) / h0;
    const double h1 = (d1 <= 1e-15 && d2 <= 1e-15) ? fmax(1e-6, h0 * 1e-3) : pow(0.01 / fmax(d1, d2), 0.2);
    return fmin(fmin(100 * h0, h1), t_end);
}

// The per-ray solve over all nine rows (k_propagate's SP_METHOD_RK45X loop, rk45x_integrate) restricted to a window:
// the loop of dp5_window with the same record, parking rule and votes.  y (9 rows: p, v in the kernel frame, amp, phase,
// pol) is read and written -- amp and pol are integrated, so they carry over from slab to slab like the position.  On
// resume the FSAL derivative is recomputed with deriv9 at the committed state through a fresh CellCache: a fresh lookup
// is the cached one bit for bit (tests/test_out_of_core_channels.py pins it for ext_eval), so every committed attempt
// does the in-core arithmetic.
template <bool PHASE, bool AUX64, bool STAGED = false>
SP_HD int dp5x_window(const FieldView<double>& F, const ExtView& X, const Window& W, double omega, bool with_phase, double t_end,
                      double rtol, double atol, unsigned cap, bool early, unsigned lanes, double* y, WinCtl& c, unsigned& acc,
                      unsigned& capped, StageStore<double> G = StageStore<double>()) {
    int touched = 0;
    const bool skip = (c.flags & SP_CTL_FINISHED) != 0;
    const bool held = STAGED && !skip && (c.flags & SP_CTL_STAGED) != 0;
    const int row = held ? staged_row(c.flags) : 0;
    int s_first = row >= 1 ? row : 1, s_park = 0, park_row = -1;
    double pw = NAN;
    if (skip) pw = 0.0;
    else if (!held && outside(W, F, y)) pw = y[2];
    double K[STAGED ? 7 : 1][9];                           // STAGED: the attempt's stage matrix, saved at a park
    double t = c.t, h_abs = c.h;
    unsigned n_att = c.n_att;
    bool failed = false, rejected = (c.flags & SP_CTL_PENDING) != 0, fresh = !rejected, started = (c.flags & SP_CTL_STARTED) != 0;
    double min_step = 10.0 * (nextafter(t, (double)INFINITY) - t);
    CellCache<double, PHASE> cc;
    double f[9], yn[9], fn[9];
    for (int i = 0; i < 9; ++i) f[i] = 0.0;
    if (pw != pw) {
        if constexpr (STAGED) {
            if (held) {
                for (int j = 0; j < (row > 1 ? row : 1); ++j)
                    for (int i = 0; i < 9; ++i) K[j][i] = G.get(9 * j + i);
                for (int i = 0; i < 9; ++i) f[i] = K[0][i];
            } else {
                touched += deriv9<PHASE, AUX64>(F, X, cc, omega, with_phase, y, f);
            }
        } else {
            touched += deriv9<PHASE, AUX64>(F, X, cc, omega, with_phase, y, f);
        }
        if (!started) {
            const double h0 = dp5_initial_step9<PHASE, AUX64, true>(F, X, cc, omega, with_phase, t_end, rtol, atol, y, f, touched, &W, &pw);
            if (pw != pw) { h_abs = h0; started = true; }
            if constexpr (STAGED) if (pw == pw) park_row = 0;
        }
    }
    for (;;) {
        bool go = (pw != pw) && (t < t_end) && !failed;
        const double h_top = h_abs;
        const bool fresh_top = fresh;
        if (go && fresh) {
            bool out = false;
            if (early) {
                Ray<double> q;
                for (int k = 0; k < 3; ++k) { q.p[k] = y[k]; q.v[k] = y[3 + k]; }
                out = STAGED ? escaped_grid(F, W, q) : escaped(F, q);
            }
            if (out) go = false;
            else {
                min_step = 10.0 * (nextafter(t, (double)INFINITY) - t);
                if (h_abs < min_step) h_abs = min_step;
                rejected = false; fresh = false;
            }
        }
        if (go && (n_att >= cap || h_abs < min_step)) { failed = true; capped += 1; go = false; }
        if (!SP_WIN_VOTE(lanes, go)) break;
        if (go) {
            double t_new = t + h_abs;
            if (t_new - t_end > 0.0) t_new = t_end;
            const double h = t_new - t;
            h_abs = fabs(h);
            double esq;
            if constexpr (STAGED) {
                touched += dp5_attempt9<PHASE, AUX64, true, true>(F, X, cc, omega, with_phase, h, rtol, atol, y, f, yn, fn, esq, &W,
                                                                  &pw, s_first, &s_park, &K[0][0]);
                s_first = 1;
                if (pw == pw) park_row = s_park;
            } else {
                touched += dp5_attempt9<PHASE, AUX64, true>(F, X, cc, omega, with_phase, h, rtol, atol, y, f, yn, fn, esq, &W, &pw);
            }
            if (pw == pw) { h_abs = h_top; fresh = fresh_top; }          // parked: the record as at the top of this iteration
            else {
                ++n_att;
                const double en = sqrt(esq / 9.0);
                if (!(en == en)) { failed = true; capped += 1; }
                else if (en < 1.0) {
                    h_abs *= dp5_factor<double>(en, true, rejected);
                    t = t_new; acc += 1;
                    for (int i = 0; i < 9; ++i) { y[i] = yn[i]; f[i] = fn[i]; }
                    fresh = true;
                } else {
                    h_abs *= dp5_factor<double>(en, false, rejected);
                    rejected = true;
                }
            }
        }
    }
    if (skip) return touched;
    c.t = t; c.h = h_abs; c.n_att = n_att; c.w_park = pw;
    c.flags = (started ? SP_CTL_STARTED : 0u) | (fresh ? 0u : SP_CTL_PENDING) | (pw != pw ? SP_CTL_FINISHED : 0u) | (failed ? SP_CTL_FAILED : 0u);
    if constexpr (STAGED) if (pw == pw && park_row >= 0) {
        c.flags |= SP_CTL_STAGED | ((unsigned)park_row << SP_CTL_ROW_SHIFT);
        for (int i = 0; i < 9; ++i) G.set(i, f[i]);        // K1 (for the probe: f0)
        for (int j = 1; j < park_row; ++j)
            for (int i = 0; i < 9; ++i) G.set(9 * j + i, K[j][i]);
    }
    return touched;
}

// ---- exit plane ------------------------------------------------------------------------------------------
// ray_to_Jonesvector (full_solver.py:838-894): back-project to the plane coord[p] = extent; angles atan(v_a/v_p).
// kp/ka/kb are kernel-frame indices of the probing axis and of the axes that land in rf rows (0,1) / (2,3).
// (components are picked with selects, not r.p[k]: a dynamically indexed member would force the whole ray
// state into local memory and cost six local stores per integration step)
template <typename T> SP_HD T pick3(const T* a, int k) { return k == 0 ? a[0] : (k == 1 ? a[1] : a[2]); }

template <typename T>
SP_HD void exit_project(const Ray<T>& r, int kp, int ka, int kb, T extent, T& xa, T& tha, T& xb, T& thb) {
    const T pp = pick3(r.p, kp), vp = pick3(r.v, kp);
    const T pa = pick3(r.p, ka), va = pick3(r.v, ka), pb = pick3(r.p, kb), vb = pick3(r.v, kb);
    const T tbp = (pp - extent) / vp;
    xa = pa - va * tbp;
    xb = pb - vb * tbp;
    tha = atan(va / vp);
    thb = atan(vb / vp);
}

// ---- optics ------------------------------------------------------------------------------------------------
struct OpticOp { int kind; int pad; double p0, p1, p2; };
enum { OP_TRAVEL = 0, OP_TRAVEL_NOE = 1, OP_LENS = 2, OP_CIRC_AP = 3, OP_CIRC_STOP = 4, OP_RECT_AP = 5,
       OP_KNIFE = 6, OP_REF_BEAM = 7 };

struct DetRay {
    double x, th, y, ph;      // mm, rad
    double ex_re, ex_im, ey_re, ey_im;
    bool alive;
};

SP_HD void sp_sincos(double a, double* s, double* c) {
#if defined(__CUDA_ARCH__)
    sincos(a, s, c);
#else
    *s = sin(a); *c = cos(a);
#endif
}

SP_HD void cmul_phase(double& re, double& im, double arg) {
    double s, c; sp_sincos(arg, &s, &c);
    const double r = re * c - im * s, i = re * s + im * c;   // (re + i im)(c + i s), numpy's complex product
    re = r; im = i;
}

// Applies the optical train to one ray.  rf (metres) -> m_to_mm -> ops.  Matrix elements are applied as the
// reference's np.matmul of a block-diagonal 4x4 does: x' = 1*x + d*th (products then sum).  Rejected rays
// are flagged dead (the reference sets the column to NaN; every later element keeps it NaN).
// E advances by exp(i k sqrt(dx^2 + dy^2)) across TRAVEL (k = 2 pi / wavelength, positions in mm: the
// reference's own unit mix, diagnostics.py:315-321).  Across a lens dx = dy = 0 so the factor is exactly 1.
SP_HD void run_optics(DetRay& d, double x_m, double y_m, const OpticOp* ops, int n_ops, bool with_E, double kwave) {
    for (int i = 0; i < n_ops && d.alive; ++i) {
        const OpticOp op = ops[i];
        switch (op.kind) {
            case OP_TRAVEL:
            case OP_TRAVEL_NOE: {
                const double nx = add_rn(d.x, mul_rn(op.p0, d.th));
                const double ny = add_rn(d.y, mul_rn(op.p0, d.ph));
                if (with_E && op.kind == OP_TRAVEL) {
                    const double dx = nx - d.x, dy = ny - d.y;
                    const double arg = mul_rn(kwave, sqrt(add_rn(mul_rn(dx, dx), mul_rn(dy, dy))));
                    cmul_phase(d.ex_re, d.ex_im, arg);
                    cmul_phase(d.ey_re, d.ey_im, arg);
                }
                d.x = nx; d.y = ny;
            } break;
            case OP_LENS:
                d.th = add_rn(mul_rn(-1.0 / op.p0, d.x), d.th);
                d.ph = add_rn(mul_rn(-1.0 / op.p1, d.y), d.ph);
                break;
            case OP_CIRC_AP:
                if (add_rn(mul_rn(d.x, d.x), mul_rn(d.y, d.y)) > op.p0 * op.p0) d.alive = false;
                break;
            case OP_CIRC_STOP:
                if (add_rn(mul_rn(d.x, d.x), mul_rn(d.y, d.y)) < op.p0 * op.p0) d.alive = false;
                break;
            case OP_RECT_AP:   // only rays outside BOTH half-widths are rejected (rtm_solver.py:114-117)
                if (d.x * d.x > op.p0 * op.p0 && d.y * d.y > op.p1 * op.p1) d.alive = false;
                break;
            case OP_KNIFE: {
                const double c = (op.p1 < 1.0) ? d.x : d.y;
                if (op.p2 > 0 ? (c > op.p0) : (c < op.p0)) d.alive = false;
            } break;
            case OP_REF_BEAM: {   // diagnostics.py:559-581 (uses exit positions in METRES)
                double deg = op.p1;
                if (deg >= 45.0) deg = -fabs(deg - 90.0);
                const double rad = deg * 3.14159265358979323846 / 180.0;
                const double yw = atan(rad), xw = sqrt(1.0 - yw * yw);
                double s, c; sp_sincos(2.0 * op.p0 / 3.0 * (xw * x_m + yw * y_m), &s, &c);
                d.ey_re += c; d.ey_im += s;
            } break;
            default: break;
        }
        // NaN positions: comparisons above are false, as in NumPy; the ray stays "alive" but can never be
        // binned (bin search fails on NaN), matching the reference's isnan filter.
    }
}

// ---- detector bins ---------------------------------------------------------------------------------------
// np.linspace(lo, hi, nb+1)[i] = i * step + lo with step = (hi - lo) / nb, last edge forced to hi.
SP_HD double lin_edge(double lo, double hi, double step, int nb, int i) {
    return (i >= nb) ? hi : add_rn(mul_rn((double)i, step), lo);
}

// histogram mode: index of the bin with edge[i] <= v < edge[i+1], v == hi -> nb-1  (np.histogram2d);
// digitize mode : np.digitize(v, edges) - 1 must be in [0, nb-1], so v == hi is OUT (rtm_solver.py:439-444).
// Returns -1 when the value is not binned (outside, NaN).
SP_HD int bin_index(double v, double lo, double hi, int nb, bool right_inclusive) {
    if (!(v >= lo) || !(v <= hi)) return -1;
    if (v == hi) return right_inclusive ? nb - 1 : -1;
    const double step = (hi - lo) / (double)nb;
    int i = floor_to_int((v - lo) / step);
    i = i < 0 ? 0 : (i > nb - 1 ? nb - 1 : i);
    while (i > 0 && v < lin_edge(lo, hi, step, nb, i)) --i;
    while (i < nb - 1 && v >= lin_edge(lo, hi, step, nb, i + 1)) ++i;
    return i;
}

// ---- Philox4x32-10 beam generator ---------------------------------------------------------------------------
struct Philox {
    uint32_t k0, k1;
    SP_HD static void mulhilo(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
        const uint64_t p = (uint64_t)a * b;
        hi = (uint32_t)(p >> 32); lo = (uint32_t)p;
    }
    SP_HD void block(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t out[4]) const {
        uint32_t a = k0, b = k1;
#pragma unroll
        for (int r = 0; r < 10; ++r) {
            uint32_t h0, l0, h1, l1;
            mulhilo(0xD2511F53u, c0, h0, l0);
            mulhilo(0xCD9E8D57u, c2, h1, l1);
            const uint32_t n0 = h1 ^ c1 ^ a, n2 = h0 ^ c3 ^ b;
            c0 = n0; c1 = l1; c2 = n2; c3 = l0;
            a += 0x9E3779B9u; b += 0xBB67AE85u;
        }
        out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
    }
};

SP_HD double u53(uint32_t hi, uint32_t lo) {   // uniform in [0,1) with 53 random bits, like NumPy's random_sample
    return (double)((((uint64_t)hi << 32) | lo) >> 11) * (1.0 / 9007199254740992.0);
}

struct BeamSpec { int beam_type, probing_axis; double size_a, size_b, divergence, start; uint64_t seed; };
enum { BEAM_CIRC_FOLD = 0, BEAM_CIRC_POW2 = 1, BEAM_SQUARE = 2, BEAM_RECT = 3, BEAM_LINEAR = 4 };

// Initial state of global ray `idx` in the CALLER's frame: s[0..5] = x,y,z,vx,vy,vz; amp = 1, phase = pol = 0.
// Distributions follow init_beam (full_solver.py:547-835) / Beam.init_beam (beam.py:35-303).
SP_HD void beam_ray(const BeamSpec& B, uint64_t idx, double s[6]) {
    const double C = 299792458.0, PI = 3.14159265358979323846;
    Philox ph; ph.k0 = (uint32_t)B.seed; ph.k1 = (uint32_t)(B.seed >> 32);
    uint32_t r0[4], r1[4], r2[4];
    ph.block((uint32_t)idx, (uint32_t)(idx >> 32), 0u, 0x5eedu, r0);
    ph.block((uint32_t)idx, (uint32_t)(idx >> 32), 1u, 0x5eedu, r1);
    ph.block((uint32_t)idx, (uint32_t)(idx >> 32), 2u, 0x5eedu, r2);
    const double U0 = u53(r0[0], r0[1]), U1 = u53(r0[2], r0[3]), U2 = u53(r1[0], r1[1]);
    const double U3 = u53(r1[2], r1[3]), U4 = u53(r2[0], r2[1]), U5 = u53(r2[2], r2[3]);
    // chi ~ divergence * N(0,1)  (Box-Muller);  phi ~ U[0, pi)
    const double chi = B.divergence * sqrt(-2.0 * log(1.0 - U4)) * cos(2.0 * PI * U5);
    const double phi = PI * U3;
    double a, b;
    double vpar = C * cos(chi), v1 = C * sin(chi) * cos(phi), v2 = C * sin(chi) * sin(phi);
    switch (B.beam_type) {
        case BEAM_CIRC_FOLD: {
            const double t = 2.0 * PI * U0;
            double u = U1 + U2; if (u > 1.0) u = 2.0 - u;
            a = B.size_a * u * cos(t); b = B.size_a * u * sin(t);
        } break;
        case BEAM_CIRC_POW2: {
            const double t = 2.0 * PI * U0, u = sqrt(U1);
            a = B.size_a * u * cos(t); b = B.size_a * u * sin(t);
        } break;
        case BEAM_SQUARE: a = B.size_a * (2.0 * U1 - 1.0); b = B.size_a * (2.0 * U0 - 1.0); break;
        case BEAM_RECT: a = B.size_a * (2.0 * U1 - 1.0); b = B.size_b * (2.0 * U0 - 1.0); break;
        default: /* BEAM_LINEAR: x-z plane only (full_solver.py:707-720) */
            s[0] = B.size_a * (2.0 * U0 - 1.0); s[1] = 0.0; s[2] = B.start;
            s[3] = C * sin(chi); s[4] = 0.0; s[5] = C * cos(chi);
            return;
    }
    if (B.probing_axis == 0) { s[0] = B.start; s[1] = a; s[2] = b; s[3] = vpar; s[4] = v1; s[5] = v2; }
    else if (B.probing_axis == 2) { s[0] = a; s[1] = b; s[2] = B.start; s[3] = v1; s[4] = v2; s[5] = vpar; }
    else { s[0] = a; s[1] = B.start; s[2] = b; s[3] = v1; s[4] = vpar; s[5] = v2; }
}

}  // namespace sp
