/*
 * gf_physics.cuh -- per-point flavor physics of the GolemFlavor log-posterior path,
 * written for one parameter point per CUDA thread with everything in registers.
 *
 * All functions are `__host__ __device__` so that the HOST side of the library can
 * precompute per-model constants (texture matrix, bin factors) with the very same
 * arithmetic; the host never evaluates parameter points -- there is no CPU
 * compute path behind the C ABI.
 *
 * Reference formulas restated here (ShiveshM/GolemFlavor, golemflavor/fr.py):
 *   angles_to_u          fr.py:116-162   (closed-form product R23.R13(dcp).R12)
 *   params_to_BSMu       fr.py:317-400   (H = U M U^+/(2E) + E^(d-3) N S N^+)
 *   cardano_eqn          fr.py:170-237   (eigenvectors of a 3x3 Hermitian matrix)
 *   u_to_fr              fr.py:502-536   (fr_b = sum_ai |U_ai|^2 |U_bi|^2 s_a / sum s)
 *   flux_averaged_BSMu   fr.py:403-458   (bin-width weighted mean, renormalised)
 *   angles_to_fr         fr.py:82-113
 * The reference evaluates these in x87 80-bit arithmetic with a cancellation-prone
 * eigenvector formula.  Here the eigen stage works on the trace-free, norm-scaled
 * matrix: eigenvalues by the trigonometric (Cardano) solution with the cos(phi/3)
 * branch obtained trig-free (fp32-seeded Newton on the cubic), squared eigenvector moduli
 * from the eigenvector-eigenvalue identity, and a cyclic complex Jacobi solver as
 * the fallback whenever two eigenvalues approach each other.
 */
#ifndef GF_PHYSICS_CUH
#define GF_PHYSICS_CUH

#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define GF_HD __host__ __device__ __forceinline__
#define GF_HD_NOINLINE inline __host__ __device__ __noinline__
#else
#define GF_HD inline
#define GF_HD_NOINLINE inline
#endif

/* Developer build only (-DGF_ENS_PROFILE): clock64 stage probes of the sampler's critical path, accumulated by thread 0
 * of block 0 and printed by the cluster kernel.  Compiles to nothing otherwise. */
#if defined(GF_ENS_PROFILE) && defined(__CUDACC__)
static __device__ long long gf_stage_acc[16];
static __device__ long long gf_stage_last;
#endif
#if defined(GF_ENS_PROFILE) && defined(__CUDA_ARCH__)
#define GF_STAGE(i)                                       \
    do {                                                  \
        if (threadIdx.x == 0 && blockIdx.x == 0) {        \
            const long long n_ = clock64();               \
            gf_stage_acc[i] += n_ - gf_stage_last;        \
            gf_stage_last = n_;                           \
        }                                                 \
    } while (0)
#else
#define GF_STAGE(i)
#endif

/* status bits -- must equal GF_ST_* of include/golemflavor_b200.h */
#define GFP_ST_OUT_OF_PRIOR 1u
#define GFP_ST_NON_UNITARY 2u
#define GFP_ST_NON_FINITE 4u
#define GFP_ST_ILL_COND 8u
#define GFP_ST_REFINED 16u

/* The mass-squared differences (~1e-21 GeV^2) and the BSM coupling are multiplied by this
 * exact power of two so that every intermediate of the eigen stage stays far from the
 * subnormal range.  Eigenvectors are invariant under the scaling. */
#define GFP_MASS_SCALE 1180591620717411303424.0 /* 2^70 */

/* sin^2(phi/3) below which the closed-form path hands the bin over to the deflation refinement: the closed form loses
 * accuracy like eps/relgap^2, the refinement like eps/relgap (relgap = closest pair's splitting / spectral spread =
 * (2/sqrt(3)) sin(phi/3) for a close pair).  4.7e-6 is relgap 2.5e-3, where the closed form's worst |V|^2 error over
 * 1e6 Haar-random spectra is 3.8e-11; at the former 1.4e-6 (relgap 1.37e-3) it was 1.29e-10, above the 1e-10
 * tolerance on fr (tests/test_eigen_conditioning.py::test_harness_closed_form_error_at_the_fast_path_cut). */
#ifndef GFP_FAST_MIN_SIN2
#define GFP_FAST_MIN_SIN2 4.7e-6
#endif
#define GFP_ILL_GAP 1e-6

/* High 32-bit word of a positive, normal double at compile time (exact: scaling by two and the mantissa's top 20 bits
 * are exact operations).  The device compares sin^2(phi/3) with the threshold on this word. */
constexpr unsigned gfp_hiword_pos(double x) {
    int e = 0;
    while (x >= 2.0) { x *= 0.5; ++e; }
    while (x < 1.0) { x *= 2.0; --e; }
    return ((unsigned)(e + 1023) << 20) | (unsigned)((x - 1.0) * 1048576.0);
}
constexpr unsigned GFP_FAST_MIN_SIN2_HI = gfp_hiword_pos(GFP_FAST_MIN_SIN2);
static_assert(GFP_FAST_MIN_SIN2_HI > 0x00100000u && GFP_FAST_MIN_SIN2_HI < 0x7FF00000u, "the fast-path threshold must be positive and finite");

/* ------------------------------------------------------------------ fast fp64 helpers */

/* 1/x for normal, finite x (device: MUFU.RCP64H seed, ~2^-20, + one cubic step: e' ~ e^3). */
GF_HD double gfp_rcp(double x) {
#ifdef __CUDA_ARCH__
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    const double e = fma(-x, y, 1.0);
    return fma(y, fma(e, e, e), y);
#else
    return 1.0 / x;
#endif
}

/* 1/sqrt(x) for normal, finite x > 0 (device: MUFU.RSQ64H seed + one cubic step
 * y (1 + e/2 + 3 e^2/8), e = 1 - x y^2: e' ~ 5/16 e^3). */
GF_HD double gfp_rsqrt(double x) {
#ifdef __CUDA_ARCH__
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    const double e = fma(-x * y, y, 1.0);
    return fma(y * e, fma(0.375, e, 0.5), y);
#else
    return 1.0 / sqrt(x);
#endif
}

/* sqrt(x) for the mixing-angle coordinates (x in [0, 1] inside the prior box): x * rsqrt(x), one
 * multiplication on top of the MUFU-seeded rsqrt instead of the ~12 fp64 instructions of the IEEE
 * routine; accurate to ~1 ulp.  Zero, tiny and out-of-domain arguments take the library path
 * (negative -> NaN like the reference's sqrt, fr.py:146-152). */
#ifdef __CUDACC__
/* the IEEE routine, out of line: its inlined body (Newton steps, a scaling branch, a call of its own) put two levels of
 * divergence bookkeeping around every gfp_sqrt01 */
static __device__ __noinline__ double gfp_sqrt_lib(double x) { return sqrt(x); }
#endif

GF_HD double gfp_sqrt01(double x) {
#ifdef __CUDA_ARCH__
    /* 1e-290 < x < 1e290 tested on the exponent field with integer instructions (two fp64 compares would
     * sit on the pipe every kernel here is bound by): the unsigned subtraction sends negative numbers,
     * zeros, subnormals, infinities and NaNs to the library path in one comparison.  The fast value is computed
     * unconditionally (garbage, never a trap, outside the range) and replaced on the rare path: the common path is the
     * fall-through and pays one predicated branch. */
    const unsigned hi = (unsigned)__double2hiint(x);
    double r = x * gfp_rsqrt(x);
    if (!(hi - 0x03D00000u < 0x7C200000u - 0x03D00000u)) r = gfp_sqrt_lib(x); /* outside 2^-962 <= x < 2^963 */
    return r;
#else
    return sqrt(x);
#endif
}

/*
 * sin / cos of the CP phase.  The library routines fetch their polynomial coefficients from a table in
 * global memory (LDG): harmless in the throughput kernels, but a ~300-cycle stall on the critical path of
 * the ensemble sampler, which runs about one warp per SM.  Same algorithm with immediate coefficients:
 * Cody-Waite reduction by pi/2 in three parts, then the fdlibm minimax polynomials on [-pi/4, pi/4]
 * (|error| < 1 ulp of the result scale).  |x| >= 1e5 or non-finite arguments -- never inside a prior box --
 * take the library routine.
 */
#define GFP_S1 -1.66666666666666324348e-01
#define GFP_S2 8.33333333332248946124e-03
#define GFP_S3 -1.98412698298579493134e-04
#define GFP_S4 2.75573137070700676789e-06
#define GFP_S5 -2.50507602534068634195e-08
#define GFP_S6 1.58969099521155010221e-10
#define GFP_C1 4.16666666666666019037e-02
#define GFP_C2 -1.38888888888741095749e-03
#define GFP_C3 2.48015872894767294178e-05
#define GFP_C4 -2.75573143513906633035e-07
#define GFP_C5 2.08757232129817482790e-09
#define GFP_C6 -1.13596475577881948265e-11

#ifdef __CUDACC__
/* 2/pi and the three-part split of -pi/2 (1.5707963267948966 + 6.123233995736757e-17 + 8.478427660368898e-32), in constant
 * memory: a 64-bit literal costs two moves per use, a constant-bank word is a direct DFMA operand */
static __constant__ double gfp_pio2_tab[4] = {0.63661977236758138, -1.5707963267948966, -6.123233995736757e-17, -8.478427660368898e-32};
#endif
#ifdef __CUDA_ARCH__
/* r = x - k pi/2 with k = rint(x 2/pi); returns k */
__device__ __forceinline__ int gfp_reduce_pio2(double x, double& r) {
    const double kd = rint(x * gfp_pio2_tab[0]);
    r = fma(kd, gfp_pio2_tab[1], x);
    r = fma(kd, gfp_pio2_tab[2], r);
    r = fma(kd, gfp_pio2_tab[3], r);
    return (int)kd;
}
#endif

#ifdef __CUDACC__
/* Horner coefficients of gfp_cos by quadrant parity (row 0: cos r = 1 + z (-1/2 + z (C1 + ... + z C6)); row 1:
 * sin r = r + r z (S1 + ... + z S6), led by a zero so that both rows take the same seven steps).  In constant memory
 * the row is picked by ONE index: seven LDC.64 instead of fourteen FSEL plus the moves that materialise both
 * coefficient sets -- a twentieth of the SM-only kernel's instructions. */
static __constant__ double gfp_cos_tab[2][8] = {{GFP_C6, GFP_C5, GFP_C4, GFP_C3, GFP_C2, GFP_C1, -0.5, 0.0},
                                                {0.0, GFP_S6, GFP_S5, GFP_S4, GFP_S3, GFP_S2, GFP_S1, 0.0}};
#endif

GF_HD void gfp_sincos(double x, double* sn, double* cs) {
#ifdef __CUDA_ARCH__
    if (!(fabs(x) < 1e5)) {
        sincos(x, sn, cs);
        return;
    }
    double r;
    const int k = gfp_reduce_pio2(x, r);
    const double z = r * r;
    /* coefficients as constant-bank operands (gfp_cos_tab, compile-time indices): a 64-bit literal is two moves per use */
    const double* __restrict__ kc = gfp_cos_tab[0];
    const double* __restrict__ ks = gfp_cos_tab[1];
    const double ps = fma(fma(fma(fma(fma(ks[1], z, ks[2]), z, ks[3]), z, ks[4]), z, ks[5]), z, ks[6]);
    const double pc = fma(fma(fma(fma(fma(kc[0], z, kc[1]), z, kc[2]), z, kc[3]), z, kc[4]), z, kc[5]);
    const double s = fma(r * z, ps, r);
    const double c = fma(z, fma(z, pc, -0.5), 1.0);
    /* quadrant: (sin, cos)(x) = (s, c), (c, -s), (-s, -c), (-c, s) for k mod 4 = 0..3 */
    const double a = (k & 1) ? c : s, b = (k & 1) ? s : c;
    *sn = (k & 2) ? -a : a;
    *cs = ((k + 1) & 2) ? -b : b;
#else
    *sn = sin(x);
    *cs = cos(x);
#endif
}

GF_HD double gfp_cos(double x) {
#ifdef __CUDA_ARCH__
    if (!(fabs(x) < 1e5)) return cos(x);
    double r;
    const int k = gfp_reduce_pio2(x, r);
    const double z = r * r;
    const bool odd = k & 1;
    const double* __restrict__ c = gfp_cos_tab[k & 1];
    double p = c[0];
    p = fma(p, z, c[1]);
    p = fma(p, z, c[2]);
    p = fma(p, z, c[3]);
    p = fma(p, z, c[4]);
    p = fma(p, z, c[5]);
    p = fma(p, z, c[6]);
    const double v = fma(odd ? r * z : z, p, odd ? r : 1.0);
    /* cos x = c, -s, -c, s for k mod 4 = 0..3 */
    return ((k + 1) & 2) ? -v : v;
#else
    return cos(x);
#endif
}

/* ln(x) for positive, normal, finite x (the sampler's ln z and ln u): the fdlibm algorithm (x = 2^k m,
 * m in [sqrt(1/2), sqrt(2)), s = f / (2 + f), ln m = f - f^2/2 + s (f^2/2 + R(s^2))), < 1 ulp, with the
 * MUFU-seeded reciprocal instead of the division and no special-case branches -- about two thirds of the
 * library routine's instructions on the sampler's critical path. */
GF_HD double gfp_log_pos(double x) {
#ifdef __CUDA_ARCH__
    int hx = __double2hiint(x);
    int k = (hx >> 20) - 1023;
    hx &= 0x000fffff;
    const int i = (hx + 0x95f64) & 0x100000;
    const double m = __hiloint2double(hx | (i ^ 0x3ff00000), __double2loint(x));
    k += i >> 20;
    const double dk = (double)k;
    const double f = m - 1.0;
    const double s = f * gfp_rcp(2.0 + f);
    const double z = s * s, w = z * z;
    const double t1 = w * fma(w, fma(w, 1.531383769920937332e-01, 2.222219843214978396e-01), 3.999999999940941908e-01);
    const double t2 = z * fma(w, fma(w, fma(w, 1.479819860511658591e-01, 1.818357216161805012e-01), 2.857142874366239149e-01), 6.666666666666735130e-01);
    const double R = t2 + t1;
    const double hfsq = 0.5 * f * f;
    return dk * 6.93147180369123816490e-01 - ((hfsq - fma(s, hfsq + R, dk * 1.90821492927058770002e-10)) - f);
#else
    return log(x);
#endif
}

/* ------------------------------------------------------------------ 3x3 Hermitian */

/* Hermitian matrix: real diagonal d0,d1,d2 and the upper triangle a = H01, b = H02, c = H12. */
struct gfp_herm3 {
    double d0, d1, d2;
    double ar, ai, br, bi, cr, ci;
};

/*
 * w = 1 - cos(phi/3): the smallest root of g(w) = 4w^3 - 12w^2 + 9w - delta with delta = 1 - |cos(phi)|
 * in [0, 1] (w in [0, 0.134]).  This replaces acos + cos of the reference's trigonometric root formula
 * (fr.py:216-221) and keeps full RELATIVE accuracy of w as delta -> 0 (near-degenerate pairs).
 *
 * The fp64 pipe is the bottleneck of every kernel here while the fp32 pipe idles, so the root is
 * SEEDED in single precision -- a degree-6 polynomial for w/delta (Chebyshev fit in t = 2 delta - 1,
 * scratch/fit_w32.py, relative error 3.4e-7) and the reciprocal slope r ~ 1/g'(w0) -- and polished in fp64
 * with the frozen slope, w <- w - r g(w).  Error recursion e' = e (1 - r g') + O(e^2): 3.4e-7 -> 1e-13
 * -> 2e-20 relative.  ONE step is taken by default: 1e-13 RELATIVE error of w means 5e-14 relative error
 * of the eigenvalue gap at every gap size (an absolute error far below one ulp of the matrix scale once the
 * pair is close), i.e. ~1e-13 on |V|^2 -- three orders inside the 1e-10 tolerance and below the closed form's
 * own conditioning error (parity at scale unchanged at ~3e-12 worst) -- and the second step is 4 of the 83
 * fp64 instructions of an energy bin (K2 0.596 -> 0.578 ms).  GFP_CUBIC_NEWTON_STEPS=2 restores it.
 */
#ifndef GFP_CUBIC_NEWTON_STEPS
#define GFP_CUBIC_NEWTON_STEPS 1
#endif
GF_HD double gfp_cubic_w(double delta) {
    const float d = (float)delta;
    const float t = fmaf(2.0f, d, -1.0f);
    float p = 6.536684850e-06f;
    p = fmaf(p, t, 2.486253834e-05f);
    p = fmaf(p, t, 8.752417489e-05f);
    p = fmaf(p, t, 3.777995007e-04f);
    p = fmaf(p, t, 1.834025956e-03f);
    p = fmaf(p, t, 1.102905069e-02f);
    p = fmaf(p, t, 1.206147596e-01f);
    const float w0 = d * p;
    const float slope = fmaf(fmaf(12.0f, w0, -24.0f), w0, 9.0f); /* g'(w0) in [6, 9] */
#ifdef __CUDA_ARCH__
    float rf;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rf) : "f"(slope));
#else
    const float rf = 1.0f / slope;
#endif
    const double r = (double)rf;
    double w = (double)w0;
    w = fma(-r, fma(fma(fma(4.0, w, -12.0), w, 9.0), w, -delta), w);
#if GFP_CUBIC_NEWTON_STEPS > 1
    w = fma(-r, fma(fma(fma(4.0, w, -12.0), w, 9.0), w, -delta), w);
#endif
    return w;
}

/* The four independent entries of the doubly stochastic matrix |V_ai|^2:
 * x00 = |V_00|^2, x01 = |V_01|^2, x10 = |V_10|^2, x11 = |V_11|^2 (rows = flavors e, mu; columns =
 * the isolated eigenvalue and the upper member of the remaining pair). */
struct gfp_x4 {
    double x00, x01, x10, x11;
};

/*
 * Closed-form |V_ai|^2 from the invariants of a TRACE-FREE Hermitian 3x3 matrix: diagonal entries e0, e1, the
 * diagonal COFACTORS k0 = e1 e2 - |H12|^2, k1 = e0 e2 - |H02|^2, Q = tr(H^2)/6 and det H.
 * Eigenvalues 2 sqrt(Q) cos((phi + 2 pi k)/3) with cos(phi) = det / (2 Q^(3/2)); squared eigenvector moduli from
 * the eigenvector-eigenvalue identity |V_ai|^2 p'(l_i) = det(l_i - M_a) (M_a = 2x2 principal minor).  With
 * e0 + e1 + e2 = 0 the minor determinants are (l - e1)(l - e2) - |H12|^2 = l (l + e0) + k0 and
 * (l - e0)(l - e2) - |H02|^2 = l (l + e1) + k1: one addition and one FMA each, and neither e2 nor the squared
 * off-diagonal moduli are needed per matrix.  Returns false -- the caller then discards `out` -- when the closest
 * eigenvalue pair is nearer than the fast-path limit or the input is degenerate / non-finite; the caller then
 * runs the deflation fallback.
 */
GF_HD bool gfp_eig_core(double e0, double e1, double k0, double k1, double Q, double hdet, gfp_x4& out) {
    /* hdet = det / 2.  Straight-line code on purpose (no early exit): the caller evaluates two energy
     * bins back to back and the compiler interleaves their independent dependency chains -- with 16
     * resident warps per SM the kernels are bound by the latency of this chain.  Degenerate or
     * non-finite inputs simply produce garbage that the returned flag tells the caller to discard. */
    const double rs = gfp_rsqrt(Q);
    const double r = (hdet * rs) * (rs * rs); /* cos(phi) */
    const double delta = 1.0 - fabs(r);       /* a rounding-negative delta gives s2 < 0 and takes the fallback */
    const double w = gfp_cubic_w(delta);
    const double s2 = w * (2.0 - w); /* sin^2(phi/3) */
    const double sq = 2.0 * Q * rs;                     /* 2 sqrt(Q) */
    const double l0 = copysign(sq - sq * w, r);         /* 2 sqrt(Q) cos(phi/3), isolated eigenvalue */
    const double half_gap = (0.8660254037844386 * sq) * (s2 * gfp_rsqrt(s2));
    const double l1 = fma(-0.5, l0, half_gap);
    /* eigenvector-eigenvalue identity for rows a = 0, 1; for the trace-free cubic p'(l) = 3 (l^2 - Q): no third
     * minor, and the operands stay register-light (a DFMA reading three distinct register pairs issues at 2/3
     * rate on B200) */
    const double n00 = fma(l0, l0 + e0, k0), n10 = fma(l0, l0 + e1, k1);
    const double n01 = fma(l1, l1 + e0, k0), n11 = fma(l1, l1 + e1, k1);
    const double p0 = fma(l0, l0, -Q), p1 = fma(l1, l1, -Q); /* p'(l_i) / 3 */
    const double q = gfp_rcp(3.0 * (p0 * p1));
    const double i0 = q * p1, i1 = q * p0;
    out.x00 = n00 * i0;
    out.x10 = n10 * i0;
    out.x01 = n01 * i1;
    out.x11 = n11 * i1;
    /* Q > tiny also rejects NaN; s2 >= limit rejects close pairs, NaN and negative round-off.  On the device
     * both tests read the exponent fields with integer instructions (unsigned range checks: positive, finite,
     * above the threshold's high word) instead of two compares on the fp64 pipe.  The high word ignores the low 32 bits
     * of the threshold: the device's cut sits at most 2^-20 relative below the host's. */
#if defined(__CUDA_ARCH__)
    const unsigned hq = (unsigned)__double2hiint(Q), hs = (unsigned)__double2hiint(s2);
    return (hq - 0x05E00000u < 0x7FF00000u - 0x05E00000u) && (hs - GFP_FAST_MIN_SIN2_HI < 0x7FF00000u - GFP_FAST_MIN_SIN2_HI); /* Q > ~1e-280, s2 >= GFP_FAST_MIN_SIN2 */
#else
    return (Q > 1e-280) && (s2 >= GFP_FAST_MIN_SIN2);
#endif
}

/* Invariants of one matrix computed directly (single-matrix entry points and tests). */
GF_HD bool gfp_herm3_x4_fast(const gfp_herm3& h, gfp_x4& out) {
    const double mu = (h.d0 + h.d1 + h.d2) * (1.0 / 3.0);
    const double e0 = h.d0 - mu, e1 = h.d1 - mu, e2 = h.d2 - mu;
    const double a2 = fma(h.ar, h.ar, h.ai * h.ai);
    const double b2 = fma(h.br, h.br, h.bi * h.bi);
    const double c2 = fma(h.cr, h.cr, h.ci * h.ci);
    const double p2 = fma(2.0, a2 + b2 + c2, fma(e0, e0, fma(e1, e1, e2 * e2)));
    /* det = e0 e1 e2 + 2 Re(a c conj(b)) - e0 |c|^2 - e1 |b|^2 - e2 |a|^2 */
    const double acr = fma(h.ar, h.cr, -(h.ai * h.ci));
    const double aci = fma(h.ar, h.ci, h.ai * h.cr);
    const double tri = fma(acr, h.br, aci * h.bi);
    const double det = fma(2.0, tri, e0 * e1 * e2) - fma(e0, c2, fma(e1, b2, e2 * a2));
    return gfp_eig_core(e0, e1, fma(e1, e2, -c2), fma(e0, e2, -b2), p2 * (1.0 / 6.0), 0.5 * det, out);
}

/*
 * The matrix pencil H(rho) = H0 + rho T of the energy-bin loop (fr.py:441-452: only the scalar
 * rho = 10^logLam * 2 E^(d-2) changes from bin to bin).  Every invariant gfp_eig_core needs is a
 * polynomial in rho -- the trace-free diagonal (degree 1), the diagonal cofactors and Q (degree 2), the
 * determinant (degree 3) -- so a bin costs 11 FMAs for the invariants instead of rebuilding the matrix and
 * its determinant.  The coefficients split into a part that depends on T alone (gfp_pencil_T: a
 * model constant for the fixed textures, then read straight from the constant bank) and a per-point
 * part (gfp_pencil_P).
 */
struct gfp_pencil_T {
    double te[3];        /* trace-free diagonal of T                                              */
    double kt0, kt1;     /* diagonal cofactors of T': te1 te2 - |T12|^2, te0 te2 - |T02|^2         */
    double q2, d3;       /* tr(T'^2)/6, det(T')/2                                                 */
};
struct gfp_pencil_P {
    double e[2];                 /* trace-free diagonal of H0: e_k(rho) = e[k] + rho te[k], k = 0, 1   */
    double k0[2], k1[2];         /* cofactors: k_a(rho) = k_a[0] + rho (k_a[1] + rho kt_a)             */
    double q[2];                 /* Q(rho) = q[0] + rho (q[1] + rho q2)                                */
    double d[3];                 /* det(rho)/2 = d[0] + rho (d[1] + rho (d[2] + rho d3))               */
};

/* Adjugate of a trace-free Hermitian matrix A = (ea, A.offdiag): real diagonal cofactors k and the
 * upper triangle j01, j02, j12.  For the fixed textures adj(T') is a model constant (host). */
struct gfp_adj3 {
    double k0, k1, k2;
    double j01r, j01i, j02r, j02i, j12r, j12i;
};

GF_HD gfp_adj3 gfp_adj_tf(const double* ea, const gfp_herm3& A) {
    gfp_adj3 j;
    const double a2 = fma(A.ar, A.ar, A.ai * A.ai), b2 = fma(A.br, A.br, A.bi * A.bi), c2 = fma(A.cr, A.cr, A.ci * A.ci);
    j.k0 = fma(ea[1], ea[2], -c2); j.k1 = fma(ea[0], ea[2], -b2); j.k2 = fma(ea[0], ea[1], -a2);
    /* adj_01 = b conj(c) - a e2 ; adj_02 = a c - b e1 ; adj_12 = conj(a) b - e0 c */
    j.j01r = fma(A.br, A.cr, A.bi * A.ci) - A.ar * ea[2]; j.j01i = fma(A.bi, A.cr, -(A.br * A.ci)) - A.ai * ea[2];
    j.j02r = fma(A.ar, A.cr, -(A.ai * A.ci)) - A.br * ea[1]; j.j02i = fma(A.ar, A.ci, A.ai * A.cr) - A.bi * ea[1];
    j.j12r = fma(A.ar, A.br, A.ai * A.bi) - ea[0] * A.cr; j.j12i = fma(A.ar, A.bi, -(A.ai * A.br)) - ea[0] * A.ci;
    return j;
}

/* tr(adj(A) B) = sum_i k_i B_ii + 2 Re(adj_01 conj(B_01) + adj_02 conj(B_02) + adj_12 conj(B_12)): the
 * coefficient of rho in det(A + rho B) for trace-free Hermitian A, B = (eb, B.offdiag). */
GF_HD double gfp_tr_adj_pre(const gfp_adj3& j, const double* eb, const gfp_herm3& B) {
    const double off = fma(j.j01r, B.ar, j.j01i * B.ai) + fma(j.j02r, B.br, j.j02i * B.bi) + fma(j.j12r, B.cr, j.j12i * B.ci);
    return fma(2.0, off, fma(j.k0, eb[0], fma(j.k1, eb[1], j.k2 * eb[2])));
}

/* Q = tr(H'^2)/6 and det(H')/2 of a Hermitian matrix with eigenvalues (0, m1, m2): they depend on the
 * spectrum alone, not on the mixing -- for H0 = U diag(0, m21, m3x) U^+ on the mass-squared differences
 * only, for T = N diag(0, 1/100, 1) N^+ they are constants of the model whatever the NP angles. */
GF_HD void gfp_spectrum_invariants(double m1, double m2, double& q, double& hdet) {
    const double mu = (m1 + m2) * (1.0 / 3.0);
    const double l0 = -mu, l1 = m1 - mu, l2 = m2 - mu;
    q = (1.0 / 6.0) * fma(l0, l0, fma(l1, l1, l2 * l2));
    hdet = 0.5 * (l0 * l1 * l2);
}

#define GFP_T_EIG1 0.01 /* sc1 = sc2 / 100, fr.py:381 */
#define GFP_T_EIG2 1.0

GF_HD gfp_pencil_T gfp_make_pencil_T(const gfp_herm3& T) {
    gfp_pencil_T t;
    const double mut = (T.d0 + T.d1 + T.d2) * (1.0 / 3.0);
    t.te[0] = T.d0 - mut; t.te[1] = T.d1 - mut; t.te[2] = T.d2 - mut;
    t.kt0 = fma(t.te[1], t.te[2], -fma(T.cr, T.cr, T.ci * T.ci));
    t.kt1 = fma(t.te[0], t.te[2], -fma(T.br, T.br, T.bi * T.bi));
    gfp_spectrum_invariants(GFP_T_EIG1, GFP_T_EIG2, t.q2, t.d3);
    return t;
}

/* h0 = U diag(0, m1, m2) U^+ (its spectrum-only invariants come from m1, m2), T with trace-free diagonal
 * te; adjT = gfp_adj_tf(te, T) (a constant for the fixed textures). */
GF_HD gfp_pencil_P gfp_make_pencil_P(const gfp_herm3& h0, double m1, double m2, const gfp_herm3& T, const double* te, const gfp_adj3& adjT) {
    gfp_pencil_P p;
    const double mu0 = (h0.d0 + h0.d1 + h0.d2) * (1.0 / 3.0);
    const double pe[3] = {h0.d0 - mu0, h0.d1 - mu0, h0.d2 - mu0};
    p.e[0] = pe[0]; p.e[1] = pe[1];
    /* rho-linear coefficients of |H01|^2, |H02|^2, |H12|^2: 2 Re(H0_ab conj(T_ab)) */
    const double a21 = 2.0 * fma(h0.ar, T.ar, h0.ai * T.ai);
    const double b21 = 2.0 * fma(h0.br, T.br, h0.bi * T.bi);
    const double c21 = 2.0 * fma(h0.cr, T.cr, h0.ci * T.ci);
    const gfp_adj3 adjH = gfp_adj_tf(pe, h0);
    /* diagonal cofactors e1 e2 - |H12|^2 and e0 e2 - |H02|^2 of H0' + rho T': the constant terms are those of adj(H0'),
     * the rho^2 terms those of adj(T') (gfp_pencil_T / the model constant adjT) */
    p.k0[0] = adjH.k0; p.k0[1] = fma(pe[1], te[2], fma(pe[2], te[1], -c21));
    p.k1[0] = adjH.k1; p.k1[1] = fma(pe[0], te[2], fma(pe[2], te[0], -b21));
    gfp_spectrum_invariants(m1, m2, p.q[0], p.d[0]);
    p.q[1] = (1.0 / 6.0) * fma(2.0, a21 + b21 + c21, 2.0 * fma(pe[0], te[0], fma(pe[1], te[1], pe[2] * te[2])));
    p.d[1] = 0.5 * gfp_tr_adj_pre(adjH, te, T);
    p.d[2] = 0.5 * gfp_tr_adj_pre(adjT, pe, h0);
    return p;
}

GF_HD bool gfp_pencil_x4_fast(const gfp_pencil_P& p, const gfp_pencil_T& t, double rho, gfp_x4& out) {
    const double e0 = fma(rho, t.te[0], p.e[0]), e1 = fma(rho, t.te[1], p.e[1]);
    const double k0 = fma(fma(t.kt0, rho, p.k0[1]), rho, p.k0[0]);
    const double k1 = fma(fma(t.kt1, rho, p.k1[1]), rho, p.k1[0]);
    const double Q = fma(fma(t.q2, rho, p.q[1]), rho, p.q[0]);
    const double hdet = fma(fma(fma(t.d3, rho, p.d[2]), rho, p.d[1]), rho, p.d[0]);
    return gfp_eig_core(e0, e1, k0, k1, Q, hdet, out);
}

/*
 * Cyclic Jacobi eigensolver for a complex Hermitian 3x3 matrix (the refinement / fallback
 * stage).  On return lam[i] are the eigenvalues (unsorted) and V = (vr + i vi)[3*a + i] the
 * eigenvector matrix (columns = eigenvectors).  Accuracy eps*|H| for eigenvalues and
 * eps/gap for eigenvectors.  Returns the smallest eigenvalue gap divided by the spectral
 * spread (0 for an exactly degenerate input).
 */
GF_HD_NOINLINE double gfp_herm3_jacobi(const gfp_herm3& h, double* lam, double* vr, double* vi) {
    double hr[9], hi[9];
    /* scale the largest entry into [1, 2) by an EXACT power of two 2^-ex taken from its exponent (subnormals included):
     * the squares of the rotations can then neither overflow nor underflow at any input scale, the eigenvectors are
     * the same bits at every power-of-two scale, and the eigenvalues are rescaled exactly.  A reciprocal of the
     * largest entry would overflow for a subnormal one and round the entries.  Non-finite input is not scaled
     * (ex = 0) and comes out non-finite. */
    double mx = fmax(fmax(fabs(h.d0), fabs(h.d1)), fabs(h.d2));
    mx = fmax(mx, fmax(fmax(fabs(h.ar), fabs(h.ai)), fmax(fmax(fabs(h.br), fabs(h.bi)), fmax(fabs(h.cr), fabs(h.ci)))));
    const int ex = (mx > 0.0 && mx <= 1.7976931348623157e308) ? ilogb(mx) : 0;
    hr[0] = scalbn(h.d0, -ex); hi[0] = 0.0;
    hr[4] = scalbn(h.d1, -ex); hi[4] = 0.0;
    hr[8] = scalbn(h.d2, -ex); hi[8] = 0.0;
    hr[1] = scalbn(h.ar, -ex); hi[1] = scalbn(h.ai, -ex); hr[3] = hr[1]; hi[3] = -hi[1];
    hr[2] = scalbn(h.br, -ex); hi[2] = scalbn(h.bi, -ex); hr[6] = hr[2]; hi[6] = -hi[2];
    hr[5] = scalbn(h.cr, -ex); hi[5] = scalbn(h.ci, -ex); hr[7] = hr[5]; hi[7] = -hi[5];
    for (int k = 0; k < 9; ++k) { vr[k] = (k % 4 == 0) ? 1.0 : 0.0; vi[k] = 0.0; }

    for (int sweep = 0; sweep < 24; ++sweep) {
        const double off = hr[1] * hr[1] + hi[1] * hi[1] + hr[2] * hr[2] + hi[2] * hi[2] + hr[5] * hr[5] + hi[5] * hi[5];
        if (!(off > 1e-40)) break; /* also leaves on NaN */
        for (int pair = 0; pair < 3; ++pair) {
            const int p = (pair == 2) ? 1 : 0;
            const int q = (pair == 0) ? 1 : 2;
            const int r = 3 - p - q;
            const double xr = hr[3 * p + q], xi = hi[3 * p + q];
            const double ah2 = xr * xr + xi * xi;
            if (!(ah2 > 1e-300)) continue;
            const double ah = sqrt(ah2);
            const double er = xr / ah, ei = xi / ah; /* e^{i phi} = H_pq / |H_pq| */
            const double tau = (hr[4 * q] - hr[4 * p]) / (2.0 * ah);
            const double t = (tau >= 0.0 ? 1.0 : -1.0) / (fabs(tau) + sqrt(fma(tau, tau, 1.0)));
            const double c = 1.0 / sqrt(fma(t, t, 1.0));
            const double s = t * c;
            /* G = [[c, s], [-s e^{-i phi}, c e^{-i phi}]] on (p,q);  H <- G^+ H G */
            hr[4 * p] -= t * ah;
            hr[4 * q] += t * ah;
            hr[3 * p + q] = hi[3 * p + q] = hr[3 * q + p] = hi[3 * q + p] = 0.0;
            /* third index r: H'_rp = c H_rp - s e^{-i phi} H_rq ; H'_rq = s H_rp + c e^{-i phi} H_rq */
            {
                const double rpr = hr[3 * r + p], rpi = hi[3 * r + p];
                const double rqr = hr[3 * r + q], rqi = hi[3 * r + q];
                /* e^{-i phi} H_rq */
                const double wr = er * rqr + ei * rqi, wi = er * rqi - ei * rqr;
                const double npr = c * rpr - s * wr, npi = c * rpi - s * wi;
                const double nqr = s * rpr + c * wr, nqi = s * rpi + c * wi;
                hr[3 * r + p] = npr; hi[3 * r + p] = npi; hr[3 * p + r] = npr; hi[3 * p + r] = -npi;
                hr[3 * r + q] = nqr; hi[3 * r + q] = nqi; hr[3 * q + r] = nqr; hi[3 * q + r] = -nqi;
            }
            /* V <- V G */
            for (int k = 0; k < 3; ++k) {
                const double kpr = vr[3 * k + p], kpi = vi[3 * k + p];
                const double kqr = vr[3 * k + q], kqi = vi[3 * k + q];
                const double wr = er * kqr + ei * kqi, wi = er * kqi - ei * kqr;
                vr[3 * k + p] = c * kpr - s * wr; vi[3 * k + p] = c * kpi - s * wi;
                vr[3 * k + q] = s * kpr + c * wr; vi[3 * k + q] = s * kpi + c * wi;
            }
        }
    }
    const double l0 = hr[0], l1 = hr[4], l2 = hr[8];
    lam[0] = scalbn(l0, ex); lam[1] = scalbn(l1, ex); lam[2] = scalbn(l2, ex);
    const double g01 = fabs(l0 - l1), g02 = fabs(l0 - l2), g12 = fabs(l1 - l2);
    const double spread = fmax(g01, fmax(g02, g12));
    const double gmin = fmin(g01, fmin(g02, g12));
    return spread > 0.0 ? gmin / spread : 0.0;
}

/*
 * Refinement of a near-degenerate eigenvalue pair by DEFLATION (single matrix).
 *
 * The closed form loses accuracy like eps/gap^2 when two eigenvalues approach each other -- through the
 * characteristic polynomial, whose close roots are ill-conditioned in its coefficients.  The ISOLATED
 * eigenvalue l0 and its eigenvector stay well-conditioned, so the matrix itself is used for the pair:
 *   A = H' - l0, adj(A) = p'(l0) v0 v0^+  (exact for the exact l0)  =>  W = v0 v0^+ = adj(A) / tr adj(A);
 *   with m = -l0/2 the pair's midpoint, F = (H' - m) - (3/2) l0 W = h (v1 v1^+ - v2 v2^+),
 *   h^2 = tr(F^2)/2 (half the pair's splitting), and on the diagonal F_aa = h (|V_a1|^2 - |V_a2|^2).
 * Every entry of F is a difference of O(|H|) terms formed once, so |V_a1|^2, |V_a2|^2 come out with error
 * eps |H| / h -- the conditioning of the eigenvectors themselves, which is also what Jacobi delivers, at
 * ~150 instead of several thousand fp64 operations and without loops or local-memory arrays.
 * Returns status bits; GFP_ST_NON_FINITE asks the caller for the Jacobi solver (degenerate scale, NaN).
 */
GF_HD unsigned gfp_herm3_x4_deflate(const gfp_herm3& h, gfp_x4& out) {
    const double mu = (h.d0 + h.d1 + h.d2) * (1.0 / 3.0);
    const double e0 = h.d0 - mu, e1 = h.d1 - mu, e2 = h.d2 - mu;
    const double a2 = fma(h.ar, h.ar, h.ai * h.ai), b2 = fma(h.br, h.br, h.bi * h.bi), c2 = fma(h.cr, h.cr, h.ci * h.ci);
    const double Q = (1.0 / 6.0) * fma(2.0, a2 + b2 + c2, fma(e0, e0, fma(e1, e1, e2 * e2)));
    if (!(Q > 1e-280 && Q < 1e280)) return GFP_ST_NON_FINITE;
    const double acr = fma(h.ar, h.cr, -(h.ai * h.ci)), aci = fma(h.ar, h.ci, h.ai * h.cr);
    const double tri = fma(acr, h.br, aci * h.bi);
    const double hdet = 0.5 * (fma(2.0, tri, e0 * e1 * e2) - fma(e0, c2, fma(e1, b2, e2 * a2)));
    const double rs = gfp_rsqrt(Q);
    const double r = (hdet * rs) * (rs * rs);
    const double delta = fmax(1.0 - fabs(r), 0.0);
    const double w = gfp_cubic_w(delta);
    const double sq = 2.0 * Q * rs;
    const double l0 = copysign(sq - sq * w, r); /* isolated eigenvalue, absolute error ~ eps sqrt(Q) */
    /* adj(H' - l0): real diagonal cofactors and the upper triangle */
    const double g0 = e0 - l0, g1 = e1 - l0, g2 = e2 - l0;
    const double k0 = fma(g1, g2, -c2), k1 = fma(g0, g2, -b2), k2 = fma(g0, g1, -a2);
    const double j01r = fma(h.br, h.cr, h.bi * h.ci) - h.ar * g2, j01i = fma(h.bi, h.cr, -(h.br * h.ci)) - h.ai * g2;
    const double j02r = acr - h.br * g1, j02i = aci - h.bi * g1;
    const double j12r = fma(h.ar, h.br, h.ai * h.bi) - g0 * h.cr, j12i = fma(h.ar, h.bi, -(h.ai * h.br)) - g0 * h.ci;
    const double ip = gfp_rcp(k0 + k1 + k2); /* tr adj = p'(l0) = (l0 - l1)(l0 - l2) in [6 Q, 9 Q] */
    const double t = 1.5 * l0 * ip;
    const double m = -0.5 * l0;
    /* F = (H' - m) - (3/2) l0 W */
    const double n0 = fma(-t, k0, e0 - m), n1 = fma(-t, k1, e1 - m), n2 = fma(-t, k2, e2 - m);
    const double f01r = fma(-t, j01r, h.ar), f01i = fma(-t, j01i, h.ai);
    const double f02r = fma(-t, j02r, h.br), f02i = fma(-t, j02i, h.bi);
    const double f12r = fma(-t, j12r, h.cr), f12i = fma(-t, j12i, h.ci);
    const double h2 = fma(0.5, fma(n0, n0, fma(n1, n1, n2 * n2)),
                          fma(f01r, f01r, f01i * f01i) + fma(f02r, f02r, f02i * f02i) + fma(f12r, f12r, f12i * f12i));
    const double hh = sqrt(h2);
    const double ih = hh > 0.0 ? 1.0 / hh : 0.0; /* exactly degenerate pair: split it evenly */
    const double x00 = k0 * ip, x10 = k1 * ip;
    out.x00 = x00;
    out.x10 = x10;
    /* |V_a1|^2 - |V_a2|^2 = n_a / h lies in [-(1 - x_a0), 1 - x_a0]; round-off of a (nearly) degenerate
     * pair must not leave that range */
    out.x01 = fmin(fmax(0.5 * fma(n0, ih, 1.0 - x00), 0.0), fmax(1.0 - x00, 0.0));
    out.x11 = fmin(fmax(0.5 * fma(n1, ih, 1.0 - x10), 0.0), fmax(1.0 - x10, 0.0));
    unsigned st = GFP_ST_REFINED;
    const double relgap = 2.0 * hh / (1.5 * fabs(l0) + hh);
    if (!(relgap >= GFP_ILL_GAP)) st |= GFP_ST_ILL_COND;
    if (!(fabs(out.x00) + fabs(out.x01) + fabs(out.x10) + fabs(out.x11) < 1e300)) st |= GFP_ST_NON_FINITE;
    return st;
}

/* Fallback of the energy-bin loop: rebuild H = H0 + rho T and refine by deflation (Jacobi only for a
 * degenerate scale or non-finite input), return the same four entries as the fast path.  Out of line,
 * operands by pointer: only the rare slow path pays for the memory round trip.  Returns status bits
 * (REFINED / ILL_COND / NON_FINITE). */
GF_HD_NOINLINE unsigned gfp_pencil_x4_refine(const gfp_herm3* h0, const gfp_herm3* T, double rho, gfp_x4* out) {
    gfp_herm3 h;
    h.d0 = fma(rho, T->d0, h0->d0);
    h.d1 = fma(rho, T->d1, h0->d1);
    h.d2 = fma(rho, T->d2, h0->d2);
    h.ar = fma(rho, T->ar, h0->ar);
    h.ai = fma(rho, T->ai, h0->ai);
    h.br = fma(rho, T->br, h0->br);
    h.bi = fma(rho, T->bi, h0->bi);
    h.cr = fma(rho, T->cr, h0->cr);
    h.ci = fma(rho, T->ci, h0->ci);
    gfp_x4 x;
    unsigned st = gfp_herm3_x4_deflate(h, x);
    if (st & GFP_ST_NON_FINITE) {
        double lam[3], vr[9], vi[9];
        const double relgap = gfp_herm3_jacobi(h, lam, vr, vi);
        st = GFP_ST_REFINED;
        x.x00 = fma(vr[0], vr[0], vi[0] * vi[0]);
        x.x01 = fma(vr[1], vr[1], vi[1] * vi[1]);
        x.x10 = fma(vr[3], vr[3], vi[3] * vi[3]);
        x.x11 = fma(vr[4], vr[4], vi[4] * vi[4]);
        if (!(relgap >= GFP_ILL_GAP)) st |= GFP_ST_ILL_COND;
        if (!(fabs(x.x00) + fabs(x.x01) + fabs(x.x10) + fabs(x.x11) < 1e300)) st |= GFP_ST_NON_FINITE;
    }
    *out = x;
    return st;
}

/* ------------------------------------------------------------------ mixing matrices */

/* Columns 1 and 2 of U = R23 R13(dcp) R12 (column 0 multiplies the zero eigenvalue and is
 * never needed for the Hamiltonians).  fr.py:138-162 with sin(asin(x)) = x folded. */
struct gfp_cols12 {
    double u01;        /* c13 s12                     (real) */
    double u11r, u11i; /* c23 c12 - s23 s13 s12 e^{i d} */
    double u21r, u21i; /* -s23 c12 - c23 s13 s12 e^{i d} */
    double u02r, u02i; /* s13 e^{-i d}                 */
    double u12, u22;   /* s23 c13, c23 c13            (real) */
};

struct gfp_trig {
    double s12, c12, s13, c13, s23, c23, sd, cd;
};

GF_HD gfp_trig gfp_angles_trig(double s12_2, double c13_4, double s23_2, double dcp) {
    gfp_trig t;
    t.s12 = gfp_sqrt01(s12_2);
    t.c12 = gfp_sqrt01(1.0 - s12_2);
    const double c13_2 = gfp_sqrt01(c13_4);
    t.c13 = gfp_sqrt01(c13_2);
    t.s13 = gfp_sqrt01(1.0 - c13_2);
    t.s23 = gfp_sqrt01(s23_2);
    t.c23 = gfp_sqrt01(1.0 - s23_2);
    gfp_sincos(dcp, &t.sd, &t.cd);
    return t;
}

GF_HD gfp_cols12 gfp_cols_from_trig(const gfp_trig& t) {
    gfp_cols12 u;
    const double k = t.s13 * t.s12; /* multiplies e^{i d} in rows 1,2 of column 1 */
    u.u01 = t.c13 * t.s12;
    u.u11r = fma(-t.s23 * k, t.cd, t.c23 * t.c12);
    u.u11i = -t.s23 * k * t.sd;
    u.u21r = fma(-t.c23 * k, t.cd, -(t.s23 * t.c12));
    u.u21i = -t.c23 * k * t.sd;
    u.u02r = t.s13 * t.cd;
    u.u02i = -t.s13 * t.sd;
    u.u12 = t.s23 * t.c13;
    u.u22 = t.c23 * t.c13;
    return u;
}

/* Full U (row-major [3][3], re/im interleaved) -- fr.angles_to_u. */
GF_HD void gfp_full_u(const gfp_trig& t, double* u /*[18]*/) {
    const double er = t.cd, ei = t.sd; /* e^{+i d} */
    const double k12 = t.s13 * t.c12, k = t.s13 * t.s12;
    u[0] = t.c13 * t.c12; u[1] = 0.0;
    u[2] = t.c13 * t.s12; u[3] = 0.0;
    u[4] = t.s13 * er;    u[5] = -t.s13 * ei;
    u[6] = -t.c23 * t.s12 - t.s23 * k12 * er; u[7] = -t.s23 * k12 * ei;
    u[8] = t.c23 * t.c12 - t.s23 * k * er;    u[9] = -t.s23 * k * ei;
    u[10] = t.s23 * t.c13; u[11] = 0.0;
    u[12] = t.s23 * t.s12 - t.c23 * k12 * er; u[13] = -t.c23 * k12 * ei;
    u[14] = -t.s23 * t.c12 - t.c23 * k * er;  u[15] = -t.c23 * k * ei;
    u[16] = t.c23 * t.c13; u[17] = 0.0;
}

/* |U_ai|^2 of the PMNS-like matrix without any complex arithmetic (only cos(dcp) enters). */
GF_HD void gfp_pmns_abs2(const gfp_trig& t, double* X) {
    const double s12_2 = t.s12 * t.s12, c12_2 = t.c12 * t.c12;
    const double s13_2 = t.s13 * t.s13, c13_2 = t.c13 * t.c13;
    const double s23_2 = t.s23 * t.s23, c23_2 = t.c23 * t.c23;
    const double cross = 2.0 * t.c23 * t.s23 * t.s12 * t.c12 * t.s13 * t.cd;
    X[0] = c13_2 * c12_2;
    X[1] = c13_2 * s12_2;
    X[2] = s13_2;
    X[3] = fma(c23_2, s12_2, s23_2 * s13_2 * c12_2) + cross;
    X[4] = fma(c23_2, c12_2, s23_2 * s13_2 * s12_2) - cross;
    X[5] = s23_2 * c13_2;
    X[6] = fma(s23_2, s12_2, c23_2 * s13_2 * c12_2) - cross;
    X[7] = fma(s23_2, c12_2, c23_2 * s13_2 * s12_2) + cross;
    X[8] = c23_2 * c13_2;
}

/* |U_ai|^2 straight from the Haar-flat coordinates (s12^2, c13^4, s23^2, dcp): the squared sines and
 * cosines ARE the coordinates (fr.py:146-155 round-trips them through asin / sin), so the SM-only
 * models need two square roots -- c13^2 = sqrt(c13^4) and the interference term -- and cos(dcp) only.
 * |U|^2 is doubly stochastic, so only its four independent entries (rows e, mu; columns 1, 2 -- the layout
 * of gfp_x4) are formed; gfp_mix4 writes the transition in them (9 + 14 fp64 instructions instead of 22 + 18
 * for the nine entries and the full double sum: the SM-only kernel is bound by its instruction count). */
GF_HD gfp_x4 gfp_pmns_abs2_coords4(double s12_2, double c13_4, double s23_2, double dcp) {
    const double c12_2 = 1.0 - s12_2, c23_2 = 1.0 - s23_2;
    const double c13_2 = gfp_sqrt01(c13_4), s13_2 = 1.0 - c13_2;
    /* 2 c23 s23 s12 c12 s13 cos(dcp); every factor is a non-negative root inside the prior box, a
     * negative coordinate makes the product's root NaN exactly where the reference's sqrt is NaN */
    const bool valid = s12_2 >= 0.0 && c12_2 >= 0.0 && s23_2 >= 0.0 && c23_2 >= 0.0 && s13_2 >= 0.0;
    const double prod = (c23_2 * s23_2) * (s12_2 * c12_2) * s13_2;
    const double cross = valid ? 2.0 * gfp_sqrt01(prod) * gfp_cos(dcp) : NAN;
    const double t = s23_2 * s13_2;
    gfp_x4 x;
    x.x00 = c13_2 * c12_2;                                  /* |U_e1|^2  */
    x.x01 = c13_2 * s12_2;                                  /* |U_e2|^2  */
    x.x10 = fma(c23_2, s12_2, t * c12_2) + cross;           /* |U_mu1|^2 */
    x.x11 = fma(c23_2, c12_2, t * s12_2) - cross;           /* |U_mu2|^2 */
    return x;
}

/* H = m1 u1 u1^+ + m2 u2 u2^+ for the columns above (U diag(0,m1,m2) U^+, fr.py:383-394). */
GF_HD gfp_herm3 gfp_herm_from_cols(const gfp_cols12& u, double m1, double m2) {
    gfp_herm3 h;
    h.d0 = fma(m1, u.u01 * u.u01, m2 * fma(u.u02r, u.u02r, u.u02i * u.u02i));
    h.d1 = fma(m1, fma(u.u11r, u.u11r, u.u11i * u.u11i), m2 * u.u12 * u.u12);
    h.d2 = fma(m1, fma(u.u21r, u.u21r, u.u21i * u.u21i), m2 * u.u22 * u.u22);
    /* a = H01 = m1 u01 conj(u11) + m2 u02 u12 */
    h.ar = fma(m1 * u.u01, u.u11r, m2 * u.u12 * u.u02r);
    h.ai = fma(-m1 * u.u01, u.u11i, m2 * u.u12 * u.u02i);
    /* b = H02 = m1 u01 conj(u21) + m2 u02 u22 */
    h.br = fma(m1 * u.u01, u.u21r, m2 * u.u22 * u.u02r);
    h.bi = fma(-m1 * u.u01, u.u21i, m2 * u.u22 * u.u02i);
    /* c = H12 = m1 u11 conj(u21) + m2 u12 u22 */
    h.cr = fma(m1, fma(u.u11r, u.u21r, u.u11i * u.u21i), m2 * u.u12 * u.u22);
    h.ci = m1 * fma(u.u11i, u.u21r, -(u.u11r * u.u21i));
    return h;
}

/* (sin^4 phi, cos 2psi) -> (f_e, f_mu, f_tau); fr.py:101-113 with sin^2(acos(c)/2) = (1-c)/2. */
GF_HD void gfp_angles_to_fr(double sphi4, double c2psi, double* f) {
    const double sphi2 = gfp_sqrt01(sphi4);
    const double cphi2 = 1.0 - sphi2;
    double spsi2 = 0.5 * (1.0 - c2psi);
    if (!(fabs(c2psi) <= 1.0)) spsi2 = NAN; /* acos domain of the reference */
    const double cpsi2 = 1.0 - spsi2;
    f[0] = fabs(sphi2 * cpsi2);
    f[1] = fabs(sphi2 * spsi2);
    f[2] = fabs(cphi2);
}

/* Transition with the four independent entries of the doubly stochastic X (rows and columns sum
 * to one): f_b = sum_i X_bi w_i, w_i = sum_a X_ai s_a.  sd0 = s0 - s2, sd1 = s1 - s2, S = s0+s1+s2.
 * Returns f_e and f_mu (NOT divided by S); f_tau = S - f_e - f_mu. */
GF_HD void gfp_mix4(const gfp_x4& x, double s2, double sd0, double sd1, double S, double& f0, double& f1) {
    const double w0 = fma(x.x00, sd0, fma(x.x10, sd1, s2));
    const double w1 = fma(x.x01, sd0, fma(x.x11, sd1, s2));
    const double w2 = S - w0 - w1;
    const double u0 = w0 - w2, u1 = w1 - w2;
    f0 = fma(x.x00, u0, fma(x.x01, u1, w2));
    f1 = fma(x.x10, u0, fma(x.x11, u1, w2));
}

/* The flavor transition P = X X^T of a doubly stochastic X is symmetric and doubly stochastic, so three numbers determine
 * it: P00 = sum_i X_0i^2, P01 = sum_i X_0i X_1i, P11 = sum_i X_1i^2 (the third row and column follow from the unit sums).
 * From the four independent entries of gfp_x4; X_a2 = 1 - X_a0 - X_a1. */
GF_HD void gfp_x4_transition(const gfp_x4& x, double& p00, double& p01, double& p11) {
    const double x02 = 1.0 - x.x00 - x.x01, x12 = 1.0 - x.x10 - x.x11;
    p00 = fma(x.x00, x.x00, fma(x.x01, x.x01, x02 * x02));
    p01 = fma(x.x00, x.x10, fma(x.x01, x.x11, x02 * x12));
    p11 = fma(x.x10, x.x10, fma(x.x11, x.x11, x12 * x12));
}

/* A source composition s in the form gfp_transition_fr consumes, for bin-width sums W = sum_b w_b:
 * sd0 = s0 - s2, sd1 = s1 - s2, ws2 = W s2, inv_sw = 1 / (S W) with S = s0 + s1 + s2. */
struct gfp_src_consts {
    double sd0, sd1, ws2, inv_sw;
};
GF_HD gfp_src_consts gfp_source_consts(double s0, double s1, double s2, double W) {
    gfp_src_consts c;
    c.sd0 = s0 - s2;
    c.sd1 = s1 - s2;
    c.ws2 = W * s2;
    c.inv_sw = 1.0 / ((s0 + s1 + s2) * W);
    return c;
}

/* flux_averaged_BSMu (fr.py:441-457) of ANY source from the bin-width-weighted transition sums A = (A00, A01, A11),
 * A_ab = sum_b w_b P_ab:  fr_0 = (A00 s0 + A01 s1 + (W - A00 - A01) s2) / (S W), fr_1 likewise with (A01, A11),
 * fr_2 = 1 - fr_0 - fr_1.  Equal to the per-bin gfp_mix4 accumulation of gf_bin_loop up to rounding. */
GF_HD void gfp_transition_fr(const double* A, const gfp_src_consts& c, double* fr) {
    fr[0] = fma(A[0], c.sd0, fma(A[1], c.sd1, c.ws2)) * c.inv_sw;
    fr[1] = fma(A[1], c.sd0, fma(A[2], c.sd1, c.ws2)) * c.inv_sw;
    fr[2] = 1.0 - fr[0] - fr[1];
}

/* fr_b = sum_i X_bi (sum_a X_ai s_a)  -- NOT divided by sum(s). */
GF_HD void gfp_mix(const double* X, double s0, double s1, double s2, double* f) {
    const double w0 = fma(X[0], s0, fma(X[3], s1, X[6] * s2));
    const double w1 = fma(X[1], s0, fma(X[4], s1, X[7] * s2));
    const double w2 = fma(X[2], s0, fma(X[5], s1, X[8] * s2));
    f[0] = fma(X[0], w0, fma(X[1], w1, X[2] * w2));
    f[1] = fma(X[3], w0, fma(X[4], w1, X[5] * w2));
    f[2] = fma(X[6], w0, fma(X[7], w1, X[8] * w2));
}

/* H_ab = m1 U_a1 conj(U_b1) + m2 U_a2 conj(U_b2) for a general complex matrix U given row-major
 * with interleaved (re, im) -- `sm_u` of fr.params_to_BSMu (fr.py:383-386). */
GF_HD gfp_herm3 gfp_herm_from_u(const double* u /*[18]*/, double m1, double m2) {
    gfp_herm3 h;
#define GFP_UR(a, i) u[2 * (3 * (a) + (i))]
#define GFP_UI(a, i) u[2 * (3 * (a) + (i)) + 1]
#define GFP_ABS2(a, i) fma(GFP_UR(a, i), GFP_UR(a, i), GFP_UI(a, i) * GFP_UI(a, i))
#define GFP_PR(a, b, i) fma(GFP_UR(a, i), GFP_UR(b, i), GFP_UI(a, i) * GFP_UI(b, i))   /* Re u_a conj(u_b) */
#define GFP_PI(a, b, i) fma(GFP_UI(a, i), GFP_UR(b, i), -(GFP_UR(a, i) * GFP_UI(b, i))) /* Im u_a conj(u_b) */
    h.d0 = fma(m1, GFP_ABS2(0, 1), m2 * GFP_ABS2(0, 2));
    h.d1 = fma(m1, GFP_ABS2(1, 1), m2 * GFP_ABS2(1, 2));
    h.d2 = fma(m1, GFP_ABS2(2, 1), m2 * GFP_ABS2(2, 2));
    h.ar = fma(m1, GFP_PR(0, 1, 1), m2 * GFP_PR(0, 1, 2));
    h.ai = fma(m1, GFP_PI(0, 1, 1), m2 * GFP_PI(0, 1, 2));
    h.br = fma(m1, GFP_PR(0, 2, 1), m2 * GFP_PR(0, 2, 2));
    h.bi = fma(m1, GFP_PI(0, 2, 1), m2 * GFP_PI(0, 2, 2));
    h.cr = fma(m1, GFP_PR(1, 2, 1), m2 * GFP_PR(1, 2, 2));
    h.ci = fma(m1, GFP_PI(1, 2, 1), m2 * GFP_PI(1, 2, 2));
#undef GFP_UR
#undef GFP_UI
#undef GFP_ABS2
#undef GFP_PR
#undef GFP_PI
    return h;
}

/* Full eigen-decomposition with columns ordered by ascending eigenvalue.  out_v: row-major
 * [3][3] interleaved (re, im); returns the relative gap of gfp_herm3_jacobi. */
GF_HD double gfp_herm3_eig_sorted(const gfp_herm3& h, double* lam, double* out_v /*[18]*/) {
    double l[3], vr[9], vi[9];
    const double relgap = gfp_herm3_jacobi(h, l, vr, vi);
    int i0 = 0, i1 = 1, i2 = 2, t;
    if (l[i0] > l[i1]) { t = i0; i0 = i1; i1 = t; }
    if (l[i1] > l[i2]) { t = i1; i1 = i2; i2 = t; }
    if (l[i0] > l[i1]) { t = i0; i0 = i1; i1 = t; }
    const int ord[3] = {i0, i1, i2};
    for (int c = 0; c < 3; ++c) {
        lam[c] = l[ord[c]];
        for (int a = 0; a < 3; ++a) {
            out_v[2 * (3 * a + c)] = vr[3 * a + ord[c]];
            out_v[2 * (3 * a + c) + 1] = vi[3 * a + ord[c]];
        }
    }
    return relgap;
}

#endif /* GF_PHYSICS_CUH */
