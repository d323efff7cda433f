/*
 * gf_model.cuh -- device-side flattening of the reference's ln_prob closure
 * (`partial(ln_prob, args=..., asimov_paramset=..., llh_paramset=...)`,
 * scripts/fr.py:182-187) and the per-point evaluation built on gf_physics.cuh.
 *
 * gf_dev_model is passed to every kernel BY VALUE as a __grid_constant__ parameter
 * (constant bank, uniform access, no global symbol => concurrent launches with
 * different models on different streams are safe).
 */
#ifndef GF_MODEL_CUH
#define GF_MODEL_CUH

#include <type_traits>

#include "../../include/golemflavor_b200.h"
#include "gf_physics.cuh"

struct gf_dev_model {
    int32_t ndim, no_bsm, nbins, llh_kind, emulate_underflow, np_free;
    int32_t col_sm[4], col_mass[2], col_src[2], col_np[4], col_scale, col_x, col_src3[3];
    double fixed_sm[4], fixed_mass[2], fixed_src[3], fixed_np[4], fixed_loglam;
    gfp_herm3 T;                /* N diag(0,.01,1) N^+ for the fixed NP angles          */
    gfp_pencil_T penT;          /* its pencil coefficients (fixed textures)              */
    gfp_adj3 adjT;              /* adj(T'), the rho^2 coefficient of det is tr(adj(T') H0')/2 */
    double wsum;                /* sum of the bin widths                                 */
    double inv_S_wsum;          /* fixed source: 1 / (src_S wsum)                        */
    double src_S, src_sd0, src_sd1; /* fixed source: s0+s1+s2, s0-s2, s1-s2              */
    double g[GF_MAX_BINS];      /* 2 Ec^(dim-2) 2^70: H*2E = H0 + 10^logLam g T          */
    double width[GF_MAX_BINS];  /* |E_hi - E_lo|                          (fr.py:414)    */
    double fr_bf[3];
    double half_inv_s2;         /* 1/(2 sigma^2)                                        */
    double lognorm3;            /* -1.5 log(2 pi sigma^2)                               */
    double offset, underflow_logpdf, llh_const, epsilon;
    double lo[GF_MAX_DIM], hi[GF_MAX_DIM], mu[GF_MAX_DIM], inv_sigma[GF_MAX_DIM]; /* inv_sigma = 0: uniform */
    double lognorm_total;       /* sum of the Gaussian dimensions' log-normalisers       */
    double cdf_lo[GF_MAX_DIM], cdf_span[GF_MAX_DIM], sigma[GF_MAX_DIM]; /* scans: inverse-CDF draws */
    int32_t kind[GF_MAX_DIM];
};

/* strided accessor for theta (see include/golemflavor_b200.h "theta") */
struct gf_theta_view {
    const double* p;
    int64_t ld_point, ld_dim;
    GF_HD double at(int64_t i, int k) const { return p[i * ld_point + (int64_t)k * ld_dim]; }
};

/* Physical inputs of one parameter point. */
struct gf_point {
    double sm[4], mass[2], np[4], loglam, src[3];
    bool src_unit; /* the source sums to one by construction (SM-only path: no division by sum(source), see gf_point_fr) */
};

/* (sin^4 phi, cos 2psi) -> source composition.  Its entries sum to one -- sin^2 phi (cos^2 psi + sin^2 psi) + cos^2 phi --
 * as long as sin^4 phi <= 1 (beyond, fr.py:101-113 takes |cos^2 phi| and the sum is 2 sin^2 phi - 1). */
GF_HD void gf_source_from_angles(double sphi4, double c2psi, gf_point& q) {
    gfp_angles_to_fr(sphi4, c2psi, q.src);
    q.src_unit = sphi4 <= 1.0;
}

/*
 * Kernel specialisations (compile-time, chosen by the host from the model):
 *   GF_SPEC_GENERIC : every model; which quantities are sampled is decided by uniform branches.
 *   GF_SPEC_SM      : models without the BSM path (m.no_bsm); the kernel then carries none of the
 *                     eigen-stage code or registers and runs at full occupancy (HBM / latency bound).
 *   GF_SPEC_FIXED   : the production BSM shape -- fixed texture AND fixed source composition
 *                     (scripts/fr.py, mc_texture.py).  The texture part of the pencil and the
 *                     source constants are then read from the constant bank as direct DFMA operands:
 *                     fewer registers and fewer three-register DFMAs (which issue at 2/3 rate on B200).
 */
#define GF_SPEC_GENERIC 0
#define GF_SPEC_FIXED 1
#define GF_SPEC_SM 2 /* no_bsm models (notebook SM fit, unitary / x scans): no BSM code, light on registers */
/*   GF_SPEC_NPFREE  : Haar-random NP mixing (4 sampled NP angles) with a FIXED source composition -- the
 *                     anarchic scan.  The source constants come from the constant bank, which frees the
 *                     registers the second interleaved bin chain needs.  Scan kernels only; the
 *                     log-posterior launcher serves such models with GF_SPEC_GENERIC. */
#define GF_SPEC_NPFREE 3
/*   GF_SPEC_SM6     : the SM-only model in the reference's own column layout (examples/inference.ipynb:
 *                     columns 0-3 = s12^2, c13^4, s23^2, dcp, columns 4-5 = the two source angles, ndim = 6).
 *                     Every theta read has a compile-time index, so the point lives in registers from the
 *                     load to the likelihood: no shared-memory staging, no column-map lookups.  Other SM-only
 *                     layouts run GF_SPEC_SM. */
#define GF_SPEC_SM6 4
#define GF_SPEC_IS_SM(SPEC) ((SPEC) == GF_SPEC_SM || (SPEC) == GF_SPEC_SM6)
/*   GF_SPEC_FIXED7  : GF_SPEC_FIXED in the column layout of scripts/fr.py (columns 0-3 = the four mixing
 *                     coordinates, 4-5 = the mass-squared differences, 6 = logLam, ndim = 7): compile-time
 *                     theta indices as in GF_SPEC_SM6.  Log-posterior and sampler kernels; the scans run it
 *                     as GF_SPEC_FIXED. */
#define GF_SPEC_FIXED7 5
/*   GF_SPEC_FIXED12 : the same with the five GolemFit nuisance columns of scripts/fr.py:54-60 between the
 *                     masses and logLam (columns 6-10 carry priors only, logLam is column 11, ndim = 12) --
 *                     the reference's production parameter set. */
#define GF_SPEC_FIXED12 6
#define GF_SPEC_IS_FIXED(SPEC) ((SPEC) == GF_SPEC_FIXED || (SPEC) == GF_SPEC_FIXED7 || (SPEC) == GF_SPEC_FIXED12)
/*   GF_SPEC_SM4, GF_SPEC_NPFREE11 : scan kernels only -- the unitary scan (columns 0-3 = the mixing
 *                     coordinates, fixed source, ndim = 4) and the anarchic scan (0-3 mixing, 4-5 masses,
 *                     6-9 NP mixing, 10 logLam, fixed source, ndim = 11) in the layouts scan.scan_paramset
 *                     produces; the texture scan is GF_SPEC_FIXED7.  The drawn sample stays in registers. */
#define GF_SPEC_SM4 7
#define GF_SPEC_NPFREE11 8
#define GF_SPEC_SM5X 9 /* the x scan: columns 0-3 = the mixing coordinates, 4 = x with source (x, 1-x, 0), ndim = 5 */
#undef GF_SPEC_IS_SM
#define GF_SPEC_IS_SM(SPEC) ((SPEC) == GF_SPEC_SM || (SPEC) == GF_SPEC_SM6 || (SPEC) == GF_SPEC_SM4 || (SPEC) == GF_SPEC_SM5X)
#define GF_SPEC_IS_NPFREE(SPEC) ((SPEC) == GF_SPEC_NPFREE || (SPEC) == GF_SPEC_NPFREE11)
#define GF_SPEC_STATIC_NDIM(SPEC)                                                                                  \
    ((SPEC) == GF_SPEC_SM6 ? 6 : (SPEC) == GF_SPEC_FIXED7 ? 7 : (SPEC) == GF_SPEC_FIXED12 ? 12 : (SPEC) == GF_SPEC_SM4 ? 4 : \
     (SPEC) == GF_SPEC_NPFREE11 ? 11 : (SPEC) == GF_SPEC_SM5X ? 5 : 0)

/* Which dimensions carry a (truncated) Gaussian prior term, as a compile-time bit mask (bit k = dimension k), for the
 * specialisations that are the reference's own parameter sets: examples/inference.ipynb (three LIMITEDGAUSS mixing
 * coordinates, flat dcp, flat source angles) and scripts/fr.py:30-104 (the same four, two GAUSSIAN mass-squared
 * differences, flat logLam).  The prior loop then has no per-dimension kind test at all -- the SM-only kernel is bound by
 * its instruction count and the runtime tests were a tenth of it.  -1: kinds read from the model at run time.  A model
 * in one of these column layouts but with other prior kinds is served by the corresponding runtime-layout specialisation
 * (gf_model_spec). */
#define GF_SPEC_STATIC_GMASK(SPEC) ((SPEC) == GF_SPEC_SM6 ? 0x07 : (SPEC) == GF_SPEC_FIXED7 ? 0x37 : -1)
GF_HD int gf_model_gauss_mask(const gf_dev_model& m);
GF_HD bool gf_model_is_fixed_spec(const gf_dev_model& m);
GF_HD bool gf_model_has_fixed_source(const gf_dev_model& m);
GF_HD int gf_model_spec(const gf_dev_model& m);
GF_HD int gf_model_layout_spec(const gf_dev_model& m);
GF_HD int gf_model_grid_spec(const gf_dev_model& m);

/* the general case: runtime column map */
template <int SPEC, class Get>
GF_HD void gf_resolve_point_mapped(const gf_dev_model& m, Get get, gf_point& q) {
#pragma unroll
    for (int k = 0; k < 4; ++k) q.sm[k] = m.col_sm[k] >= 0 ? get(m.col_sm[k]) : m.fixed_sm[k];
    if (SPEC != GF_SPEC_SM) {
#pragma unroll
        for (int k = 0; k < 2; ++k) q.mass[k] = m.col_mass[k] >= 0 ? get(m.col_mass[k]) : m.fixed_mass[k];
    }
    if ((SPEC == GF_SPEC_GENERIC && m.np_free) || GF_SPEC_IS_NPFREE(SPEC)) {
#pragma unroll
        for (int k = 0; k < 4; ++k) q.np[k] = m.col_np[k] >= 0 ? get(m.col_np[k]) : m.fixed_np[k];
    }
    if (SPEC != GF_SPEC_SM) q.loglam = m.col_scale >= 0 ? get(m.col_scale) : m.fixed_loglam;
    q.src_unit = false;
    if (GF_SPEC_IS_FIXED(SPEC) || GF_SPEC_IS_NPFREE(SPEC)) return; /* the source (and for FIXED the NP mixing) comes from the constant bank */
    if (m.col_src[0] >= 0) {
        gf_source_from_angles(get(m.col_src[0]), get(m.col_src[1]), q);
    } else if (m.col_src3[0] >= 0) {
        q.src[0] = get(m.col_src3[0]);
        q.src[1] = get(m.col_src3[1]);
        q.src[2] = get(m.col_src3[2]);
    } else if (m.col_x >= 0) {
        const double x = get(m.col_x); /* scripts/mc_x.py:187: source = (x, 1-x, 0) */
        q.src[0] = x;
        q.src[1] = 1.0 - x;
        q.src[2] = 0.0;
        q.src_unit = true;
    } else {
        q.src[0] = m.fixed_src[0];
        q.src[1] = m.fixed_src[1];
        q.src[2] = m.fixed_src[2];
        q.src_unit = m.src_S == 1.0; /* a normalised fixed source ((1,2,0)/3, (1,0,0), ...): dividing by exactly 1 is the identity */
    }
}

/* Resolve theta columns / fixed values -> physical inputs (fr.py:421-435, llh notebook model). */
template <int SPEC = GF_SPEC_GENERIC, class Get>
GF_HD void gf_resolve_point(const gf_dev_model& m, Get get, gf_point& q) {
    q.src_unit = false;
    if constexpr (SPEC == GF_SPEC_SM6) {
        q.sm[0] = get(0);
        q.sm[1] = get(1);
        q.sm[2] = get(2);
        q.sm[3] = get(3);
        gf_source_from_angles(get(4), get(5), q);
    } else if constexpr (SPEC == GF_SPEC_SM4) {
        q.sm[0] = get(0);
        q.sm[1] = get(1);
        q.sm[2] = get(2);
        q.sm[3] = get(3);
        q.src[0] = m.fixed_src[0];
        q.src[1] = m.fixed_src[1];
        q.src[2] = m.fixed_src[2];
        q.src_unit = m.src_S == 1.0; /* a normalised fixed source: dividing by exactly 1 is the identity */
    } else if constexpr (SPEC == GF_SPEC_SM5X) {
        q.sm[0] = get(0);
        q.sm[1] = get(1);
        q.sm[2] = get(2);
        q.sm[3] = get(3);
        const double x = get(4); /* scripts/mc_x.py:187 */
        q.src[0] = x;
        q.src[1] = 1.0 - x;
        q.src[2] = 0.0;
        q.src_unit = true;
    } else if constexpr (SPEC == GF_SPEC_NPFREE11) {
        q.sm[0] = get(0);
        q.sm[1] = get(1);
        q.sm[2] = get(2);
        q.sm[3] = get(3);
        q.mass[0] = get(4);
        q.mass[1] = get(5);
        q.np[0] = get(6);
        q.np[1] = get(7);
        q.np[2] = get(8);
        q.np[3] = get(9);
        q.loglam = get(10);
    } else if constexpr (SPEC == GF_SPEC_FIXED7 || SPEC == GF_SPEC_FIXED12) {
        q.sm[0] = get(0);
        q.sm[1] = get(1);
        q.sm[2] = get(2);
        q.sm[3] = get(3);
        q.mass[0] = get(4);
        q.mass[1] = get(5);
        q.loglam = get(SPEC == GF_SPEC_FIXED12 ? 11 : 6);
    } else {
        gf_resolve_point_mapped<SPEC>(m, get, q);
    }
}


/*
 * Measured flavor composition of one point.
 *   no_bsm : fr = u_to_fr(source, angles_to_u(sm))                (notebook SM model)
 *   else   : flux_averaged_BSMu -- per energy bin H*2E = H0 + rho_b T, |V|^2, u_to_fr,
 *            bin-width weighted mean, renormalised                  (fr.py:441-457)
 * The source normalisation 1/sum(s) and the 1/(E_max-E_min) factor cancel in the final
 * renormalisation and are not applied per bin.
 */
/* H0 = U diag(0, m21, m3x) U^+ (scaled by 2^70) and the new-physics matrix T = N diag(0, 1/100, 1) N^+ of one point. */
template <int SPEC>
GF_HD void gf_point_matrices(const gf_dev_model& m, const gf_point& q, gfp_herm3& h0, gfp_herm3& T, double& m1, double& m2) {
    const gfp_trig t = gfp_angles_trig(q.sm[0], q.sm[1], q.sm[2], q.sm[3]);
    GF_STAGE(4);
    const gfp_cols12 u = gfp_cols_from_trig(t);
    m1 = q.mass[0] * GFP_MASS_SCALE;
    m2 = q.mass[1] * GFP_MASS_SCALE;
    h0 = gfp_herm_from_cols(u, m1, m2);
    GF_STAGE(5);
    if (!GF_SPEC_IS_FIXED(SPEC) && (GF_SPEC_IS_NPFREE(SPEC) || m.np_free)) {
        const gfp_trig tn = gfp_angles_trig(q.np[0], q.np[1], q.np[2], q.np[3]);
        T = gfp_herm_from_cols(gfp_cols_from_trig(tn), GFP_T_EIG1, GFP_T_EIG2);
    } else {
        T = m.T;
    }
}

/*
 * Where the RARE refinement path of the bin loop (two eigenvalues closer than the fast path tolerates: 0.02-1.4 % of
 * the points) gets H0 and T from.  The closed form only needs the pencil's polynomial coefficients, so a kernel that
 * kept the two matrices around for the fallback paid 18 local-memory stores per point for them.
 *   gf_mats_ptr     : the caller keeps both in memory (sampler, single-sample entry points: latency-bound or tiny).
 *   gf_mats_rebuild : nothing is kept -- the fallback RECOMPUTES them from the point's theta, which the log-posterior
 *                     kernel can always get back (it re-reads the row from global memory): a few hundred instructions
 *                     on a path taken by < 1 % of the warps' bins.  Same functions, same inputs: the rebuilt matrices
 *                     are the original bits.  k_lnprob: no local store left in the point loop, -0.8 %.  The scan kernels
 *                     could re-draw the sample from its Philox counter the same way; measured, the extra live state
 *                     (seed, index, model pointer across three call sites) made them spill and cost 2 %: they keep
 *                     gf_mats_ptr.
 */
struct gf_mats_ptr {
    const gfp_herm3* h0;
    const gfp_herm3* T;
};
template <int SPEC, class ThetaSrc>
struct gf_mats_rebuild {
    const gf_dev_model* m;
    ThetaSrc src; /* void operator()(const gf_dev_model&, double* theta) const */
};
struct gf_no_src {}; /* tag: keep the matrices in memory */

/* theta of a point from a (strided) row in memory */
struct gf_src_row {
    const double* row;
    int64_t ld;
    GF_HD void operator()(const gf_dev_model& m, double* th) const {
        for (int k = 0; k < m.ndim; ++k) th[k] = row[(int64_t)k * ld];
    }
};

GF_HD unsigned gf_refine_bin(const gf_mats_ptr& p, double rho, gfp_x4* out) { return gfp_pencil_x4_refine(p.h0, p.T, rho, out); }

template <int SPEC, class ThetaSrc>
GF_HD_NOINLINE unsigned gf_refine_bin(const gf_mats_rebuild<SPEC, ThetaSrc> r, double rho, gfp_x4* out) {
    double th[GF_MAX_DIM];
    r.src(*r.m, th);
    gf_point q;
    gf_resolve_point<SPEC>(*r.m, [&](int k) { return th[k]; }, q);
    gfp_herm3 h0, T;
    double m1, m2;
    gf_point_matrices<SPEC>(*r.m, q, h0, T, m1, m2);
    return gfp_pencil_x4_refine(&h0, &T, rho, out);
}

/* The energy-bin loop: per bin the invariants of the pencil, the closed-form |V|^2 (deflation
 * fallback), the transition in its four independent entries and the width-weighted sums.
 *
 * LANES = 1: one thread runs all bins of its point in increasing order (log-posterior kernel, scans, evidence).
 * LANES = 2 (device-resident sampler): the two adjacent lanes 2w, 2w+1 of a warp evaluate ONE point together; lane
 * `lane` (= threadIdx.x & 1) runs the bins of its own parity in increasing order, and the two partial sums are
 * exchanged with one __shfl_xor_sync each -- addition commutes, so both lanes hold the same bits afterwards and take
 * the same accept / reject decision.  Every launch shape of the sampler uses the same split, hence identical chains.
 * The sampler is bound by the latency of one thread's instruction stream (gf_ensemble.cu); halving the bin work per
 * thread shortens that stream by ~40 %. */
template <int ILP, int LANES, class TPART, class MATS>
GF_HD unsigned gf_bin_loop(const gf_dev_model& m, const gfp_pencil_P& pp, const TPART& pt, const MATS& mats,
                           double lam, double s2, double sd0, double sd1, double inv_norm, double S, double* fr, int lane = 0) {
    static_assert(LANES == 1 || LANES == 2, "one thread or a pair of lanes per point");
    unsigned st = 0u;
    double a0 = 0.0, a1 = 0.0;
    /* ILP bins per iteration, i.e. ILP independent fast-path chains in flight per thread.  2: +10 % on
     * k_lnprob, which is bound by the latency of that chain at 16 warps per SM; 1: kernels whose extra
     * per-thread state would make the second chain spill; 4-5: the ensemble sampler, where one or two warps
     * per SM sub-partition run the chain and latency is all that matters */
    constexpr int STEP = LANES;
    int b = LANES == 2 ? lane : 0;
    if (ILP > 1) {
        for (; b + STEP * (ILP - 1) < m.nbins; b += STEP * ILP) {
            gfp_x4 x[ILP];
            bool ok = true;
#pragma unroll
            for (int i = 0; i < ILP; ++i) ok = gfp_pencil_x4_fast(pp, pt, lam * m.g[b + STEP * i], x[i]) && ok;
            if (!ok) { /* rare: refine whichever bin failed (re-tested: the flags are not kept in registers) */
#pragma unroll
                for (int i = 0; i < ILP; ++i) {
                    gfp_x4 again;
                    if (!gfp_pencil_x4_fast(pp, pt, lam * m.g[b + STEP * i], again)) {
                        gfp_x4 slow; /* a separate object keeps x[] in registers */
                        st |= gf_refine_bin(mats, lam * m.g[b + STEP * i], &slow);
                        x[i] = slow;
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < ILP; ++i) {
                double f0, f1;
                gfp_mix4(x[i], s2, sd0, sd1, S, f0, f1);
                const double wd = m.width[b + STEP * i];
                a0 = fma(wd, f0, a0);
                a1 = fma(wd, f1, a1);
            }
        }
    }
    for (; b < m.nbins; b += STEP) { /* ILP = 1, or the remaining bins */
        const double rho = lam * m.g[b];
        gfp_x4 x;
        if (!gfp_pencil_x4_fast(pp, pt, rho, x)) {
            gfp_x4 slow;
            st |= gf_refine_bin(mats, rho, &slow);
            x = slow;
        }
        double f0, f1;
        gfp_mix4(x, s2, sd0, sd1, S, f0, f1);
        const double wd = m.width[b];
        a0 = fma(wd, f0, a0);
        a1 = fma(wd, f1, a1);
    }
#ifdef __CUDA_ARCH__
    if (LANES == 2) {
        /* the mask names just the two lanes of the pair (lane == threadIdx.x & 1 by contract): they follow the same
         * control flow up to here -- other pairs of the warp may have left early (out-of-prior proposal) */
        const unsigned mask = 3u << (((unsigned)threadIdx.x & 31u) & ~1u);
        a0 += __shfl_xor_sync(mask, a0, 1);
        a1 += __shfl_xor_sync(mask, a1, 1);
        st |= __shfl_xor_sync(mask, st, 1);
    }
#endif
    /* sum_b f_b = S in every bin, so the normalisation of fr.py:455-457 is inv_norm = 1 / (S sum(width)) */
    fr[0] = a0 * inv_norm;
    fr[1] = a1 * inv_norm;
    fr[2] = 1.0 - fr[0] - fr[1];
    return st;
}

template <int SPEC = GF_SPEC_GENERIC, int ILP = 1, int LANES = 1, class ThetaSrc = gf_no_src>
GF_HD unsigned gf_point_fr(const gf_dev_model& m, const gf_point& q, double* fr, int lane = 0, const ThetaSrc& src = ThetaSrc()) {
    unsigned st = 0u;
    if (GF_SPEC_IS_SM(SPEC) || (SPEC == GF_SPEC_GENERIC && m.no_bsm)) {
        /* fr = u_to_fr(source, angles_to_u(sm)) in the four independent entries of |U|^2.  A source built from the two
         * source angles or from x sums to one by construction (q.src_unit): the division by sum(source) of fr.py:535
         * is then a division by 1 +- 1 ulp and is not carried out; raw source ratios (config 1), fixed sources and
         * source angles outside their natural box are normalised. */
        const gfp_x4 x = gfp_pmns_abs2_coords4(q.sm[0], q.sm[1], q.sm[2], q.sm[3]);
        const bool unit_sum = q.src_unit;
        const double S = unit_sum ? 1.0 : q.src[0] + q.src[1] + q.src[2];
        double f0, f1;
        gfp_mix4(x, q.src[2], q.src[0] - q.src[2], q.src[1] - q.src[2], S, f0, f1);
        if (!unit_sum) {
            const double inv = gfp_rcp(S); /* fr.py:535 */
            f0 *= inv;
            f1 *= inv;
        }
        fr[0] = f0;
        fr[1] = f1;
        fr[2] = 1.0 - f0 - f1;
    } else if (!GF_SPEC_IS_SM(SPEC)) {
        /* the loop runs on the polynomial invariants of the pencil H0 + rho T; the matrices themselves are only needed
         * by the rare refinement path (see gf_mats_ptr / gf_mats_rebuild) */
        gfp_herm3 h0, T;
        double m1, m2;
        gf_point_matrices<SPEC>(m, q, h0, T, m1, m2);
#ifdef __CUDA_ARCH__
        const double lam = exp10(q.loglam);
#else
        const double lam = pow(10.0, q.loglam);
#endif
        GF_STAGE(6);
        /* gf_mats_ptr: taking the addresses parks h0 / T in local memory; gf_mats_rebuild: they die after the pencil */
        auto run = [&](const auto& mats) {
            if (GF_SPEC_IS_FIXED(SPEC)) {
                const gfp_pencil_P pp = gfp_make_pencil_P(h0, m1, m2, m.T, m.penT.te, m.adjT);
                GF_STAGE(7);
                st = gf_bin_loop<ILP, LANES>(m, pp, m.penT, mats, lam, m.fixed_src[2], m.src_sd0, m.src_sd1, m.inv_S_wsum, m.src_S, fr, lane);
                GF_STAGE(8);
            } else {
                const bool npf = GF_SPEC_IS_NPFREE(SPEC) || m.np_free;
                const gfp_pencil_T pt = gfp_make_pencil_T(T);
                const gfp_pencil_P pp = gfp_make_pencil_P(h0, m1, m2, T, pt.te, npf ? gfp_adj_tf(pt.te, T) : m.adjT);
                if (GF_SPEC_IS_NPFREE(SPEC)) {
                    st = gf_bin_loop<ILP, LANES>(m, pp, pt, mats, lam, m.fixed_src[2], m.src_sd0, m.src_sd1, m.inv_S_wsum, m.src_S, fr, lane);
                } else {
                    const double S = q.src[0] + q.src[1] + q.src[2];
                    st = gf_bin_loop<ILP, LANES>(m, pp, pt, mats, lam, q.src[2], q.src[0] - q.src[2], q.src[1] - q.src[2], gfp_rcp(S * m.wsum), S, fr, lane);
                }
            }
        };
        if constexpr (std::is_same<ThetaSrc, gf_no_src>::value) {
            /* the fixed texture is read where it lives -- the kernel parameter (constant bank; the address of a
             * __grid_constant__ parameter may be taken): no per-point copy */
            run(gf_mats_ptr{&h0, GF_SPEC_IS_FIXED(SPEC) ? &m.T : &T});
        } else {
            run(gf_mats_rebuild<SPEC, ThetaSrc>{&m, src});
        }
        /* |V|^2 must be doubly stochastic, hence 0 <= fr <= 1: a violation beyond epsilon is the
         * analogue of the reference's failed unitarity assertion (fr.py:489-498) */
        const double mn = fmin(fr[0], fmin(fr[1], fr[2]));
        if (!(mn >= -m.epsilon)) st |= GFP_ST_NON_UNITARY;
    }
    if (!(fabs(fr[0]) + fabs(fr[1]) + fabs(fr[2]) < 1e300)) st |= GFP_ST_NON_FINITE;
    return st;
}

/*
 * The binned BSM composition of ONE point at SEVERAL new-physics scales (the sensitivity grid of
 * scripts/sens.py:232-294 evaluates the same prior sample at every grid value of log10(Lambda)): everything that does not
 * depend on the scale -- the PMNS columns, H0, the new-physics matrix T and the pencil coefficients -- is built once, then
 * `emit(s, fr, status)` is called with the composition at lam_of(s) = 10^logLam_s for s = 0 .. ns-1.  Same arithmetic per
 * scale as gf_point_fr (which is the ns = 1 case with lam = exp10(q.loglam)).
 */
template <int SPEC, int ILP, class LamOf, class Emit, class ThetaSrc = gf_no_src>
GF_HD void gf_point_fr_scales(const gf_dev_model& m, const gf_point& q, int ns, LamOf lam_of, Emit emit, const ThetaSrc& src = ThetaSrc()) {
    static_assert(!GF_SPEC_IS_SM(SPEC), "the scale grid needs the BSM path");
    gfp_herm3 h0, T;
    double m1, m2;
    gf_point_matrices<SPEC>(m, q, h0, T, m1, m2);
    auto finish = [&](int s, unsigned st, double* fr) {
        const double mn = fmin(fr[0], fmin(fr[1], fr[2]));
        if (!(mn >= -m.epsilon)) st |= GFP_ST_NON_UNITARY;
        if (!(fabs(fr[0]) + fabs(fr[1]) + fabs(fr[2]) < 1e300)) st |= GFP_ST_NON_FINITE;
        emit(s, fr, st);
    };
    auto run = [&](const auto& mats) {
        if (GF_SPEC_IS_FIXED(SPEC)) {
            const gfp_pencil_P pp = gfp_make_pencil_P(h0, m1, m2, m.T, m.penT.te, m.adjT);
            for (int s = 0; s < ns; ++s) {
                double fr[3];
                const unsigned st = gf_bin_loop<ILP, 1>(m, pp, m.penT, mats, lam_of(s), m.fixed_src[2], m.src_sd0, m.src_sd1, m.inv_S_wsum, m.src_S, fr);
                finish(s, st, fr);
            }
        } else {
            const bool npf = GF_SPEC_IS_NPFREE(SPEC) || m.np_free;
            const gfp_pencil_T pt = gfp_make_pencil_T(T);
            const gfp_pencil_P pp = gfp_make_pencil_P(h0, m1, m2, T, pt.te, npf ? gfp_adj_tf(pt.te, T) : m.adjT);
            const bool fixed_src = GF_SPEC_IS_NPFREE(SPEC) || gf_model_has_fixed_source(m);
            const double S = fixed_src ? m.src_S : q.src[0] + q.src[1] + q.src[2];
            const double s2 = fixed_src ? m.fixed_src[2] : q.src[2];
            const double sd0 = fixed_src ? m.src_sd0 : q.src[0] - q.src[2], sd1 = fixed_src ? m.src_sd1 : q.src[1] - q.src[2];
            const double inv_norm = fixed_src ? m.inv_S_wsum : gfp_rcp(S * m.wsum);
            for (int s = 0; s < ns; ++s) {
                double fr[3];
                const unsigned st = gf_bin_loop<ILP, 1>(m, pp, pt, mats, lam_of(s), s2, sd0, sd1, inv_norm, S, fr);
                finish(s, st, fr);
            }
        }
    };
    if constexpr (std::is_same<ThetaSrc, gf_no_src>::value) {
        run(gf_mats_ptr{&h0, GF_SPEC_IS_FIXED(SPEC) ? &m.T : &T});
    } else {
        run(gf_mats_rebuild<SPEC, ThetaSrc>{&m, src});
    }
}

/*
 * The energy-bin loop of gf_bin_loop (same fast path, same rare refinement, ILP interleaved chains, LANES = 1) with a
 * source-independent result: the bin-width-weighted sums of the transition P = X X^T in its three independent entries,
 * A[0..2] = sum_b w_b (P00, P01, P11) (gfp_x4_transition).  gfp_transition_fr turns them into the composition of any
 * source.  Returns the status bits of the eigen stage.
 */
template <int ILP, class TPART, class MATS>
GF_HD unsigned gf_bin_loop_transition(const gf_dev_model& m, const gfp_pencil_P& pp, const TPART& pt, const MATS& mats, double lam, double* A) {
    unsigned st = 0u;
    double a00 = 0.0, a01 = 0.0, a11 = 0.0;
    int b = 0;
    if (ILP > 1) {
        for (; b + ILP - 1 < m.nbins; b += ILP) {
            gfp_x4 x[ILP];
            bool ok = true;
#pragma unroll
            for (int i = 0; i < ILP; ++i) ok = gfp_pencil_x4_fast(pp, pt, lam * m.g[b + i], x[i]) && ok;
            if (!ok) {
#pragma unroll
                for (int i = 0; i < ILP; ++i) {
                    gfp_x4 again;
                    if (!gfp_pencil_x4_fast(pp, pt, lam * m.g[b + i], again)) {
                        gfp_x4 slow;
                        st |= gf_refine_bin(mats, lam * m.g[b + i], &slow);
                        x[i] = slow;
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < ILP; ++i) {
                double p00, p01, p11;
                gfp_x4_transition(x[i], p00, p01, p11);
                const double wd = m.width[b + i];
                a00 = fma(wd, p00, a00);
                a01 = fma(wd, p01, a01);
                a11 = fma(wd, p11, a11);
            }
        }
    }
    for (; b < m.nbins; ++b) {
        const double rho = lam * m.g[b];
        gfp_x4 x;
        if (!gfp_pencil_x4_fast(pp, pt, rho, x)) {
            gfp_x4 slow;
            st |= gf_refine_bin(mats, rho, &slow);
            x = slow;
        }
        double p00, p01, p11;
        gfp_x4_transition(x, p00, p01, p11);
        const double wd = m.width[b];
        a00 = fma(wd, p00, a00);
        a01 = fma(wd, p01, a01);
        a11 = fma(wd, p11, a11);
    }
    A[0] = a00;
    A[1] = a01;
    A[2] = a11;
    return st;
}

/*
 * The twin of gf_point_fr_scales for many sources at once: the same once-per-point set-up (PMNS, H0, T, pencil, refinement
 * matrices), then `emit(s, A, status)` per scale with the transition sums A of gf_bin_loop_transition at lam_of(s).  The
 * model's source (fixed_src, sampled source columns) is not used.  status carries the eigen-stage bits and
 * GFP_ST_NON_FINITE; unitarity is a property of a composition, hence of a source, and is not tested here.
 */
template <int SPEC, int ILP, class LamOf, class Emit, class ThetaSrc = gf_no_src>
GF_HD void gf_point_transition_scales(const gf_dev_model& m, const gf_point& q, int ns, LamOf lam_of, Emit emit, const ThetaSrc& src = ThetaSrc()) {
    static_assert(!GF_SPEC_IS_SM(SPEC), "the scale grid needs the BSM path");
    gfp_herm3 h0, T;
    double m1, m2;
    gf_point_matrices<SPEC>(m, q, h0, T, m1, m2);
    auto finish = [&](int s, unsigned st, double* A) {
        if (!(fabs(A[0]) + fabs(A[1]) + fabs(A[2]) < 1e300)) st |= GFP_ST_NON_FINITE;
        emit(s, A, st);
    };
    auto run = [&](const auto& mats) {
        if (GF_SPEC_IS_FIXED(SPEC)) {
            const gfp_pencil_P pp = gfp_make_pencil_P(h0, m1, m2, m.T, m.penT.te, m.adjT);
            for (int s = 0; s < ns; ++s) {
                double A[3];
                const unsigned st = gf_bin_loop_transition<ILP>(m, pp, m.penT, mats, lam_of(s), A);
                finish(s, st, A);
            }
        } else {
            const bool npf = GF_SPEC_IS_NPFREE(SPEC) || m.np_free;
            const gfp_pencil_T pt = gfp_make_pencil_T(T);
            const gfp_pencil_P pp = gfp_make_pencil_P(h0, m1, m2, T, pt.te, npf ? gfp_adj_tf(pt.te, T) : m.adjT);
            for (int s = 0; s < ns; ++s) {
                double A[3];
                const unsigned st = gf_bin_loop_transition<ILP>(m, pp, pt, mats, lam_of(s), A);
                finish(s, st, A);
            }
        }
    };
    if constexpr (std::is_same<ThetaSrc, gf_no_src>::value) {
        run(gf_mats_ptr{&h0, GF_SPEC_IS_FIXED(SPEC) ? &m.T : &T});
    } else {
        run(gf_mats_rebuild<SPEC, ThetaSrc>{&m, src});
    }
}

GF_HD int gf_model_gauss_mask(const gf_dev_model& m) {
    int mask = 0;
    for (int k = 0; k < m.ndim; ++k) mask |= (m.kind[k] != GF_PRIOR_UNIFORM) << k;
    return mask;
}

GF_HD bool gf_model_has_fixed_source(const gf_dev_model& m) { return m.col_src[0] < 0 && m.col_x < 0 && m.col_src3[0] < 0; }

GF_HD bool gf_model_is_fixed_spec(const gf_dev_model& m) { return !m.no_bsm && !m.np_free && gf_model_has_fixed_source(m); }

/* columns 0-3 the mixing coordinates, 4-5 the mass splittings: the head of the layout of sens.py */
GF_HD bool gf_model_has_head6(const gf_dev_model& m) {
    return m.col_sm[0] == 0 && m.col_sm[1] == 1 && m.col_sm[2] == 2 && m.col_sm[3] == 3 && m.col_mass[0] == 4 && m.col_mass[1] == 5;
}

/* the specialisation a model's COLUMN LAYOUT allows (kernels without a GF_SPEC_NPFREE instance map it to GF_SPEC_GENERIC) */
GF_HD int gf_model_layout_spec(const gf_dev_model& m) {
    if (m.no_bsm) {
        const bool canon = m.ndim == 6 && m.col_sm[0] == 0 && m.col_sm[1] == 1 && m.col_sm[2] == 2 && m.col_sm[3] == 3 &&
                           m.col_src[0] == 4 && m.col_src[1] == 5 && m.col_x < 0 && m.col_src3[0] < 0;
        return canon ? GF_SPEC_SM6 : GF_SPEC_SM;
    }
    if (!gf_model_has_fixed_source(m)) return GF_SPEC_GENERIC;
    if (m.np_free) return GF_SPEC_NPFREE;
    const bool head = gf_model_has_head6(m);
    if (head && m.ndim == 7 && m.col_scale == 6) return GF_SPEC_FIXED7;
    if (head && m.ndim == 12 && m.col_scale == 11) return GF_SPEC_FIXED12;
    return GF_SPEC_FIXED;
}

/* which instance the frozen-scale grid kernels (k_evidence_grid, k_evidence_sources, k_profile, k_profile_sources) launch:
 * 2 = <GF_SPEC_FIXED, STATIC6> for the six columns of sens.py, 1 = <GF_SPEC_FIXED, false>, 0 = <GF_SPEC_GENERIC, false> */
GF_HD int gf_model_grid_spec(const gf_dev_model& m) {
    const bool fixed = gf_model_is_fixed_spec(m);
    return fixed && m.ndim == 6 && gf_model_has_head6(m) ? 2 : fixed ? 1 : 0;
}

/* which specialisation the log-posterior and sampler kernels launch: the layout's, unless it also fixes the prior kinds at
 * compile time (GF_SPEC_STATIC_GMASK) and the model's differ -- then the runtime-layout sibling */
GF_HD int gf_model_spec(const gf_dev_model& m) {
    const int spec = gf_model_layout_spec(m);
    if (spec == GF_SPEC_SM6 && gf_model_gauss_mask(m) != GF_SPEC_STATIC_GMASK(GF_SPEC_SM6)) return GF_SPEC_SM;
    if (spec == GF_SPEC_FIXED7 && gf_model_gauss_mask(m) != GF_SPEC_STATIC_GMASK(GF_SPEC_FIXED7)) return GF_SPEC_FIXED;
    return spec;
}

/* which specialisation the scan kernels launch: their own compile-time layouts where the model has one */
GF_HD int gf_model_scan_spec(const gf_dev_model& m) {
    const int spec = gf_model_layout_spec(m); /* the scans draw from the priors: no prior-kind specialisation */
    const bool sm03 = m.col_sm[0] == 0 && m.col_sm[1] == 1 && m.col_sm[2] == 2 && m.col_sm[3] == 3;
    if (spec == GF_SPEC_SM6) return GF_SPEC_SM;
    if (spec == GF_SPEC_SM) {
        if (sm03 && m.ndim == 4 && gf_model_has_fixed_source(m)) return GF_SPEC_SM4;
        if (sm03 && m.ndim == 5 && m.col_x == 4) return GF_SPEC_SM5X;
        return GF_SPEC_SM;
    }
    if (spec == GF_SPEC_FIXED12) return GF_SPEC_FIXED;
    if (spec == GF_SPEC_NPFREE) {
        const bool canon = sm03 && m.ndim == 11 && m.col_mass[0] == 4 && m.col_mass[1] == 5 && m.col_np[0] == 6 && m.col_np[1] == 7 &&
                           m.col_np[2] == 8 && m.col_np[3] == 9 && m.col_scale == 10;
        return canon ? GF_SPEC_NPFREE11 : GF_SPEC_NPFREE;
    }
    return spec; /* GENERIC, FIXED, FIXED7 */
}

/* llh.lnprior (llh.py:74-90): -inf outside the box, sum of (truncated) Gaussian log-pdfs inside.
 * The normalisers of all Gaussian dimensions are pre-summed on the host (m.lognorm_total).  Uniform
 * dimensions (llh.py:80-81: they contribute nothing) skip the Gaussian term on a WARP-UNIFORM predicate --
 * m.kind[k] is a constant-bank word and k a compile-time index, so the test runs on the uniform datapath and
 * saves three fp64-pipe instructions per uniform dimension; it also keeps an infinite coordinate inside an
 * unbounded box from turning into inf * 0 = NaN. */
template <int NDIM = 0, int GMASK = -1, class Get>
GF_HD double gf_point_lnprior(const gf_dev_model& m, Get get) {
    double acc = 0.0;
    bool inside = true;
    /* fully unrolled with an early exit on the (warp-uniform) dimension count: with a compile-time k the
     * prior tables are constant-bank operands of the compares and the FMA instead of indexed constant
     * loads -- the rolled loop was 21 % of the instructions of the SM-only kernel */
#pragma unroll
    for (int k = 0; k < (NDIM > 0 ? NDIM : GF_MAX_DIM); ++k) {
        if (NDIM == 0 && k >= m.ndim) break;
        const double v = get(k);
        inside = inside & (v >= m.lo[k]) & (v <= m.hi[k]); /* no short circuit: twelve chained compares, no branches */
        if (GMASK >= 0 ? ((GMASK >> k) & 1) != 0 : m.kind[k] != GF_PRIOR_UNIFORM) {
            const double z = (v - m.mu[k]) * m.inv_sigma[k];
            acc = fma(z, z, acc);
        }
    }
    return inside ? fma(-0.5, acc, m.lognorm_total) : -INFINITY;
}

/* llh.multi_gaussian (llh.py:53-54) in closed form, with the pdf-underflow -> -inf emulation. */
GF_HD double gf_multi_gaussian(const double* fr, const double* bf, double half_inv_s2, double lognorm3, double offset,
                               int emulate_underflow, double underflow_logpdf) {
    const double d0 = fr[0] - bf[0], d1 = fr[1] - bf[1], d2 = fr[2] - bf[2];
    const double logpdf = fma(-half_inv_s2, fma(d0, d0, fma(d1, d1, d2 * d2)), lognorm3);
    if (emulate_underflow && logpdf < underflow_logpdf) return -INFINITY;
    return logpdf + offset;
}

/* llh.ln_prob (llh.py:121-130) with the Gaussian (or flat) likelihood. */
template <int SPEC = GF_SPEC_GENERIC, int ILP = 1, int LANES = 1, class Get, class ThetaSrc = gf_no_src>
GF_HD double gf_point_lnprob(const gf_dev_model& m, Get get, double* fr, unsigned& st, int lane = 0, const ThetaSrc& src = ThetaSrc()) {
    const double lp = gf_point_lnprior<GF_SPEC_STATIC_NDIM(SPEC), GF_SPEC_STATIC_GMASK(SPEC)>(m, get);
    GF_STAGE(3);
    if (!(lp > -INFINITY)) { /* -inf, or NaN from a NaN theta */
        fr[0] = fr[1] = fr[2] = NAN;
        st = (lp != lp) ? (GFP_ST_NON_FINITE | GFP_ST_OUT_OF_PRIOR) : GFP_ST_OUT_OF_PRIOR;
        return (lp != lp) ? NAN : -INFINITY;
    }
    gf_point q;
    gf_resolve_point<SPEC>(m, get, q);
    st = gf_point_fr<SPEC, ILP, LANES>(m, q, fr, lane, src);
    /* scripts/mc_*.py triangle_llh: parameters are only stored, "return 1. # Flat LLH" */
    if (m.llh_kind == GF_LLH_FLAT) return lp + m.llh_const;
    const double out = lp + gf_multi_gaussian(fr, m.fr_bf, m.half_inv_s2, m.lognorm3, m.offset, m.emulate_underflow, m.underflow_logpdf);
    GF_STAGE(9);
    return out;
}

#endif /* GF_MODEL_CUH */
