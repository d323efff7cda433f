/*
 * gf_sources_dev.cuh -- per-sample pieces of the evidence grid over many source compositions (k_evidence_sources,
 * gf_sources.cu): the source table passed by value, the physics of one prior sample at several scales, the likelihood of
 * one (sample, scale, source) and the running log-sum-exp.  __host__ __device__, so that the host harness runs the same
 * code sequentially.
 *
 * The reference's sensitivity study runs scripts/sens.py once per (dimension, texture, source composition, Lambda
 * segment) (submitter/sens_dag.py:8-16, 38-61, 76-95).  The eigen stage of a sample does not depend on the source: it
 * enters only through fr_b = sum_a P_ba s_a (fr.py:441-457), and the transition sums of gf_bin_loop_transition give that
 * for every source at the cost of a few instructions each.
 */
#ifndef GF_SOURCES_DEV_CUH
#define GF_SOURCES_DEV_CUH

#include "gf_scan_dev.cuh"

/* sources per launch: 56 bytes each in the kernel parameter, 14 KB of the 32 KB sm_100 allows */
#define GF_SRC_MAX 256

/* one source: its composition in the form of gfp_transition_fr and the injected composition it is scored against */
struct gf_src_rec {
    gfp_src_consts c;
    double bf[3];
};

struct gf_src_table {
    gf_src_rec src[GF_SRC_MAX];
    int32_t nsrc, reserved;
};

/* Normalise source s and injected composition inj as model.flatten normalises them (x / sum(x)) and derive the record for
 * bin-width sum W.  false (nothing written) for a negative or non-finite entry or a zero sum. */
GF_HD bool gf_src_record(const double* s, const double* inj, double W, gf_src_rec* out) {
    for (int k = 0; k < 3; ++k)
        if (!(s[k] >= 0.0 && s[k] < 1e300 && inj[k] >= 0.0 && inj[k] < 1e300)) return false;
    const double S = s[0] + s[1] + s[2], I = inj[0] + inj[1] + inj[2];
    if (!(S > 0.0 && S < 1e300 && I > 0.0 && I < 1e300)) return false;
    const double n0 = s[0] / S, n1 = s[1] / S, n2 = s[2] / S;
    out->c = gfp_source_consts(n0, n1, n2, W);
    for (int k = 0; k < 3; ++k) out->bf[k] = inj[k] / I;
    return true;
}

/* The source table of a source-list entry point `who` (host): refuses a model that samples the source or has no Gaussian
 * likelihood, and a composition gf_src_record refuses; fills S from sources[nsrc][3] / injected[nsrc][3] otherwise. */
int gf_src_table_fill(const char* who, const gf_dev_model& d, const double* sources, const double* injected, int nsrc, gf_src_table* S);

/* llh.multi_gaussian of source r's composition fr (written) from the transition sums A of one (sample, scale) */
GF_HD double gf_src_llh(const gf_dev_model& m, const gf_src_rec& r, const double* A, double* fr) {
    gfp_transition_fr(A, r.c, fr);
    return gf_multi_gaussian(fr, r.bf, m.half_inv_s2, m.lognorm3, m.offset, m.emulate_underflow, m.underflow_logpdf);
}

GF_HD double gf_src_llh(const gf_dev_model& m, const gf_src_rec& r, const double* A) {
    double fr[3];
    return gf_src_llh(m, r, A, fr);
}

/* the running log-sum-exp of one (scale, source) pair: gf_lse_push, under the name the source grid's host harness calls */
GF_HD void gf_src_lse_push(double& mo, double& so, double ll) { gf_lse_push(mo, so, ll); }

/* The physics of prior sample `index` (the draw of gf_scan_evidence_grid) at the ns scales lam[0..ns-1]:
 * emit(k, A, status) per scale.  STATIC6: the layout of sens.py, columns 0-3 mixing coordinates, 4-5 mass splittings. */
template <int SPEC, bool STATIC6, int ILP, class Emit>
GF_HD void gf_src_sample(const gf_dev_model& m, uint64_t seed, uint64_t index, int ns, const double* lam, Emit emit) {
    double theta[GF_MAX_DIM];
    gf_point q;
    if constexpr (STATIC6) {
        gf_draw_theta<true, 6>(m, seed, index, theta);
        q.sm[0] = theta[0]; q.sm[1] = theta[1]; q.sm[2] = theta[2]; q.sm[3] = theta[3];
        q.mass[0] = theta[4]; q.mass[1] = theta[5];
    } else {
        gf_draw_theta(m, seed, index, theta);
        gf_resolve_point<SPEC>(m, [&](int k) { return theta[k]; }, q);
    }
    gf_point_transition_scales<SPEC, ILP>(m, q, ns, [&](int k) { return lam[k]; }, emit);
}

#endif /* GF_SOURCES_DEV_CUH */
