/*
 * TEST INFRASTRUCTURE ONLY -- never linked into libgolemflavor_b200.so, never imported by the product package.
 *
 * Host instantiation of the per-sample code of gf_scan_evidence_sources (golemflavor_b200/csrc/gf_sources_dev.cuh): the
 * transition sums of one point and the composition of a source from them, and the whole task (draw, eigen stage per scale,
 * likelihood per source, running log-sum-exp in sample order) run sequentially, so that the CPU test-suite checks the
 * algorithm before any GPU time is spent.  Built like harness.cu (g++, -ffp-contract=off).
 */
#include <string.h>

#include <vector>

#include "../../golemflavor_b200/csrc/gf_common.cuh"
#include "../../golemflavor_b200/csrc/gf_sources_dev.cuh"

/* For every point (its own logLam): the transition sums A[n][3] and fr[n][nsrc][3] of each source through
 * gfp_transition_fr.  spec: 1 = FIXED, 0 = GENERIC, -1 = as the library chooses. */
extern "C" int hh_transition_fr(const gf_model* model, const double* theta, int64_t n, const double* sources, int nsrc, int spec, double* A,
                                double* fr, uint8_t* st) {
    gf_dev_model d;
    if (int rc = gf_build_dev_model(model, &d)) return rc;
    if (d.no_bsm) return GF_ERR_ARG;
    const bool fixed = spec < 0 ? gf_model_is_fixed_spec(d) : spec == 1;
    std::vector<gf_src_rec> rec(nsrc);
    const double one[3] = {1.0, 1.0, 1.0};
    for (int j = 0; j < nsrc; ++j)
        if (!gf_src_record(sources + 3 * j, one, d.wsum, &rec[j])) return GF_ERR_ARG;
    for (int64_t i = 0; i < n; ++i) {
        auto get = [&](int k) { return theta[i * d.ndim + k]; };
        gf_point q;
        auto emit = [&](int, const double* a, unsigned s) {
            memcpy(A + 3 * i, a, 3 * sizeof(double));
            st[i] = (uint8_t)s;
            for (int j = 0; j < nsrc; ++j) gfp_transition_fr(a, rec[j].c, fr + 3 * (i * nsrc + j));
        };
        if (fixed) {
            gf_resolve_point<GF_SPEC_FIXED>(d, get, q);
            const double lam = pow(10.0, q.loglam);
            gf_point_transition_scales<GF_SPEC_FIXED, 2>(d, q, 1, [&](int) { return lam; }, emit);
        } else {
            gf_resolve_point<GF_SPEC_GENERIC>(d, get, q);
            const double lam = pow(10.0, q.loglam);
            gf_point_transition_scales<GF_SPEC_GENERIC, 1>(d, q, 1, [&](int) { return lam; }, emit);
        }
    }
    return 0;
}

/* The task of gf_scan_evidence_sources for samples first .. first + count - 1 in index order: lse[nsrc][ns][2] accumulates
 * (max, sum) like the device (initialise to {-inf, 0}).  The same refusals as the entry point, as GF_ERR_ARG. */
extern "C" int hh_evidence_sources(const gf_model* model, uint64_t seed, uint64_t first, int64_t count, const double* scales, int ns,
                                   const double* sources, const double* injected, int nsrc, double* lse) {
    gf_dev_model d;
    if (int rc = gf_build_dev_model(model, &d)) return rc;
    if (d.no_bsm || d.col_scale >= 0 || !gf_model_has_fixed_source(d) || d.llh_kind != GF_LLH_GAUSSIAN) return GF_ERR_ARG;
    std::vector<gf_src_rec> rec(nsrc);
    for (int j = 0; j < nsrc; ++j)
        if (!gf_src_record(sources + 3 * j, injected + 3 * j, d.wsum, &rec[j])) return GF_ERR_ARG;
    std::vector<double> lam(ns);
    for (int k = 0; k < ns; ++k) lam[k] = pow(10.0, scales[k]);
    const bool fixed = gf_model_is_fixed_spec(d);
    const bool static6 = fixed && d.ndim == 6 && d.col_sm[0] == 0 && d.col_sm[1] == 1 && d.col_sm[2] == 2 && d.col_sm[3] == 3 &&
                         d.col_mass[0] == 4 && d.col_mass[1] == 5;
    for (int64_t i = 0; i < count; ++i) {
        auto emit = [&](int k, const double* A, unsigned st) {
            for (int j = 0; j < nsrc; ++j) {
                const double ll = (st & GFP_ST_NON_FINITE) ? NAN : gf_src_llh(d, rec[j], A);
                double* o = lse + 2 * ((size_t)j * ns + k);
                gf_src_lse_push(o[0], o[1], ll);
            }
        };
        if (static6) gf_src_sample<GF_SPEC_FIXED, true, 2>(d, seed, first + (uint64_t)i, ns, lam.data(), emit);
        else if (fixed) gf_src_sample<GF_SPEC_FIXED, false, 2>(d, seed, first + (uint64_t)i, ns, lam.data(), emit);
        else gf_src_sample<GF_SPEC_GENERIC, false, 1>(d, seed, first + (uint64_t)i, ns, lam.data(), emit);
    }
    return 0;
}
