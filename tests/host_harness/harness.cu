/*
 * TEST INFRASTRUCTURE ONLY -- never linked into libgolemflavor_b200.so, never imported by the
 * product package.
 *
 * The per-point functions of golemflavor_b200/csrc/gf_*.cuh are `__host__ __device__` (the library
 * uses the host instantiation for model constants such as the texture matrix).  This harness
 * instantiates them on the host in a plain loop so that the CPU test-suite (`-m "not gpu"`, no GPU
 * in the build container) can compare the kernels' ALGORITHM -- closed-form eigen stage, Jacobi
 * fallback thresholds, prior / likelihood composition, Philox stream, histogram bin index -- with
 * the oracle before any GPU time is spent.  The GPU parity tests (`-m gpu`) remain the parity
 * tests proper and go through the C ABI.
 */
#include <string.h>

#include "../../golemflavor_b200/csrc/gf_common.cuh"
#include "../../golemflavor_b200/csrc/gf_ensemble_dev.cuh"

/* spec < 0: choose like the library does (FIXED specialisation when the model is eligible) */
static bool use_fixed(const gf_dev_model& d, int spec) { return spec < 0 ? gf_model_is_fixed_spec(d) : spec == GF_SPEC_FIXED; }

/* which specialisation gf_lnprob / the sampler would launch for the model (layout AND prior kinds) */
extern "C" int hh_model_spec(const gf_model* model, int* spec, int* layout_spec, int* gauss_mask) {
    gf_dev_model d;
    if (int rc = gf_build_dev_model(model, &d)) return rc;
    *spec = gf_model_spec(d);
    *layout_spec = gf_model_layout_spec(d);
    *gauss_mask = gf_model_gauss_mask(d);
    return 0;
}

extern "C" int hh_lnprob(const gf_model* model, const double* theta, int64_t n, double* lnp, double* fr, uint8_t* st, int spec) {
    gf_dev_model d;
    if (int rc = gf_build_dev_model(model, &d)) return rc;
    const bool fixed = use_fixed(d, spec);
    for (int64_t i = 0; i < n; ++i) {
        auto get = [&](int k) { return theta[i * d.ndim + k]; };
        unsigned s = 0u;
        double f[3];
        /* the compile-time layouts (and prior-kind masks) on request: the caller vouches for the model's layout */
        if (spec == GF_SPEC_SM6) lnp[i] = gf_point_lnprob<GF_SPEC_SM6, 1>(d, get, f, s);
        else if (spec == GF_SPEC_SM) lnp[i] = gf_point_lnprob<GF_SPEC_SM, 1>(d, get, f, s);
        else if (spec == GF_SPEC_FIXED7) lnp[i] = gf_point_lnprob<GF_SPEC_FIXED7, 2>(d, get, f, s);
        else
        lnp[i] = fixed ? gf_point_lnprob<GF_SPEC_FIXED, 2>(d, get, f, s) : gf_point_lnprob<GF_SPEC_GENERIC, 2>(d, get, f, s); /* as k_lnprob */
        if (fr) memcpy(fr + 3 * i, f, sizeof(f));
        if (st) st[i] = (uint8_t)s;
    }
    return 0;
}

extern "C" int hh_fr(const gf_model* model, const double* theta, int64_t n, double* fr, uint8_t* st, int spec) {
    gf_dev_model d;
    if (int rc = gf_build_dev_model(model, &d)) return rc;
    const bool fixed = use_fixed(d, spec);
    for (int64_t i = 0; i < n; ++i) {
        auto get = [&](int k) { return theta[i * d.ndim + k]; };
        gf_point q;
        unsigned s;
        if (fixed) {
            gf_resolve_point<GF_SPEC_FIXED>(d, get, q);
            s = gf_point_fr<GF_SPEC_FIXED>(d, q, fr + 3 * i);
        } else {
            gf_resolve_point<GF_SPEC_GENERIC>(d, get, q);
            s = gf_point_fr<GF_SPEC_GENERIC>(d, q, fr + 3 * i);
        }
        if (st) st[i] = (uint8_t)s;
    }
    return 0;
}

extern "C" int hh_lnprior(const gf_model* model, const double* theta, int64_t n, double* lnp) {
    gf_dev_model d;
    if (int rc = gf_build_dev_model(model, &d)) return rc;
    for (int64_t i = 0; i < n; ++i) lnp[i] = gf_point_lnprior(d, [&](int k) { return theta[i * d.ndim + k]; });
    return 0;
}

extern "C" void hh_philox(const uint32_t* ctr /*[n][4]*/, int64_t n, uint32_t k0, uint32_t k1, uint32_t* out /*[n][4]*/) {
    for (int64_t i = 0; i < n; ++i) {
        const gf_u4 r = gf_philox4x32_10(ctr[4 * i], ctr[4 * i + 1], ctr[4 * i + 2], ctr[4 * i + 3], k0, k1);
        out[4 * i] = r.x; out[4 * i + 1] = r.y; out[4 * i + 2] = r.z; out[4 * i + 3] = r.w;
    }
}

extern "C" int hh_draw(const gf_model* model, uint64_t seed, uint64_t first, int64_t n, double* theta) {
    gf_dev_model d;
    if (int rc = gf_build_dev_model(model, &d)) return rc;
    for (int64_t i = 0; i < n; ++i) gf_draw_theta(d, seed, first + (uint64_t)i, theta + i * d.ndim);
    return 0;
}

extern "C" void hh_hist(const double* fr, int64_t n, int nb, unsigned long long* hist) {
    const int nb1 = nb + 1;
    const double step = 1.0 / (double)nb1;
    for (int64_t i = 0; i < n; ++i) {
        const int c = gf_cell_index(fr + 3 * i, nb1, step);
        if (c >= 0) ++hist[c];
    }
}

extern "C" void hh_eig(const double* ham /*[n][18]*/, int64_t n, double* lam, double* vec, double* x_fast /*[n][4]*/, uint8_t* fast_ok) {
    for (int64_t i = 0; i < n; ++i) {
        const double* h = ham + 18 * i;
        gfp_herm3 m;
        m.d0 = h[0]; m.d1 = h[8]; m.d2 = h[16];
        m.ar = h[2]; m.ai = h[3]; m.br = h[4]; m.bi = h[5]; m.cr = h[10]; m.ci = h[11];
        gfp_herm3_eig_sorted(m, lam + 3 * i, vec + 18 * i);
        gfp_x4 x = {NAN, NAN, NAN, NAN};
        fast_ok[i] = gfp_herm3_x4_fast(m, x) ? 1 : 0;
        x_fast[4 * i] = x.x00; x_fast[4 * i + 1] = x.x01; x_fast[4 * i + 2] = x.x10; x_fast[4 * i + 3] = x.x11;
    }
}

/* deflation refinement of single matrices: x4 = (|V_00|^2, |V_01|^2, |V_10|^2, |V_11|^2), status bits */
extern "C" void hh_deflate(const double* ham /*[n][18]*/, int64_t n, double* x4 /*[n][4]*/, uint8_t* st) {
    for (int64_t i = 0; i < n; ++i) {
        const double* h = ham + 18 * i;
        gfp_herm3 m;
        m.d0 = h[0]; m.d1 = h[8]; m.d2 = h[16];
        m.ar = h[2]; m.ai = h[3]; m.br = h[4]; m.bi = h[5]; m.cr = h[10]; m.ci = h[11];
        gfp_x4 x = {NAN, NAN, NAN, NAN};
        st[i] = (uint8_t)gfp_herm3_x4_deflate(m, x);
        x4[4 * i] = x.x00; x4[4 * i + 1] = x.x01; x4[4 * i + 2] = x.x10; x4[4 * i + 3] = x.x11;
    }
}

/* sequential replay of gf_ensemble_run: same update function, same order of half-steps */
extern "C" int hh_ensemble(const gf_model* model, const gf_ensemble_config* cfg, double* pos, double* lnp, double* chain,
                           double* lnp_chain, unsigned long long* naccept) {
    gf_dev_model d;
    if (int rc = gf_build_dev_model(model, &d)) return rc;
    gf_ens_args A;
    A.nchains = cfg->nchains; A.nsteps = cfg->nsteps; A.step0 = cfg->step0; A.thin = cfg->thin;
    A.nwalkers = cfg->nwalkers; A.nfree = cfg->nfree; A.a = cfg->a; A.seed = cfg->seed; A.chain0 = cfg->chain0;
    A.pos = pos; A.lnp = lnp; A.chain = chain; A.lnp_chain = lnp_chain; A.naccept = naccept;
    const int half = cfg->nwalkers / 2;
    const int64_t nstore = cfg->nsteps / cfg->thin;
    for (int64_t s = 0; s < cfg->nsteps; ++s) {
        for (int h = 0; h < 2; ++h) {
            /* the whole half proposes from the state BEFORE any walker of that half moved: partners
             * come from the other half, so updating in place is equivalent */
            for (int64_t c = 0; c < cfg->nchains; ++c)
                for (int w = 0; w < half; ++w) {
                    const unsigned acc = gf_ens_update(d, A, c, h * half + w, h, cfg->step0 + s);
                    if (naccept) naccept[c * cfg->nwalkers + h * half + w] += acc;
                }
        }
        if ((s + 1) % cfg->thin == 0 && (s + 1) / cfg->thin <= nstore)
            for (int64_t c = 0; c < cfg->nchains; ++c)
                for (int k = 0; k < cfg->nwalkers; ++k) gf_ens_store(d, A, c, k, (s + 1) / cfg->thin - 1, nstore);
    }
    return 0;
}

extern "C" void hh_cubic_w(const double* delta, int64_t n, double* w) {
    for (int64_t i = 0; i < n; ++i) w[i] = gfp_cubic_w(delta[i]);
}

/* the multi-scale evaluation of the evidence grid: fr[n][ns][3] at logLam = scales[s] for every point (the model's own
 * scale column / fixed_loglam is ignored) */
extern "C" int hh_fr_scales(const gf_model* model, const double* theta, int64_t n, const double* scales, int ns, double* fr, uint8_t* st) {
    gf_dev_model d;
    if (int rc = gf_build_dev_model(model, &d)) return rc;
    const bool fixed = gf_model_is_fixed_spec(d);
    for (int64_t i = 0; i < n; ++i) {
        auto get = [&](int k) { return theta[i * d.ndim + k]; };
        gf_point q;
        auto lam_of = [&](int s) { return pow(10.0, scales[s]); };
        auto emit = [&](int s, const double* f, unsigned status) {
            memcpy(fr + 3 * (i * ns + s), f, 3 * sizeof(double));
            if (st) st[i * ns + s] = (uint8_t)status;
        };
        if (fixed) {
            gf_resolve_point<GF_SPEC_FIXED>(d, get, q);
            gf_point_fr_scales<GF_SPEC_FIXED, 2>(d, q, ns, lam_of, emit);
        } else {
            gf_resolve_point<GF_SPEC_GENERIC>(d, get, q);
            gf_point_fr_scales<GF_SPEC_GENERIC, 1>(d, q, ns, lam_of, emit);
        }
    }
    return 0;
}

/* the table-based inverse normal CDF of the prior draws: z[i] and whether the table covered p[i] */
extern "C" void hh_ndtri(const double* p, int64_t n, double* z, uint8_t* covered) {
    for (int64_t i = 0; i < n; ++i) {
        double v = NAN;
        covered[i] = gf_ndtri_table(p[i], &v) ? 1 : 0;
        z[i] = v;
    }
}

/* the log-posterior with the refinement path REBUILDING H0 / T from the row (as k_lnprob does) instead of keeping them */
extern "C" int hh_lnprob_rebuild(const gf_model* model, const double* theta, int64_t n, double* lnp, double* fr, uint8_t* st, int spec) {
    gf_dev_model d;
    if (int rc = gf_build_dev_model(model, &d)) return rc;
    const bool fixed = use_fixed(d, spec);
    for (int64_t i = 0; i < n; ++i) {
        const double* row = theta + i * d.ndim;
        auto get = [&](int k) { return row[k]; };
        const gf_src_row again{row, 1};
        unsigned s = 0u;
        double f[3];
        lnp[i] = fixed ? gf_point_lnprob<GF_SPEC_FIXED, 2, 1>(d, get, f, s, 0, again) : gf_point_lnprob<GF_SPEC_GENERIC, 2, 1>(d, get, f, s, 0, again);
        if (fr) memcpy(fr + 3 * i, f, sizeof(f));
        if (st) st[i] = (uint8_t)s;
    }
    return 0;
}

/* the fast path's sin^2(phi/3) threshold and the high word the device compares with */
extern "C" unsigned hh_fast_min_sin2(double* thr) {
    *thr = GFP_FAST_MIN_SIN2;
    return GFP_FAST_MIN_SIN2_HI;
}
