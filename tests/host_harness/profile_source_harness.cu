/*
 * TEST INFRASTRUCTURE ONLY -- never linked into libgolemflavor_b200.so, never imported by the product package.
 *
 * Host instantiation of the task of gf_profile_sources (golemflavor_b200/csrc/gf_profile_dev.cuh, gf_profile_src_obj): the
 * source objective at given points next to the single-source objective of gf_profile_grid, and the whole profile of every
 * (source, scale) run sequentially, so that the CPU test-suite checks the source path before any GPU time is spent.  Built
 * like harness.cu (g++, -ffp-contract=off).
 */
#include <string.h>

#include <vector>

#include "../../golemflavor_b200/csrc/gf_common.cuh"
#include "../../golemflavor_b200/csrc/gf_profile_dev.cuh"

namespace {

/* spec as the library chooses it for d (2 = static 6-column layout, 1 = FIXED, 0 = GENERIC), or -1 if d does not fit `want` */
int hh_spec(const gf_dev_model& d, int want) {
    const bool fixed = gf_model_is_fixed_spec(d);
    const bool static6 = fixed && d.ndim == 6 && d.col_sm[0] == 0 && d.col_sm[1] == 1 && d.col_sm[2] == 2 && d.col_sm[3] == 3 &&
                         d.col_mass[0] == 4 && d.col_mass[1] == 5;
    const int best = static6 ? 2 : fixed ? 1 : 0;
    return want < 0 ? best : want <= best ? want : -1;
}

template <class Obj>
void hh_objective(Obj& obj, const double* theta, int64_t n, double* lnp, double* fr, uint8_t* st) {
    for (int64_t i = 0; i < n; ++i) {
        obj.st = 0u;
        lnp[i] = obj.lnprob(theta + i * obj.m.ndim);
        memcpy(fr + 3 * i, obj.fr, sizeof(obj.fr));
        st[i] = (uint8_t)obj.st;
    }
}

template <int SPEC, bool STATIC6, int ILP>
void hh_objectives(const gf_dev_model& d, const double* theta, int64_t n, double scale, const gf_src_rec* rec, double* lnp, double* fr,
                   uint8_t* st) {
    if (rec) {
        gf_profile_src_obj<SPEC, STATIC6, ILP> obj{{d, gf_exp10(scale)}, rec};
        hh_objective(obj, theta, n, lnp, fr, st);
    } else {
        gf_profile_obj<SPEC, STATIC6, ILP> obj{d, gf_exp10(scale)};
        hh_objective(obj, theta, n, lnp, fr, st);
    }
}

/* one (source, scale) row: the starts in thread order, the first strict improvement wins (ties stay with the lower k) */
template <int SPEC, bool STATIC6, int ILP>
void hh_profile_row(const gf_dev_model& d, const gf_profile_config* cfg, double scale, int64_t task, const gf_src_rec* rec, double* best,
                    double* argmax, double* fr, uint8_t* st, int64_t* counts) {
    const int n = d.ndim;
    const gf_nm_opts o{cfg->ftol, cfg->xtol, cfg->max_evals};
    std::vector<double> S((size_t)(n + 1) * (n + 1));
    double fbest = 0.0;
    int64_t nev = 0, nconv = 0;
    unsigned nonfinite = 0u;
    for (int k = 0; k < cfg->nstarts; ++k) {
        gf_profile_src_obj<SPEC, STATIC6, ILP> obj{{d, gf_exp10(scale)}, rec};
        const gf_nm_out r = gf_profile_task(obj, cfg->seed, (uint64_t)task, cfg->nstarts, k, o, S.data(), 1);
        const double f = -S[(size_t)(n + 1) * n + r.best];
        nev += r.nevals;
        nconv += r.converged;
        nonfinite |= obj.nonfinite;
        if (k == 0 || f > fbest) {
            fbest = f;
            for (int j = 0; j < n; ++j) argmax[j] = obj.theta(S[(size_t)r.best * n + j], j);
            memcpy(fr, obj.fr, sizeof(obj.fr));
            *st = (uint8_t)obj.st;
        }
    }
    *best = fbest;
    *st |= (uint8_t)nonfinite;
    counts[0] = nev;
    counts[1] = nconv;
}

}  // namespace

/* ln_prob at theta[n][ndim] with the scale frozen at `scale`: of gf_profile_src_obj for each source (lnp[nsrc][n],
 * fr[nsrc][n][3], st[nsrc][n]), or of the single-source gf_profile_obj of the model itself when sources is NULL (nsrc rows of
 * the same values).  spec as hh_profile_sources. */
extern "C" int hh_profile_objective(const gf_model* model, const double* theta, int64_t n, double scale, const double* sources,
                                    const double* injected, int nsrc, int spec, double* lnp, double* fr, uint8_t* st) {
    gf_dev_model d;
    if (int rc = gf_build_dev_model(model, &d)) return rc;
    spec = hh_spec(d, spec);
    if (d.no_bsm || d.col_scale >= 0 || spec < 0) return GF_ERR_ARG;
    for (int j = 0; j < nsrc; ++j) {
        gf_src_rec rec;
        if (sources && !gf_src_record(sources + 3 * j, injected + 3 * j, d.wsum, &rec)) return GF_ERR_ARG;
        const gf_src_rec* r = sources ? &rec : nullptr;
        double* l = lnp + j * n;
        double* f = fr + 3 * j * n;
        uint8_t* s = st + j * n;
        if (spec == 2) hh_objectives<GF_SPEC_FIXED, true, 2>(d, theta, n, scale, r, l, f, s);
        else if (spec == 1) hh_objectives<GF_SPEC_FIXED, false, 2>(d, theta, n, scale, r, l, f, s);
        else hh_objectives<GF_SPEC_GENERIC, false, 1>(d, theta, n, scale, r, l, f, s);
    }
    return 0;
}

/* gf_profile_sources run sequentially: outputs [nsrc][nscales]...; spec: -1 = as the library chooses, 2 = static 6-column
 * layout, 1 = FIXED, 0 = GENERIC.  The refusals of the model as GF_ERR_ARG. */
extern "C" int hh_profile_sources(const gf_model* model, const gf_profile_config* cfg, const double* scales, int32_t nscales, const double* sources,
                                  const double* injected, int32_t nsrc, double* best, double* argmax, double* fr, uint8_t* st, int64_t* counts,
                                  int spec) {
    gf_dev_model d;
    if (int rc = gf_build_dev_model(model, &d)) return rc;
    spec = hh_spec(d, spec);
    if (d.no_bsm || d.col_scale >= 0 || spec < 0 || !gf_model_has_fixed_source(d) || d.llh_kind != GF_LLH_GAUSSIAN) return GF_ERR_ARG;
    for (int32_t j = 0; j < nsrc; ++j) {
        gf_src_rec rec;
        if (!gf_src_record(sources + 3 * j, injected + 3 * j, d.wsum, &rec)) return GF_ERR_ARG;
        for (int32_t s = 0; s < nscales; ++s) {
            const int64_t task = cfg->task0 + s, row = (int64_t)j * nscales + s;
            double* a = argmax + row * d.ndim;
            if (spec == 2) hh_profile_row<GF_SPEC_FIXED, true, 2>(d, cfg, scales[s], task, &rec, best + row, a, fr + 3 * row, st + row, counts + 2 * row);
            else if (spec == 1) hh_profile_row<GF_SPEC_FIXED, false, 2>(d, cfg, scales[s], task, &rec, best + row, a, fr + 3 * row, st + row, counts + 2 * row);
            else hh_profile_row<GF_SPEC_GENERIC, false, 1>(d, cfg, scales[s], task, &rec, best + row, a, fr + 3 * row, st + row, counts + 2 * row);
        }
    }
    return 0;
}
