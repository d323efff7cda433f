/*
 * TEST INFRASTRUCTURE ONLY -- never linked into libgolemflavor_b200.so, never imported by the product package.
 *
 * Host instantiation of the profile-likelihood task of gf_profile_grid (golemflavor_b200/csrc/gf_profile_dev.cuh): the
 * same per-task function run sequentially, and the Nelder-Mead core alone on an analytic objective, so that the CPU
 * test-suite checks the optimiser before any GPU time is spent.  Built like harness.cu (g++, -ffp-contract=off).
 */
#include <string.h>

#include <vector>

#include "../../golemflavor_b200/csrc/gf_common.cuh"
#include "../../golemflavor_b200/csrc/gf_profile_dev.cuh"

/* ------------------------------------------------------------------ profile likelihood (gf_profile_dev.cuh) */

template <int SPEC, bool STATIC6, int ILP>
static void hh_profile_scale(const gf_dev_model& d, const gf_profile_config* cfg, double scale, int64_t task, double* best, double* argmax,
                             double* fr, uint8_t* st, int64_t* counts) {
    const int n = d.ndim;
    const gf_nm_opts o{cfg->ftol, cfg->xtol, cfg->max_evals};
    std::vector<double> S((size_t)(n + 1) * (n + 1));
    double fbest = 0.0;
    int64_t nev = 0, nconv = 0;
    unsigned nonfinite = 0u;
    for (int k = 0; k < cfg->nstarts; ++k) { /* thread order: the first strict improvement wins, ties stay with the lower k */
        gf_profile_obj<SPEC, STATIC6, ILP> obj{d, gf_exp10(scale)};
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

/* gf_profile_grid run sequentially; spec: -1 = as the library chooses, 2 = static 6-column layout, 1 = FIXED, 0 = GENERIC */
extern "C" int hh_profile(const gf_model* model, const gf_profile_config* cfg, const double* scales, int32_t nscales, double* best,
                          double* argmax, double* fr, uint8_t* st, int64_t* counts, int spec) {
    gf_dev_model d;
    if (int rc = gf_build_dev_model(model, &d)) return rc;
    const bool fixed = gf_model_is_fixed_spec(d);
    const bool static6 = fixed && d.ndim == 6 && d.col_sm[0] == 0 && d.col_sm[1] == 1 && d.col_sm[2] == 2 && d.col_sm[3] == 3 &&
                         d.col_mass[0] == 4 && d.col_mass[1] == 5;
    if (spec < 0) spec = static6 ? 2 : fixed ? 1 : 0;
    if (d.no_bsm || d.col_scale >= 0 || (spec == 2 && !static6) || (spec == 1 && !fixed)) return GF_ERR_ARG;
    for (int32_t s = 0; s < nscales; ++s) {
        const int64_t task = cfg->task0 + s;
        double* a = argmax + (size_t)s * d.ndim;
        if (spec == 2) hh_profile_scale<GF_SPEC_FIXED, true, 2>(d, cfg, scales[s], task, best + s, a, fr + 3 * s, st + s, counts + 2 * s);
        else if (spec == 1) hh_profile_scale<GF_SPEC_FIXED, false, 2>(d, cfg, scales[s], task, best + s, a, fr + 3 * s, st + s, counts + 2 * s);
        else hh_profile_scale<GF_SPEC_GENERIC, false, 1>(d, cfg, scales[s], task, best + s, a, fr + 3 * s, st + s, counts + 2 * s);
    }
    return 0;
}

/* the optimiser core alone on g(x) = sum_k a_k (x_k - c_k)^2 over the box [lo, hi] */
struct hh_box_quadratic {
    const double *a, *c, *blo, *bhi;
    int n;
    int64_t calls = 0;
    double lo(int k) const { return blo[k]; }
    double hi(int k) const { return bhi[k]; }
    double operator()(const double* x) {
        ++calls;
        double g = 0.0;
        for (int k = 0; k < n; ++k) g += a[k] * (x[k] - c[k]) * (x[k] - c[k]);
        return g;
    }
};

extern "C" void hh_nm_box_quadratic(int n, const double* a, const double* c, const double* lo, const double* hi, const double* x0, double ftol,
                                    double xtol, int max_evals, double* xbest, double* gbest, int64_t* nevals, int* converged) {
    hh_box_quadratic q{a, c, lo, hi, n};
    std::vector<double> S((size_t)(n + 1) * (n + 1));
    const gf_nm_out r = gf_nm_minimize<0>(q, n, x0, S.data(), 1, gf_nm_opts{ftol, xtol, max_evals});
    for (int k = 0; k < n; ++k) xbest[k] = S[(size_t)r.best * n + k];
    *gbest = S[(size_t)(n + 1) * n + r.best];
    nevals[0] = r.nevals;
    nevals[1] = q.calls;
    *converged = r.converged;
}
