/*
 * gf_profile.cu -- the frequentist statistic of scripts/sens.py (StatCateg.FREQUENTIST, gf.get_llh_freq): the profile
 * likelihood max over the nuisance parameters of ln_prob at each frozen log10(Lambda), by bounded Nelder-Mead from
 * `nstarts` starts per scale (gf_profile_dev.cuh), one block per scale and one thread per start.
 */
#include <atomic>
#include <stdlib.h>
#include <string.h>

#include "gf_common.cuh"
#include "gf_profile_dev.cuh"

extern std::atomic<unsigned long long> g_gf_launches;

#define GF_PROFILE_MAX_STARTS 256

/* (f, k) of the better start: larger ln_prob, ties to the lower start index (f is never NaN here) */
__device__ __forceinline__ void gf_profile_pick(double& f, int& k, double f2, int k2) {
    if (f2 > f || (f2 == f && k2 < k)) {
        f = f2;
        k = k2;
    }
}

template <int SPEC, bool STATIC6>
__global__ void __launch_bounds__(GF_PROFILE_MAX_STARTS, 1)
    k_profile(const __grid_constant__ gf_dev_model m, const gf_profile_config c, const double* __restrict__ scales,
              double* __restrict__ best, double* __restrict__ argmax, double* __restrict__ fr_out, uint8_t* __restrict__ status,
              int64_t* __restrict__ counts) {
    extern __shared__ double sh_nm[]; /* [(ndim+1)^2][nstarts]: element e of start k at e * nstarts + k */
    __shared__ double sh_f[GF_PROFILE_MAX_STARTS / 32];
    __shared__ int sh_k[GF_PROFILE_MAX_STARTS / 32];
    __shared__ unsigned long long sh_nev[GF_PROFILE_MAX_STARTS / 32], sh_conv[GF_PROFILE_MAX_STARTS / 32];
    __shared__ int sh_win;
    const int s = blockIdx.x, k = threadIdx.x, T = blockDim.x, n = m.ndim;
    gf_profile_obj<SPEC, STATIC6, GF_SPEC_IS_FIXED(SPEC) ? 2 : 1> obj{m, gf_exp10(scales[s])};
    const gf_nm_opts o{c.ftol, c.xtol, c.max_evals};
    const gf_nm_out r = gf_profile_task(obj, c.seed, (uint64_t)(c.task0 + s), c.nstarts, k, o, sh_nm + k, T);
    double f = -sh_nm[(size_t)((n + 1) * n + r.best) * T + k];
    int kk = k;
    unsigned long long nev = (unsigned long long)r.nevals, conv = r.converged ? 1ull : 0ull;
    /* thread order: lanes by shuffle, then warps in order */
    for (int off = 16; off > 0; off >>= 1) {
        gf_profile_pick(f, kk, __shfl_down_sync(0xffffffffu, f, off), __shfl_down_sync(0xffffffffu, kk, off));
        nev += __shfl_down_sync(0xffffffffu, nev, off);
        conv += __shfl_down_sync(0xffffffffu, conv, off);
    }
    const int lane = k & 31, warp = k >> 5;
    if (lane == 0) {
        sh_f[warp] = f;
        sh_k[warp] = kk;
        sh_nev[warp] = nev;
        sh_conv[warp] = conv;
    }
    const unsigned nonfinite = __syncthreads_or((int)obj.nonfinite) ? GFP_ST_NON_FINITE : 0u;
    if (k == 0) {
        for (int w = 1; w < T / 32; ++w) {
            gf_profile_pick(f, kk, sh_f[w], sh_k[w]);
            nev += sh_nev[w];
            conv += sh_conv[w];
        }
        sh_win = kk;
        best[s] = f;
        if (counts) {
            counts[2 * s] = (int64_t)nev;
            counts[2 * s + 1] = (int64_t)conv;
        }
    }
    __syncthreads();
    if (k != sh_win) return;
    const double* xb = sh_nm + (size_t)(r.best * n) * T + k;
    if (argmax)
        for (int d = 0; d < n; ++d) argmax[(size_t)s * n + d] = obj.theta(xb[(size_t)d * T], d);
    if (fr_out) {
        fr_out[3 * s] = obj.fr[0];
        fr_out[3 * s + 1] = obj.fr[1];
        fr_out[3 * s + 2] = obj.fr[2];
    }
    if (status) status[s] = (uint8_t)(obj.st | nonfinite);
}

extern "C" int gf_profile_grid(const gf_model* model, const gf_profile_config* cfg, const double* d_scales, int32_t nscales, double* d_best,
                               double* d_argmax, double* d_fr, uint8_t* d_status, int64_t* d_counts, void* stream) {
    GF_REQUIRE(cfg != nullptr && d_best != nullptr && d_scales != nullptr, "gf_profile_grid: null pointer");
    GF_REQUIRE(nscales >= 0 && nscales <= (1 << 30), "gf_profile_grid: nscales = %d outside [0, 2^30]", nscales);
    gf_dev_model d;
    if (int rc = gf_build_dev_model(model, &d)) return rc;
    GF_REQUIRE(!d.no_bsm, "gf_profile_grid: the model has no BSM path (no_bsm = 1)");
    GF_REQUIRE(d.col_scale < 0, "gf_profile_grid: the scale must not be a sampled column (col_scale = %d): it is frozen at the grid values", d.col_scale);
    GF_REQUIRE(cfg->nstarts >= 32 && cfg->nstarts <= GF_PROFILE_MAX_STARTS && cfg->nstarts % 32 == 0,
               "gf_profile_grid: nstarts = %d must be a multiple of 32 in [32, %d]", cfg->nstarts, GF_PROFILE_MAX_STARTS);
    GF_REQUIRE(cfg->max_evals >= 1, "gf_profile_grid: max_evals = %d must be positive", cfg->max_evals);
    GF_REQUIRE(cfg->task0 >= 0, "gf_profile_grid: task0 = %lld is negative", (long long)cfg->task0);
    GF_REQUIRE(cfg->ftol >= 0.0 && cfg->xtol >= 0.0, "gf_profile_grid: ftol = %g and xtol = %g must be non-negative", cfg->ftol, cfg->xtol);
    for (int k = 0; k < d.ndim; ++k)
        GF_REQUIRE(d.kind[k] != GF_PRIOR_UNIFORM || (isfinite(d.lo[k]) && isfinite(d.hi[k]) && d.hi[k] > d.lo[k]),
                   "gf_profile_grid: uniform prior %d needs a finite box of positive width, got (%g, %g)", k, d.lo[k], d.hi[k]);
    if (nscales == 0) return GF_OK;
    const bool fixed = gf_model_is_fixed_spec(d);
    const bool static6 = fixed && d.ndim == 6 && d.col_sm[0] == 0 && d.col_sm[1] == 1 && d.col_sm[2] == 2 && d.col_sm[3] == 3 &&
                         d.col_mass[0] == 4 && d.col_mass[1] == 5;
    /* GF_PROFILE_SPEC = static6 / fixed / generic: run a specialisation the model also fits (tests compare them) */
    int spec = static6 ? 2 : fixed ? 1 : 0;
    if (const char* env = getenv("GF_PROFILE_SPEC")) {
        const int want = !strcmp(env, "static6") ? 2 : !strcmp(env, "fixed") ? 1 : !strcmp(env, "generic") ? 0 : -1;
        GF_REQUIRE(want >= 0 && want <= spec, "gf_profile_grid: GF_PROFILE_SPEC = '%s' is not a specialisation this model fits", env);
        spec = want;
    }
    auto kern = spec == 2 ? k_profile<GF_SPEC_FIXED, true> : spec == 1 ? k_profile<GF_SPEC_FIXED, false> : k_profile<GF_SPEC_GENERIC, false>;
    const size_t smem = (size_t)(d.ndim + 1) * (d.ndim + 1) * cfg->nstarts * sizeof(double);
    int dev = 0, optin = 0;
    GF_CUDA(cudaGetDevice(&dev));
    GF_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    cudaFuncAttributes fa;
    GF_CUDA(cudaFuncGetAttributes(&fa, kern));
    const size_t avail = (size_t)optin - fa.sharedSizeBytes; /* less the static reduction arrays */
    GF_REQUIRE(smem <= avail, "gf_profile_grid: the simplices of %d starts in %d dimensions need %zu B of shared memory per block, at most %zu B "
               "fit: (ndim + 1)^2 * nstarts * 8 <= %zu", cfg->nstarts, d.ndim, smem, avail, avail);
    GF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<(unsigned)nscales, (unsigned)cfg->nstarts, smem, (cudaStream_t)stream>>>(d, *cfg, d_scales, d_best, d_argmax, d_fr, d_status, d_counts);
    ++g_gf_launches;
    GF_LAUNCH_CHECK("gf_profile_grid");
    return GF_OK;
}
