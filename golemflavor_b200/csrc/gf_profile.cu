/*
 * gf_profile.cu -- the frequentist statistic of scripts/sens.py (StatCateg.FREQUENTIST, gf.get_llh_freq): the profile
 * likelihood max over the nuisance parameters of ln_prob at each frozen log10(Lambda), by bounded Nelder-Mead from
 * `nstarts` starts per scale (gf_profile_dev.cuh), one block per scale and one thread per start; k_profile_sources does
 * the same for many source compositions in one launch, one block per (scale, source).
 */
#include <atomic>
#include <stdlib.h>
#include <string.h>

#include "gf_common.cuh"
#include "gf_profile_dev.cuh"

extern std::atomic<unsigned long long> g_gf_launches;

#define GF_PROFILE_MAX_STARTS 256
/* register cap of k_profile_sources (DESIGN.md K3e; -D overrides it for A/B builds) */
#ifndef GF_PROFILE_SRC_REGS
#define GF_PROFILE_SRC_REGS 152
#endif

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

/*
 * gf_profile_sources: block (s, j) = scale s of source j, thread k = start k, so every source starts from the points
 * k_profile uses at that scale.  The registers are capped at GF_PROFILE_SRC_REGS = 152: 6 blocks of 64 starts per SM
 * (k_profile: 230 registers, 4 blocks).  The static 6-column kernel then spills 210 B per thread; of the caps measured
 * (128: 8 blocks, 390 B of spills; 152; 192: 5 blocks, no spills) 152 ran the 30-source grid fastest (DESIGN.md K3e).
 */
template <int SPEC, bool STATIC6>
__global__ void __maxnreg__(GF_PROFILE_SRC_REGS)
    k_profile_sources(const __grid_constant__ gf_dev_model m, const __grid_constant__ gf_src_table S, const gf_profile_config c,
                      const double* __restrict__ scales, double* __restrict__ best, double* __restrict__ argmax, double* __restrict__ fr_out,
                      uint8_t* __restrict__ status, int64_t* __restrict__ counts) {
    extern __shared__ double sh_nm[]; /* [(ndim+1)^2][nstarts]: element e of start k at e * nstarts + k */
    __shared__ double sh_f[GF_PROFILE_MAX_STARTS / 32];
    __shared__ int sh_k[GF_PROFILE_MAX_STARTS / 32];
    __shared__ unsigned long long sh_nev[GF_PROFILE_MAX_STARTS / 32], sh_conv[GF_PROFILE_MAX_STARTS / 32];
    __shared__ int sh_win;
    const int s = blockIdx.x, j = blockIdx.y, k = threadIdx.x, T = blockDim.x, n = m.ndim;
    const size_t row = (size_t)j * gridDim.x + s; /* output row [j][s] */
    gf_profile_src_obj<SPEC, STATIC6, GF_SPEC_IS_FIXED(SPEC) ? 2 : 1> obj{{m, gf_exp10(scales[s])}, &S.src[j]};
    const gf_nm_opts o{c.ftol, c.xtol, c.max_evals};
    const gf_nm_out r = gf_profile_task(obj, c.seed, (uint64_t)(c.task0 + s), c.nstarts, k, o, sh_nm + k, T);
    /* from here on k_profile's reduction (its body is left as it is, so that its code stays unchanged) */
    double f = -sh_nm[(size_t)((n + 1) * n + r.best) * T + k];
    int kk = k;
    unsigned long long nev = (unsigned long long)r.nevals, conv = r.converged ? 1ull : 0ull;
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
        best[row] = f;
        if (counts) {
            counts[2 * row] = (int64_t)nev;
            counts[2 * row + 1] = (int64_t)conv;
        }
    }
    __syncthreads();
    if (k != sh_win) return;
    const double* xb = sh_nm + (size_t)(r.best * n) * T + k;
    if (argmax)
        for (int d = 0; d < n; ++d) argmax[row * n + d] = obj.theta(xb[(size_t)d * T], d);
    if (fr_out) {
        fr_out[3 * row] = obj.fr[0];
        fr_out[3 * row + 1] = obj.fr[1];
        fr_out[3 * row + 2] = obj.fr[2];
    }
    if (status) status[row] = (uint8_t)(obj.st | nonfinite);
}

namespace {

/* The checks gf_profile_grid and gf_profile_sources share; d = the device model. */
int profile_prepare(const char* who, const gf_model* model, const gf_profile_config* cfg, gf_dev_model* d) {
    if (int rc = gf_build_dev_model(model, d)) return rc;
    GF_REQUIRE(!d->no_bsm, "%s: the model has no BSM path (no_bsm = 1)", who);
    GF_REQUIRE(d->col_scale < 0, "%s: the scale must not be a sampled column (col_scale = %d): it is frozen at the grid values", who, d->col_scale);
    GF_REQUIRE(cfg->nstarts >= 32 && cfg->nstarts <= GF_PROFILE_MAX_STARTS && cfg->nstarts % 32 == 0,
               "%s: nstarts = %d must be a multiple of 32 in [32, %d]", who, cfg->nstarts, GF_PROFILE_MAX_STARTS);
    GF_REQUIRE(cfg->max_evals >= 1, "%s: max_evals = %d must be positive", who, cfg->max_evals);
    GF_REQUIRE(cfg->task0 >= 0, "%s: task0 = %lld is negative", who, (long long)cfg->task0);
    GF_REQUIRE(cfg->ftol >= 0.0 && cfg->xtol >= 0.0, "%s: ftol = %g and xtol = %g must be non-negative", who, cfg->ftol, cfg->xtol);
    for (int k = 0; k < d->ndim; ++k)
        GF_REQUIRE(d->kind[k] != GF_PRIOR_UNIFORM || (isfinite(d->lo[k]) && isfinite(d->hi[k]) && d->hi[k] > d->lo[k]),
                   "%s: uniform prior %d needs a finite box of positive width, got (%g, %g)", who, k, d->lo[k], d->hi[k]);
    return GF_OK;
}

/* The specialisation (2 = static6, 1 = FIXED, 0 = GENERIC) of the model, or the one GF_PROFILE_SPEC = static6 / fixed / generic
 * selects among those the model also fits (tests compare them). */
int profile_spec(const char* who, const gf_dev_model* d, int* spec) {
    const bool fixed = gf_model_is_fixed_spec(*d);
    const bool static6 = fixed && d->ndim == 6 && d->col_sm[0] == 0 && d->col_sm[1] == 1 && d->col_sm[2] == 2 && d->col_sm[3] == 3 &&
                         d->col_mass[0] == 4 && d->col_mass[1] == 5;
    *spec = static6 ? 2 : fixed ? 1 : 0;
    if (const char* env = getenv("GF_PROFILE_SPEC")) {
        const int want = !strcmp(env, "static6") ? 2 : !strcmp(env, "fixed") ? 1 : !strcmp(env, "generic") ? 0 : -1;
        GF_REQUIRE(want >= 0 && want <= *spec, "%s: GF_PROFILE_SPEC = '%s' is not a specialisation this model fits", who, env);
        *spec = want;
    }
    return GF_OK;
}

/* Dynamic shared memory of kern for the simplices of cfg->nstarts starts in d.ndim dimensions, refused beyond the device's
 * opt-in limit less the kernel's static reduction arrays; sets the kernel's limit to it. */
template <class Kern>
int profile_smem(const char* who, Kern kern, const gf_dev_model& d, const gf_profile_config* cfg, size_t* smem) {
    *smem = (size_t)(d.ndim + 1) * (d.ndim + 1) * cfg->nstarts * sizeof(double);
    int dev = 0, optin = 0;
    GF_CUDA(cudaGetDevice(&dev));
    GF_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    cudaFuncAttributes fa;
    GF_CUDA(cudaFuncGetAttributes(&fa, kern));
    const size_t avail = (size_t)optin - fa.sharedSizeBytes; /* less the static reduction arrays */
    GF_REQUIRE(*smem <= avail, "%s: the simplices of %d starts in %d dimensions need %zu B of shared memory per block, at most %zu B "
               "fit: (ndim + 1)^2 * nstarts * 8 <= %zu", who, cfg->nstarts, d.ndim, *smem, avail, avail);
    GF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)*smem));
    return GF_OK;
}

}  // namespace

extern "C" int gf_profile_grid(const gf_model* model, const gf_profile_config* cfg, const double* d_scales, int32_t nscales, double* d_best,
                               double* d_argmax, double* d_fr, uint8_t* d_status, int64_t* d_counts, void* stream) {
    GF_REQUIRE(cfg != nullptr && d_best != nullptr && d_scales != nullptr, "gf_profile_grid: null pointer");
    GF_REQUIRE(nscales >= 0 && nscales <= (1 << 30), "gf_profile_grid: nscales = %d outside [0, 2^30]", nscales);
    gf_dev_model d;
    if (int rc = profile_prepare("gf_profile_grid", model, cfg, &d)) return rc;
    if (nscales == 0) return GF_OK;
    int spec = 0;
    if (int rc = profile_spec("gf_profile_grid", &d, &spec)) return rc;
    auto kern = spec == 2 ? k_profile<GF_SPEC_FIXED, true> : spec == 1 ? k_profile<GF_SPEC_FIXED, false> : k_profile<GF_SPEC_GENERIC, false>;
    size_t smem = 0;
    if (int rc = profile_smem("gf_profile_grid", kern, d, cfg, &smem)) return rc;
    kern<<<(unsigned)nscales, (unsigned)cfg->nstarts, smem, (cudaStream_t)stream>>>(d, *cfg, d_scales, d_best, d_argmax, d_fr, d_status, d_counts);
    ++g_gf_launches;
    GF_LAUNCH_CHECK("gf_profile_grid");
    return GF_OK;
}

extern "C" int gf_profile_sources(const gf_model* model, const gf_profile_config* cfg, const double* d_scales, int32_t nscales, const double* sources,
                                  const double* injected, int32_t nsrc, double* d_best, double* d_argmax, double* d_fr, uint8_t* d_status,
                                  int64_t* d_counts, void* stream) {
    GF_REQUIRE(model != nullptr && cfg != nullptr && d_scales != nullptr && sources != nullptr && injected != nullptr && d_best != nullptr,
               "gf_profile_sources: null pointer");
    GF_REQUIRE(nscales >= 0 && nscales <= (1 << 30), "gf_profile_sources: nscales = %d outside [0, 2^30]", nscales);
    GF_REQUIRE(nsrc >= 1 && nsrc <= GF_SRC_MAX, "gf_profile_sources: nsrc = %d outside [1, %d]", nsrc, GF_SRC_MAX);
    gf_dev_model d;
    if (int rc = profile_prepare("gf_profile_sources", model, cfg, &d)) return rc;
    GF_REQUIRE(gf_model_has_fixed_source(d), "gf_profile_sources: the model samples the source (col_src / col_x / col_src3): the sources are "
               "the launch's own list");
    GF_REQUIRE(d.llh_kind == GF_LLH_GAUSSIAN, "gf_profile_sources: llh_kind = %d, the Gaussian likelihood (GF_LLH_GAUSSIAN) is required", d.llh_kind);
    gf_src_table tab; /* 14 KB, copied into the kernel parameter buffer by the launch */
    tab.nsrc = nsrc;
    tab.reserved = 0;
    for (int j = 0; j < nsrc; ++j)
        GF_REQUIRE(gf_src_record(sources + 3 * j, injected + 3 * j, d.wsum, &tab.src[j]),
                   "gf_profile_sources: source %d = (%g, %g, %g) / injected (%g, %g, %g): entries must be finite and non-negative with a "
                   "positive sum",
                   j, sources[3 * j], sources[3 * j + 1], sources[3 * j + 2], injected[3 * j], injected[3 * j + 1], injected[3 * j + 2]);
    int spec = 0;
    if (int rc = profile_spec("gf_profile_sources", &d, &spec)) return rc;
    auto kern = spec == 2 ? k_profile_sources<GF_SPEC_FIXED, true> : spec == 1 ? k_profile_sources<GF_SPEC_FIXED, false>
                                                                                : k_profile_sources<GF_SPEC_GENERIC, false>;
    size_t smem = 0;
    if (int rc = profile_smem("gf_profile_sources", kern, d, cfg, &smem)) return rc;
    if (nscales == 0) return GF_OK;
    kern<<<dim3((unsigned)nscales, (unsigned)nsrc), (unsigned)cfg->nstarts, smem, (cudaStream_t)stream>>>(d, tab, *cfg, d_scales, d_best, d_argmax,
                                                                                                         d_fr, d_status, d_counts);
    ++g_gf_launches;
    GF_LAUNCH_CHECK("gf_profile_sources");
    return GF_OK;
}
