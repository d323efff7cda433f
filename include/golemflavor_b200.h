/*
 * golemflavor_b200 -- C ABI of the B200-native log-posterior hot path.
 *
 * Every entry point is `extern "C"`, takes plain pointers and sizes and returns
 * an int status (GF_OK = 0; on error `gf_last_error()` describes it).  Pointers
 * named `d_*` are DEVICE pointers (cudaMalloc / torch tensors), pointers named
 * `h_*` are HOST pointers; `stream` is a `cudaStream_t` passed as `void*`
 * (NULL = the legacy default stream).  Nothing here allocates on the caller's
 * behalf except the `*_host` convenience calls, which own their staging buffers.
 * There is NO CPU implementation behind this ABI: without a CUDA device every
 * compute call returns GF_ERR_CUDA.
 *
 * Each function cites the reference interface it replaces
 * (ShiveshM/GolemFlavor, paths relative to its repository root).
 *
 * Layout conventions
 *   complex matrices : [n][3][3][2] doubles (re, im) == NumPy complex128 C-order
 *   theta            : element (point i, parameter k) at theta[i*ld_point + k*ld_dim]
 *                      (row-major emcee layout: ld_point = ndim, ld_dim = 1;
 *                       SoA layout: ld_point = 1, ld_dim = n)
 *   fr               : [n][3] doubles (nu_e, nu_mu, nu_tau)
 *   status           : one byte per point, bit mask GF_ST_*
 */
#ifndef GOLEMFLAVOR_B200_H
#define GOLEMFLAVOR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GF_ABI_VERSION 1

#define GF_MAX_DIM 16   /* parameters per point   */
#define GF_MAX_BINS 64  /* energy bins per point  */

/* return codes */
#define GF_OK 0
#define GF_ERR_ARG 1   /* bad argument (the reference raises ValueError/AssertionError) */
#define GF_ERR_CUDA 2  /* CUDA runtime error / no device */

/* per-point status bits (the reference raises or returns -inf mid-loop instead) */
#define GF_ST_OUT_OF_PRIOR 1u /* lnprior = -inf        (llh.py:74-78)                  */
#define GF_ST_NON_UNITARY 2u  /* unitarity residual > epsilon (fr.py:493-498 asserts)  */
#define GF_ST_NON_FINITE 4u   /* NaN/Inf encountered (invalid angles, ...)             */
#define GF_ST_ILL_COND 8u     /* eigen-gap below 1e-6: result limited by fp64 inputs   */
#define GF_ST_REFINED 16u     /* informational: Jacobi refinement path was taken        */

/* prior kinds == golemflavor/enums.py:38-41 (PriorsCateg) minus one */
#define GF_PRIOR_UNIFORM 0
#define GF_PRIOR_GAUSSIAN 1
#define GF_PRIOR_LIMITEDGAUSS 2

/* likelihood kinds */
#define GF_LLH_FLAT 0     /* ln_prob = lnprior + llh_const  (scripts/mc_*.py: "return 1. # Flat LLH") */
#define GF_LLH_GAUSSIAN 1 /* llh.multi_gaussian (llh.py:32-54)                                        */

/* One sampled parameter: param.Param (param.py:24-91) flattened. */
typedef struct gf_prior_dim {
    double lo, hi;    /* Param.ranges                               */
    double mu, sigma; /* Param.nominal_value, Param.std             */
    int32_t kind;     /* GF_PRIOR_*                                 */
    int32_t reserved;
} gf_prior_dim;

/*
 * The closure `partial(ln_prob, args=..., asimov_paramset=..., llh_paramset=...)`
 * (scripts/fr.py:182-187, examples/inference.ipynb cell 23) flattened:
 * which theta column feeds which physical quantity, the fixed values of the
 * quantities that are not sampled, the energy binning, the priors and the
 * Gaussian likelihood constants.
 */
typedef struct gf_model {
    int32_t ndim;         /* len(llh_paramset)                                            */
    int32_t col_sm[4];    /* theta columns of s_12_2, c_13_4, s_23_2, dcp; -1 = fixed_sm  */
    int32_t col_mass[2];  /* theta columns of m21_2, m3x_2;              -1 = fixed_mass  */
    int32_t col_src[2];   /* theta columns of the SRCANGLES (sin^4 phi, cos 2psi);
                             -1 = use fixed_src (args.source_ratio)                        */
    int32_t col_np[4];    /* theta columns of the MMANGLES (NP mixing);   -1 = fixed_np   */
    int32_t col_scale;    /* theta column of logLam (SCALE tag); -1 = fixed_loglam        */
    int32_t col_x;        /* theta column of x, source = (x, 1-x, 0) (scripts/mc_x.py:187); -1 = unused */
    int32_t col_src3[3];  /* theta columns of three raw source ratios (normalised by u_to_fr, fr.py:535;
                             BASELINE config 1: "3 source-flavor params, fixed PMNS"); -1 = unused */
    int32_t no_bsm;       /* 1: skip the BSM path, fr = u_to_fr(source, sm_u) (notebook SM model) */
    int32_t dimension;    /* args.dimension (3..8)                                         */
    int32_t nbins;        /* len(args.binning) - 1                                         */
    int32_t llh_kind;     /* GF_LLH_*                                                      */
    int32_t emulate_underflow; /* 1: multi_gaussian returns -inf where the reference's pdf underflows */
    double fixed_sm[4];   /* default NUFIT angles (fr.py:313)                              */
    double fixed_mass[2]; /* default MASS_EIGENVALUES (fr.py:42)                           */
    double fixed_src[3];  /* args.source_ratio (need not be normalised)                    */
    double fixed_np[4];   /* texture angles (fr.py:370-376)                                */
    double fixed_loglam;
    double bin_edges[GF_MAX_BINS + 1]; /* args.binning (GeV)                               */
    double fr_bf[3];      /* injected / best-fit composition                               */
    double smearing;      /* sigma of the Gaussian likelihood                              */
    double offset;        /* multi_gaussian offset (-320)                                  */
    double llh_const;     /* value of the flat likelihood (1.0 in scripts/mc_*.py)         */
    double epsilon;       /* unitarity tolerance for GF_ST_NON_UNITARY (fr.py:319: 1e-7)   */
    gf_prior_dim prior[GF_MAX_DIM];
} gf_model;

/*
 * Monte-Carlo scan: scripts/mc_unitary.py, mc_x.py, mc_texture.py + plot.py:364-370.
 * The reference draws prior samples by running emcee on a flat likelihood; here sample i draws
 * parameter k of the model directly from its prior (model.prior[k]: uniform in `ranges`, or a
 * Gaussian truncated to `ranges`, by inverse CDF) using Philox4x32-10 with
 *   key = (lo32(seed), hi32(seed)),  counter = (lo32(i), hi32(i), k / 4, 0),  word k % 4,
 *   uniform = (word + 0.5) * 2^-32,
 * so that the result is independent of the launch geometry and of the number of GPUs.
 * Which scan it is (unitary / x / texture / anarchic) is entirely a property of the model:
 *   unitary  : 4 SM_ANGLES columns, no_bsm = 1, fixed source          (mc_unitary.py:189-192)
 *   x        : unitary + col_x, source = (x, 1-x, 0)                  (mc_x.py:186-192)
 *   texture  : 6 SM columns + logLam, fixed texture angles, 20 bins   (mc_texture.py:216-221)
 *   anarchic : texture + 4 MMANGLES columns (Haar-random NP mixing)   (Texture.NONE)
 */
typedef struct gf_scan_config {
    uint64_t seed;        /* Philox4x32-10 key                                      */
    uint64_t first_index; /* global index of this shard's first sample              */
    uint64_t count;       /* samples in this shard                                  */
    int32_t nb;           /* nbins*oversample: histogram has (nb+1)^3 cells         */
    int32_t reserved;
} gf_scan_config;

/* ---- library ---------------------------------------------------------- */
int gf_abi_version(void);
/* sizeof(gf_model) / gf_scan_config / gf_prior_dim / gf_ensemble_config / gf_profile_config for which = 0 / 1 / 2 / 3 / 4: lets a
 * foreign-language binding verify its struct layout at load time. */
uint64_t gf_sizeof(int32_t which);
const char* gf_last_error(void);
/* sm_count, compute capability and the SM clock (kHz) of the current device */
int gf_device_info(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor, int32_t* clock_khz);
/* Page-locked host buffers for the *_host calls (pageable buffers work too, through an internal
 * pinned staging ring, at memcpy speed). */
int gf_host_alloc(void** h_ptr, uint64_t bytes);
/* The same, write-combined: for INPUT buffers the host only writes (theta): the DMA engine reads them without snooping
 * the CPU caches, which matters when several GPUs pull from one host; host reads of such memory are slow. */
int gf_host_alloc_wc(void** h_ptr, uint64_t bytes);
int gf_host_free(void* h_ptr);
/* Validate a model without launching anything (same checks as every compute call). */
int gf_model_check(const gf_model* model);

/* ---- fr.py ------------------------------------------------------------ */
/* fr.angles_to_u(bsm_angles)                                   fr.py:116-162 */
int gf_angles_to_u(const double* d_angles /*[n][4]*/, int64_t n, double* d_u /*[n][3][3][2]*/, void* stream);
/* fr.angles_to_fr(src_angles)                                  fr.py:82-113  */
int gf_angles_to_fr(const double* d_src_angles /*[n][2]*/, int64_t n, double* d_fr /*[n][3]*/, void* stream);
/* fr.u_to_fr(source_fr, matrix)                                fr.py:502-536
 * source_stride = 3 for one source per point, 0 for a single shared source. */
int gf_u_to_fr(const double* d_source, int64_t source_stride, const double* d_u /*[n][3][3][2]*/, int64_t n,
               double* d_fr /*[n][3]*/, void* stream);
/* fr.cardano_eqn(ham)                                          fr.py:170-237
 * Eigenvector matrices (columns = eigenvectors, ascending eigenvalue) and
 * optionally the eigenvalues [n][3]; status gets GF_ST_NON_FINITE / ILL_COND. */
int gf_eigvec_herm3(const double* d_ham /*[n][3][3][2]*/, int64_t n, double* d_vec /*[n][3][3][2]*/,
                    double* d_eigval /*[n][3] or NULL*/, uint8_t* d_status /*[n] or NULL*/, void* stream);
/* fr.params_to_BSMu(bsm_angles, dim, energy, mass_eigenvalues, sm_u, no_bsm, texture, check_uni, epsilon)
 *                                                              fr.py:317-400
 * bsm[n][5] = (np_s12_2, np_c13_4, np_s23_2, np_dcp, logLam) -- textures resolved by the caller
 * (fr.py:370-376); mass_stride / smu_stride = 0 share one value across the batch. */
int gf_params_to_bsmu(const double* d_bsm /*[n][5]*/, int32_t dim, const double* d_energy /*[n]*/,
                      const double* d_mass, int64_t mass_stride /*2 or 0*/,
                      const double* d_sm_u, int64_t smu_stride /*18 or 0*/, int32_t no_bsm, double epsilon,
                      int64_t n, double* d_vec /*[n][3][3][2]*/, uint8_t* d_status /*[n] or NULL*/, void* stream);
/* fr.flux_averaged_BSMu(theta, args, spectral_index, llh_paramset)  fr.py:403-458 */
int gf_flux_averaged_fr(const gf_model* model, const double* d_theta, int64_t n, int64_t ld_point, int64_t ld_dim,
                        double* d_fr /*[n][3]*/, uint8_t* d_status /*[n] or NULL*/, void* stream);

/* ---- llh.py ----------------------------------------------------------- */
/* llh.lnprior(theta, paramset)                                 llh.py:65-91  */
int gf_lnprior(const gf_model* model, const double* d_theta, int64_t n, int64_t ld_point, int64_t ld_dim,
               double* d_lnprior /*[n]*/, void* stream);
/* llh.multi_gaussian(fr, fr_bf, smearing, offset)              llh.py:32-54  */
int gf_multi_gaussian(const double* d_fr /*[n][3]*/, int64_t n, const double* h_fr_bf /*[3]*/, double smearing,
                      double offset, int32_t emulate_underflow, double* d_llh /*[n]*/, void* stream);
/* llh.ln_prob(theta, args, asimov_paramset, llh_paramset)      llh.py:121-130
 * with the Gaussian flavor-ratio likelihood (examples/inference.ipynb cells 21-23).
 * d_fr (optional) receives the measured composition of every in-prior point. */
int gf_lnprob(const gf_model* model, const double* d_theta, int64_t n, int64_t ld_point, int64_t ld_dim,
              double* d_lnprob /*[n]*/, double* d_fr /*[n][3] or NULL*/, uint8_t* d_status /*[n] or NULL*/,
              void* stream);
/* Same call on HOST buffers (row-major theta[n][ndim]): chunked H2D -> kernel -> D2H
 * pipeline on internal streams; returns after the results are in h_lnprob. */
int gf_lnprob_host(const gf_model* model, const double* h_theta, int64_t n, double* h_lnprob,
                   double* h_fr /*or NULL*/, uint8_t* h_status /*or NULL*/);

/* ---- Monte-Carlo scans ------------------------------------------------ */
/* Draw `count` samples with Philox4x32-10 (counter = global sample index), push them through the
 * flavor path selected by cfg->mode and accumulate the ternary histogram
 * np.histogramdd(frs, bins=(nb+1,)*3, range=((0,1),)*3) (plot.py:364-370) into d_hist (ADDS to it).
 * d_accepted (optional, 1 counter) ADDS the number of samples inside the prior box. */
int gf_scan_hist(const gf_model* model, const gf_scan_config* cfg, unsigned long long* d_hist /*[(nb+1)^3]*/,
                 unsigned long long* d_accepted /*[1] or NULL*/, void* stream);
/* Same sampler, but writes the drawn theta [count][ndim] and fr [count][3] (parity/debug; cfg->nb unused). */
int gf_scan_samples(const gf_model* model, const gf_scan_config* cfg, double* d_theta /*[count][ndim] or NULL*/,
                    double* d_fr /*[count][3] or NULL*/, uint8_t* d_status /*[count] or NULL*/, void* stream);
/* Histogram of given compositions (bit-exact np.histogramdd), ADDS into d_hist. */
int gf_ternary_hist(const double* d_fr /*[n][3]*/, int64_t n, int32_t nb, unsigned long long* d_hist, void* stream);

/* Prior-sample Monte-Carlo evidence (the quantity scripts/sens.py:232-294 gets from MultiNest per
 * (dimension, scale) grid point): draws `cfg->count` samples from the priors exactly like gf_scan_hist,
 * evaluates the likelihood L (model.llh_kind) and accumulates log-sum-exp partials with warp shuffles:
 * d_lse[0] = max ln L, d_lse[1] = sum exp(ln L - max), merged with the values already stored there
 * (initialise to {-inf, 0}); ln mean(L) = d_lse[0] + log(d_lse[1]) - log(N).  cfg->nb is unused. */
int gf_scan_evidence(const gf_model* model, const gf_scan_config* cfg, double* d_lse /*[2]*/, void* stream);
/* The whole scale grid of one operator dimension in ONE launch (scripts/sens.py:199-201, 232-294: `eval_scales` x one
 * MultiNest run each): the model's scale is NOT sampled (col_scale = -1); every prior sample is drawn once and evaluated at
 * each of the `nscales` frozen values d_scales[s] = log10(Lambda_s), and d_lse[s][0..1] accumulates (max ln L, sum exp) per
 * scale exactly like gf_scan_evidence (initialise to {-inf, 0}; the values already there are merged).  d_work is scratch
 * of at least gf_scan_evidence_grid_workspace(nscales) bytes (any contents; reusable by the next call on the same stream). */
uint64_t gf_scan_evidence_grid_workspace(int32_t nscales);
int gf_scan_evidence_grid(const gf_model* model, const gf_scan_config* cfg, const double* d_scales /*[nscales]*/, int32_t nscales,
                          double* d_lse /*[nscales][2]*/, void* d_work, uint64_t work_bytes, void* stream);
/*
 * The same grid for many SOURCE COMPOSITIONS in one launch (the reference runs scripts/sens.py once per (dimension, texture,
 * source composition, Lambda segment), 30 compositions per texture: submitter/sens_dag.py:8-16, 38-61, 76-95).  Each prior
 * sample is drawn exactly as gf_scan_evidence_grid draws it and its eigen stage is run once per scale; the source enters only
 * through fr_b = sum_a P_ba s_a with the bin-width-averaged transition P = X X^T of flux_averaged_BSMu (fr.py:441-457), so
 * every source is then scored at a few instructions.  `sources` and `injected` are HOST arrays [nsrc][3] (source composition
 * and the injected composition it is scored against; each row normalised to unit sum inside); the model's own fixed_src and
 * fr_bf are ignored.  d_lse[j][s][0..1] accumulates (max ln L, sum exp) of source j at scale d_scales[s] exactly like
 * gf_scan_evidence_grid (initialise to {-inf, 0}; the values already there are merged).  d_work is scratch of at least
 * gf_scan_evidence_sources_workspace(nscales, nsrc) bytes (any contents; reusable by the next call on the same stream).
 * GF_ERR_ARG, with nothing enqueued, for: a null pointer; nscales outside [1, 65535]; nsrc outside [1, GF_SRC_MAX = 256];
 * a sampled scale (col_scale >= 0); no_bsm; a sampled source (col_src / col_x / col_src3); llh_kind other than
 * GF_LLH_GAUSSIAN; a source or injected row with a negative or non-finite entry or a zero sum; a workspace too small.
 * cfg->count = 0 is a no-op.  The result is the same for any order of the sources (row j depends on row j's compositions only).
 */
uint64_t gf_scan_evidence_sources_workspace(int32_t nscales, int32_t nsrc);
int gf_scan_evidence_sources(const gf_model* model, const gf_scan_config* cfg, const double* d_scales /*[nscales]*/, int32_t nscales,
                             const double* sources /*HOST [nsrc][3]*/, const double* injected /*HOST [nsrc][3]*/, int32_t nsrc,
                             double* d_lse /*[nsrc][nscales][2]*/, void* d_work, uint64_t work_bytes, void* stream);
/*
 * Grouped evidence grids: the Monte-Carlo error of lnZ by a delete-one-group jackknife.  The samples are split into `groups`
 * fixed groups, a power of two in [2, 32]: sample i (global Philox index cfg->first_index + j) is in group i mod groups, so the
 * grouping does not depend on the launch geometry or on how the index range is sharded.  d_lse gains a group axis and
 * accumulates (max ln L, sum exp) per (scale, group) with the rules of the ungrouped calls (NaN and -inf carry no weight;
 * initialise to {-inf, 0}; the values already there are merged).  Merging the groups gives the ungrouped result up to
 * rounding.  Same launch count as the ungrouped calls, one per call.  GF_ERR_ARG, with nothing enqueued, for everything the
 * ungrouped call refuses, and for `groups` not a power of two in [2, 32], a workspace smaller than the `_workspace` size, and
 * (source grid) nsrc * groups > 4096: one launch takes at most 4096 / groups sources (all 256 up to 16 groups, 128 at 32).
 */
uint64_t gf_scan_evidence_grid_groups_workspace(int32_t nscales, int32_t groups);
int gf_scan_evidence_grid_groups(const gf_model* model, const gf_scan_config* cfg, const double* d_scales /*[nscales]*/, int32_t nscales,
                                 int32_t groups, double* d_lse /*[nscales][groups][2]*/, void* d_work, uint64_t work_bytes, void* stream);
uint64_t gf_scan_evidence_sources_groups_workspace(int32_t nscales, int32_t nsrc, int32_t groups);
int gf_scan_evidence_sources_groups(const gf_model* model, const gf_scan_config* cfg, const double* d_scales /*[nscales]*/, int32_t nscales,
                                    const double* sources /*HOST [nsrc][3]*/, const double* injected /*HOST [nsrc][3]*/, int32_t nsrc,
                                    int32_t groups, double* d_lse /*[nsrc][nscales][groups][2]*/, void* d_work, uint64_t work_bytes,
                                    void* stream);
/*
 * Profile likelihood on the same grid: the frequentist statistic of scripts/sens.py (StatCateg.FREQUENTIST, whose value the
 * reference takes from GolemFit's profiled fit, gf.get_llh_freq / Likelihood.GF_FREQ).  For each frozen scale
 * d_scales[s] = log10(Lambda_s) of a model that does not sample the scale (col_scale = -1), d_best[s] = the maximum of ln_prob
 * (llh.ln_prob: prior terms included) over every model column inside its prior box.  Task (s, k) is bounded Nelder-Mead
 * (Gao & Han's adaptive coefficients) in coordinates scaled per column (sigma of a Gaussian prior, a tenth of a uniform box)
 * from start k: start 0 = the prior means clipped to the box (the centre of a uniform box), start k >= 1 = the prior draw of
 * the scans with sample index (task0 + s) * nstarts + k (see gf_scan_config).  It converges when the spread of ln_prob over
 * the simplex is <= ftol and its extent <= xtol in every scaled coordinate, restarts from the best vertex with a fresh
 * simplex, and stops when a restart gains < ftol or after max_evals evaluations.  The best start wins (ties: the lower k),
 * so a scale's result depends on (seed, task0 + s, nstarts) only: not on how the scales are split over calls or GPUs.
 * Optional outputs: d_argmax[s] = the maximising theta, d_fr[s] = its measured composition, d_status[s] = its status bits
 * (| GF_ST_NON_FINITE if any evaluation of the scale was not finite; such values count as -inf), d_counts[s] =
 * {evaluations over all starts, starts that converged before max_evals}.  One launch: one block per scale, one thread per
 * start; the simplices take (ndim + 1)^2 * nstarts * 8 bytes of shared memory per block (GF_ERR_ARG beyond the device's limit).
 */
typedef struct gf_profile_config {
    uint64_t seed;      /* Philox key of the starts                                   */
    int64_t task0;      /* global index of d_scales[0]: shard / split offset          */
    int32_t nstarts;    /* starts per scale, multiple of 32, <= 256                   */
    int32_t max_evals;  /* objective evaluations per start                            */
    double ftol;        /* spread of ln_prob over the simplex                         */
    double xtol;        /* simplex diameter in scaled coordinates                     */
} gf_profile_config;
int gf_profile_grid(const gf_model* model, const gf_profile_config* cfg, const double* d_scales, int32_t nscales,
                    double* d_best /*[nscales]*/, double* d_argmax /*[nscales][ndim] or NULL*/,
                    double* d_fr /*[nscales][3] or NULL*/, uint8_t* d_status /*[nscales] or NULL*/,
                    int64_t* d_counts /*[nscales][2] or NULL: evaluations, starts that converged*/, void* stream);
/*
 * The profile likelihood for many SOURCE COMPOSITIONS in one launch: the frequentist column of the reference's sensitivity
 * table (scripts/sens.py with StatCateg.FREQUENTIST, run once per source composition, 30 per texture: submitter/sens_dag.py).
 * Row (j, s) is gf_profile_grid's task with source j: d_best[j][s] = the maximum over the model's columns inside their prior
 * box of ln_prob at log10 Lambda = d_scales[s], with sources[j] as the source composition and injected[j] as the injected
 * composition the Gaussian likelihood scores it against.  `sources` and `injected` are HOST arrays [nsrc][3], each row
 * normalised to unit sum inside; the model's own fixed_src and fr_bf are ignored.  The composition comes from the eigen
 * stage's transition sums (as gf_scan_evidence_sources), which differ from gf_profile_grid's per-bin mix in rounding only.
 * The optimiser, the starts and the configuration are gf_profile_grid's: start 0 = the nominal point, start k >= 1 = the prior
 * draw with sample index (task0 + s) * nstarts + k for every source, the best start wins (ties: the lower k).  A row
 * therefore depends on (seed, task0 + s, nstarts, source j, injected j) only: not on the other sources, their order, or how
 * the scales are split over calls or GPUs.  Optional outputs as gf_profile_grid's, per row: d_argmax[j][s], d_fr[j][s],
 * d_status[j][s], d_counts[j][s].  One launch: one block per (scale, source), one thread per start.
 * GF_ERR_ARG, with nothing enqueued, for: a null pointer; nscales outside [0, 2^30]; nsrc outside [1, GF_SRC_MAX = 256];
 * a sampled scale; no_bsm; a sampled source; llh_kind other than GF_LLH_GAUSSIAN; a source or injected row with a negative or
 * non-finite entry or a zero sum; nstarts not a multiple of 32 in [32, 256]; max_evals < 1; ftol or xtol negative;
 * task0 < 0; a uniform prior without a finite box; simplices that do not fit in shared memory.  nscales = 0 is a no-op.
 */
int gf_profile_sources(const gf_model* model, const gf_profile_config* cfg, const double* d_scales /*[nscales]*/, int32_t nscales,
                       const double* sources /*HOST [nsrc][3]*/, const double* injected /*HOST [nsrc][3]*/, int32_t nsrc,
                       double* d_best /*[nsrc][nscales]*/, double* d_argmax /*[nsrc][nscales][ndim] or NULL*/,
                       double* d_fr /*[nsrc][nscales][3] or NULL*/, uint8_t* d_status /*[nsrc][nscales] or NULL*/,
                       int64_t* d_counts /*[nsrc][nscales][2] or NULL*/, void* stream);
/* Highest-density coverage region of a histogram (plot.flavor_contour, plot.py:372-384: normalise,
 * sort cells by content, cumulative sum, `thres = searchsorted(cumsum, coverage/100)`, mask the first
 * `thres` cells).  d_mask[i] = 1 for the cells inside the region.  h_info (host, optional) receives
 * {count of the first excluded cell c*, number of masked cells, number of masked cells with count == c*}.
 * Cells tied at c* are taken in flat-index order (the reference's order among ties is that of an
 * unstable sort).  The 3-D Gaussian filter of plot.py:375 has sigma = 0.05 bins, i.e. a one-tap kernel:
 * it is the identity and is not applied.  Synchronises `stream`. */
int gf_coverage_mask(const unsigned long long* d_hist, int64_t cells, double coverage_percent, uint8_t* d_mask,
                     unsigned long long* h_info /*[3] or NULL*/, void* stream);

/* The smoothing step of the same function for hist_smooth values that are not the identity (plot.py:372-375:
 * `H = H / np.sum(H); H_s = gaussian_filter(H, sigma=hist_smooth)`): d_out[n1^3] = the normalised histogram filtered along
 * the three axes with SciPy's conventions (separable, boundary mode 'reflect', symmetric-kernel accumulation order of
 * scipy.ndimage, no FMA contraction: bit-identical to SciPy for the same weights).  `h_weights[0..radius]` (host) are the
 * normalised Gaussian weights from the outermost tap to the centre, radius = int(4 sigma + 0.5) <= 64 -- SciPy's
 * `_gaussian_kernel1d(sigma, 0, radius)[:radius + 1]`; `total` = the sum of the counts; d_work[n1^3] is scratch. */
int gf_hist_smooth(const unsigned long long* d_hist /*[n1^3]*/, int32_t n1, unsigned long long total, const double* h_weights,
                   int32_t radius, double* d_out /*[n1^3]*/, double* d_work /*[n1^3]*/, void* stream);

/* gf_coverage_mask for a non-negative float field (the smoothed histogram of gf_hist_smooth): mask of the cells that
 * precede `searchsorted(cumsum(sorted descending), coverage/100)` (plot.py:377-384; the threshold is the absolute fraction
 * coverage/100 of a field that sums to one).  *h_cstar (host, optional) = value of the first excluded cell, h_counts =
 * {number of masked cells, number of masked cells tied with it}.  Deterministic (fixed reduction order).  Synchronises `stream`. */
int gf_coverage_mask_f64(const double* d_field, int64_t cells, double coverage_percent, uint8_t* d_mask, double* h_cstar /*or NULL*/,
                         unsigned long long* h_counts /*[2] or NULL*/, void* stream);

/* ---- ensemble sampler --------------------------------------------------- */
/*
 * Device-resident affine-invariant ensemble sampler: the stretch move of emcee's EnsembleSampler
 * (Goodman & Weare 2010; red/blue half-ensembles, parameter a) that golemflavor/mcmc.py:27-53 drives
 * from Python, for `nchains` INDEPENDENT ensembles of `nwalkers` walkers at once (one thread per
 * walker pair; ensembles of up to 4096 walkers (8192 for SM-only models) live in the distributed shared memory of one thread-block
 * cluster per chain and synchronise with the hardware cluster barrier; the other shapes -- one block per
 * chain with global-memory positions, one cooperative launch with a grid barrier per half-step when the
 * batch is co-resident, one launch per half-step otherwise -- remain selectable; all shapes give
 * identical chains).
 *
 * Randomness (reproducible on the CPU, see tests): walker k of chain c at global step s uses
 * Philox4x32-10 with key = (lo32(seed), hi32(seed)), counter = ((chain0 + c)*nwalkers + k, lo32(s), hi32(s), 0)
 * (chain0 = global index of this call's first chain, so that a set of chains gives the same result
 * however it is sharded over calls or GPUs):
 *   word 0 -> z = ((a-1) u + 1)^2 / a,  word 1 -> partner j = floor(u * nwalkers/2) in the other half,
 *   word 2 -> accept iff (nfree-1) ln z + lnp(q) - lnp(p) > ln u;   u = (word + 0.5) 2^-32,
 *   proposal q = c_j - z (c_j - p_k), evaluated without FMA contraction.
 * Columns whose value is identical in all walkers of a chain stay frozen (q = c - z*0); `nfree` is
 * the number of sampled dimensions that enters the acceptance factor.
 */
typedef struct gf_ensemble_config {
    int64_t nchains;     /* independent ensembles                                   */
    int32_t nwalkers;    /* walkers per ensemble (even, >= 2)                       */
    int32_t nfree;       /* dimensions that actually move (<= model.ndim)           */
    int64_t nsteps;      /* steps to advance                                        */
    int64_t step0;       /* global index of the first step (RNG counter offset)     */
    int64_t thin;        /* store every thin-th step                                */
    double a;            /* stretch scale (emcee default 2.0)                       */
    uint64_t seed;
    int64_t chain0;      /* global index of the first chain (RNG counter offset)    */
    int32_t mode;        /* 0 = auto; 1 = grid-wide barrier per half-step (one cooperative launch, or one
                            launch per half-step when not co-resident); 2 = one block per chain;
                            3 = one thread-block cluster per chain, ensemble in distributed shared memory */
    int32_t cluster_blocks; /* mode 0 / 3: CTAs per cluster (rounded up to a power of two, <= 16); 0 = auto */
} gf_ensemble_config;
/* d_pos [nchains][nwalkers][ndim] and d_lnp [nchains][nwalkers] are updated in place (d_lnp must hold
 * ln_prob(d_pos) on entry: call gf_lnprob first).  Optional outputs: d_chain
 * [nchains][nwalkers][nsteps/thin][ndim] (emcee's `chain` layout, mcmc.py:44), d_lnp_chain
 * [nchains][nwalkers][nsteps/thin], d_naccept [nchains][nwalkers] (ADDS accepted-move counts). */
int gf_ensemble_run(const gf_model* model, const gf_ensemble_config* cfg, double* d_pos, double* d_lnp, double* d_chain,
                    double* d_lnp_chain, unsigned long long* d_naccept, void* stream);
/*
 * Integrated autocorrelation time of stored chains (emcee's get_autocorr_time, golemflavor/mcmc.py:46-49), for every chain
 * and parameter of d_chain[nchains][nwalkers][nsteps][ndim] (gf_ensemble_run's layout).  For chain c, parameter d and
 * walker w with y = x_w - mean(x_w): a_w(t) = sum_{i < nsteps-t} y_i y_{i+t}; rho_w(t) = a_w(t) / a_w(0) if a_w(0) > 0,
 * else 0; acf(t) = the mean of rho_w(t) over all walkers; tau(t) = 2 sum_{s <= t} acf(s) - 1.  d_window[c][d] = m, the
 * first t with t >= c * tau(t) (nsteps - 1 if there is none), and d_tau[c][d] = tau(m).  A walker whose values are
 * bitwise equal contributes rho = 0, so a parameter constant in every walker gets tau = -1 at m = 0.  Lags are computed
 * in tiles of 256 and stop at the tile holding every pair's window: 1 + 2 ceil(nsteps / 256) launches at most, no host
 * synchronisation, no float atomics (bit-identical results; a chain's result does not depend on the other chains).
 * d_work is scratch of at least gf_autocorr_time_workspace(...) bytes (0 for a shape the call refuses).  GF_ERR_ARG, with
 * nothing enqueued, for: a null pointer; nchains < 1, nwalkers < 1 or nsteps < 2; ndim outside [1, GF_MAX_DIM];
 * nchains * nwalkers > 2^31 - 1; c not finite and positive; a workspace too small.
 */
uint64_t gf_autocorr_time_workspace(int64_t nchains, int32_t nwalkers, int64_t nsteps, int32_t ndim);
int gf_autocorr_time(const double* d_chain /*[nchains][nwalkers][nsteps][ndim]*/, int64_t nchains, int32_t nwalkers, int64_t nsteps,
                     int32_t ndim, double c, double* d_tau /*[nchains][ndim]*/, int64_t* d_window /*[nchains][ndim]*/, void* d_work,
                     uint64_t work_bytes, void* stream);

/* ---- measurement helper ----------------------------------------------- */
/* fp64 throughput microbenchmarks: `iters` dependent FMAs x 8 chains per thread on a full grid;
 * *flops receives the number of fp64 FLOPs issued (2 per FMA, 1 per MUL); time it with CUDA events
 * on `stream`.  mode 0 (operands: 1 register pair + uniform constants) is the roofline peak;
 * modes 1-3 probe the register-file operand bandwidth (3 distinct register pairs per DFMA,
 * DMUL with 2 register pairs, DFMA with operands shared between consecutive instructions). */
int gf_fp64_peak_probe(int32_t mode, int64_t iters, double* d_sink /*[>= 1]*/, double* flops, void* stream);
/* Device self-test of the MUFU-seeded helpers of the eigen stage: rsqrt_out[i] ~ 1/sqrt(x[i]),
 * rcp_out[i] ~ 1/x[i] for normal positive x (tests/test_gpu_parity.py checks them to 1e-15). */
int gf_selftest_math(const double* d_x, int64_t n, double* d_rsqrt_out, double* d_rcp_out, void* stream);
/* Device self-test of the table-free sin / cos of the CP phase (fr.py:157-159 evaluates them with NumPy):
 * sin_out, cos_out from the joint routine, cos_only_out from the cosine-only one. */
int gf_selftest_trig(const double* d_x, int64_t n, double* d_sin_out, double* d_cos_out, double* d_cos_only_out, void* stream);
/* Device self-test of the table-free logarithm of the sampler's acceptance test: log_out[i] ~ ln x[i] for
 * positive normal x. */
int gf_selftest_log(const double* d_x, int64_t n, double* d_log_out, void* stream);
/* Number of kernels this library has launched in the calling process (bench.py's gpu_launches). */
uint64_t gf_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* GOLEMFLAVOR_B200_H */
