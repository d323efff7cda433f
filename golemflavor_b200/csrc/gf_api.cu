/*
 * gf_api.cu -- library glue, model flattening and the element-wise entry points of the C ABI
 * (fr.angles_to_u, fr.angles_to_fr, fr.u_to_fr, fr.cardano_eqn, fr.params_to_BSMu,
 * llh.multi_gaussian, plus the fp64 peak probe).  The log-posterior kernel lives in
 * gf_lnprob.cu, the Monte-Carlo scans in gf_scan.cu.
 */
#include <atomic>
#include <math.h>
#include <string.h>

#include "gf_common.cuh"

/* ------------------------------------------------------------------ glue */

static thread_local char g_last_error[512] = "";
std::atomic<unsigned long long> g_gf_launches{0};

int gf_fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_last_error, sizeof(g_last_error), fmt, ap);
    va_end(ap);
    return code;
}

int gf_sm_count(int* sms) {
    /* cached per device ordinal: a process may drive several GPUs */
    constexpr int kMaxDevices = 64;
    static std::atomic<int> cached[kMaxDevices];
    int dev = 0;
    GF_CUDA(cudaGetDevice(&dev));
    int n = (dev >= 0 && dev < kMaxDevices) ? cached[dev].load(std::memory_order_relaxed) : 0;
    if (!n) {
        GF_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
        if (dev >= 0 && dev < kMaxDevices) cached[dev].store(n, std::memory_order_relaxed);
    }
    *sms = n;
    return GF_OK;
}

extern "C" int gf_abi_version(void) { return GF_ABI_VERSION; }
extern "C" const char* gf_last_error(void) { return g_last_error; }
extern "C" uint64_t gf_launch_count(void) { return g_gf_launches.load(); }
extern "C" uint64_t gf_sizeof(int32_t which) {
    return which == 0 ? sizeof(gf_model) : which == 1 ? sizeof(gf_scan_config) : which == 2 ? sizeof(gf_prior_dim) : which == 3 ? sizeof(gf_ensemble_config)
         : which == 4 ? sizeof(gf_profile_config) : 0;
}

extern "C" int gf_device_info(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor, int32_t* clock_khz) {
    int dev = 0, v = 0;
    GF_CUDA(cudaGetDevice(&dev));
    GF_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev));
    if (sm_count) *sm_count = v;
    GF_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrComputeCapabilityMajor, dev));
    if (cc_major) *cc_major = v;
    GF_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrComputeCapabilityMinor, dev));
    if (cc_minor) *cc_minor = v;
    GF_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrClockRate, dev));
    if (clock_khz) *clock_khz = v;
    return GF_OK;
}

extern "C" int gf_host_alloc(void** h_ptr, uint64_t bytes) {
    GF_REQUIRE(h_ptr != nullptr, "gf_host_alloc: null output pointer");
    GF_CUDA(cudaHostAlloc(h_ptr, bytes ? bytes : 1, cudaHostAllocDefault));
    return GF_OK;
}

extern "C" int gf_host_alloc_wc(void** h_ptr, uint64_t bytes) {
    GF_REQUIRE(h_ptr != nullptr, "gf_host_alloc_wc: null output pointer");
    GF_CUDA(cudaHostAlloc(h_ptr, bytes ? bytes : 1, cudaHostAllocWriteCombined));
    return GF_OK;
}

extern "C" int gf_host_free(void* h_ptr) {
    if (h_ptr) GF_CUDA(cudaFreeHost(h_ptr));
    return GF_OK;
}

/* ------------------------------------------------------------------ model flattening */

/* log(Phi(b) - Phi(a)) for a < b, evaluated on the side of the distribution where the
 * difference does not cancel (closed form of the normaliser of scipy.stats.truncnorm,
 * llh.py:25-29). */
static double log_gauss_mass(double a, double b) {
    const double r = 0.70710678118654752440;
    if (a == -INFINITY && b == INFINITY) return 0.0;
    if (b <= 0.0) return log(0.5 * (erfc(-b * r) - erfc(-a * r)));
    if (a >= 0.0) return log(0.5 * (erfc(a * r) - erfc(b * r)));
    return log1p(-0.5 * (erfc(-a * r) + erfc(b * r)));
}

static double gauss_cdf(double x) { return 0.5 * erfc(-x * 0.70710678118654752440); }

int gf_build_dev_model(const gf_model* m, gf_dev_model* d) {
    GF_REQUIRE(m != nullptr, "model is NULL");
    GF_REQUIRE(m->ndim >= 1 && m->ndim <= GF_MAX_DIM, "model.ndim = %d outside [1, %d]", m->ndim, GF_MAX_DIM);
    memset(d, 0, sizeof(*d));
    d->ndim = m->ndim;
    d->no_bsm = m->no_bsm ? 1 : 0;
    d->llh_kind = m->llh_kind;
    GF_REQUIRE(m->llh_kind == GF_LLH_FLAT || m->llh_kind == GF_LLH_GAUSSIAN, "model.llh_kind = %d is not a GF_LLH_* value", m->llh_kind);
    d->emulate_underflow = m->emulate_underflow ? 1 : 0;

    struct { const int32_t* src; int32_t* dst; int n; const char* name; } cols[] = {
        {m->col_sm, d->col_sm, 4, "col_sm"},       {m->col_mass, d->col_mass, 2, "col_mass"},
        {m->col_src, d->col_src, 2, "col_src"},    {m->col_np, d->col_np, 4, "col_np"},
        {&m->col_scale, &d->col_scale, 1, "col_scale"}, {&m->col_x, &d->col_x, 1, "col_x"},
        {m->col_src3, d->col_src3, 3, "col_src3"}};
    for (auto& c : cols)
        for (int k = 0; k < c.n; ++k) {
            GF_REQUIRE(c.src[k] >= -1 && c.src[k] < m->ndim, "model.%s[%d] = %d outside [-1, ndim)", c.name, k, c.src[k]);
            c.dst[k] = c.src[k];
        }
    GF_REQUIRE((m->col_src[0] >= 0) == (m->col_src[1] >= 0), "model.col_src: both source angles must be sampled or neither");
    GF_REQUIRE(!(m->col_src[0] >= 0 && m->col_x >= 0), "model: col_src and col_x are mutually exclusive");
    GF_REQUIRE((m->col_src3[0] >= 0) == (m->col_src3[1] >= 0) && (m->col_src3[0] >= 0) == (m->col_src3[2] >= 0),
               "model.col_src3: all three source ratios must be sampled or none");
    GF_REQUIRE(!(m->col_src3[0] >= 0 && (m->col_src[0] >= 0 || m->col_x >= 0)), "model: col_src3 excludes col_src and col_x");
    d->np_free = 0;
    for (int k = 0; k < 4; ++k) d->np_free |= (m->col_np[k] >= 0);

    memcpy(d->fixed_sm, m->fixed_sm, sizeof(d->fixed_sm));
    memcpy(d->fixed_mass, m->fixed_mass, sizeof(d->fixed_mass));
    memcpy(d->fixed_src, m->fixed_src, sizeof(d->fixed_src));
    memcpy(d->fixed_np, m->fixed_np, sizeof(d->fixed_np));
    d->fixed_loglam = m->fixed_loglam;
    d->src_S = m->fixed_src[0] + m->fixed_src[1] + m->fixed_src[2];
    d->src_sd0 = m->fixed_src[0] - m->fixed_src[2];
    d->src_sd1 = m->fixed_src[1] - m->fixed_src[2];
    if (m->col_src[0] < 0 && m->col_x < 0 && m->col_src3[0] < 0) {
        const double s = m->fixed_src[0] + m->fixed_src[1] + m->fixed_src[2];
        GF_REQUIRE(isfinite(s) && s != 0.0, "model.fixed_src sums to %g", s);
    }

    if (!d->no_bsm) {
        GF_REQUIRE(m->dimension >= 3 && m->dimension <= 8, "model.dimension = %d outside [3, 8] (fr.SCALE_BOUNDARIES)", m->dimension);
        GF_REQUIRE(m->nbins >= 1 && m->nbins <= GF_MAX_BINS, "model.nbins = %d outside [1, %d]", m->nbins, GF_MAX_BINS);
        d->nbins = m->nbins;
        for (int b = 0; b < m->nbins; ++b) {
            const double lo = m->bin_edges[b], hi = m->bin_edges[b + 1];
            GF_REQUIRE(lo > 0.0 && hi > 0.0 && isfinite(lo) && isfinite(hi), "model.bin_edges[%d..%d] = (%g, %g) must be positive", b, b + 1, lo, hi);
            const double ec = sqrt(lo * hi);                                   /* fr.py:413 */
            d->g[b] = 2.0 * pow(ec, (double)(m->dimension - 2)) * GFP_MASS_SCALE; /* 2E * E^(d-3), fr.py:386,394 */
            d->width[b] = fabs(hi - lo);                                       /* fr.py:414 */
            d->wsum += d->width[b];
        }
        GF_REQUIRE(d->wsum > 0.0 && isfinite(d->wsum), "model.bin_edges: the bins have no width");
        d->inv_S_wsum = 1.0 / (d->src_S * d->wsum);
        /* fixed new-physics mixing: T = N diag(0, 1/100, 1) N^+  (fr.py:380-381, 390-394) */
        const gfp_trig tn = gfp_angles_trig(m->fixed_np[0], m->fixed_np[1], m->fixed_np[2], m->fixed_np[3]);
        d->T = gfp_herm_from_cols(gfp_cols_from_trig(tn), GFP_T_EIG1, GFP_T_EIG2);
        if (!d->np_free) GF_REQUIRE(isfinite(d->T.d0 + d->T.d1 + d->T.d2), "model.fixed_np does not describe mixing angles");
        d->penT = gfp_make_pencil_T(d->T);
        d->adjT = gfp_adj_tf(d->penT.te, d->T);
    }

    d->fr_bf[0] = m->fr_bf[0];
    d->fr_bf[1] = m->fr_bf[1];
    d->fr_bf[2] = m->fr_bf[2];
    if (m->llh_kind == GF_LLH_GAUSSIAN) {
        GF_REQUIRE(m->smearing > 0.0 && isfinite(m->smearing), "model.smearing = %g must be positive", m->smearing);
        d->half_inv_s2 = 0.5 / (m->smearing * m->smearing);
        d->lognorm3 = -1.5 * log(2.0 * M_PI * m->smearing * m->smearing);
    }
    d->offset = m->offset;
    d->underflow_logpdf = -1075.0 * M_LN2; /* exp() rounds to +0 below log(2^-1075) */
    d->llh_const = m->llh_const;
    d->epsilon = m->epsilon > 0.0 ? m->epsilon : 1e-7;

    for (int k = 0; k < m->ndim; ++k) {
        const gf_prior_dim& p = m->prior[k];
        GF_REQUIRE(p.lo <= p.hi, "model.prior[%d]: ranges (%g, %g) are not ordered", k, p.lo, p.hi);
        d->lo[k] = p.lo;
        d->hi[k] = p.hi;
        d->kind[k] = p.kind;
        d->cdf_lo[k] = 0.0;
        d->cdf_span[k] = 1.0;
        if (p.kind == GF_PRIOR_UNIFORM) continue;
        GF_REQUIRE(p.kind == GF_PRIOR_GAUSSIAN || p.kind == GF_PRIOR_LIMITEDGAUSS, "model.prior[%d].kind = %d is not a GF_PRIOR_* value", k, p.kind);
        GF_REQUIRE(p.sigma > 0.0 && isfinite(p.sigma) && isfinite(p.mu), "model.prior[%d]: Gaussian prior needs finite mu and sigma > 0", k);
        d->mu[k] = p.mu;
        d->sigma[k] = p.sigma;
        d->inv_sigma[k] = 1.0 / p.sigma;
        const double a = (p.lo - p.mu) / p.sigma, b = (p.hi - p.mu) / p.sigma;
        const double lognorm_free = -log(p.sigma * sqrt(2.0 * M_PI));
        /* llh.py:82-85: GAUSSIAN is an unbounded normal; llh.py:86-90: LIMITEDGAUSS is truncated to ranges */
        d->lognorm_total += (p.kind == GF_PRIOR_GAUSSIAN) ? lognorm_free : lognorm_free - log_gauss_mass(a, b);
        /* scans draw inside `ranges` for both kinds (the box check of llh.py:74-78 applies to both) */
        d->cdf_lo[k] = gauss_cdf(a);
        d->cdf_span[k] = gauss_cdf(b) - gauss_cdf(a);
    }
    return GF_OK;
}

extern "C" int gf_model_check(const gf_model* model) {
    gf_dev_model d;
    return gf_build_dev_model(model, &d);
}

/* ------------------------------------------------------------------ element-wise kernels */

#define GF_EW_THREADS 128

__global__ void __launch_bounds__(GF_EW_THREADS) k_angles_to_u(const double* __restrict__ ang, int64_t n, double* __restrict__ u) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const gfp_trig t = gfp_angles_trig(ang[4 * i], ang[4 * i + 1], ang[4 * i + 2], ang[4 * i + 3]);
    double m[18];
    gfp_full_u(t, m);
    double2* o = reinterpret_cast<double2*>(u + 18 * i);
#pragma unroll
    for (int k = 0; k < 9; ++k) o[k] = make_double2(m[2 * k], m[2 * k + 1]);
}

__global__ void __launch_bounds__(GF_EW_THREADS) k_angles_to_fr(const double* __restrict__ src, int64_t n, double* __restrict__ fr) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double f[3];
    gfp_angles_to_fr(src[2 * i], src[2 * i + 1], f);
    fr[3 * i] = f[0];
    fr[3 * i + 1] = f[1];
    fr[3 * i + 2] = f[2];
}

__global__ void __launch_bounds__(GF_EW_THREADS)
    k_u_to_fr(const double* __restrict__ source, int64_t source_stride, const double* __restrict__ u, int64_t n, double* __restrict__ fr) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double2* m = reinterpret_cast<const double2*>(u + 18 * i);
    double X[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        const double2 z = m[k];
        X[k] = fma(z.x, z.x, z.y * z.y);
    }
    const double s0 = source[i * source_stride], s1 = source[i * source_stride + 1], s2 = source[i * source_stride + 2];
    double f[3];
    gfp_mix(X, s0, s1, s2, f);
    const double inv = 1.0 / (s0 + s1 + s2); /* fr.py:535 */
    fr[3 * i] = f[0] * inv;
    fr[3 * i + 1] = f[1] * inv;
    fr[3 * i + 2] = f[2] * inv;
}

__device__ __forceinline__ gfp_herm3 load_herm(const double* h /*[18]*/) {
    /* Hermitian part of the input: real diagonal, upper triangle averaged with the conjugate lower one */
    gfp_herm3 r;
    r.d0 = h[0];
    r.d1 = h[8];
    r.d2 = h[16];
    r.ar = 0.5 * (h[2] + h[6]);
    r.ai = 0.5 * (h[3] - h[7]);
    r.br = 0.5 * (h[4] + h[12]);
    r.bi = 0.5 * (h[5] - h[13]);
    r.cr = 0.5 * (h[10] + h[14]);
    r.ci = 0.5 * (h[11] - h[15]);
    return r;
}

__global__ void __launch_bounds__(GF_EW_THREADS)
    k_eigvec_herm3(const double* __restrict__ ham, int64_t n, double* __restrict__ vec, double* __restrict__ eigval, uint8_t* __restrict__ status) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const gfp_herm3 h = load_herm(ham + 18 * i);
    double lam[3], v[18];
    const double relgap = gfp_herm3_eig_sorted(h, lam, v);
    unsigned st = 0u;
    if (!(relgap >= GFP_ILL_GAP)) st |= GFP_ST_ILL_COND;
    double acc = 0.0;
#pragma unroll
    for (int k = 0; k < 18; ++k) {
        vec[18 * i + k] = v[k];
        acc += fabs(v[k]);
    }
    if (!(acc < 1e300)) st |= GFP_ST_NON_FINITE;
    if (eigval) {
        eigval[3 * i] = lam[0];
        eigval[3 * i + 1] = lam[1];
        eigval[3 * i + 2] = lam[2];
    }
    if (status) status[i] = (uint8_t)st;
}

__global__ void __launch_bounds__(GF_EW_THREADS)
    k_params_to_bsmu(const double* __restrict__ bsm, int dim, const double* __restrict__ energy, const double* __restrict__ mass,
                     int64_t mass_stride, const double* __restrict__ sm_u, int64_t smu_stride, int no_bsm, double epsilon, int64_t n,
                     double* __restrict__ vec, uint8_t* __restrict__ status) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double u[18];
#pragma unroll
    for (int k = 0; k < 18; ++k) u[k] = sm_u[i * smu_stride + k];
    const double e = energy[i];
    /* 2E * 2^70 * H = U diag(0, m21, m3x) U^+ 2^70 + 2 E^(d-2) 2^70 N diag(0, L/100, L) N^+  (fr.py:380-395) */
    gfp_herm3 h = gfp_herm_from_u(u, mass[i * mass_stride] * GFP_MASS_SCALE, mass[i * mass_stride + 1] * GFP_MASS_SCALE);
    if (!no_bsm) {
        const gfp_trig tn = gfp_angles_trig(bsm[5 * i], bsm[5 * i + 1], bsm[5 * i + 2], bsm[5 * i + 3]);
        const gfp_herm3 T = gfp_herm_from_cols(gfp_cols_from_trig(tn), 0.01, 1.0);
        const double rho = exp10(bsm[5 * i + 4]) * 2.0 * pow(e, (double)(dim - 2)) * GFP_MASS_SCALE;
        h.d0 = fma(rho, T.d0, h.d0);
        h.d1 = fma(rho, T.d1, h.d1);
        h.d2 = fma(rho, T.d2, h.d2);
        h.ar = fma(rho, T.ar, h.ar);
        h.ai = fma(rho, T.ai, h.ai);
        h.br = fma(rho, T.br, h.br);
        h.bi = fma(rho, T.bi, h.bi);
        h.cr = fma(rho, T.cr, h.cr);
        h.ci = fma(rho, T.ci, h.ci);
    }
    double lam[3], v[18];
    const double relgap = gfp_herm3_eig_sorted(h, lam, v);
    unsigned st = 0u;
    if (!(relgap >= GFP_ILL_GAP)) st |= GFP_ST_ILL_COND;
    double acc = 0.0;
#pragma unroll
    for (int k = 0; k < 18; ++k) {
        vec[18 * i + k] = v[k];
        acc += fabs(v[k]);
    }
    if (!(acc < 1e300)) st |= GFP_ST_NON_FINITE | GFP_ST_NON_UNITARY;
    /* fr.test_unitarity (fr.py:489-498): f = |V V^+|, |tr f - 3| and |sum f - 3| against epsilon */
    double tr = 0.0, sum = 0.0;
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = 0; b < 3; ++b) {
            double re = 0.0, im = 0.0;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const double ar = v[2 * (3 * a + c)], ai = v[2 * (3 * a + c) + 1], br = v[2 * (3 * b + c)], bi = v[2 * (3 * b + c) + 1];
                re += ar * br + ai * bi;
                im += ai * br - ar * bi;
            }
            const double f = sqrt(re * re + im * im);
            sum += f;
            if (a == b) tr += f;
        }
    if (!(fabs(tr - 3.0) < epsilon && fabs(sum - 3.0) < epsilon)) st |= GFP_ST_NON_UNITARY;
    if (status) status[i] = (uint8_t)st;
}

__global__ void __launch_bounds__(GF_EW_THREADS)
    k_multi_gaussian(const double* __restrict__ fr, int64_t n, double b0, double b1, double b2, double half_inv_s2, double lognorm3,
                     double offset, int emulate_underflow, double underflow_logpdf, double* __restrict__ llh) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double f[3] = {fr[3 * i], fr[3 * i + 1], fr[3 * i + 2]};
    const double bf[3] = {b0, b1, b2};
    llh[i] = gf_multi_gaussian(f, bf, half_inv_s2, lognorm3, offset, emulate_underflow, underflow_logpdf);
}

/* fp64 throughput probes: 8 independent dependent-chains per thread, nothing else in the loop.
 *   mode 0: a = fma(a, m, b)      m, b uniform constants (2 register-file operands)  -- the roofline peak
 *   mode 1: a = fma(a, b_c, d_c)  three distinct per-thread register pairs per instruction
 *   mode 2: a = a * b_c           DMUL, two distinct register pairs
 *   mode 3: a = fma(a, b, d)      b, d per-thread registers shared by all chains (operand-reuse friendly)
 */
#define GF_PROBE_CHAINS 8
#define GF_PROBE_THREADS 256
#define GF_PROBE_BLOCKS_PER_SM 8
template <int MODE>
__global__ void __launch_bounds__(GF_PROBE_THREADS) k_fp64_probe(int64_t iters, double seed, double* __restrict__ sink) {
    double a[GF_PROBE_CHAINS], b[GF_PROBE_CHAINS], d[GF_PROBE_CHAINS];
#pragma unroll
    for (int c = 0; c < GF_PROBE_CHAINS; ++c) {
        a[c] = seed + 1e-3 * (threadIdx.x + c);
        b[c] = 1.0 - 1e-9 * (1 + ((threadIdx.x + c) & 7)) * seed * 2.0; /* per-thread values: stay in registers */
        d[c] = 1e-9 * (1 + ((threadIdx.x * 3 + c) & 7)) * seed * 2.0;
    }
    const double m = 1.0 - 1e-9, k = 1e-9;
    for (int64_t it = 0; it < iters; ++it) {
#pragma unroll
        for (int c = 0; c < GF_PROBE_CHAINS; ++c) {
            if (MODE == 0) a[c] = fma(a[c], m, k);
            if (MODE == 1) a[c] = fma(a[c], b[c], d[c]);
            if (MODE == 2) a[c] = a[c] * b[c];
            if (MODE == 3) a[c] = fma(a[c], b[0], d[0]);
        }
    }
    double s = 0.0;
#pragma unroll
    for (int c = 0; c < GF_PROBE_CHAINS; ++c) s += a[c] + b[c] + d[c];
    if (s == 12345.6789) sink[0] = s; /* never true: keeps the chains alive */
}

__global__ void __launch_bounds__(GF_EW_THREADS) k_selftest_math(const double* __restrict__ x, int64_t n, double* __restrict__ rs, double* __restrict__ rc) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    rs[i] = gfp_rsqrt(x[i]);
    rc[i] = gfp_rcp(x[i]);
}

__global__ void __launch_bounds__(GF_EW_THREADS)
    k_selftest_trig(const double* __restrict__ x, int64_t n, double* __restrict__ sn, double* __restrict__ cs, double* __restrict__ cs_only) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double s, c;
    gfp_sincos(x[i], &s, &c);
    sn[i] = s;
    cs[i] = c;
    cs_only[i] = gfp_cos(x[i]);
}

__global__ void __launch_bounds__(GF_EW_THREADS) k_selftest_log(const double* __restrict__ x, int64_t n, double* __restrict__ lg) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) lg[i] = gfp_log_pos(x[i]);
}

/* ------------------------------------------------------------------ C ABI */

extern "C" int gf_selftest_log(const double* d_x, int64_t n, double* d_log, void* stream) {
    GF_REQUIRE(n >= 0, "gf_selftest_log: n = %lld", (long long)n);
    if (n == 0) return GF_OK;
    GF_REQUIRE(d_x && d_log, "gf_selftest_log: null pointer");
    k_selftest_log<<<gf_blocks_for(n, GF_EW_THREADS), GF_EW_THREADS, 0, (cudaStream_t)stream>>>(d_x, n, d_log);
    ++g_gf_launches;
    GF_LAUNCH_CHECK("k_selftest_log");
    return GF_OK;
}

extern "C" int gf_selftest_trig(const double* d_x, int64_t n, double* d_sin, double* d_cos, double* d_cos_only, void* stream) {
    GF_REQUIRE(n >= 0, "gf_selftest_trig: n = %lld", (long long)n);
    if (n == 0) return GF_OK;
    GF_REQUIRE(d_x && d_sin && d_cos && d_cos_only, "gf_selftest_trig: null pointer");
    k_selftest_trig<<<gf_blocks_for(n, GF_EW_THREADS), GF_EW_THREADS, 0, (cudaStream_t)stream>>>(d_x, n, d_sin, d_cos, d_cos_only);
    ++g_gf_launches;
    GF_LAUNCH_CHECK("k_selftest_trig");
    return GF_OK;
}

extern "C" int gf_selftest_math(const double* d_x, int64_t n, double* d_rsqrt_out, double* d_rcp_out, void* stream) {
    GF_REQUIRE(n >= 0, "gf_selftest_math: n = %lld", (long long)n);
    if (n == 0) return GF_OK;
    GF_REQUIRE(d_x && d_rsqrt_out && d_rcp_out, "gf_selftest_math: null pointer");
    k_selftest_math<<<gf_blocks_for(n, GF_EW_THREADS), GF_EW_THREADS, 0, (cudaStream_t)stream>>>(d_x, n, d_rsqrt_out, d_rcp_out);
    ++g_gf_launches;
    GF_LAUNCH_CHECK("k_selftest_math");
    return GF_OK;
}

extern "C" int gf_angles_to_u(const double* d_angles, int64_t n, double* d_u, void* stream) {
    GF_REQUIRE(n >= 0, "gf_angles_to_u: n = %lld", (long long)n);
    if (n == 0) return GF_OK;
    GF_REQUIRE(d_angles && d_u, "gf_angles_to_u: null pointer");
    k_angles_to_u<<<gf_blocks_for(n, GF_EW_THREADS), GF_EW_THREADS, 0, (cudaStream_t)stream>>>(d_angles, n, d_u);
    ++g_gf_launches;
    GF_LAUNCH_CHECK("k_angles_to_u");
    return GF_OK;
}

extern "C" int gf_angles_to_fr(const double* d_src_angles, int64_t n, double* d_fr, void* stream) {
    GF_REQUIRE(n >= 0, "gf_angles_to_fr: n = %lld", (long long)n);
    if (n == 0) return GF_OK;
    GF_REQUIRE(d_src_angles && d_fr, "gf_angles_to_fr: null pointer");
    k_angles_to_fr<<<gf_blocks_for(n, GF_EW_THREADS), GF_EW_THREADS, 0, (cudaStream_t)stream>>>(d_src_angles, n, d_fr);
    ++g_gf_launches;
    GF_LAUNCH_CHECK("k_angles_to_fr");
    return GF_OK;
}

extern "C" int gf_u_to_fr(const double* d_source, int64_t source_stride, const double* d_u, int64_t n, double* d_fr, void* stream) {
    GF_REQUIRE(n >= 0, "gf_u_to_fr: n = %lld", (long long)n);
    GF_REQUIRE(source_stride == 0 || source_stride == 3, "gf_u_to_fr: source_stride must be 0 or 3, got %lld", (long long)source_stride);
    if (n == 0) return GF_OK;
    GF_REQUIRE(d_source && d_u && d_fr, "gf_u_to_fr: null pointer");
    k_u_to_fr<<<gf_blocks_for(n, GF_EW_THREADS), GF_EW_THREADS, 0, (cudaStream_t)stream>>>(d_source, source_stride, d_u, n, d_fr);
    ++g_gf_launches;
    GF_LAUNCH_CHECK("k_u_to_fr");
    return GF_OK;
}

extern "C" int gf_eigvec_herm3(const double* d_ham, int64_t n, double* d_vec, double* d_eigval, uint8_t* d_status, void* stream) {
    GF_REQUIRE(n >= 0, "gf_eigvec_herm3: n = %lld", (long long)n);
    if (n == 0) return GF_OK;
    GF_REQUIRE(d_ham && d_vec, "gf_eigvec_herm3: null pointer");
    k_eigvec_herm3<<<gf_blocks_for(n, GF_EW_THREADS), GF_EW_THREADS, 0, (cudaStream_t)stream>>>(d_ham, n, d_vec, d_eigval, d_status);
    ++g_gf_launches;
    GF_LAUNCH_CHECK("k_eigvec_herm3");
    return GF_OK;
}

extern "C" int gf_params_to_bsmu(const double* d_bsm, int32_t dim, const double* d_energy, const double* d_mass, int64_t mass_stride,
                                 const double* d_sm_u, int64_t smu_stride, int32_t no_bsm, double epsilon, int64_t n, double* d_vec,
                                 uint8_t* d_status, void* stream) {
    if (!(epsilon > 0.0)) epsilon = 1e-7; /* fr.py:319 default; the Jacobi eigenvectors are unitary to rounding, so only a
                                            * caller-tightened epsilon (or a non-finite input) ever raises the flag */
    GF_REQUIRE(n >= 0, "gf_params_to_bsmu: n = %lld", (long long)n);
    GF_REQUIRE(mass_stride == 0 || mass_stride == 2, "gf_params_to_bsmu: mass_stride must be 0 or 2");
    GF_REQUIRE(smu_stride == 0 || smu_stride == 18, "gf_params_to_bsmu: smu_stride must be 0 or 18");
    GF_REQUIRE(no_bsm || (dim >= 3 && dim <= 8), "gf_params_to_bsmu: dim = %d outside [3, 8]", dim);
    if (n == 0) return GF_OK;
    GF_REQUIRE(d_energy && d_mass && d_sm_u && d_vec && (no_bsm || d_bsm), "gf_params_to_bsmu: null pointer");
    k_params_to_bsmu<<<gf_blocks_for(n, GF_EW_THREADS), GF_EW_THREADS, 0, (cudaStream_t)stream>>>(
        d_bsm, dim, d_energy, d_mass, mass_stride, d_sm_u, smu_stride, no_bsm, epsilon, n, d_vec, d_status);
    ++g_gf_launches;
    GF_LAUNCH_CHECK("k_params_to_bsmu");
    return GF_OK;
}

extern "C" int gf_multi_gaussian(const double* d_fr, int64_t n, const double* h_fr_bf, double smearing, double offset,
                                 int32_t emulate_underflow, double* d_llh, void* stream) {
    GF_REQUIRE(n >= 0, "gf_multi_gaussian: n = %lld", (long long)n);
    GF_REQUIRE(smearing > 0.0 && isfinite(smearing), "gf_multi_gaussian: smearing = %g must be positive", smearing);
    GF_REQUIRE(h_fr_bf != nullptr, "gf_multi_gaussian: fr_bf is NULL");
    if (n == 0) return GF_OK;
    GF_REQUIRE(d_fr && d_llh, "gf_multi_gaussian: null pointer");
    const double half_inv_s2 = 0.5 / (smearing * smearing);
    const double lognorm3 = -1.5 * log(2.0 * M_PI * smearing * smearing);
    k_multi_gaussian<<<gf_blocks_for(n, GF_EW_THREADS), GF_EW_THREADS, 0, (cudaStream_t)stream>>>(
        d_fr, n, h_fr_bf[0], h_fr_bf[1], h_fr_bf[2], half_inv_s2, lognorm3, offset, emulate_underflow, -1075.0 * M_LN2, d_llh);
    ++g_gf_launches;
    GF_LAUNCH_CHECK("k_multi_gaussian");
    return GF_OK;
}

extern "C" int gf_fp64_peak_probe(int32_t mode, int64_t iters, double* d_sink, double* flops, void* stream) {
    GF_REQUIRE(iters > 0 && d_sink != nullptr, "gf_fp64_peak_probe: bad arguments");
    GF_REQUIRE(mode >= 0 && mode <= 3, "gf_fp64_peak_probe: mode = %d outside [0, 3]", mode);
    int sms = 0;
    if (int rc = gf_sm_count(&sms)) return rc;
    const unsigned blocks = (unsigned)(sms * GF_PROBE_BLOCKS_PER_SM);
    cudaStream_t st = (cudaStream_t)stream;
    if (mode == 0) k_fp64_probe<0><<<blocks, GF_PROBE_THREADS, 0, st>>>(iters, 0.5, d_sink);
    if (mode == 1) k_fp64_probe<1><<<blocks, GF_PROBE_THREADS, 0, st>>>(iters, 0.5, d_sink);
    if (mode == 2) k_fp64_probe<2><<<blocks, GF_PROBE_THREADS, 0, st>>>(iters, 0.5, d_sink);
    if (mode == 3) k_fp64_probe<3><<<blocks, GF_PROBE_THREADS, 0, st>>>(iters, 0.5, d_sink);
    ++g_gf_launches;
    GF_LAUNCH_CHECK("k_fp64_probe");
    /* flops: 2 per FMA, 1 per MUL */
    if (flops) *flops = (mode == 2 ? 1.0 : 2.0) * (double)iters * GF_PROBE_CHAINS * GF_PROBE_THREADS * (double)blocks;
    return GF_OK;
}
