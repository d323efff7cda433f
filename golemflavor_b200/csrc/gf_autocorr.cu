/*
 * gf_autocorr.cu -- integrated autocorrelation time of stored ensemble chains (emcee's `get_autocorr_time`, the
 * `sampler.acor` that golemflavor/mcmc.py:46-49 prints), for many chains in one call.
 *
 * For chain c, parameter d and walker w with y = x_w - mean(x_w):
 *   a_w(t) = sum_{i < N-t} y_i y_{i+t},   rho_w(t) = a_w(t) / a_w(0) if a_w(0) > 0 else 0,
 *   acf(t) = (1/W) sum_w rho_w(t),        tau(t) = 2 sum_{s <= t} acf(s) - 1,
 * window m = the first t with t >= c tau(t) (N - 1 if there is none), result tau(m).  This is the FFT estimator of
 * mcmc.integrated_time as a direct lag sum: the zero-padded FFT product is the exact linear autocorrelation, and only the
 * lags up to m are needed (typically 5 tau << N).  A walker whose N values are bitwise equal has y = 0 exactly (its mean
 * is taken to be that value) and contributes rho = 0.
 *
 * Launches, all on `stream`, no host synchronisation:
 *   k_acor_mean                  per-walker means (fixed-order sums) and the open flags of every (chain, parameter) pair;
 *   (k_acor_tile, k_acor_decide) for each tile of GF_ACOR_T lags: every walker's rho_w(t) of the tile into the workspace,
 *                                then the fixed-order walker sum, the running tau(t) and the window test per open pair.
 * A tile whose pairs are all closed returns at once.  No float atomics: every sum has one fixed order, so results are
 * bit-identical from run to run and a chain's result does not depend on the other chains of the call.
 */
#include <atomic>
#include <math.h>

#include "gf_common.cuh"

extern std::atomic<unsigned long long> g_gf_launches;

#define GF_ACOR_L 8                          /* lags per thread: T = 32 L lags per tile, one warp per parameter   */
#define GF_ACOR_T (32 * GF_ACOR_L)           /* 256                                                              */
#define GF_ACOR_S 512                        /* steps per shared-memory chunk (a multiple of 32 L)               */
#define GF_ACOR_SB (GF_ACOR_S + GF_ACOR_T + 32) /* lagged window: the chunk shifted by t0, plus the register window's overrun */

static_assert(GF_ACOR_S % (32 * GF_ACOR_L) == 0, "the unrolled step loop needs S / 32 to be a multiple of L");

/* block = one (chain, walker), warp d = parameter d */
__global__ void __launch_bounds__(32 * GF_MAX_DIM) k_acor_mean(const double* __restrict__ chain, int nwalkers, int64_t nsteps, int ndim,
                                                              double* __restrict__ mean, int* __restrict__ open, double* __restrict__ run) {
    const int64_t cw = blockIdx.x;
    const int d = threadIdx.x >> 5, j = threadIdx.x & 31;
    const double* x = chain + cw * nsteps * ndim + d;
    const long long x0 = __double_as_longlong(x[0]);
    double s = 0.0;
    bool same = true;
    for (int64_t i = j; i < nsteps; i += 32) {
        const double v = x[i * ndim];
        s += v;
        same &= __double_as_longlong(v) == x0;
    }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    same = __all_sync(0xffffffffu, same);
    if (j == 0) {
        mean[cw * ndim + d] = same ? x[0] : s / (double)nsteps;
        if (cw % nwalkers == 0) {
            const int64_t p = (cw / nwalkers) * ndim + d;
            open[p] = 1;
            run[p] = 0.0;
        }
    }
}

/*
 * Lags [t0, t0 + T) of one (chain, walker), all parameters.  Lane j of warp d owns the lags t0 + j + 32 l, l < L.  The
 * steps of a chunk are visited as i = r + 32 k (r = 0..31 outer, k inner): the value that lag l needs at step k is
 * the one lag l + 1 needed at step k - 1, so each k costs one broadcast load of y_i and one new load of the L-value
 * register window for L FMAs.  Samples beyond the chain are zeros in shared memory, which ends every sum at i = N-1-t.
 */
__global__ void __launch_bounds__(32 * GF_MAX_DIM) k_acor_tile(const double* __restrict__ chain, int nwalkers, int64_t nsteps, int ndim, int64_t t0,
                                                              const double* __restrict__ mean, const int* __restrict__ open,
                                                              double* __restrict__ a0, double* __restrict__ rho) {
    extern __shared__ double sm[];
    double* A = sm;                                /* [ndim][S]  y[i0 + s]       */
    double* B = sm + ndim * GF_ACOR_S;             /* [ndim][SB] y[i0 + t0 + s]  */
    __shared__ double mu[GF_MAX_DIM];
    const int64_t cw = blockIdx.x, c = cw / nwalkers, w = cw % nwalkers;
    const int d = threadIdx.x >> 5, j = threadIdx.x & 31;
    const int64_t p = c * ndim + d;
    const bool mine = open[p] != 0;
    if (!__syncthreads_or(mine)) return;
    if (threadIdx.x < ndim) mu[threadIdx.x] = mean[cw * ndim + threadIdx.x];
    const double* x = chain + cw * nsteps * ndim;
    double acc[GF_ACOR_L];
#pragma unroll
    for (int l = 0; l < GF_ACOR_L; ++l) acc[l] = 0.0;
    for (int64_t i0 = 0; i0 < nsteps - t0; i0 += GF_ACOR_S) {
        __syncthreads();
        for (int e = threadIdx.x; e < GF_ACOR_S * ndim; e += blockDim.x) {
            const int s = e / ndim, dd = e - s * ndim;
            const int64_t n = i0 + s;
            A[dd * GF_ACOR_S + s] = n < nsteps ? x[n * ndim + dd] - mu[dd] : 0.0;
        }
        for (int e = threadIdx.x; e < GF_ACOR_SB * ndim; e += blockDim.x) {
            const int s = e / ndim, dd = e - s * ndim;
            const int64_t n = i0 + t0 + s;
            B[dd * GF_ACOR_SB + s] = n < nsteps ? x[n * ndim + dd] - mu[dd] : 0.0;
        }
        __syncthreads();
        if (!mine) continue;
        for (int r = 0; r < 32; ++r) {
            const double* a = A + d * GF_ACOR_S + r;
            const double* b = B + d * GF_ACOR_SB + r + j;
            double win[GF_ACOR_L]; /* win[(k + l) % L] = y at step k, lag l */
#pragma unroll
            for (int l = 0; l < GF_ACOR_L; ++l) win[l] = b[32 * l];
            for (int k0 = 0; k0 < GF_ACOR_S / 32; k0 += GF_ACOR_L) {
#pragma unroll
                for (int kk = 0; kk < GF_ACOR_L; ++kk) {
                    const double yi = a[32 * (k0 + kk)];
#pragma unroll
                    for (int l = 0; l < GF_ACOR_L; ++l) acc[l] = fma(yi, win[(kk + l) % GF_ACOR_L], acc[l]);
                    win[kk] = b[32 * (k0 + kk + GF_ACOR_L)];
                }
            }
        }
    }
    if (!mine) return;
    /* a_w(0) is lane 0's first lag of tile 0; later tiles read it back */
    const double z = t0 == 0 ? __shfl_sync(0xffffffffu, acc[0], 0) : a0[p * nwalkers + w];
    if (t0 == 0 && j == 0) a0[p * nwalkers + w] = z;
    double* out = rho + (p * nwalkers + w) * GF_ACOR_T + j;
#pragma unroll
    for (int l = 0; l < GF_ACOR_L; ++l) out[32 * l] = z > 0.0 ? acc[l] / z : 0.0;
}

/* block = one (chain, parameter) pair, thread t = lag t0 + t: walker sum in walker order, then one thread extends the
 * running tau(t) in lag order and closes the pair at its window */
__global__ void __launch_bounds__(GF_ACOR_T) k_acor_decide(int nwalkers, int64_t nsteps, int64_t t0, double c, const double* __restrict__ rho,
                                                          int* __restrict__ open, double* __restrict__ run, double* __restrict__ tau,
                                                          int64_t* __restrict__ window) {
    __shared__ double acf[GF_ACOR_T];
    const int64_t p = blockIdx.x;
    if (!open[p]) return;
    const int t = threadIdx.x;
    const double* a = rho + p * nwalkers * GF_ACOR_T + t;
    double s = 0.0;
#pragma unroll 8
    for (int w = 0; w < nwalkers; ++w) s += a[(int64_t)w * GF_ACOR_T];
    acf[t] = s / (double)nwalkers;
    __syncthreads();
    if (t != 0) return;
    double r = run[p];
    const int64_t n = nsteps - t0 < GF_ACOR_T ? nsteps - t0 : GF_ACOR_T;
    for (int k = 0; k < n; ++k) {
        r += acf[k];
        const double tt = 2.0 * r - 1.0;
        const int64_t lag = t0 + k;
        if ((double)lag >= c * tt || lag == nsteps - 1) {
            tau[p] = tt;
            window[p] = lag;
            open[p] = 0;
            return;
        }
    }
    run[p] = r;
}

/* ------------------------------------------------------------------ C ABI */

static inline uint64_t acor_align(uint64_t b) { return (b + 255u) & ~(uint64_t)255u; }

struct acor_layout {
    uint64_t mean, a0, rho, run, open, total;
};

static acor_layout acor_plan(int64_t nchains, int32_t nwalkers, int32_t ndim) {
    acor_layout L;
    const uint64_t pairs = (uint64_t)nchains * (uint64_t)ndim, walkers = pairs * (uint64_t)nwalkers;
    L.mean = 0;
    L.a0 = L.mean + acor_align(walkers * sizeof(double));
    L.rho = L.a0 + acor_align(walkers * sizeof(double));
    L.run = L.rho + acor_align(walkers * GF_ACOR_T * sizeof(double));
    L.open = L.run + acor_align(pairs * sizeof(double));
    L.total = L.open + acor_align(pairs * sizeof(int));
    return L;
}

static bool acor_shape_ok(int64_t nchains, int32_t nwalkers, int64_t nsteps, int32_t ndim) {
    return nchains >= 1 && nwalkers >= 1 && nsteps >= 2 && ndim >= 1 && ndim <= GF_MAX_DIM && nchains * (int64_t)nwalkers <= INT32_MAX;
}

extern "C" uint64_t gf_autocorr_time_workspace(int64_t nchains, int32_t nwalkers, int64_t nsteps, int32_t ndim) {
    if (!acor_shape_ok(nchains, nwalkers, nsteps, ndim)) return 0;
    return acor_plan(nchains, nwalkers, ndim).total;
}

extern "C" int gf_autocorr_time(const double* d_chain, int64_t nchains, int32_t nwalkers, int64_t nsteps, int32_t ndim, double c, double* d_tau,
                                int64_t* d_window, void* d_work, uint64_t work_bytes, void* stream) {
    GF_REQUIRE(d_chain && d_tau && d_window && d_work, "gf_autocorr_time: null pointer");
    GF_REQUIRE(nchains >= 1 && nwalkers >= 1 && nsteps >= 2, "gf_autocorr_time: nchains = %lld, nwalkers = %d, nsteps = %lld (need >= 1, >= 1, >= 2)",
               (long long)nchains, nwalkers, (long long)nsteps);
    GF_REQUIRE(ndim >= 1 && ndim <= GF_MAX_DIM, "gf_autocorr_time: ndim = %d outside [1, %d]", ndim, GF_MAX_DIM);
    GF_REQUIRE(nchains * (int64_t)nwalkers <= INT32_MAX, "gf_autocorr_time: nchains * nwalkers = %lld exceeds 2^31 - 1",
               (long long)(nchains * (int64_t)nwalkers));
    GF_REQUIRE(isfinite(c) && c > 0.0, "gf_autocorr_time: c = %g must be finite and positive", c);
    const acor_layout L = acor_plan(nchains, nwalkers, ndim);
    GF_REQUIRE(work_bytes >= L.total, "gf_autocorr_time: workspace of %llu bytes, need %llu (gf_autocorr_time_workspace)",
               (unsigned long long)work_bytes, (unsigned long long)L.total);
    char* ws = (char*)d_work;
    double* mean = (double*)(ws + L.mean);
    double* a0 = (double*)(ws + L.a0);
    double* rho = (double*)(ws + L.rho);
    double* run = (double*)(ws + L.run);
    int* open = (int*)(ws + L.open);
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned blocks = (unsigned)(nchains * nwalkers), threads = 32u * (unsigned)ndim;
    const size_t smem = (size_t)ndim * (GF_ACOR_S + GF_ACOR_SB) * sizeof(double);
    GF_CUDA(cudaFuncSetAttribute(k_acor_tile, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(GF_MAX_DIM * (GF_ACOR_S + GF_ACOR_SB) * sizeof(double))));
    k_acor_mean<<<blocks, threads, 0, st>>>(d_chain, nwalkers, nsteps, ndim, mean, open, run);
    ++g_gf_launches;
    GF_LAUNCH_CHECK("k_acor_mean");
    const unsigned pairs = (unsigned)(nchains * ndim);
    for (int64_t t0 = 0; t0 < nsteps; t0 += GF_ACOR_T) {
        k_acor_tile<<<blocks, threads, smem, st>>>(d_chain, nwalkers, nsteps, ndim, t0, mean, open, a0, rho);
        k_acor_decide<<<pairs, GF_ACOR_T, 0, st>>>(nwalkers, nsteps, t0, c, rho, open, run, d_tau, d_window);
        g_gf_launches += 2;
        GF_LAUNCH_CHECK("k_acor_tile / k_acor_decide");
    }
    return GF_OK;
}
