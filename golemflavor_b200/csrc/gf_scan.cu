/*
 * gf_scan.cu -- Monte-Carlo prior scans (scripts/mc_unitary.py, mc_x.py, mc_texture.py) fused
 * with the ternary flavor histogram of plot.flavor_contour (plot.py:364-370).
 *
 * The reference draws prior samples by running emcee on a flat likelihood, maps the flavor
 * functions over the chain in Python and histograms later.  Here every sample is drawn directly
 * from the priors with a counter-based Philox4x32-10 stream (counter = global sample index, so
 * the result does not depend on launch geometry or on how the index range is sharded over GPUs),
 * pushed through the same per-point physics as the log-posterior kernel and counted into a
 * block-private shared-memory histogram; nothing but the final counts touches HBM.
 */
#include <atomic>
#include <string.h>

#include "gf_common.cuh"
#include "gf_scan_dev.cuh"

extern std::atomic<unsigned long long> g_gf_launches;

#ifndef GF_SCAN_THREADS
#define GF_SCAN_THREADS 256
#endif
/* bins interleaved per thread in the scan kernels (see gf_bin_loop): two independent chains wherever
 * they fit into 128 registers without spilling -- the specialisations that keep the source (and the
 * texture) in the constant bank; GF_SPEC_GENERIC (sampled source) spills with two and keeps one */
#ifndef GF_SCAN_ILP
#define GF_SCAN_ILP 2
#endif
#define GF_SCAN_ILP_FOR(SPEC) ((SPEC) == GF_SPEC_GENERIC ? 1 : GF_SCAN_ILP)
#ifndef GF_SCAN_MIN_BLOCKS
#define GF_SCAN_MIN_BLOCKS 2
#endif
/* The SM-only scans (unitary, x) are register-light (~50), but the 70 KB block-private histogram allows three blocks per SM:
 * at 256 threads that is 24 warps per SM and the fixed-latency `wait` stall leads (profiles/r02c_hist_unitary.md).  Larger
 * blocks share one histogram among more warps: 512 threads x 2 blocks = 32 warps per SM (unitary 6.36 -> 6.70e10, x 3.96 ->
 * 4.20e10 samples/s; 384 x 3: 6.54 / 4.18).  Grids too fine for a shared-memory histogram (global atomics) keep 256 threads:
 * larger blocks lose 4 % there. */
#ifndef GF_SCAN_THREADS_SM
#define GF_SCAN_THREADS_SM 512
#endif
#ifndef GF_SCAN_BLOCKS_SM
#define GF_SCAN_BLOCKS_SM 2
#endif
#define GF_SCAN_THREADS_FOR(SPEC) (GF_SPEC_IS_SM(SPEC) ? GF_SCAN_THREADS_SM : GF_SCAN_THREADS)

/* ------------------------------------------------------------------ kernels */

/* Source of compositions: drawn samples (SCAN) or a given array (GIVEN). */
template <bool SCAN, bool SMEM_HIST, int SPEC>
__global__ void __launch_bounds__(GF_SCAN_THREADS_FOR(SPEC), GF_SPEC_IS_SM(SPEC) ? GF_SCAN_BLOCKS_SM : GF_SCAN_MIN_BLOCKS) /* BSM: <= 128 registers, two 256-thread blocks (2 x 70 KB histograms) per SM; SM-only: three larger ones */
    k_hist(const __grid_constant__ gf_dev_model m, const uint64_t seed, const uint64_t first_index, const uint64_t count,
           const double* __restrict__ fr_in, const int nb1, const double step, unsigned long long* __restrict__ hist,
           unsigned long long* __restrict__ accepted) {
    extern __shared__ unsigned int sh_hist[];
    const int cells = nb1 * nb1 * nb1;
    if (SMEM_HIST) {
        for (int c = threadIdx.x; c < cells; c += blockDim.x) sh_hist[c] = 0u;
        __syncthreads();
    }
    unsigned int kept = 0u;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < count; j += stride) {
        double fr[3];
        if (SCAN) {
            double theta[GF_MAX_DIM];
            gf_draw_theta<GF_SPEC_IS_SM(SPEC) || (GF_SPEC_STATIC_NDIM(SPEC) > 0), GF_SPEC_STATIC_NDIM(SPEC)>(m, seed, first_index + j, theta);
            gf_point q;
            gf_resolve_point<SPEC>(m, [&](int k) { return theta[k]; }, q);
            gf_point_fr<SPEC, GF_SCAN_ILP_FOR(SPEC)>(m, q, fr);
        } else {
            fr[0] = fr_in[3 * j];
            fr[1] = fr_in[3 * j + 1];
            fr[2] = fr_in[3 * j + 2];
        }
        const int cell = gf_cell_index(fr, nb1, step);
        if (cell >= 0) ++kept;
        if (SMEM_HIST) {
            if (cell >= 0) atomicAdd(&sh_hist[cell], 1u);
        } else {
            /* no block-private copy for oversampled grids: aggregate equal cells inside the warp
             * first (prior scans put most samples into a handful of cells, and L2 serialises atomics
             * per address), one 64-bit atomic per distinct cell and warp */
            const unsigned peers = __match_any_sync(__activemask(), cell);
            if (cell >= 0 && (threadIdx.x & 31) == (unsigned)(__ffs(peers) - 1)) atomicAdd(&hist[cell], (unsigned long long)__popc(peers));
        }
    }
    if (SMEM_HIST) {
        __syncthreads();
        for (int c = threadIdx.x; c < cells; c += blockDim.x) {
            const unsigned int v = sh_hist[c];
            if (v) atomicAdd(&hist[c], (unsigned long long)v);
        }
    }
    if (accepted) {
        /* warp-shuffle reduction, one atomic per warp */
        for (int o = 16; o > 0; o >>= 1) kept += __shfl_down_sync(0xffffffffu, kept, o);
        if ((threadIdx.x & 31) == 0 && kept) atomicAdd(accepted, (unsigned long long)kept);
    }
}

__global__ void __launch_bounds__(GF_SCAN_THREADS)
    k_scan_samples(const __grid_constant__ gf_dev_model m, const uint64_t seed, const uint64_t first_index, const uint64_t count,
                   double* __restrict__ theta_out, double* __restrict__ fr_out, uint8_t* __restrict__ status) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= count) return;
    double theta[GF_MAX_DIM];
    gf_draw_theta(m, seed, first_index + j, theta);
    gf_point q;
    gf_resolve_point(m, [&](int k) { return theta[k]; }, q);
    double fr[3];
    const unsigned st = gf_point_fr(m, q, fr);
    if (theta_out)
        for (int k = 0; k < m.ndim; ++k) theta_out[j * m.ndim + k] = theta[k];
    if (fr_out) {
        fr_out[3 * j] = fr[0];
        fr_out[3 * j + 1] = fr[1];
        fr_out[3 * j + 2] = fr[2];
    }
    if (status) status[j] = (uint8_t)st;
}

/* ------------------------------------------------------------------ C ABI */

namespace {

/* samples per launch: keeps the 32-bit block-private counters far from overflow */
constexpr uint64_t kMaxPerLaunch = 1ull << 36;
constexpr size_t kSmemHistLimit = 200 * 1024;

template <bool SCAN>
int launch_hist(const char* fn, const gf_dev_model& d, uint64_t seed, uint64_t first, uint64_t count, const double* d_fr, int nb,
                unsigned long long* d_hist, unsigned long long* d_accepted, cudaStream_t stream) {
    GF_REQUIRE(nb >= 0 && nb <= 1023, "%s: nb = %d outside [0, 1023]", fn, nb);
    GF_REQUIRE(d_hist != nullptr, "%s: histogram is NULL", fn);
    if (count == 0) return GF_OK;
    const int nb1 = nb + 1;
    const double step = 1.0 / (double)nb1;
    const size_t smem = (size_t)nb1 * nb1 * nb1 * sizeof(unsigned int);
    const bool use_smem = smem <= kSmemHistLimit;
    int sms = 0;
    if (int rc = gf_sm_count(&sms)) return rc;
    const int spec = SCAN ? gf_model_scan_spec(d) : GF_SPEC_GENERIC;
#define GF_HIST_KERNEL(SMEM)                                                                  \
    (spec == GF_SPEC_FIXED      ? k_hist<SCAN, SMEM, GF_SPEC_FIXED>                           \
     : spec == GF_SPEC_FIXED7   ? k_hist<SCAN, SMEM, GF_SPEC_FIXED7>                          \
     : spec == GF_SPEC_SM       ? k_hist<SCAN, SMEM, GF_SPEC_SM>                              \
     : spec == GF_SPEC_SM4      ? k_hist<SCAN, SMEM, GF_SPEC_SM4>                             \
     : spec == GF_SPEC_SM5X     ? k_hist<SCAN, SMEM, GF_SPEC_SM5X>                            \
     : spec == GF_SPEC_NPFREE   ? k_hist<SCAN, SMEM, GF_SPEC_NPFREE>                          \
     : spec == GF_SPEC_NPFREE11 ? k_hist<SCAN, SMEM, GF_SPEC_NPFREE11>                        \
                                : k_hist<SCAN, SMEM, GF_SPEC_GENERIC>)
    auto kern_s = GF_HIST_KERNEL(true);
    auto kern_g = GF_HIST_KERNEL(false);
#undef GF_HIST_KERNEL
    const int threads = (SCAN && use_smem && GF_SPEC_IS_SM(spec)) ? GF_SCAN_THREADS_SM : GF_SCAN_THREADS; /* <= GF_SCAN_THREADS_FOR of the launched instance */
    int per_sm = 1;
    if (use_smem) {
        GF_CUDA(cudaFuncSetAttribute(kern_s, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        GF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern_s, threads, smem));
    } else {
        GF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern_g, threads, 0));
    }
    GF_REQUIRE(per_sm >= 1, "%s: kernel does not fit on an SM (smem %zu B)", fn, smem);
    for (uint64_t done = 0; done < count; done += kMaxPerLaunch) {
        const uint64_t cnt = (count - done < kMaxPerLaunch) ? count - done : kMaxPerLaunch;
        uint64_t want = (cnt + threads - 1) / threads;
        const uint64_t persistent = (uint64_t)sms * per_sm;
        const unsigned blocks = (unsigned)(want < persistent ? want : persistent);
        const double* frp = d_fr ? d_fr + 3 * done : nullptr;
        if (use_smem)
            kern_s<<<blocks, threads, smem, stream>>>(d, seed, first + done, cnt, frp, nb1, step, d_hist, d_accepted);
        else
            kern_g<<<blocks, threads, 0, stream>>>(d, seed, first + done, cnt, frp, nb1, step, d_hist, d_accepted);
        ++g_gf_launches;
        GF_LAUNCH_CHECK(fn);
    }
    return GF_OK;
}

}  // namespace

extern "C" int gf_scan_hist(const gf_model* model, const gf_scan_config* cfg, unsigned long long* d_hist,
                            unsigned long long* d_accepted, void* stream) {
    GF_REQUIRE(cfg != nullptr, "gf_scan_hist: cfg is NULL");
    gf_dev_model d;
    if (int rc = gf_build_dev_model(model, &d)) return rc;
    return launch_hist<true>("gf_scan_hist", d, cfg->seed, cfg->first_index, cfg->count, nullptr, cfg->nb, d_hist, d_accepted,
                             (cudaStream_t)stream);
}

extern "C" int gf_ternary_hist(const double* d_fr, int64_t n, int32_t nb, unsigned long long* d_hist, void* stream) {
    GF_REQUIRE(n >= 0, "gf_ternary_hist: n = %lld", (long long)n);
    GF_REQUIRE(n == 0 || d_fr != nullptr, "gf_ternary_hist: fr is NULL");
    gf_dev_model d;
    memset(&d, 0, sizeof(d));
    return launch_hist<false>("gf_ternary_hist", d, 0, 0, (uint64_t)n, d_fr, nb, d_hist, nullptr, (cudaStream_t)stream);
}

extern "C" int gf_scan_samples(const gf_model* model, const gf_scan_config* cfg, double* d_theta, double* d_fr, uint8_t* d_status,
                               void* stream) {
    GF_REQUIRE(cfg != nullptr, "gf_scan_samples: cfg is NULL");
    gf_dev_model d;
    if (int rc = gf_build_dev_model(model, &d)) return rc;
    if (cfg->count == 0) return GF_OK;
    GF_REQUIRE(cfg->count < (1ull << 40), "gf_scan_samples: count too large");
    k_scan_samples<<<gf_blocks_for((int64_t)cfg->count, GF_SCAN_THREADS), GF_SCAN_THREADS, 0, (cudaStream_t)stream>>>(
        d, cfg->seed, cfg->first_index, cfg->count, d_theta, d_fr, d_status);
    ++g_gf_launches;
    GF_LAUNCH_CHECK("gf_scan_samples");
    return GF_OK;
}

/* ------------------------------------------------------------------ coverage region (plot.py:372-384) */

/*
 * Sorted by content, a cell is inside the region while the inclusive cumulative sum stays below need = coverage * total
 * (np.searchsorted(cumsum, coverage), plot.py:380-382).  With G(c) = sum of the counts > c, the content of the first
 * excluded cell is c* = min{c : G(c) < need}: a bisection on c with one multi-block reduction per probe.  The whole
 * search runs ON THE DEVICE -- the bisection state lives in a small stream-ordered workspace, every probe is a
 * (reduce, decide) pair of launches without a host round trip -- and only the three result numbers are read back at the end.
 *
 * ws[0] gt   : sum of counts > probe          ws[4] ngt : #cells > probe         ws[8]  probe   ws[11] take
 * ws[1] eq   : #cells == probe                ws[5] lo                           ws[9]  phase   ws[12] n_gt
 * ws[2] max  : largest count                  ws[6] hi                           ws[10] cstar
 * ws[3] tot  : sum of all counts              ws[7] (unused)
 */
enum { COV_GT = 0, COV_EQ = 1, COV_MAX = 2, COV_TOT = 3, COV_NGT = 4, COV_LO = 5, COV_HI = 6, COV_PROBE = 8, COV_PHASE = 9, COV_CSTAR = 10,
       COV_TAKE = 11, COV_NGT_FINAL = 12, COV_WORDS = 16 };

__global__ void __launch_bounds__(256) k_cov_reduce(const unsigned long long* __restrict__ hist, int64_t cells, unsigned long long* __restrict__ ws) {
    const unsigned long long c = ws[COV_PROBE], phase = ws[COV_PHASE];
    if (phase == 3ull) return; /* search finished: the remaining probes of the fixed-length schedule are no-ops */
    unsigned long long gt = 0ull, eq = 0ull, mx = 0ull, tot = 0ull, ngt = 0ull;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < cells; i += (int64_t)gridDim.x * blockDim.x) {
        const unsigned long long v = hist[i];
        gt += v > c ? v : 0ull;
        ngt += v > c ? 1ull : 0ull;
        eq += v == c ? 1ull : 0ull;
        mx = v > mx ? v : mx;
        tot += v;
    }
    for (int o = 16; o > 0; o >>= 1) {
        gt += __shfl_down_sync(0xffffffffu, gt, o);
        ngt += __shfl_down_sync(0xffffffffu, ngt, o);
        eq += __shfl_down_sync(0xffffffffu, eq, o);
        tot += __shfl_down_sync(0xffffffffu, tot, o);
        const unsigned long long other = __shfl_down_sync(0xffffffffu, mx, o);
        mx = other > mx ? other : mx;
    }
    if ((threadIdx.x & 31) == 0) {
        if (gt) atomicAdd(ws + COV_GT, gt);
        if (eq) atomicAdd(ws + COV_EQ, eq);
        if (phase == 0ull) { /* total and maximum: first pass only (later probes would add them again) */
            atomicMax(ws + COV_MAX, mx);
            if (tot) atomicAdd(ws + COV_TOT, tot);
        }
        if (ngt) atomicAdd(ws + COV_NGT, ngt);
    }
}

/* one thread: digest the probe that just ran, choose the next one.  phase 0: first pass (probe 0: total and maximum),
 * 1: bisection, 2: final probe at c*, 3: done */
__global__ void k_cov_decide(unsigned long long* __restrict__ ws, double coverage_fraction) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const unsigned long long phase = ws[COV_PHASE];
    if (phase == 3ull) return;
    const double need = coverage_fraction * (double)ws[COV_TOT];
    const double g = (double)ws[COV_GT];
    if (phase == 0ull) {
        if (ws[COV_TOT] == 0ull || !(need > 0.0)) { /* empty histogram or zero coverage: nothing is masked */
            ws[COV_CSTAR] = ws[COV_MAX];
            ws[COV_TAKE] = 0ull;
            ws[COV_NGT_FINAL] = 0ull;
            ws[COV_PHASE] = 3ull;
            return;
        }
        ws[COV_LO] = 0ull; /* G(0) = total >= need */
        ws[COV_HI] = ws[COV_MAX];
        ws[COV_PHASE] = 1ull;
    } else if (phase == 1ull) {
        if (g < need) ws[COV_HI] = ws[COV_PROBE]; else ws[COV_LO] = ws[COV_PROBE];
    } else { /* phase 2: the probe was c* itself */
        const unsigned long long cstar = ws[COV_PROBE];
        /* tied cells j = 1, 2, ... are inside while g + j c* < need */
        unsigned long long m = (unsigned long long)floor((need - g) / (double)cstar);
        while (g + (double)(m + 1ull) * (double)cstar < need) ++m;
        while (m > 0ull && !(g + (double)m * (double)cstar < need)) --m;
        ws[COV_CSTAR] = cstar;
        ws[COV_TAKE] = m < ws[COV_EQ] ? m : ws[COV_EQ];
        ws[COV_NGT_FINAL] = ws[COV_NGT];
        ws[COV_PHASE] = 3ull;
        return;
    }
    const unsigned long long lo = ws[COV_LO], hi = ws[COV_HI];
    if (hi - lo > 1ull) {
        ws[COV_PROBE] = lo + (hi - lo) / 2ull;
    } else {
        ws[COV_PROBE] = hi; /* c* = hi: probe it once more for g, the tie count and the number of cells above it */
        ws[COV_PHASE] = 2ull;
    }
    ws[COV_GT] = ws[COV_EQ] = ws[COV_NGT] = 0ull; /* total and maximum are kept from the first pass */
}

/* one block walks the cells in order: mask = count > c*, plus the first `take` cells with count == c* */
__global__ void __launch_bounds__(1024) k_cov_mask(const unsigned long long* __restrict__ hist, int64_t cells, const unsigned long long* __restrict__ ws,
                                                   uint8_t* __restrict__ mask) {
    __shared__ unsigned int warp_ties[32];
    __shared__ unsigned long long base;
    const unsigned long long c = ws[COV_CSTAR], take = ws[COV_TAKE];
    const bool nothing = ws[COV_NGT_FINAL] == 0ull && take == 0ull;
    if (threadIdx.x == 0) base = 0ull;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int64_t start = 0; start < cells; start += blockDim.x) {
        const int64_t i = start + threadIdx.x;
        const unsigned long long v = i < cells ? hist[i] : 0ull;
        const bool tie = !nothing && i < cells && v == c && c > 0ull;
        const unsigned ballot = __ballot_sync(0xffffffffu, tie);
        if (lane == 0) warp_ties[warp] = __popc(ballot);
        __syncthreads();
        unsigned before = __popc(ballot & ((1u << lane) - 1u));
        for (int w = 0; w < warp; ++w) before += warp_ties[w];
        const unsigned long long rank = base + before; /* number of tied cells ahead of this one */
        if (i < cells) mask[i] = (!nothing && (v > c || (tie && rank < take))) ? 1 : 0;
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned t = 0;
            for (int w = 0; w < 32; ++w) t += warp_ties[w];
            base += t;
        }
        __syncthreads();
    }
}

extern "C" int gf_coverage_mask(const unsigned long long* d_hist, int64_t cells, double coverage_percent, uint8_t* d_mask,
                                unsigned long long* h_info, void* stream) {
    GF_REQUIRE(cells >= 1 && d_hist && d_mask, "gf_coverage_mask: bad arguments");
    GF_REQUIRE(coverage_percent >= 0.0 && coverage_percent <= 100.0, "gf_coverage_mask: coverage = %g outside [0, 100]", coverage_percent);
    cudaStream_t st = (cudaStream_t)stream;
    int sms = 0;
    if (int rc = gf_sm_count(&sms)) return rc;
    const int64_t want = (cells + 255) / 256;
    const unsigned blocks = (unsigned)(want < (int64_t)sms * 8 ? want : (int64_t)sms * 8);
    unsigned long long* ws = nullptr;
    GF_CUDA(cudaMallocAsync(&ws, COV_WORDS * sizeof(unsigned long long), st)); /* stream-ordered: no device-wide synchronisation */
    GF_CUDA(cudaMemsetAsync(ws, 0, COV_WORDS * sizeof(unsigned long long), st));
    /* 1 first pass + at most 64 bisection probes (64-bit counts) + 1 final probe: a fixed schedule, probes after the end are no-ops */
    for (int it = 0; it < 66; ++it) {
        k_cov_reduce<<<blocks, 256, 0, st>>>(d_hist, cells, ws);
        k_cov_decide<<<1, 32, 0, st>>>(ws, coverage_percent / 100.0);
        g_gf_launches += 2;
    }
    k_cov_mask<<<1, 1024, 0, st>>>(d_hist, cells, ws, d_mask);
    ++g_gf_launches;
    cudaError_t e = cudaGetLastError();
    unsigned long long h[COV_WORDS] = {};
    if (e == cudaSuccess && h_info) e = cudaMemcpyAsync(h, ws, sizeof(h), cudaMemcpyDeviceToHost, st);
    cudaFreeAsync(ws, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return gf_fail(GF_ERR_CUDA, "gf_coverage_mask: %s", cudaGetErrorString(e));
    if (h_info) {
        h_info[0] = h[COV_CSTAR];
        h_info[1] = h[COV_NGT_FINAL] + h[COV_TAKE];
        h_info[2] = h[COV_TAKE];
    }
    return GF_OK;
}

/* ------------------------------------------------------------------ smoothed coverage region (plot.py:372-384, hist_smooth > 1/8 bin) */

/*
 * plot.flavor_contour smooths the normalised histogram with scipy.ndimage.gaussian_filter(H, sigma = hist_smooth) before it
 * looks for the coverage region.  The default sigma = 0.05 bins truncates to a one-tap kernel (radius int(4 sigma + 1/2) = 0:
 * the identity, served by the integer path above); any sigma >= 0.125 is a real separable filter.  One pass per axis with
 * SciPy's own conventions -- boundary mode 'reflect' (d c b a | a b c d | d c b a), and for its symmetric kernels the
 * accumulation order of ni_filters.c: centre tap first, then (left + right) pairs from the outside in, no FMA contraction
 * -- so the smoothed field equals SciPy's bit for bit given the same weights (the caller passes SciPy's weights).
 */
#define GF_SMOOTH_MAX_RADIUS 64
struct gf_smooth_weights {
    double w[GF_SMOOTH_MAX_RADIUS + 1]; /* w[k] = weight at distance radius - k ... w[radius] = centre: SciPy's fw[0 .. size1] */
};

template <bool FROM_COUNTS>
__global__ void __launch_bounds__(256) k_smooth_axis(const void* __restrict__ in_, double* __restrict__ out, int n1, int axis, int radius,
                                                     const __grid_constant__ gf_smooth_weights W, double total) {
    const int64_t cells = (int64_t)n1 * n1 * n1;
    const int64_t stride = axis == 0 ? (int64_t)n1 * n1 : axis == 1 ? n1 : 1;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < cells; i += (int64_t)gridDim.x * blockDim.x) {
        const int l = (int)((i / stride) % n1);
        const int64_t base = i - (int64_t)l * stride;
        auto at = [&](int k) -> double { /* 'reflect': -1 -> 0, -2 -> 1, n -> n - 1, n + 1 -> n - 2, periodically for long kernels */
            const int period = 2 * n1;
            int m = k % period;
            if (m < 0) m += period;
            if (m >= n1) m = period - 1 - m;
            const int64_t j = base + (int64_t)m * stride;
            if (FROM_COUNTS) return __ddiv_rn((double)static_cast<const unsigned long long*>(in_)[j], total); /* H / np.sum(H) */
            return static_cast<const double*>(in_)[j];
        };
        double tmp = __dmul_rn(at(l), W.w[radius]);
        for (int ii = -radius; ii < 0; ++ii) tmp = __dadd_rn(tmp, __dmul_rn(__dadd_rn(at(l + ii), at(l - ii)), W.w[ii + radius]));
        out[i] = tmp;
    }
}

extern "C" int gf_hist_smooth(const unsigned long long* d_hist, int32_t n1, unsigned long long total, const double* h_weights, int32_t radius,
                              double* d_out, double* d_work, void* stream) {
    GF_REQUIRE(d_hist && d_out && d_work && h_weights, "gf_hist_smooth: null pointer");
    GF_REQUIRE(n1 >= 1 && n1 <= 1024, "gf_hist_smooth: %d cells per axis outside [1, 1024]", n1);
    GF_REQUIRE(radius >= 0 && radius <= GF_SMOOTH_MAX_RADIUS, "gf_hist_smooth: kernel radius %d outside [0, %d]", radius, GF_SMOOTH_MAX_RADIUS);
    GF_REQUIRE(total > 0ull, "gf_hist_smooth: empty histogram");
    gf_smooth_weights W;
    for (int k = 0; k <= radius; ++k) W.w[k] = h_weights[k];
    cudaStream_t st = (cudaStream_t)stream;
    int sms = 0;
    if (int rc = gf_sm_count(&sms)) return rc;
    const int64_t cells = (int64_t)n1 * n1 * n1, want = (cells + 255) / 256;
    const unsigned blocks = (unsigned)(want < (int64_t)sms * 8 ? want : (int64_t)sms * 8);
    /* axes 0, 1, 2 in SciPy's order: counts -> out -> work -> out */
    k_smooth_axis<true><<<blocks, 256, 0, st>>>(d_hist, d_out, n1, 0, radius, W, (double)total);
    k_smooth_axis<false><<<blocks, 256, 0, st>>>(d_out, d_work, n1, 1, radius, W, 0.0);
    k_smooth_axis<false><<<blocks, 256, 0, st>>>(d_work, d_out, n1, 2, radius, W, 0.0);
    g_gf_launches += 3;
    GF_LAUNCH_CHECK("gf_hist_smooth");
    return GF_OK;
}

/*
 * Coverage region of a non-negative float field (the smoothed histogram): the same definition and the same sort-free search
 * as gf_coverage_mask.  Non-negative doubles order like their bit patterns, so the bisection runs on the 64-bit keys
 * (at most 64 probes); G(c) = sum of the values with key > c is accumulated in double with a FIXED reduction tree (per-block
 * partials summed in block order by the deciding thread): the same field gives the same mask on every run.
 * wsd: [0] g  [1] total  [2] need;  wsu: as the integer path (counts of cells, keys)
 */
__global__ void __launch_bounds__(256) k_covf_reduce(const double* __restrict__ h, int64_t cells, const unsigned long long* __restrict__ wsu,
                                                     double* __restrict__ part /*[gridDim.x][2]*/, unsigned long long* __restrict__ cnt /*[gridDim.x][3]*/) {
    __shared__ double sg[8], stot[8];
    __shared__ unsigned long long sn[8], se[8], smx[8];
    const unsigned long long c = wsu[COV_PROBE], phase = wsu[COV_PHASE];
    if (phase == 3ull) return;
    double g = 0.0, tot = 0.0;
    unsigned long long ngt = 0ull, eq = 0ull, mx = 0ull;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < cells; i += (int64_t)gridDim.x * blockDim.x) {
        const double v = h[i];
        const unsigned long long key = (unsigned long long)__double_as_longlong(v > 0.0 ? v : 0.0); /* -0, NaN and negatives count as 0 */
        g += key > c ? v : 0.0;
        ngt += key > c ? 1ull : 0ull;
        eq += key == c ? 1ull : 0ull;
        mx = key > mx ? key : mx;
        tot += v > 0.0 ? v : 0.0;
    }
    for (int o = 16; o > 0; o >>= 1) {
        g += __shfl_down_sync(0xffffffffu, g, o);
        tot += __shfl_down_sync(0xffffffffu, tot, o);
        ngt += __shfl_down_sync(0xffffffffu, ngt, o);
        eq += __shfl_down_sync(0xffffffffu, eq, o);
        const unsigned long long other = __shfl_down_sync(0xffffffffu, mx, o);
        mx = other > mx ? other : mx;
    }
    const int warp = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) { sg[warp] = g; stot[warp] = tot; sn[warp] = ngt; se[warp] = eq; smx[warp] = mx; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) { g += sg[w]; tot += stot[w]; ngt += sn[w]; eq += se[w]; mx = smx[w] > mx ? smx[w] : mx; }
        part[2 * blockIdx.x] = g; part[2 * blockIdx.x + 1] = tot;
        cnt[3 * blockIdx.x] = ngt; cnt[3 * blockIdx.x + 1] = eq; cnt[3 * blockIdx.x + 2] = mx;
    }
}

__global__ void k_covf_decide(unsigned long long* __restrict__ wsu, double* __restrict__ wsd, const double* __restrict__ part,
                              const unsigned long long* __restrict__ cnt, int nblocks, double coverage_fraction) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const unsigned long long phase = wsu[COV_PHASE];
    if (phase == 3ull) return;
    double g = 0.0, tot = 0.0;
    unsigned long long ngt = 0ull, eq = 0ull, mx = 0ull;
    for (int b = 0; b < nblocks; ++b) { /* block order: a fixed summation tree */
        g += part[2 * b]; tot += part[2 * b + 1];
        ngt += cnt[3 * b]; eq += cnt[3 * b + 1]; mx = cnt[3 * b + 2] > mx ? cnt[3 * b + 2] : mx;
    }
    if (phase == 0ull) {
        /* plot.py:381: searchsorted(cumsum(sorted H_s), coverage / 100) on the field itself (its sum is 1 up to rounding) */
        wsd[1] = tot; wsd[2] = coverage_fraction;
        wsu[COV_MAX] = mx;
        if (!(tot > 0.0) || !(coverage_fraction > 0.0)) {
            wsu[COV_CSTAR] = mx; wsu[COV_TAKE] = 0ull; wsu[COV_NGT_FINAL] = 0ull; wsu[COV_PHASE] = 3ull;
            return;
        }
        wsu[COV_LO] = 0ull; /* G(key 0) = total: all positive cells */
        wsu[COV_HI] = mx;
        wsu[COV_PHASE] = 1ull;
        if (!(tot >= coverage_fraction)) { /* the whole field holds less than the requested fraction: every positive cell is inside */
            wsu[COV_CSTAR] = 0ull; wsu[COV_TAKE] = 0ull; wsu[COV_NGT_FINAL] = ngt; wsu[COV_PHASE] = 3ull;
            return;
        }
    } else if (phase == 1ull) {
        if (g < wsd[2]) wsu[COV_HI] = wsu[COV_PROBE]; else wsu[COV_LO] = wsu[COV_PROBE];
    } else {
        const unsigned long long ckey = wsu[COV_PROBE];
        const double cstar = __longlong_as_double((long long)ckey), need = wsd[2];
        unsigned long long m = 0ull; /* tied cells j = 1, 2, ... are inside while g + j c* < need */
        if (cstar > 0.0) {
            m = (unsigned long long)fmax(floor((need - g) / cstar), 0.0);
            while (g + (double)(m + 1ull) * cstar < need) ++m;
            while (m > 0ull && !(g + (double)m * cstar < need)) --m;
        }
        wsu[COV_CSTAR] = ckey;
        wsu[COV_TAKE] = m < eq ? m : eq;
        wsu[COV_NGT_FINAL] = ngt;
        wsu[COV_PHASE] = 3ull;
        wsd[0] = g;
        return;
    }
    const unsigned long long lo = wsu[COV_LO], hi = wsu[COV_HI];
    if (hi - lo > 1ull) {
        wsu[COV_PROBE] = lo + (hi - lo) / 2ull;
    } else {
        wsu[COV_PROBE] = hi;
        wsu[COV_PHASE] = 2ull;
    }
}

__global__ void __launch_bounds__(1024) k_covf_mask(const double* __restrict__ h, int64_t cells, const unsigned long long* __restrict__ ws,
                                                    uint8_t* __restrict__ mask) {
    __shared__ unsigned int warp_ties[32];
    __shared__ unsigned long long base;
    const unsigned long long c = ws[COV_CSTAR], take = ws[COV_TAKE];
    const bool nothing = ws[COV_NGT_FINAL] == 0ull && take == 0ull;
    if (threadIdx.x == 0) base = 0ull;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int64_t start = 0; start < cells; start += blockDim.x) {
        const int64_t i = start + threadIdx.x;
        const double v = i < cells ? h[i] : 0.0;
        const unsigned long long key = (unsigned long long)__double_as_longlong(v > 0.0 ? v : 0.0);
        const bool tie = !nothing && i < cells && key == c && c > 0ull;
        const unsigned ballot = __ballot_sync(0xffffffffu, tie);
        if (lane == 0) warp_ties[warp] = __popc(ballot);
        __syncthreads();
        unsigned before = __popc(ballot & ((1u << lane) - 1u));
        for (int w = 0; w < warp; ++w) before += warp_ties[w];
        const unsigned long long rank = base + before;
        if (i < cells) mask[i] = (!nothing && (key > c || (tie && rank < take))) ? 1 : 0;
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned t = 0;
            for (int w = 0; w < 32; ++w) t += warp_ties[w];
            base += t;
        }
        __syncthreads();
    }
}

extern "C" int gf_coverage_mask_f64(const double* d_field, int64_t cells, double coverage_percent, uint8_t* d_mask, double* h_cstar,
                                    unsigned long long* h_counts /*[2] or NULL*/, void* stream) {
    GF_REQUIRE(cells >= 1 && d_field && d_mask, "gf_coverage_mask_f64: bad arguments");
    GF_REQUIRE(coverage_percent >= 0.0 && coverage_percent <= 100.0, "gf_coverage_mask_f64: coverage = %g outside [0, 100]", coverage_percent);
    cudaStream_t st = (cudaStream_t)stream;
    int sms = 0;
    if (int rc = gf_sm_count(&sms)) return rc;
    const int64_t want = (cells + 255) / 256;
    const int blocks = (int)(want < (int64_t)sms * 8 ? want : (int64_t)sms * 8);
    /* one stream-ordered allocation: integer state | double state | per-block partials */
    const size_t bytes = (COV_WORDS + 4 + (size_t)blocks * 5) * 8;
    unsigned long long* wsu = nullptr;
    GF_CUDA(cudaMallocAsync(&wsu, bytes, st));
    GF_CUDA(cudaMemsetAsync(wsu, 0, bytes, st));
    double* wsd = reinterpret_cast<double*>(wsu + COV_WORDS);
    double* part = wsd + 4;
    unsigned long long* cnt = reinterpret_cast<unsigned long long*>(part + 2 * (size_t)blocks);
    for (int it = 0; it < 66; ++it) { /* first pass + <= 64 probes of the key bisection + the final probe; later ones are no-ops */
        k_covf_reduce<<<blocks, 256, 0, st>>>(d_field, cells, wsu, part, cnt);
        k_covf_decide<<<1, 32, 0, st>>>(wsu, wsd, part, cnt, blocks, coverage_percent / 100.0);
        g_gf_launches += 2;
    }
    k_covf_mask<<<1, 1024, 0, st>>>(d_field, cells, wsu, d_mask);
    ++g_gf_launches;
    cudaError_t e = cudaGetLastError();
    unsigned long long h[COV_WORDS] = {};
    if (e == cudaSuccess) e = cudaMemcpyAsync(h, wsu, sizeof(h), cudaMemcpyDeviceToHost, st);
    cudaFreeAsync(wsu, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return gf_fail(GF_ERR_CUDA, "gf_coverage_mask_f64: %s", cudaGetErrorString(e));
    if (h_cstar) memcpy(h_cstar, &h[COV_CSTAR], sizeof(double));
    if (h_counts) {
        h_counts[0] = h[COV_NGT_FINAL] + h[COV_TAKE];
        h_counts[1] = h[COV_TAKE];
    }
    return GF_OK;
}

/* ------------------------------------------------------------------ Monte-Carlo evidence */

template <int SPEC>
__global__ void __launch_bounds__(GF_SCAN_THREADS, GF_SCAN_MIN_BLOCKS)
    k_evidence(const __grid_constant__ gf_dev_model m, const uint64_t seed, const uint64_t first_index, const uint64_t count,
               double* __restrict__ partials /*[gridDim.x][2]*/) {
    __shared__ double sh_m[GF_SCAN_THREADS / 32], sh_s[GF_SCAN_THREADS / 32];
    double mx = -INFINITY, sm = 0.0;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < count; j += stride) {
        double theta[GF_MAX_DIM], fr[3];
        gf_draw_theta(m, seed, first_index + j, theta);
        gf_point q;
        gf_resolve_point<SPEC>(m, [&](int k) { return theta[k]; }, q);
        gf_point_fr<SPEC, GF_SCAN_ILP_FOR(SPEC)>(m, q, fr);
        const double ll = m.llh_kind == GF_LLH_FLAT
                              ? m.llh_const
                              : gf_multi_gaussian(fr, m.fr_bf, m.half_inv_s2, m.lognorm3, m.offset, m.emulate_underflow, m.underflow_logpdf);
        if (ll == ll) gf_lse_merge(mx, sm, ll, 1.0); /* NaN samples carry no weight */
    }
    for (int o = 16; o > 0; o >>= 1) {
        const double m2 = __shfl_down_sync(0xffffffffu, mx, o), s2 = __shfl_down_sync(0xffffffffu, sm, o);
        gf_lse_merge(mx, sm, m2, s2);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) {
        sh_m[warp] = mx;
        sh_s[warp] = sm;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < GF_SCAN_THREADS / 32; ++w) gf_lse_merge(mx, sm, sh_m[w], sh_s[w]);
        partials[2 * blockIdx.x] = mx;
        partials[2 * blockIdx.x + 1] = sm;
    }
}

__global__ void k_lse_finish(const double* __restrict__ partials, int n, double* __restrict__ lse) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    double mx = lse[0], sm = lse[1];
    for (int b = 0; b < n; ++b) gf_lse_merge(mx, sm, partials[2 * b], partials[2 * b + 1]); /* fixed order: deterministic */
    lse[0] = mx;
    lse[1] = sm;
}

extern "C" int gf_scan_evidence(const gf_model* model, const gf_scan_config* cfg, double* d_lse, void* stream) {
    GF_REQUIRE(cfg != nullptr && d_lse != nullptr, "gf_scan_evidence: null pointer");
    gf_dev_model d;
    if (int rc = gf_build_dev_model(model, &d)) return rc;
    if (cfg->count == 0) return GF_OK;
    cudaStream_t st = (cudaStream_t)stream;
    int sms = 0;
    if (int rc = gf_sm_count(&sms)) return rc;
    const bool fixed = gf_model_is_fixed_spec(d);
    auto kern = fixed ? k_evidence<GF_SPEC_FIXED> : k_evidence<GF_SPEC_GENERIC>;
    int per_sm = 1;
    GF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, GF_SCAN_THREADS, 0));
    const uint64_t want = (cfg->count + GF_SCAN_THREADS - 1) / GF_SCAN_THREADS, persistent = (uint64_t)sms * (per_sm > 0 ? per_sm : 1);
    const unsigned blocks = (unsigned)(want < persistent ? want : persistent);
    double* d_part = nullptr;
    GF_CUDA(cudaMallocAsync(&d_part, 2 * sizeof(double) * blocks, st));
    kern<<<blocks, GF_SCAN_THREADS, 0, st>>>(d, cfg->seed, cfg->first_index, cfg->count, d_part);
    k_lse_finish<<<1, 32, 0, st>>>(d_part, (int)blocks, d_lse);
    g_gf_launches += 2;
    cudaError_t e = cudaGetLastError();
    cudaFreeAsync(d_part, st);
    if (e != cudaSuccess) return gf_fail(GF_ERR_CUDA, "gf_scan_evidence: %s", cudaGetErrorString(e));
    return GF_OK;
}

/* ------------------------------------------------------------------ evidence on a grid of scales */

/*
 * The sensitivity grid (scripts/sens.py:232-294: one MultiNest run per (dimension, scale)) as ONE launch per
 * dimension: blockIdx.y selects a group of `s_per` grid scales, blockIdx.x strides over the prior samples.  A thread
 * draws its sample once, builds everything that does not depend on the scale once (PMNS, H0, pencil coefficients) and
 * evaluates the 20-bin composition + likelihood at each scale of the group.  The running log-sum-exp (max, sum) of
 * every (thread, scale) lives in shared memory (two LDS/STS per ~1900 fp64 instructions), so the accumulators cost no
 * registers.  Per-block partials are merged by the LAST block of the group (ticket counter) in block order:
 * deterministic for a given launch geometry, no finishing kernel, no allocation.
 */
#define GF_EVG_MAX_S_PER 16

template <int SPEC, bool STATIC6>
__global__ void __launch_bounds__(GF_SCAN_THREADS, GF_SCAN_MIN_BLOCKS)
    k_evidence_grid(const __grid_constant__ gf_dev_model m, const uint64_t seed, const uint64_t first_index, const uint64_t count,
                    const double* __restrict__ scales, const int nscales, const int s_per, double* __restrict__ partials /*[nscales][gridDim.x][2]*/,
                    unsigned int* __restrict__ tickets /*[gridDim.y]*/, double* __restrict__ lse /*[nscales][2]*/) {
    extern __shared__ double sh_evg[];
    constexpr int T = GF_SCAN_THREADS, W = GF_SCAN_THREADS / 32;
    double* sh_lam = sh_evg;                        /* [GF_EVG_MAX_S_PER]        */
    double* sh_m = sh_evg + GF_EVG_MAX_S_PER;       /* [s_per][T] running max    */
    double* sh_s = sh_m + s_per * T;                /* [s_per][T] running sum    */
    __shared__ double sh_wm[GF_EVG_MAX_S_PER][W], sh_ws[GF_EVG_MAX_S_PER][W];
    __shared__ int sh_last;
    const int tid = threadIdx.x, g = blockIdx.y;
    const int s0 = g * s_per, ns = min(s_per, nscales - s0);
    if (tid < ns) sh_lam[tid] = exp10(scales[s0 + tid]); /* the same exp10 the per-point kernels apply to logLam */
    for (int k = 0; k < ns; ++k) {
        sh_m[k * T + tid] = -INFINITY;
        sh_s[k * T + tid] = 0.0;
    }
    __syncthreads();
    const uint64_t stride = (uint64_t)gridDim.x * T;
    for (uint64_t j = (uint64_t)blockIdx.x * T + tid; j < count; j += stride) {
        double theta[GF_MAX_DIM];
        gf_point q;
        if constexpr (STATIC6) { /* the layout of sens.py: columns 0-3 mixing coordinates, 4-5 mass splittings */
            gf_draw_theta<true, 6>(m, seed, first_index + j, theta);
            q.sm[0] = theta[0]; q.sm[1] = theta[1]; q.sm[2] = theta[2]; q.sm[3] = theta[3];
            q.mass[0] = theta[4]; q.mass[1] = theta[5];
        } else {
            gf_draw_theta(m, seed, first_index + j, theta);
            gf_resolve_point<SPEC>(m, [&](int k) { return theta[k]; }, q);
        }
        gf_point_fr_scales<SPEC, GF_SCAN_ILP_FOR(SPEC)>(
            m, q, ns, [&](int k) { return sh_lam[k]; },
            [&](int k, const double* fr, unsigned) {
                const double ll = m.llh_kind == GF_LLH_FLAT
                                      ? m.llh_const
                                      : gf_multi_gaussian(fr, m.fr_bf, m.half_inv_s2, m.lognorm3, m.offset, m.emulate_underflow, m.underflow_logpdf);
                if (ll > -INFINITY) { /* only the samples with weight touch shared memory */
                    double mo = sh_m[k * T + tid], so = sh_s[k * T + tid];
                    gf_lse_push(mo, so, ll);
                    sh_m[k * T + tid] = mo;
                    sh_s[k * T + tid] = so;
                }
            });
    }
    /* block reduction: lanes by shuffle, warps in order */
    const int lane = tid & 31, warp = tid >> 5;
    for (int k = 0; k < ns; ++k) {
        double mx = sh_m[k * T + tid], sm = sh_s[k * T + tid];
        for (int o = 16; o > 0; o >>= 1) {
            const double m2 = __shfl_down_sync(0xffffffffu, mx, o), s2 = __shfl_down_sync(0xffffffffu, sm, o);
            gf_lse_merge(mx, sm, m2, s2);
        }
        if (lane == 0) {
            sh_wm[k][warp] = mx;
            sh_ws[k][warp] = sm;
        }
    }
    __syncthreads();
    if (tid < ns) {
        double mx = sh_wm[tid][0], sm = sh_ws[tid][0];
        for (int w = 1; w < W; ++w) gf_lse_merge(mx, sm, sh_wm[tid][w], sh_ws[tid][w]);
        double* out = partials + 2 * ((size_t)(s0 + tid) * gridDim.x + blockIdx.x);
        out[0] = mx;
        out[1] = sm;
    }
    /* the last block of this scale group merges the per-block partials (classic ticket pattern) */
    __threadfence();
    __syncthreads();
    if (tid == 0) sh_last = atomicAdd(&tickets[g], 1u) == gridDim.x - 1;
    __syncthreads();
    if (!sh_last) return;
    __threadfence();
    if (tid < ns) {
        double mx = lse[2 * (s0 + tid)], sm = lse[2 * (s0 + tid) + 1];
        const volatile double* in = partials + 2 * (size_t)(s0 + tid) * gridDim.x;
        for (unsigned b = 0; b < gridDim.x; ++b) gf_lse_merge(mx, sm, in[2 * b], in[2 * b + 1]); /* block order: deterministic */
        lse[2 * (s0 + tid)] = mx;
        lse[2 * (s0 + tid) + 1] = sm;
    }
    if (tid == 0) tickets[g] = 0u; /* the workspace is reusable by the next launch on this stream */
}

namespace {

struct evg_geometry {
    int s_per, ny, per_sm;
    unsigned nx;
    size_t smem;
};

template <class K>
int evg_plan(K kern, int nscales, uint64_t count, evg_geometry* geo) {
    int sms = 0;
    if (int rc = gf_sm_count(&sms)) return rc;
    /* scales per block: as many as amortise the per-sample set-up while every SM still gets work; 10 scales
     * (20 KB of accumulators per block... 2 x 10 x 256 x 8 B = 40 KB) leave two blocks per SM */
    int s_per = nscales < 10 ? nscales : 10;
    const size_t smem = (size_t)(GF_EVG_MAX_S_PER + 2 * s_per * GF_SCAN_THREADS) * sizeof(double);
    GF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;
    GF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, GF_SCAN_THREADS, smem));
    GF_REQUIRE(per_sm >= 1, "gf_scan_evidence_grid: kernel does not fit on an SM (smem %zu B)", smem);
    const int ny = (nscales + s_per - 1) / s_per;
    geo->s_per = s_per; geo->ny = ny; geo->per_sm = per_sm; geo->nx = gf_evidence_nx(sms, per_sm, ny, count, GF_SCAN_THREADS); geo->smem = smem;
    return GF_OK;
}

}  // namespace

int gf_check_frozen_scale(const char* who, const gf_dev_model& d) {
    GF_REQUIRE(!d.no_bsm, "%s: the model has no BSM path (no_bsm = 1)", who);
    GF_REQUIRE(d.col_scale < 0, "%s: the scale must not be a sampled column (col_scale = %d): it is frozen at the grid values", who, d.col_scale);
    return GF_OK;
}

unsigned gf_evidence_nx(int sms, int per_sm, int ny, uint64_t count, int threads) {
    const uint64_t want = (count + threads - 1) / threads;
    uint64_t nx = ((uint64_t)sms * per_sm) / ny;
    if (nx > want) nx = want;
    if (nx < 1) nx = 1;
    return (unsigned)nx;
}

int gf_evidence_workspace(const char* who, size_t rows, unsigned nx, int ny, void* d_work, uint64_t work_bytes, cudaStream_t st, double** part,
                          unsigned int** tickets) {
    const size_t part_bytes = rows * nx * 2 * sizeof(double);
    const size_t need = part_bytes + (size_t)ny * sizeof(unsigned int);
    GF_REQUIRE(d_work != nullptr && work_bytes >= need, "%s: workspace of %llu B is too small, need %llu B (%s_workspace)", who,
               (unsigned long long)work_bytes, (unsigned long long)need, who);
    *part = static_cast<double*>(d_work);
    *tickets = reinterpret_cast<unsigned int*>(static_cast<char*>(d_work) + part_bytes);
    GF_CUDA(cudaMemsetAsync(*tickets, 0, (size_t)ny * sizeof(unsigned int), st));
    return GF_OK;
}

extern "C" uint64_t gf_scan_evidence_grid_workspace(int32_t nscales) {
    int sms = 0;
    if (nscales < 1 || gf_sm_count(&sms) != GF_OK) return 0;
    /* [nscales][blocks in x][2] partials (blocks in x <= resident blocks of the device) + one ticket per scale */
    return (uint64_t)nscales * ((uint64_t)sms * 8) * 2 * sizeof(double) + (uint64_t)nscales * sizeof(unsigned int) + 256;
}

extern "C" int gf_scan_evidence_grid(const gf_model* model, const gf_scan_config* cfg, const double* d_scales, int32_t nscales,
                                     double* d_lse, void* d_work, uint64_t work_bytes, void* stream) {
    GF_REQUIRE(cfg != nullptr && d_lse != nullptr && d_scales != nullptr, "gf_scan_evidence_grid: null pointer");
    GF_REQUIRE(nscales >= 1 && nscales <= 65535, "gf_scan_evidence_grid: nscales = %d outside [1, 65535]", nscales);
    gf_dev_model d;
    if (int rc = gf_build_dev_model(model, &d)) return rc;
    if (int rc = gf_check_frozen_scale("gf_scan_evidence_grid", d)) return rc;
    if (cfg->count == 0) return GF_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const int spec = gf_model_grid_spec(d);
    auto kern = spec == 2 ? k_evidence_grid<GF_SPEC_FIXED, true> : spec == 1 ? k_evidence_grid<GF_SPEC_FIXED, false> : k_evidence_grid<GF_SPEC_GENERIC, false>;
    evg_geometry geo;
    if (int rc = evg_plan(kern, nscales, cfg->count, &geo)) return rc;
    double* part = nullptr;
    unsigned int* tickets = nullptr;
    if (int rc = gf_evidence_workspace("gf_scan_evidence_grid", nscales, geo.nx, geo.ny, d_work, work_bytes, st, &part, &tickets)) return rc;
    kern<<<dim3(geo.nx, (unsigned)geo.ny), GF_SCAN_THREADS, geo.smem, st>>>(d, cfg->seed, cfg->first_index, cfg->count, d_scales, nscales, geo.s_per, part,
                                                                              tickets, d_lse);
    ++g_gf_launches;
    GF_LAUNCH_CHECK("gf_scan_evidence_grid");
    return GF_OK;
}
