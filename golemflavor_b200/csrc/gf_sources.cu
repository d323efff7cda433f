/*
 * gf_sources.cu -- the evidence grid of gf_scan_evidence_grid for many source compositions in ONE launch per dimension
 * (the reference runs scripts/sens.py once per source composition, submitter/sens_dag.py:8-16, 38-61, 76-95).
 *
 * k_evidence_sources keeps the grid of k_evidence_grid -- blockIdx.y = a group of s_per scales, blockIdx.x strides over the
 * prior samples in one wave, sample j drawn with gf_draw_theta(m, seed, first_index + j) -- and runs each iteration in two
 * phases separated by a barrier:
 *   physics : thread t draws sample base + t and writes the transition sums A = (A00, A01, A11) of every scale of the group
 *             into the shared tile [s_per][3][T] (NaN for a non-finite result or past the end of the shard);
 *   apply   : the block's threads are re-mapped onto (scale, source) pairs.  A pair is owned by G threads (G a power of two,
 *             G > 1 only when the pairs do not fill the block), thread c of them walks samples [c T/G, (c+1) T/G) of the tile
 *             in index order, forms fr (gfp_transition_fr), the likelihood with the source's injected composition and
 *             updates the pair's running (max, sum) in registers with the rule of k_evidence_grid.
 * Between iterations a thread's (max, sum) of each of its `slots` pairs is parked in shared memory ([slots][2][T], one entry
 * per pair and chunk, not per (thread, scale, source)), so it adds no live registers to the physics phase.  At the end the G
 * chunks of a pair are merged in chunk order, the per-block partials [nscales][nsrc][blocks][2] are merged by the last block of each scale group (ticket) in
 * block order.  The result depends on (seed, samples, the sources and scales) and on G and the launch geometry, which are
 * functions of (nscales, nsrc, count) and the device only.
 */
#include <atomic>
#include <string.h>

#include "gf_common.cuh"
#include "gf_sources_dev.cuh"

extern std::atomic<unsigned long long> g_gf_launches;

#define GF_EVS_THREADS 256
#define GF_EVS_MIN_BLOCKS 2
#define GF_EVS_MAX_S_PER 10 /* scales per block, as k_evidence_grid                     */
#define GF_EVS_MAX_SLOTS 8  /* (scale, source) pairs per thread: s_per * nsrc <= 8 * 256 */
#define GF_EVS_ILP_FOR(SPEC) ((SPEC) == GF_SPEC_GENERIC ? 1 : 2)

template <int SPEC, bool STATIC6>
__global__ void __launch_bounds__(GF_EVS_THREADS, GF_EVS_MIN_BLOCKS)
    k_evidence_sources(const __grid_constant__ gf_dev_model m, const __grid_constant__ gf_src_table S, const uint64_t seed,
                       const uint64_t first_index, const uint64_t count, const double* __restrict__ scales, const int nscales,
                       const int s_per, const int G, const int slots, double* __restrict__ partials /*[nscales][nsrc][gridDim.x][2]*/,
                       unsigned int* __restrict__ tickets /*[gridDim.y]*/, double* __restrict__ lse /*[nsrc][nscales][2]*/) {
    extern __shared__ double sh_evs[];
    constexpr int T = GF_EVS_THREADS;
    double* sh_lam = sh_evs;                      /* [GF_EVS_MAX_S_PER]                               */
    double* acc = sh_evs + GF_EVS_MAX_S_PER;      /* [slots][2][T] running (max, sum) of thread slots */
    double* tile = acc + 2 * slots * T;           /* [s_per][3][T] transition sums of the samples      */
    __shared__ int sh_last;
    const int tid = threadIdx.x, g = blockIdx.y, nsrc = S.nsrc;
    const int s0 = g * s_per, ns = min(s_per, nscales - s0), npairs = ns * nsrc, L = T / G;
    if (tid < ns) sh_lam[tid] = exp10(scales[s0 + tid]); /* the same exp10 the per-point kernels apply to logLam */
    for (int q = 0; q < slots; ++q) {
        acc[(2 * q) * T + tid] = -INFINITY;
        acc[(2 * q + 1) * T + tid] = 0.0;
    }
    __syncthreads();
    const uint64_t stride = (uint64_t)gridDim.x * T;
    for (uint64_t base = (uint64_t)blockIdx.x * T; base < count; base += stride) {
        if (base + tid < count) {
            gf_src_sample<SPEC, STATIC6, GF_EVS_ILP_FOR(SPEC)>(m, seed, first_index + base + tid, ns, sh_lam, [&](int k, const double* A, unsigned st) {
                tile[(3 * k) * T + tid] = (st & GFP_ST_NON_FINITE) ? NAN : A[0];
                tile[(3 * k + 1) * T + tid] = A[1];
                tile[(3 * k + 2) * T + tid] = A[2];
            });
        } else {
            for (int k = 0; k < ns; ++k) tile[(3 * k) * T + tid] = NAN;
        }
        __syncthreads();
        /* slot q of this thread: u = tid + q T, pair u / G, chunk u % G (G > 1 implies a single slot) */
        for (int q = 0; q < slots; ++q) {
            const int u = tid + q * T, pair = u / G;
            if (pair >= npairs) break;
            const int k = pair / nsrc, j = pair - k * nsrc, t0 = (u - pair * G) * L;
            const gf_src_rec r = S.src[j];
            const double* a = tile + 3 * k * T;
            double mq = acc[(2 * q) * T + tid], sq = acc[(2 * q + 1) * T + tid];
            for (int t = t0; t < t0 + L; ++t) {
                const double A[3] = {a[t], a[T + t], a[2 * T + t]};
                gf_lse_push(mq, sq, gf_src_llh(m, r, A)); /* a NaN marker gives a NaN likelihood: no weight */
            }
            acc[(2 * q) * T + tid] = mq;
            acc[(2 * q + 1) * T + tid] = sq;
        }
        __syncthreads();
    }
    /* the block's partial of every pair: its G chunks (threads pair G .. pair G + G - 1, slot 0) merged in chunk order */
    const size_t nx = gridDim.x;
    for (int pair = tid; pair < npairs; pair += T) {
        const int u = pair * G, q = u / T, t = u - q * T;
        double mx = acc[(2 * q) * T + t], sm = acc[(2 * q + 1) * T + t];
        for (int c = 1; c < G; ++c) gf_lse_merge(mx, sm, acc[t + c], acc[T + t + c]);
        double* o = partials + 2 * (((size_t)(s0 + pair / nsrc) * nsrc + pair % nsrc) * nx + blockIdx.x);
        o[0] = mx;
        o[1] = sm;
    }
    /* the last block of this scale group merges the per-block partials (ticket pattern of k_evidence_grid) */
    __threadfence();
    __syncthreads();
    if (tid == 0) sh_last = atomicAdd(&tickets[g], 1u) == gridDim.x - 1;
    __syncthreads();
    if (!sh_last) return;
    __threadfence();
    for (int pair = tid; pair < npairs; pair += T) {
        const int k = pair / nsrc, j = pair - k * nsrc;
        double* dst = lse + 2 * ((size_t)j * nscales + s0 + k);
        double mx = dst[0], sm = dst[1];
        const volatile double* in = partials + 2 * ((size_t)(s0 + k) * nsrc + j) * nx;
        for (unsigned b = 0; b < gridDim.x; ++b) gf_lse_merge(mx, sm, in[2 * b], in[2 * b + 1]); /* block order */
        dst[0] = mx;
        dst[1] = sm;
    }
    if (tid == 0) tickets[g] = 0u; /* the workspace is reusable by the next launch on this stream */
}

namespace {

struct evs_plan_t {
    int s_per, G, ny, slots;
};

/* Scales per block and threads per pair.  Per scale, a block spends ~1900 fp64 instructions per sample in the bin loop
 * (DESIGN.md K2/K3b) plus a share of the ~600 of the per-point set-up, and its apply phase runs ceil(pairs G / T) rounds of
 * T / G samples at ~45 instructions on the critical path of the slowest thread.  s_per minimises the sum per scale (ties:
 * the larger s_per); G is the largest power of two with pairs * G <= T. */
evs_plan_t evs_plan(int nscales, int nsrc) {
    const int T = GF_EVS_THREADS;
    evs_plan_t best{1, 1, nscales, 1};
    double best_cost = 1e300;
    for (int s = 1; s <= GF_EVS_MAX_S_PER && s <= nscales; ++s) {
        const int pairs = s * nsrc;
        if (pairs > T * GF_EVS_MAX_SLOTS) break;
        int G = 1;
        while (pairs * G * 2 <= T) G *= 2;
        const int rounds = (pairs * G + T - 1) / T;
        const double cost = (600.0 + 1900.0 * s + 45.0 * rounds * (T / G)) / s;
        if (cost <= best_cost) {
            best_cost = cost;
            best = evs_plan_t{s, G, (nscales + s - 1) / s, rounds};
        }
    }
    return best;
}

/* resident blocks per SM bound the x extent; the workspace is sized for this many */
constexpr int EVS_MAX_BLOCKS_PER_SM = 8;

size_t evs_smem(const evs_plan_t& p) { return (size_t)(GF_EVS_MAX_S_PER + (2 * p.slots + 3 * p.s_per) * GF_EVS_THREADS) * sizeof(double); }

}  // namespace

int gf_src_table_fill(const char* who, const gf_dev_model& d, const double* sources, const double* injected, int nsrc, gf_src_table* S) {
    GF_REQUIRE(gf_model_has_fixed_source(d), "%s: the model samples the source (col_src / col_x / col_src3): the sources are the launch's own list",
               who);
    GF_REQUIRE(d.llh_kind == GF_LLH_GAUSSIAN, "%s: llh_kind = %d, the Gaussian likelihood (GF_LLH_GAUSSIAN) is required", who, d.llh_kind);
    S->nsrc = nsrc;
    S->reserved = 0;
    for (int j = 0; j < nsrc; ++j)
        GF_REQUIRE(gf_src_record(sources + 3 * j, injected + 3 * j, d.wsum, &S->src[j]),
                   "%s: source %d = (%g, %g, %g) / injected (%g, %g, %g): entries must be finite and non-negative with a positive sum", who, j,
                   sources[3 * j], sources[3 * j + 1], sources[3 * j + 2], injected[3 * j], injected[3 * j + 1], injected[3 * j + 2]);
    return GF_OK;
}

extern "C" uint64_t gf_scan_evidence_sources_workspace(int32_t nscales, int32_t nsrc) {
    int sms = 0;
    if (nscales < 1 || nscales > 65535 || nsrc < 1 || nsrc > GF_SRC_MAX || gf_sm_count(&sms) != GF_OK) return 0;
    const evs_plan_t p = evs_plan(nscales, nsrc);
    uint64_t nx = (uint64_t)sms * EVS_MAX_BLOCKS_PER_SM / (uint64_t)p.ny;
    if (nx < 1) nx = 1;
    /* [nscales][nsrc][blocks in x][2] partials + one ticket per scale group */
    return (uint64_t)nscales * (uint64_t)nsrc * nx * 2 * sizeof(double) + (uint64_t)p.ny * sizeof(unsigned int) + 256;
}

extern "C" int gf_scan_evidence_sources(const gf_model* model, const gf_scan_config* cfg, const double* d_scales, int32_t nscales,
                                        const double* sources, const double* injected, int32_t nsrc, double* d_lse, void* d_work,
                                        uint64_t work_bytes, void* stream) {
    GF_REQUIRE(model != nullptr && cfg != nullptr && d_scales != nullptr && sources != nullptr && injected != nullptr && d_lse != nullptr,
               "gf_scan_evidence_sources: null pointer");
    GF_REQUIRE(nscales >= 1 && nscales <= 65535, "gf_scan_evidence_sources: nscales = %d outside [1, 65535]", nscales);
    GF_REQUIRE(nsrc >= 1 && nsrc <= GF_SRC_MAX, "gf_scan_evidence_sources: nsrc = %d outside [1, %d]", nsrc, GF_SRC_MAX);
    gf_dev_model d;
    if (int rc = gf_build_dev_model(model, &d)) return rc;
    if (int rc = gf_check_frozen_scale("gf_scan_evidence_sources", d)) return rc;
    gf_src_table tab; /* 14 KB, copied into the kernel parameter buffer by the launch */
    if (int rc = gf_src_table_fill("gf_scan_evidence_sources", d, sources, injected, nsrc, &tab)) return rc;
    const evs_plan_t p = evs_plan(nscales, nsrc);
    const int spec = gf_model_grid_spec(d);
    auto kern = spec == 2 ? k_evidence_sources<GF_SPEC_FIXED, true> : spec == 1 ? k_evidence_sources<GF_SPEC_FIXED, false>
                                                                                : k_evidence_sources<GF_SPEC_GENERIC, false>;
    const size_t smem = evs_smem(p);
    int sms = 0;
    if (int rc = gf_sm_count(&sms)) return rc;
    if (cfg->count == 0) return GF_OK;
    GF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;
    GF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, GF_EVS_THREADS, smem));
    GF_REQUIRE(per_sm >= 1, "gf_scan_evidence_sources: kernel does not fit on an SM (smem %zu B)", smem);
    /* the workspace holds EVS_MAX_BLOCKS_PER_SM blocks per SM */
    const unsigned nx = gf_evidence_nx(sms, per_sm < EVS_MAX_BLOCKS_PER_SM ? per_sm : EVS_MAX_BLOCKS_PER_SM, p.ny, cfg->count, GF_EVS_THREADS);
    cudaStream_t st = (cudaStream_t)stream;
    double* part = nullptr;
    unsigned int* tickets = nullptr;
    if (int rc = gf_evidence_workspace("gf_scan_evidence_sources", (size_t)nscales * nsrc, nx, p.ny, d_work, work_bytes, st, &part, &tickets))
        return rc;
    kern<<<dim3(nx, (unsigned)p.ny), GF_EVS_THREADS, smem, st>>>(d, tab, cfg->seed, cfg->first_index, cfg->count, d_scales, nscales, p.s_per, p.G,
                                                                 p.slots, part, tickets, d_lse);
    ++g_gf_launches;
    GF_LAUNCH_CHECK("gf_scan_evidence_sources");
    return GF_OK;
}
