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
 *
 * GROUPED: the samples are split into R = `groups` fixed groups, sample i in group i mod R (R a power of two dividing T; a
 * block's tile starts at an index that is a multiple of T, so tile sample t is in group (first_index + t) mod R).  The units
 * of the apply phase are (scale, source, group) triples instead of pairs; the G chunks of a triple split the T / R tile
 * samples of its group, which it walks with stride R in index order.  Partials and results gain a group axis:
 * [nscales][nsrc][R][blocks][2] and [nsrc][nscales][R][2].  Without GROUPED R is 1 and the kernel is the ungrouped one;
 * `groups` is never read.
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
/* (scale, source, group) triples per thread of the grouped kernel: s_per * nsrc * groups <= 16 * 256.  The kernel's registers
 * allow two blocks per SM; 16 slots (64 KB) and the tile of 8 scales (48 KB) still fit two, so 30 sources at 16 groups keep
 * the 8 scales per block of the ungrouped plan.  The grouped plan only takes shapes whose dynamic shared memory leaves room
 * for two blocks on an SM (GF_EVS_SMEM_TWO_BLOCKS): more slots or scales than that would silently halve the resident blocks */
#define GF_EVS_MAX_SLOTS_GROUPED 16
/* two blocks per SM of sm_100 (228 KB of shared memory, 1 KB of it reserved per block), less the kernel's 16 B of static memory */
#define GF_EVS_SMEM_TWO_BLOCKS ((228 * 1024) / 2 - 1024 - 16)
#define GF_EVS_ILP_FOR(SPEC) ((SPEC) == GF_SPEC_GENERIC ? 1 : 2)

template <int SPEC, bool STATIC6, bool GROUPED = false>
__global__ void __launch_bounds__(GF_EVS_THREADS, GF_EVS_MIN_BLOCKS)
    k_evidence_sources(const __grid_constant__ gf_dev_model m, const __grid_constant__ gf_src_table S, const uint64_t seed,
                       const uint64_t first_index, const uint64_t count, const double* __restrict__ scales, const int nscales,
                       const int s_per, const int G, const int slots, double* __restrict__ partials /*[nscales][nsrc][R][gridDim.x][2]*/,
                       unsigned int* __restrict__ tickets /*[gridDim.y]*/, double* __restrict__ lse /*[nsrc][nscales][R][2]*/, const int groups) {
    extern __shared__ double sh_evs[];
    constexpr int T = GF_EVS_THREADS;
    double* sh_lam = sh_evs;                      /* [GF_EVS_MAX_S_PER]                               */
    double* acc = sh_evs + GF_EVS_MAX_S_PER;      /* [slots][2][T] running (max, sum) of thread slots */
    double* tile = acc + 2 * slots * T;           /* [s_per][3][T] transition sums of the samples      */
    __shared__ int sh_last;
    const int tid = threadIdx.x, g = blockIdx.y, nsrc = S.nsrc;
    const int R = GROUPED ? groups : 1;
    /* a unit is (pair, group r, chunk c) = u / (R G), (u / G) % R, u % G; chunk c walks L samples of the group at stride R */
    const int s0 = g * s_per, ns = min(s_per, nscales - s0), npairs = ns * nsrc, L = T / (G * R);
    const int l0 = (int)(first_index & (uint64_t)(R - 1));
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
        /* slot q of this thread: unit u = tid + q T (G > 1 implies a single slot) */
        for (int q = 0; q < slots; ++q) {
            const int u = tid + q * T, v = u / G, pair = v / R;
            if (pair >= npairs) break;
            const int k = pair / nsrc, j = pair - k * nsrc, r = v - pair * R;
            const int t0 = ((r - l0) & (R - 1)) + (u - v * G) * L * R; /* first tile sample of group r in chunk u % G */
            const gf_src_rec rec = S.src[j];
            const double* a = tile + 3 * k * T;
            double mq = acc[(2 * q) * T + tid], sq = acc[(2 * q + 1) * T + tid];
            for (int t = t0; t < t0 + L * R; t += R) {
                const double A[3] = {a[t], a[T + t], a[2 * T + t]};
                gf_lse_push(mq, sq, gf_src_llh(m, rec, A)); /* a NaN marker gives a NaN likelihood: no weight */
            }
            acc[(2 * q) * T + tid] = mq;
            acc[(2 * q + 1) * T + tid] = sq;
        }
        __syncthreads();
    }
    /* the block's partial of every (pair, group): its G chunks (units v G .. v G + G - 1, slot 0 when G > 1) merged in chunk order */
    const size_t nx = gridDim.x;
    for (int v = tid; v < npairs * R; v += T) {
        const int u = v * G, q = u / T, t = u - q * T;
        double mx = acc[(2 * q) * T + t], sm = acc[(2 * q + 1) * T + t];
        for (int c = 1; c < G; ++c) gf_lse_merge(mx, sm, acc[t + c], acc[T + t + c]);
        const int pair = v / R, r = v - pair * R;
        double* o = partials + 2 * ((((size_t)(s0 + pair / nsrc) * nsrc + pair % nsrc) * R + r) * nx + blockIdx.x);
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
    for (int v = tid; v < npairs * R; v += T) {
        const int pair = v / R, r = v - pair * R, k = pair / nsrc, j = pair - k * nsrc;
        double* dst = lse + 2 * (((size_t)j * nscales + s0 + k) * R + r);
        double mx = dst[0], sm = dst[1];
        const volatile double* in = partials + 2 * ((((size_t)(s0 + k) * nsrc + j) * R + r) * nx);
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

/* Scales per block and threads per unit (a (scale, source) pair, or a (scale, source, group) triple with R groups).  Per
 * scale, a block spends ~1900 fp64 instructions per sample in the bin loop (DESIGN.md K2/K3b) plus a share of the ~600 of the
 * per-point set-up, and its apply phase runs ceil(units G / T) rounds of T / (G R) samples at ~45 instructions on the critical
 * path of the slowest thread.  s_per minimises the sum per scale (ties: the larger s_per); G is the largest power of two with
 * units * G <= T.  The grouped plan skips shapes that would not fit two blocks per SM (GF_EVS_SMEM_TWO_BLOCKS).  s_per = 0:
 * even one scale has more units than the block's slots hold (nsrc * R > 16 T). */
size_t evs_smem_of(int s_per, int slots) { return (size_t)(GF_EVS_MAX_S_PER + (2 * slots + 3 * s_per) * GF_EVS_THREADS) * sizeof(double); }

/* one scale with every slot in use always fits two blocks, so the grouped plan always finds a shape */
static_assert((GF_EVS_MAX_S_PER + (2 * GF_EVS_MAX_SLOTS_GROUPED + 3) * GF_EVS_THREADS) * sizeof(double) <= GF_EVS_SMEM_TWO_BLOCKS,
              "the grouped source plan must fit two blocks per SM at one scale per block");
/* the shape of 30 sources at 16 groups: 8 scales, 15 slots */
static_assert((GF_EVS_MAX_S_PER + (2 * 15 + 3 * 8) * GF_EVS_THREADS) * sizeof(double) <= GF_EVS_SMEM_TWO_BLOCKS,
              "30 sources at 16 groups must keep 8 scales per block at two blocks per SM");

evs_plan_t evs_plan(int nscales, int nsrc, int R = 1) {
    const int T = GF_EVS_THREADS;
    const int max_units = T * (R == 1 ? GF_EVS_MAX_SLOTS : GF_EVS_MAX_SLOTS_GROUPED);
    evs_plan_t best{R == 1 ? 1 : 0, 1, nscales, 1};
    double best_cost = 1e300;
    for (int s = 1; s <= GF_EVS_MAX_S_PER && s <= nscales; ++s) {
        const int units = s * nsrc * R;
        if (units > max_units) break;
        int G = 1;
        while (units * G * 2 <= T) G *= 2;
        const int rounds = (units * G + T - 1) / T;
        if (R > 1 && evs_smem_of(s, rounds) > GF_EVS_SMEM_TWO_BLOCKS) continue;
        const double cost = (600.0 + 1900.0 * s + 45.0 * rounds * (T / (G * R))) / s;
        if (cost <= best_cost) {
            best_cost = cost;
            best = evs_plan_t{s, G, (nscales + s - 1) / s, rounds};
        }
    }
    return best;
}

/* resident blocks per SM bound the x extent; the workspace is sized for this many */
constexpr int EVS_MAX_BLOCKS_PER_SM = 8;

size_t evs_smem(const evs_plan_t& p) { return evs_smem_of(p.s_per, p.slots); }

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

/* (scale, source, group) triples one block of the grouped kernel holds: s_per * nsrc * groups <= 16 T, so one launch takes at
 * most 4096 / groups sources (all 256 up to 16 groups, 128 at 32) */
#define GF_EVS_MAX_UNITS (GF_EVS_THREADS * GF_EVS_MAX_SLOTS_GROUPED)

namespace {

/* [nscales][nsrc][groups][blocks in x][2] partials + one ticket per scale group; 0 if refused */
uint64_t evidence_sources_workspace(int32_t nscales, int32_t nsrc, int groups) {
    int sms = 0;
    if (nscales < 1 || nscales > 65535 || nsrc < 1 || nsrc > GF_SRC_MAX || nsrc * groups > GF_EVS_MAX_UNITS || gf_sm_count(&sms) != GF_OK) return 0;
    const evs_plan_t p = evs_plan(nscales, nsrc, groups);
    uint64_t nx = (uint64_t)sms * EVS_MAX_BLOCKS_PER_SM / (uint64_t)p.ny;
    if (nx < 1) nx = 1;
    return (uint64_t)nscales * (uint64_t)nsrc * groups * nx * 2 * sizeof(double) + (uint64_t)p.ny * sizeof(unsigned int) + 256;
}

}  // namespace

extern "C" uint64_t gf_scan_evidence_sources_workspace(int32_t nscales, int32_t nsrc) { return evidence_sources_workspace(nscales, nsrc, 1); }

extern "C" uint64_t gf_scan_evidence_sources_groups_workspace(int32_t nscales, int32_t nsrc, int32_t groups) {
    return gf_evidence_groups_ok(groups) ? evidence_sources_workspace(nscales, nsrc, groups) : 0;
}

namespace {

/* gf_scan_evidence_sources (grouped = false: the ungrouped kernel, lse [nsrc][nscales][2]) and gf_scan_evidence_sources_groups
 * (lse [nsrc][nscales][groups][2]): the same checks, plan and launch */
int evidence_sources(const char* who, const gf_model* model, const gf_scan_config* cfg, const double* d_scales, int32_t nscales, const double* sources,
                     const double* injected, int32_t nsrc, bool grouped, int groups, double* d_lse, void* d_work, uint64_t work_bytes,
                     cudaStream_t st) {
    GF_REQUIRE(model != nullptr && cfg != nullptr && d_scales != nullptr && sources != nullptr && injected != nullptr && d_lse != nullptr,
               "%s: null pointer", who);
    GF_REQUIRE(nscales >= 1 && nscales <= 65535, "%s: nscales = %d outside [1, 65535]", who, nscales);
    GF_REQUIRE(nsrc >= 1 && nsrc <= GF_SRC_MAX, "%s: nsrc = %d outside [1, %d]", who, nsrc, GF_SRC_MAX);
    GF_REQUIRE(!grouped || gf_evidence_groups_ok(groups), "%s: groups = %d is not a power of two in [2, %d]", who, groups, GF_EVIDENCE_MAX_GROUPS);
    const int R = grouped ? groups : 1;
    GF_REQUIRE(!grouped || nsrc * R <= GF_EVS_MAX_UNITS, "%s: nsrc = %d with %d groups: one launch takes at most %d sources (nsrc * groups <= %d)",
               who, nsrc, R, GF_EVS_MAX_UNITS / R, GF_EVS_MAX_UNITS);
    gf_dev_model d;
    if (int rc = gf_build_dev_model(model, &d)) return rc;
    if (int rc = gf_check_frozen_scale(who, d)) return rc;
    gf_src_table tab; /* 14 KB, copied into the kernel parameter buffer by the launch */
    if (int rc = gf_src_table_fill(who, d, sources, injected, nsrc, &tab)) return rc;
    const evs_plan_t p = evs_plan(nscales, nsrc, R);
    const int spec = gf_model_grid_spec(d);
    auto kern = grouped ? (spec == 2 ? k_evidence_sources<GF_SPEC_FIXED, true, true> : spec == 1 ? k_evidence_sources<GF_SPEC_FIXED, false, true>
                                                                                                 : k_evidence_sources<GF_SPEC_GENERIC, false, true>)
                       : (spec == 2 ? k_evidence_sources<GF_SPEC_FIXED, true> : spec == 1 ? k_evidence_sources<GF_SPEC_FIXED, false>
                                                                                          : k_evidence_sources<GF_SPEC_GENERIC, false>);
    const size_t smem = evs_smem(p);
    int sms = 0;
    if (int rc = gf_sm_count(&sms)) return rc;
    if (cfg->count == 0) return GF_OK;
    GF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;
    GF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, GF_EVS_THREADS, smem));
    GF_REQUIRE(per_sm >= 1, "%s: kernel does not fit on an SM (smem %zu B)", who, smem);
    /* the workspace holds EVS_MAX_BLOCKS_PER_SM blocks per SM */
    const unsigned nx = gf_evidence_nx(sms, per_sm < EVS_MAX_BLOCKS_PER_SM ? per_sm : EVS_MAX_BLOCKS_PER_SM, p.ny, cfg->count, GF_EVS_THREADS);
    double* part = nullptr;
    unsigned int* tickets = nullptr;
    if (int rc = gf_evidence_workspace(who, (size_t)nscales * nsrc * R, nx, p.ny, d_work, work_bytes, st, &part, &tickets)) return rc;
    kern<<<dim3(nx, (unsigned)p.ny), GF_EVS_THREADS, smem, st>>>(d, tab, cfg->seed, cfg->first_index, cfg->count, d_scales, nscales, p.s_per, p.G,
                                                                 p.slots, part, tickets, d_lse, R);
    ++g_gf_launches;
    GF_LAUNCH_CHECK(who);
    return GF_OK;
}

}  // namespace

extern "C" int gf_scan_evidence_sources(const gf_model* model, const gf_scan_config* cfg, const double* d_scales, int32_t nscales,
                                        const double* sources, const double* injected, int32_t nsrc, double* d_lse, void* d_work,
                                        uint64_t work_bytes, void* stream) {
    return evidence_sources("gf_scan_evidence_sources", model, cfg, d_scales, nscales, sources, injected, nsrc, false, 1, d_lse, d_work, work_bytes,
                            (cudaStream_t)stream);
}

extern "C" int gf_scan_evidence_sources_groups(const gf_model* model, const gf_scan_config* cfg, const double* d_scales, int32_t nscales,
                                               const double* sources, const double* injected, int32_t nsrc, int32_t groups, double* d_lse,
                                               void* d_work, uint64_t work_bytes, void* stream) {
    return evidence_sources("gf_scan_evidence_sources_groups", model, cfg, d_scales, nscales, sources, injected, nsrc, true, groups, d_lse, d_work,
                            work_bytes, (cudaStream_t)stream);
}
