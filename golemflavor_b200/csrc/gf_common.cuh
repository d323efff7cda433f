/*
 * gf_common.cuh -- library-internal glue shared by the translation units of
 * libgolemflavor_b200.so: error reporting, launch geometry, and the host-side
 * flattening gf_model (C ABI) -> gf_dev_model (kernel parameter).
 */
#ifndef GF_COMMON_CUH
#define GF_COMMON_CUH

#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>

#include "gf_model.cuh"

int gf_fail(int code, const char* fmt, ...);

#define GF_CUDA(expr)                                                                            \
    do {                                                                                         \
        cudaError_t gf_e_ = (expr);                                                              \
        if (gf_e_ != cudaSuccess)                                                                \
            return gf_fail(GF_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(gf_e_));      \
    } while (0)

#define GF_REQUIRE(cond, ...)                                \
    do {                                                     \
        if (!(cond)) return gf_fail(GF_ERR_ARG, __VA_ARGS__); \
    } while (0)

/* kernel launch check: catches bad configurations immediately, execution errors surface at the
 * caller's next synchronisation (the ABI is asynchronous on `stream`). */
#define GF_LAUNCH_CHECK(name)                                                                    \
    do {                                                                                         \
        cudaError_t gf_e_ = cudaGetLastError();                                                  \
        if (gf_e_ != cudaSuccess)                                                                \
            return gf_fail(GF_ERR_CUDA, "launch of %s failed: %s", name, cudaGetErrorString(gf_e_)); \
    } while (0)

static inline unsigned gf_blocks_for(int64_t n, int threads) { return (unsigned)((n + threads - 1) / threads); }

/* Validate a gf_model and derive the kernel-side constants.  Returns GF_OK / GF_ERR_ARG. */
int gf_build_dev_model(const gf_model* m, gf_dev_model* d);

/* number of SMs of the current device (cached) */
int gf_sm_count(int* sms);

/* The refusals of every frozen-scale grid entry point `who`: the model needs a BSM path and must not sample the scale. */
int gf_check_frozen_scale(const char* who, const gf_dev_model& d);

/* Blocks in x of an evidence-grid launch of ny scale groups: as many as fit the device in ONE wave at per_sm blocks per
 * SM (every block carries the same amount of work, so blocks left for a second wave would double the time), no more than
 * the samples need, at least one. */
unsigned gf_evidence_nx(int sms, int per_sm, int ny, uint64_t count, int threads);

/* The workspace of an evidence-grid launch: per-block partials [rows][nx][2], then one ticket per scale group (ny), cleared
 * on stream st.  Refuses a workspace smaller than that (`who`_workspace gives its size). */
int gf_evidence_workspace(const char* who, size_t rows, unsigned nx, int ny, void* d_work, uint64_t work_bytes, cudaStream_t st, double** part,
                          unsigned int** tickets);

/* Sample groups of the grouped evidence grids (sample i in group i mod groups): a power of two in [2, 32], so that a group
 * is fixed per thread of the grid kernel and per lane of a warp. */
#define GF_EVIDENCE_MAX_GROUPS 32
bool gf_evidence_groups_ok(int groups);

#endif /* GF_COMMON_CUH */
