// Internal helpers shared by the translation units of libgslift.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "gslift.h"

namespace gsl {

// Thread-local message behind gsl_last_error().
void set_error(const char *fmt, ...);
int fail(int code, const char *fmt, ...);

#define GSL_CUDA_TRY(expr)                                                               \
    do {                                                                                 \
        cudaError_t _e = (expr);                                                         \
        if (_e != cudaSuccess)                                                           \
            return gsl::fail(GSL_ECUDA, "%s failed: %s (%s:%d)", #expr,                  \
                             cudaGetErrorString(_e), __FILE__, __LINE__);                \
    } while (0)

// Every kernel launch of the library passes through here; the count backs gsl_launch_count().
void count_launch();

#define GSL_LAUNCH_CHECK(name)                                                           \
    do {                                                                                 \
        gsl::count_launch();                                                             \
        cudaError_t _e = cudaGetLastError();                                             \
        if (_e != cudaSuccess)                                                           \
            return gsl::fail(GSL_ECUDA, "launch of %s failed: %s", name,                 \
                             cudaGetErrorString(_e));                                    \
    } while (0)

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Cached per-device facts (SM count) so launches can size persistent grids.
int sm_count();

// kmeans_ordered.cu: scratch for gsl_kmeans_update_ordered.
size_t ordered_workspace_bytes(int64_t N, int D, int K);

// kmeans_tc.cu: tensor-core screened assignment (K <= 64, 8 <= D <= 64).
bool tc_supported(int D, int K);
int launch_step_tc(bool accumulate, const float *data, int64_t N, int D, const float *centroids, int K,
                   int32_t *labels, double *partials, int grid, cudaStream_t st);

}  // namespace gsl
