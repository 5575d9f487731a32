// Shared helpers for libmad_b200 (sm_100a).  Internal header, not part of the C ABI.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "mad_b200.h"

void mad_set_error(const char* fmt, ...);

#define MAD_CHECK_ARG(cond)                                                        \
    do {                                                                           \
        if (!(cond)) {                                                             \
            mad_set_error("%s:%d: bad argument: %s", __FILE__, __LINE__, #cond);   \
            return MAD_ERR_ARG;                                                    \
        }                                                                          \
    } while (0)

#define MAD_CUDA(expr)                                                             \
    do {                                                                           \
        cudaError_t _e = (expr);                                                   \
        if (_e != cudaSuccess) {                                                   \
            mad_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr,            \
                          cudaGetErrorString(_e));                                 \
            return MAD_ERR_CUDA;                                                   \
        }                                                                          \
    } while (0)

#define MAD_LAUNCH_OK() MAD_CUDA(cudaGetLastError())

static inline long long mad_ceil_div(long long a, long long b) { return (a + b - 1) / b; }
static inline size_t mad_align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// SciPy `reflect` boundary (d c b a | a b c d | d c b a), valid for -n <= i < 2n.
__host__ __device__ __forceinline__ int mad_reflect(int i, int n) {
    if (i < 0) return -i - 1;
    if (i >= n) return 2 * n - 1 - i;
    return i;
}

// Segment of entry e of a batch whose G segments start at off(0) <= off(1) <= ... (off(0) <= e < total): the largest g
// with off(g) <= e, which is the non-empty segment holding e (an empty segment shares its start with the next one).
template <typename Off>
__host__ __device__ __forceinline__ int mad_segment_of(Off off, int G, long long e) {
    int lo = 0, hi = G - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (off(mid) <= e) lo = mid; else hi = mid - 1;
    }
    return lo;
}

int mad_sm_count();

// ---- launch accounting / optional per-kernel CUDA-event timing (mad_profile_*, api.cu) ----------
// Every kernel launch site of the library opens a MadProfScope: it always counts the launch
// (mad_launch_count) and, while profiling is enabled, brackets it with two events recorded on
// the launching stream.  bench.py reads the per-kernel durations from there.
struct MadProfScope {
    int slot;
    cudaStream_t st;
    MadProfScope(const char* name, cudaStream_t stream);
    ~MadProfScope();
};
#define MAD_PROF(name, stream) MadProfScope _mad_prof_scope(name, (cudaStream_t)(stream))
