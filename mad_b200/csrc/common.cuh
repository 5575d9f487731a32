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

// ---- float32 grid maximum and isovalue cut / normalisation, shared by the single-grid (dmap.cu) and batched (density.cu)
// kernels, so that a voxel of either goes through the same operations.
// order-preserving map float -> unsigned (for atomicMax on floats of either sign); 0 lies below every float's image
__device__ __forceinline__ unsigned int mad_f2ord(float f) {
    const unsigned int u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ __forceinline__ unsigned int mad_ord2bits(unsigned int ord) {
    return (ord & 0x80000000u) ? (ord & 0x7FFFFFFFu) : ~ord;
}
// v < isovalue -> 0 (mad/Dmap.py:50-54), then v / vmax with a correctly rounded float32 division (:66-67; numpy divides
// float32 by float32).  divide = 0 skips the normalisation.
__device__ __forceinline__ float mad_threshold_normalise_one(float v, float isovalue, float vmax, int divide) {
    if (v < isovalue) v = 0.f;
    if (divide) v = __fdiv_rn(v, vmax);
    return v;
}

// ---- per-map arguments of the batched orientation / description launches (mad_orient_many, mad_describe_many) ----
// The table travels as one __grid_constant__ kernel parameter, so every read of it is a constant-bank operand, as the
// single-map kernels' own arguments are; a batch of more maps is split into launches of kMadBatchMaps maps.
constexpr int kMadBatchMaps = 64;
struct MadBatchMap {
    const float4* grad[2];  // gradient of octave 0 / 1
    int n[2][3];            // dims of octave 0 / 1
    int kp0;                // first row of the map in the batch keypoint table
    int row0;               // mad_describe_many: first oriented feature of the map, counted from the launch's first map
};
struct MadBatchMaps {
    static constexpr bool kMaps = true;
    const int* kp_off;      // mad_orient_many: the batch's kp_off from the launch's first map on (device)
    int G, pad;             // maps of this launch
    MadBatchMap m[kMadBatchMaps];
};

// The table of the maps [g0, g0 + G) (G <= kMadBatchMaps) from the host arrays of a batched call: grads_host [][2]
// device addresses, dims_host [][6], and (may be NULL) kp_off_host / ori_off_host [] the batch offsets.
static inline void mad_batch_maps(MadBatchMaps& t, int g0, int G, const uint64_t* grads_host, const int* dims_host,
                                  const int* kp_off_host, const int* ori_off_host) {
    t.G = G;
    t.pad = 0;
    for (int i = 0; i < G; ++i) {
        MadBatchMap& m = t.m[i];
        for (int o = 0; o < 2; ++o) {
            m.grad[o] = reinterpret_cast<const float4*>(grads_host[2 * (g0 + i) + o]);
            for (int a = 0; a < 3; ++a) m.n[o][a] = dims_host[6 * (g0 + i) + 3 * o + a];
        }
        m.kp0 = kp_off_host ? kp_off_host[g0 + i] : 0;
        m.row0 = ori_off_host ? ori_off_host[g0 + i] - ori_off_host[g0] : 0;
    }
}

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
