// Anchor clouds of MaD._match_dsc (mad/MaD.py:427-428) and the uniform grid the repeatability kernel searches,
// built on the device so that match_dsc needs no host round trip between the matching and the per-pair loop.
//
// mad_anchor_cloud: np.unique(subv[used], axis=0) -- the distinct used rows in lexicographic (x, y, z) order.  Every
// row gets three order-preserving uint64 images of its coordinates (-0.0 keyed as +0.0, as NumPy compares them equal;
// unused rows get the largest key, so they sort behind every used row without a compaction and without a count read
// back first); three stable radix sorts, on z, then y, then x, give the lexicographic order; a flag per first row of a
// run of equal rows, an exclusive scan and a scatter give the unique cloud.  One CTA then reduces its bounds with
// exactly the float64 operations of the host construction:  org = min - cell,  dims = floor((max - org) / cell) + 2.
//
// mad_cloud_grid: the cell-sorted cloud (stable by cell id, so within a cell the cloud's own order is kept, as
// np.argsort(kind="stable") keeps it), cell_start = number of points in lower cells, and the bitmap of cells whose
// 27-cell neighbourhood holds a point.
#include <cub/cub.cuh>
#include <math.h>

#include <algorithm>
#include <utility>

#include "common.cuh"

namespace {

constexpr unsigned long long kUnusedKey = ~0ull;     // above the image of every finite double

__device__ __forceinline__ double norm_zero(double v) { return v == 0.0 ? 0.0 : v; }

// Order-preserving image of a double: a < b (as doubles, both finite) <=> img(a) < img(b) (as uint64).
__device__ __forceinline__ unsigned long long order_image(double v) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(norm_zero(v));
    return (b >> 63) ? ~b : (b | (1ull << 63));
}

__global__ void cloud_keys_kernel(const double* __restrict__ subv, const uint8_t* __restrict__ used, int n, int axis,
                                  const int* __restrict__ order, unsigned long long* __restrict__ keys,
                                  int* __restrict__ idx_out, long long* __restrict__ info) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int r = order ? order[i] : i;
    if (!order) idx_out[i] = i;
    if (!used[r]) { keys[i] = kUnusedKey; return; }
    const double v = subv[3 * (long long)r + axis];
    keys[i] = order_image(v);
    if (axis == 2 && !(isfinite(v) && isfinite(subv[3 * (long long)r]) && isfinite(subv[3 * (long long)r + 1])))
        atomicAdd((unsigned long long*)&info[1], 1ull);           // a non-finite used row: the caller refuses the set
}

__global__ void cloud_flags_kernel(const double* __restrict__ subv, const uint8_t* __restrict__ used, int n,
                                   const int* __restrict__ order, int* __restrict__ flags) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long r = order[i];
    int f = used[r] ? 1 : 0;
    if (f && i > 0) {
        const long long q = order[i - 1];               // used too: unused rows sort behind every used row
        f = !(norm_zero(subv[3 * r]) == norm_zero(subv[3 * q]) && norm_zero(subv[3 * r + 1]) == norm_zero(subv[3 * q + 1]) &&
              norm_zero(subv[3 * r + 2]) == norm_zero(subv[3 * q + 2]));
    }
    flags[i] = f;
}

__global__ void cloud_scatter_kernel(const double* __restrict__ subv, int n, const int* __restrict__ order,
                                     const int* __restrict__ flags, const int* __restrict__ pos, double* __restrict__ cloud,
                                     long long* __restrict__ info) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (i == n - 1) info[0] = pos[i] + flags[i];
    if (!flags[i]) return;
    const long long r = order[i], o = pos[i];
    for (int q = 0; q < 3; ++q) cloud[3 * o + q] = norm_zero(subv[3 * r + q]);
}

// One CTA: min / max per axis of the n = info[0] cloud rows, then org and dims (info[2..4]; org also as raw bits in
// info[5..7], so one small read brings everything the host needs).  A dims value that does not fit 2^40 is stored as 2^40.
__global__ void __launch_bounds__(1024) cloud_bounds_kernel(const double* __restrict__ cloud, double cell,
                                                            double* __restrict__ org_out, long long* __restrict__ info) {
    __shared__ double s_min[3][32], s_max[3][32];
    const long long n = info[0];
    double mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (long long i = threadIdx.x; i < n; i += blockDim.x)
        for (int q = 0; q < 3; ++q) { mn[q] = fmin(mn[q], cloud[3 * i + q]); mx[q] = fmax(mx[q], cloud[3 * i + q]); }
    for (int q = 0; q < 3; ++q)
        for (int o = 16; o > 0; o >>= 1) {
            mn[q] = fmin(mn[q], __shfl_xor_sync(0xFFFFFFFFu, mn[q], o));
            mx[q] = fmax(mx[q], __shfl_xor_sync(0xFFFFFFFFu, mx[q], o));
        }
    const int w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    if ((threadIdx.x & 31) == 0)
        for (int q = 0; q < 3; ++q) { s_min[q][w] = mn[q]; s_max[q][w] = mx[q]; }
    __syncthreads();
    if (threadIdx.x < 3) {
        const int q = threadIdx.x;
        double a = INFINITY, b = -INFINITY;
        for (int j = 0; j < nw; ++j) { a = fmin(a, s_min[q][j]); b = fmax(b, s_max[q][j]); }
        if (n == 0) { a = 0.0; b = 0.0; }
        const double org = a - cell;                               // cloud.min(0) - cell
        const double d = floor((b - org) / cell) + 2.0;            // floor((cloud.max(0) - org) / cell) + 2
        const double cap = 1099511627776.0;                        // 2^40: far beyond any grid the library accepts
        org_out[q] = org;
        info[2 + q] = n == 0 ? 0 : (long long)(d < cap ? d : cap);
        info[5 + q] = __double_as_longlong(org);
    }
}

__global__ void grid_keys_kernel(const double* __restrict__ cloud, int n, const double* __restrict__ org, double cell,
                                 int d1, int d2, int* __restrict__ keys, int* __restrict__ idx) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long cx = (long long)floor((cloud[3 * (long long)i] - org[0]) / cell);
    const long long cy = (long long)floor((cloud[3 * (long long)i + 1] - org[1]) / cell);
    const long long cz = (long long)floor((cloud[3 * (long long)i + 2] - org[2]) / cell);
    keys[i] = (int)((cx * d1 + cy) * d2 + cz);
    idx[i] = i;
}

__global__ void grid_gather_kernel(const double* __restrict__ cloud, int n, const int* __restrict__ order,
                                   double* __restrict__ sorted) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    for (int q = 0; q < 3; ++q) sorted[3 * (long long)i + q] = cloud[3 * (long long)order[i] + q];
}

// cell_start[c] = #{points in cells < c}, c = 0..ncell: a lower bound in the sorted cell ids.
__global__ void grid_cell_start_kernel(const int* __restrict__ keys, int n, long long ncell, int32_t* __restrict__ cell_start) {
    for (long long c = blockIdx.x * (long long)blockDim.x + threadIdx.x; c <= ncell; c += (long long)gridDim.x * blockDim.x) {
        int lo = 0, hi = n;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if ((long long)keys[mid] < c) lo = mid + 1; else hi = mid;
        }
        cell_start[c] = lo;
    }
}

// near_bits word w: bit b set if a cell of the 27-neighbourhood of cell 32 w + b (clipped to the grid) holds a point.
__global__ void grid_near_kernel(const int32_t* __restrict__ cell_start, int d0, int d1, int d2, long long ncell,
                                 long long n_words, uint32_t* __restrict__ near_bits) {
    for (long long w = blockIdx.x * (long long)blockDim.x + threadIdx.x; w < n_words; w += (long long)gridDim.x * blockDim.x) {
        uint32_t bits = 0;
        for (int b = 0; b < 32; ++b) {
            const long long c = 32 * w + b;
            if (c >= ncell) break;
            const int cz = (int)(c % d2), cy = (int)((c / d2) % d1), cx = (int)(c / ((long long)d1 * d2));
            bool near = false;
            for (int ix = max(cx - 1, 0); ix <= min(cx + 1, d0 - 1) && !near; ++ix)
                for (int iy = max(cy - 1, 0); iy <= min(cy + 1, d1 - 1) && !near; ++iy) {
                    const long long c0 = ((long long)ix * d1 + iy) * d2 + max(cz - 1, 0);
                    const long long c1 = ((long long)ix * d1 + iy) * d2 + min(cz + 1, d2 - 1);
                    near = cell_start[c1 + 1] > cell_start[c0];     // the z neighbours are consecutive cells
                }
            bits |= (near ? 1u : 0u) << b;
        }
        near_bits[w] = bits;
    }
}

struct CloudLayout {
    size_t keys_a, keys_b, idx_a, idx_b, flags, pos, cub, total;
};

CloudLayout cloud_layout(int n) {
    CloudLayout l;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o += mad_align_up(bytes, 256); return r; };
    const size_t nn = (size_t)(n > 0 ? n : 1);
    l.keys_a = take(nn * 8); l.keys_b = take(nn * 8);
    l.idx_a = take(nn * 4); l.idx_b = take(nn * 4);
    l.flags = take(nn * 4); l.pos = take(nn * 4);
    size_t a = 0, b = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, a, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                    (const int*)nullptr, (int*)nullptr, (int)nn);
    cub::DeviceScan::ExclusiveSum(nullptr, b, (const int*)nullptr, (int*)nullptr, (int)nn);
    l.cub = take(a > b ? a : b);
    l.total = o;
    return l;
}

struct GridLayout {
    size_t keys_in, keys_out, idx_in, idx_out, cub, total;
};

GridLayout grid_layout(int n) {
    GridLayout l;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o += mad_align_up(bytes, 256); return r; };
    const size_t nn = (size_t)(n > 0 ? n : 1);
    l.keys_in = take(nn * 4); l.keys_out = take(nn * 4);
    l.idx_in = take(nn * 4); l.idx_out = take(nn * 4);
    size_t a = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, a, (const int*)nullptr, (int*)nullptr, (const int*)nullptr, (int*)nullptr, (int)nn);
    l.cub = take(a);
    l.total = o;
    return l;
}

}  // namespace

extern "C" size_t mad_anchor_cloud_workspace_bytes(int n_rows) { return cloud_layout(n_rows).total; }

extern "C" int mad_anchor_cloud(const double* subv, const uint8_t* used, int n_rows, double cell, double* cloud,
                                double* grid_org, long long* info, void* workspace, size_t workspace_bytes, void* stream) {
    MAD_CHECK_ARG(n_rows >= 0 && info && grid_org && cell > 0.0);
    cudaStream_t st = (cudaStream_t)stream;
    MAD_CUDA(cudaMemsetAsync(info, 0, 8 * sizeof(long long), st));
    if (n_rows == 0) return MAD_OK;
    MAD_CHECK_ARG(subv && used && cloud && workspace);
    const CloudLayout l = cloud_layout(n_rows);
    MAD_CHECK_ARG(workspace_bytes >= l.total);
    char* ws = reinterpret_cast<char*>(workspace);
    auto* ka = reinterpret_cast<unsigned long long*>(ws + l.keys_a);
    auto* kb = reinterpret_cast<unsigned long long*>(ws + l.keys_b);
    int* ia = reinterpret_cast<int*>(ws + l.idx_a);
    int* ib = reinterpret_cast<int*>(ws + l.idx_b);
    int* flags = reinterpret_cast<int*>(ws + l.flags);
    int* pos = reinterpret_cast<int*>(ws + l.pos);
    const int tb = 256, nb = (int)mad_ceil_div(n_rows, tb);
    // LSD order: z, then y, then x, each sort stable -> lexicographic (x, y, z); the order travels in ia
    for (int axis = 2; axis >= 0; --axis) {
        {
            MAD_PROF("cloud_keys_kernel", st);
            cloud_keys_kernel<<<nb, tb, 0, st>>>(subv, used, n_rows, axis, axis == 2 ? nullptr : ia, ka, ia, info);
            MAD_LAUNCH_OK();
        }
        size_t cub_bytes = l.total - l.cub;
        MAD_PROF("cub_radix_sort_pairs", st);
        MAD_CUDA(cub::DeviceRadixSort::SortPairs(ws + l.cub, cub_bytes, ka, kb, ia, ib, n_rows, 0, 64, st));
        std::swap(ia, ib);
    }
    {
        MAD_PROF("cloud_flags_kernel", st);
        cloud_flags_kernel<<<nb, tb, 0, st>>>(subv, used, n_rows, ia, flags);
        MAD_LAUNCH_OK();
    }
    {
        size_t cub_bytes = l.total - l.cub;
        MAD_PROF("cub_exclusive_sum", st);
        MAD_CUDA(cub::DeviceScan::ExclusiveSum(ws + l.cub, cub_bytes, flags, pos, n_rows, st));
    }
    {
        MAD_PROF("cloud_scatter_kernel", st);
        cloud_scatter_kernel<<<nb, tb, 0, st>>>(subv, n_rows, ia, flags, pos, cloud, info);
        MAD_LAUNCH_OK();
    }
    MAD_PROF("cloud_bounds_kernel", st);
    cloud_bounds_kernel<<<1, 1024, 0, st>>>(cloud, cell, grid_org, info);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" size_t mad_cloud_grid_workspace_bytes(int n) { return grid_layout(n).total; }

extern "C" int mad_cloud_grid(const double* cloud, int n, const double* grid_org, const long long* grid_dims_host,
                              double cell, double* sorted, int32_t* cell_start, uint32_t* near_bits, void* workspace,
                              size_t workspace_bytes, void* stream) {
    MAD_CHECK_ARG(grid_dims_host);
    const long long d0 = grid_dims_host[0], d1 = grid_dims_host[1], d2 = grid_dims_host[2];
    MAD_CHECK_ARG(d0 >= 1 && d1 >= 1 && d2 >= 1);
    // the repeatability kernel indexes cells in int32: refuse a grid of 2^31 cells or more (checked before the
    // pointers, so a caller may pass none for a grid it could not allocate)
    MAD_CHECK_ARG(d0 < (1ll << 31) && d1 < (1ll << 31) && d2 < (1ll << 31) && d0 * d1 < (1ll << 31) &&
                  d0 * d1 * d2 < (1ll << 31));
    MAD_CHECK_ARG(n > 0 && cloud && grid_org && sorted && cell_start && near_bits && workspace);
    MAD_CHECK_ARG(cell > 0.0);
    const long long ncell = d0 * d1 * d2;
    const GridLayout l = grid_layout(n);
    MAD_CHECK_ARG(workspace_bytes >= l.total);
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = reinterpret_cast<char*>(workspace);
    int* keys_in = reinterpret_cast<int*>(ws + l.keys_in);
    int* keys_out = reinterpret_cast<int*>(ws + l.keys_out);
    int* idx_in = reinterpret_cast<int*>(ws + l.idx_in);
    int* idx_out = reinterpret_cast<int*>(ws + l.idx_out);
    const int tb = 256, nb = (int)mad_ceil_div(n, tb);
    {
        MAD_PROF("grid_keys_kernel", st);
        grid_keys_kernel<<<nb, tb, 0, st>>>(cloud, n, grid_org, cell, (int)d1, (int)d2, keys_in, idx_in);
        MAD_LAUNCH_OK();
    }
    {
        int end_bit = 1;
        while (end_bit < 31 && (1ll << end_bit) < ncell) ++end_bit;
        size_t cub_bytes = l.total - l.cub;
        MAD_PROF("cub_radix_sort_pairs", st);
        MAD_CUDA(cub::DeviceRadixSort::SortPairs(ws + l.cub, cub_bytes, keys_in, keys_out, idx_in, idx_out, n, 0, end_bit, st));
    }
    {
        MAD_PROF("grid_gather_kernel", st);
        grid_gather_kernel<<<nb, tb, 0, st>>>(cloud, n, idx_out, sorted);
        MAD_LAUNCH_OK();
    }
    const int cap = mad_sm_count() * 8;
    {
        MAD_PROF("grid_cell_start_kernel", st);
        grid_cell_start_kernel<<<(int)std::min<long long>(mad_ceil_div(ncell + 1, 256), cap), 256, 0, st>>>(keys_out, n, ncell,
                                                                                                           cell_start);
        MAD_LAUNCH_OK();
    }
    const long long n_words = mad_ceil_div(ncell, 32);
    MAD_PROF("grid_near_kernel", st);
    grid_near_kernel<<<(int)std::min<long long>(mad_ceil_div(n_words, 256), cap), 256, 0, st>>>(cell_start, (int)d0, (int)d1,
                                                                                                 (int)d2, ncell, n_words, near_bits);
    MAD_LAUNCH_OK();
    return MAD_OK;
}
