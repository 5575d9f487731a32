// Per-pair repeatability of MaD._match_dsc (mad/MaD.py:426-453), the loop that follows the
// descriptor contraction: for every matched pair (hi, lo) the rigid transform
//     R = inv(Rfinal_lo) . Rfinal_hi,   q = (p - subv_hi) . R^T + subv_lo
// is applied to the cloud of matched hi anchors and the share of transformed anchors that have a
// matched lo anchor within `dist` (cKDTree.query with distance_upper_bound, `distances < dist`) is
// recorded together with the pair's bookkeeping (23 float64 per pair).
//
// Two kernels share the per-pair arithmetic (pair_rotation: the roundings are the same by construction):
// repeat_counts_kernel counts the hits of the pairs [p0, p1), one CTA per pair, threads over the hi cloud; the lo cloud
// sits in a uniform grid of cell size `dist` (cell-sorted points + cell_start, mad_cloud_grid); a bitmap of the cells
// whose 27-cell neighbourhood holds any lo point rejects most transformed anchors with one probe.
// repeat_rows_kernel expands (pair, count) into the 23-column rows, one thread per output value.  Splitting the pair
// range is what lets several GPUs share the counting (mad_b200.parallel.match_dsc_sharded).
// All arithmetic is float64 like NumPy's.
#include <algorithm>

#include "common.cuh"

namespace {

struct RepeatArgs {
    const int32_t* pair_hi;
    const int32_t* pair_lo;
    const double* hi_subv;      // [Dh][3]
    const double* lo_subv;      // [Dl][3]
    const int32_t* hi_meta;     // [Dh][4] index, oct_scale, main_bin, sec_bin
    const int32_t* lo_meta;     // [Dl][4]
    const double* rf;           // [zones*zones][9] Rfinal(main, sec)
    const double* rf_inv;       // [zones*zones][9] inv(Rfinal)
    int zones;
};

// Element (i, j) = tid of R = inv(Rlo) . Rhi of the pair (h, l), row-major (np.dot of two 3x3).
__device__ __forceinline__ double pair_rotation(const RepeatArgs& a, int h, int l, int tid) {
    const double* A = a.rf_inv + ((long long)a.lo_meta[4 * l + 2] * a.zones + a.lo_meta[4 * l + 3]) * 9;
    const double* B = a.rf + ((long long)a.hi_meta[4 * h + 2] * a.zones + a.hi_meta[4 * h + 3]) * 9;
    const int i = tid / 3, j = tid % 3;
    return (A[3 * i] * B[j] + A[3 * i + 1] * B[3 + j]) + A[3 * i + 2] * B[6 + j];
}

struct CloudArgs {
    const double* hi_cloud;     // [H][3]
    int H;
    const double* lo_sorted;    // [L][3] cell-sorted lo cloud
    const int32_t* cell_start;  // [ncell + 1]
    const uint32_t* near_bits;  // [ceil(ncell / 32)]: some lo point in the 27-cell neighbourhood
    double org[3];
    int dims[3];
    double cell;                // = dist
    double dist;
};

// counts == nullptr: the count of pair p goes to results[p][1] as a double (mad_repeatability's in-place form)
__global__ void __launch_bounds__(128)
repeat_counts_kernel(RepeatArgs a, CloudArgs g, long long p0, int32_t* __restrict__ counts, double* __restrict__ results) {
    __shared__ double sR[9], shi[3], slo[3];
    __shared__ int s_count;
    const long long pi = p0 + blockIdx.x;
    const int tid = threadIdx.x;
    const int h = a.pair_hi[pi], l = a.pair_lo[pi];
    if (tid < 9) sR[tid] = pair_rotation(a, h, l, tid);
    if (tid < 3) { shi[tid] = a.hi_subv[3 * (long long)h + tid]; slo[tid] = a.lo_subv[3 * (long long)l + tid]; }
    if (tid == 0) s_count = 0;
    __syncthreads();
    int cnt = 0;
    for (int p = tid; p < g.H; p += blockDim.x) {
        const double dx = g.hi_cloud[3 * p] - shi[0], dy = g.hi_cloud[3 * p + 1] - shi[1], dz = g.hi_cloud[3 * p + 2] - shi[2];
        const double qx = ((dx * sR[0] + dy * sR[1]) + dz * sR[2]) + slo[0];
        const double qy = ((dx * sR[3] + dy * sR[4]) + dz * sR[5]) + slo[1];
        const double qz = ((dx * sR[6] + dy * sR[7]) + dz * sR[8]) + slo[2];
        const int cx = (int)floor((qx - g.org[0]) / g.cell), cy = (int)floor((qy - g.org[1]) / g.cell),
                  cz = (int)floor((qz - g.org[2]) / g.cell);
        if (cx < 0 || cy < 0 || cz < 0 || cx >= g.dims[0] || cy >= g.dims[1] || cz >= g.dims[2]) continue;
        const int c = (cx * g.dims[1] + cy) * g.dims[2] + cz;
        if (!((g.near_bits[c >> 5] >> (c & 31)) & 1u)) continue;
        bool found = false;
        for (int ix = max(cx - 1, 0); ix <= min(cx + 1, g.dims[0] - 1) && !found; ++ix)
            for (int iy = max(cy - 1, 0); iy <= min(cy + 1, g.dims[1] - 1) && !found; ++iy) {
                // the z neighbours are consecutive cells: one contiguous range of sorted points
                const int c0 = (ix * g.dims[1] + iy) * g.dims[2] + max(cz - 1, 0);
                const int c1 = (ix * g.dims[1] + iy) * g.dims[2] + min(cz + 1, g.dims[2] - 1);
                for (int s = g.cell_start[c0]; s < g.cell_start[c1 + 1]; ++s) {
                    const double ex = g.lo_sorted[3 * s] - qx, ey = g.lo_sorted[3 * s + 1] - qy, ez = g.lo_sorted[3 * s + 2] - qz;
                    if (sqrt((ex * ex + ey * ey) + ez * ez) < g.dist) { found = true; break; }
                }
            }
        cnt += found ? 1 : 0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xFFFFFFFFu, cnt, o);
    if ((tid & 31) == 0 && cnt) atomicAdd(&s_count, cnt);
    __syncthreads();
    if (tid == 0) {
        if (counts) counts[blockIdx.x] = s_count;
        else results[pi * 23 + 1] = (double)s_count;
    }
}

// counts == nullptr: the count is read from results[p][1] (where repeat_counts_kernel left it), by the thread that
// then overwrites it
__global__ void repeat_rows_kernel(RepeatArgs a, const double* __restrict__ pair_score, long long n_pairs,
                                   const int32_t* __restrict__ counts, int H, double* __restrict__ results) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n_pairs * 23; e += (long long)gridDim.x * blockDim.x) {
        const long long pi = e / 23;
        const int col = (int)(e - pi * 23);
        const int h = a.pair_hi[pi], l = a.pair_lo[pi];
        double v;
        if (col == 0) v = pair_score[pi];
        else if (col == 1) {
            const long long cnt = counts ? counts[pi] : (long long)results[e];
            v = (double)(100LL * cnt) / (double)H;                          // 100 * count / l
        }
        else if (col < 5) v = a.lo_meta[4 * l + (col - 2)];                  // lo index, oct, main
        else if (col < 8) v = a.hi_meta[4 * h + (col - 5)];                  // hi index, oct, main
        else if (col < 11) v = a.hi_subv[3 * (long long)h + (col - 8)];
        else if (col < 14) v = a.lo_subv[3 * (long long)l + (col - 11)];
        else v = pair_rotation(a, h, l, col - 14);
        results[e] = v;
    }
}

__global__ void mark_used_kernel(const int32_t* __restrict__ idx, long long n, uint8_t* __restrict__ used) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        used[idx[i]] = 1;
}

}  // namespace

extern "C" int mad_mark_used(const int32_t* idx, long long n, uint8_t* used, void* stream) {
    MAD_CHECK_ARG(n >= 0);
    if (n == 0) return MAD_OK;
    MAD_CHECK_ARG(idx && used);
    const int blocks = (int)std::min<long long>(mad_ceil_div(n, 256), (long long)mad_sm_count() * 8);
    MAD_PROF("mark_used_kernel", stream);
    mark_used_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(idx, n, used);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

namespace {

int fill_args(RepeatArgs& a, const int32_t* pair_hi, const int32_t* pair_lo, const double* hi_subv, const double* lo_subv,
              const int32_t* hi_meta, const int32_t* lo_meta, const double* rf_table, const double* rf_inv_table, int rf_zones) {
    MAD_CHECK_ARG(pair_hi && pair_lo && hi_subv && lo_subv && hi_meta && lo_meta && rf_table && rf_inv_table && rf_zones > 0);
    a.pair_hi = pair_hi; a.pair_lo = pair_lo;
    a.hi_subv = hi_subv; a.lo_subv = lo_subv; a.hi_meta = hi_meta; a.lo_meta = lo_meta;
    a.rf = rf_table; a.rf_inv = rf_inv_table; a.zones = rf_zones;
    return MAD_OK;
}

int launch_counts(const RepeatArgs& a, const double* hi_cloud, int n_hi_cloud, const double* lo_sorted, const int32_t* cell_start,
                  const uint32_t* near_bits, const double* grid_org_host, const int* grid_dims_host, double dist, long long p0,
                  long long p1, int32_t* counts, double* results, void* stream) {
    MAD_CHECK_ARG(hi_cloud && n_hi_cloud > 0 && lo_sorted && cell_start && near_bits && grid_org_host && grid_dims_host);
    MAD_CHECK_ARG(dist > 0.0);
    CloudArgs g;
    g.hi_cloud = hi_cloud; g.H = n_hi_cloud; g.lo_sorted = lo_sorted; g.cell_start = cell_start; g.near_bits = near_bits;
    for (int q = 0; q < 3; ++q) { g.org[q] = grid_org_host[q]; g.dims[q] = grid_dims_host[q]; }
    g.cell = dist; g.dist = dist;
    MAD_PROF("repeat_counts_kernel", stream);
    repeat_counts_kernel<<<(unsigned)(p1 - p0), 128, 0, (cudaStream_t)stream>>>(a, g, p0, counts, results);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

int launch_rows(const RepeatArgs& a, const double* pair_score, long long n_pairs, const int32_t* counts, int n_hi_cloud,
                double* results, void* stream) {
    MAD_CHECK_ARG(pair_score && results && n_hi_cloud > 0);
    const int blocks = (int)std::min<long long>(mad_ceil_div(n_pairs * 23, 256), (long long)mad_sm_count() * 16);
    MAD_PROF("repeat_rows_kernel", stream);
    repeat_rows_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(a, pair_score, n_pairs, counts, n_hi_cloud, results);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

}  // namespace

extern "C" int mad_repeat_counts(const int32_t* pair_hi, const int32_t* pair_lo, long long p0, long long p1,
                                 const double* hi_subv, const double* lo_subv, const int32_t* hi_meta, const int32_t* lo_meta,
                                 const double* rf_table, const double* rf_inv_table, int rf_zones,
                                 const double* hi_cloud, int n_hi_cloud, const double* lo_sorted, const int32_t* cell_start,
                                 const uint32_t* near_bits, const double* grid_org_host, const int* grid_dims_host,
                                 double dist, int32_t* counts, void* stream) {
    MAD_CHECK_ARG(p0 >= 0 && p0 <= p1 && p1 - p0 < (1LL << 31));
    if (p1 == p0) return MAD_OK;
    MAD_CHECK_ARG(counts);
    RepeatArgs a;
    int rc = fill_args(a, pair_hi, pair_lo, hi_subv, lo_subv, hi_meta, lo_meta, rf_table, rf_inv_table, rf_zones);
    if (rc != MAD_OK) return rc;
    return launch_counts(a, hi_cloud, n_hi_cloud, lo_sorted, cell_start, near_bits, grid_org_host, grid_dims_host, dist, p0, p1,
                         counts, nullptr, stream);
}

extern "C" int mad_repeat_rows(const int32_t* pair_hi, const int32_t* pair_lo, const double* pair_score, long long n_pairs,
                               const double* hi_subv, const double* lo_subv, const int32_t* hi_meta, const int32_t* lo_meta,
                               const double* rf_table, const double* rf_inv_table, int rf_zones, const int32_t* counts,
                               int n_hi_cloud, double* results, void* stream) {
    MAD_CHECK_ARG(n_pairs >= 0 && n_pairs < (1LL << 31));
    if (n_pairs == 0) return MAD_OK;
    MAD_CHECK_ARG(counts);
    RepeatArgs a;
    int rc = fill_args(a, pair_hi, pair_lo, hi_subv, lo_subv, hi_meta, lo_meta, rf_table, rf_inv_table, rf_zones);
    if (rc != MAD_OK) return rc;
    return launch_rows(a, pair_score, n_pairs, counts, n_hi_cloud, results, stream);
}

extern "C" int mad_repeatability(const int32_t* pair_hi, const int32_t* pair_lo, const double* pair_score, long long n_pairs,
                                 const double* hi_subv, const double* lo_subv, const int32_t* hi_meta, const int32_t* lo_meta,
                                 const double* rf_table, const double* rf_inv_table, int rf_zones,
                                 const double* hi_cloud, int n_hi_cloud, const double* lo_sorted, const int32_t* cell_start,
                                 const uint32_t* near_bits, const double* grid_org_host, const int* grid_dims_host,
                                 double dist, double* results, void* stream) {
    MAD_CHECK_ARG(n_pairs >= 0 && n_pairs < (1LL << 31));
    if (n_pairs == 0) return MAD_OK;
    MAD_CHECK_ARG(results);
    RepeatArgs a;
    int rc = fill_args(a, pair_hi, pair_lo, hi_subv, lo_subv, hi_meta, lo_meta, rf_table, rf_inv_table, rf_zones);
    if (rc != MAD_OK) return rc;
    // counts + rows; the counts wait in column 1 of the rows they end in (no work space)
    rc = launch_counts(a, hi_cloud, n_hi_cloud, lo_sorted, cell_start, near_bits, grid_org_host, grid_dims_host, dist, 0, n_pairs,
                       nullptr, results, stream);
    if (rc != MAD_OK) return rc;
    return launch_rows(a, pair_score, n_pairs, nullptr, n_hi_cloud, results, stream);
}
