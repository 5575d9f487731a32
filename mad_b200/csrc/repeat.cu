// Per-pair repeatability of MaD._match_dsc (mad/MaD.py:426-453), the loop that follows the
// descriptor contraction: for every matched pair (hi, lo) the rigid transform
//     R = inv(Rfinal_lo) . Rfinal_hi,   q = (p - subv_hi) . R^T + subv_lo
// is applied to the cloud of matched hi anchors and the share of transformed anchors that have a
// matched lo anchor within `dist` (cKDTree.query with distance_upper_bound, `distances < dist`) is
// recorded together with the pair's bookkeeping (23 float64 per pair).
//
// Two kernels share the per-pair arithmetic (pair_rotation: the roundings are the same by construction):
// repeat_counts_kernel counts the hits of the pairs [p0, p1), one CTA per pair, threads over the hi cloud; the lo cloud
// sits in a uniform grid of cells a little larger than `dist` (cell-sorted points + cell_start, mad_cloud_grid); a bitmap of the cells
// whose 27-cell neighbourhood holds any lo point rejects most transformed anchors with one probe.
// repeat_rows_kernel expands (pair, count) into the 23-column rows, one thread per output value.  Splitting the pair
// range is what lets several GPUs share the counting (mad_b200.parallel.match_dsc_sharded).
//
// The arithmetic is float64 with every rounding written out, so that it does not depend on nvcc's contraction choices
// (fma(a, b, c) below is rounded once, from the exact a b + c; tests/repeat_ref.py evaluates the same sequence exactly):
//     R[i][j] = fma(A[i][2], B[2][j], fma(A[i][1], B[1][j], A[i][0] B[0][j]))        A = inv(Rfinal_lo), B = Rfinal_hi
//     d = p - subv_hi,   q[i] = fma(d[2], R[i][2], fma(d[1], R[i][1], d[0] R[i][0])) + subv_lo[i]
//     e = l - q,         hit  = sqrt(fma(e[2], e[2], fma(e[1], e[1], e[0] e[0]))) < dist   (l: a lo cloud point)
// and column 1 of a row is (100 count) / H.  NumPy's plain sums differ from this by an ulp at times (the reference's
// R comes from a dgemm), which is why a count against the reference may flip when a distance is within ulps of dist.
//
// Why the 27-cell search finds every hit.  The lo grid is built with the cell c = mad_repeat_grid_cell(dist) =
// dist (1 + 2^-16), a little more than dist, while a hit still needs a distance < dist.  Let u = 2^-53, org = RN(min - c),
// dims = floor(t(max)) + 2 per axis, where t(x) = RN(RN(x - org) / c) is the cell coordinate the builder and this kernel
// both compute (cell index floor(t)).  Take a lo point l and a transformed anchor q whose computed distance is < dist:
//   (a) on each axis |l - q| < dist (1 + 3u): the computed sum is >= RN(e e) of any one axis (roundings are monotone
//       and the terms non-negative), so sqrt of it < dist gives |e| < dist (1 + u), and e = RN(l - q).
//   (b) q >= org: org is the double nearest to min - c, so a double q < org has q <= min - c, and then
//       l - q >= c > dist (1 + 3u), against (a).  So t(q) >= 0.
//   (c) t(x) = (x - org) / c (1 + th) with |th| <= 3u.  For the lo point 0 <= t(l) < dims - 1, and each dim is < 2^29
//       (the builder refuses grids of 2^31 cells or more, and every dim is >= 2), so the rounding terms add less than
//       3u (2 dims + 1) < 2^-21, and with c >= dist (1 + 2^-16) (1 - u),
//       |t(l) - t(q)| < (1 + 4u) / (1 + 2^-16) + 2^-21 < 1 - 2^-17 + 2^-21 < 1.
// So floor(t(q)) is within 1 of l's cell on every axis, and q's cell lies inside the grid (0 <= cq <= dims - 1): q is
// not skipped, its near bit is set and l's cell is among the ones searched.  With c = dist the first term of (c) is 1
// and the roundings alone can put l two cells away from q.  A q far outside (up to any finite value) is skipped by
// the range test: the float64 -> int conversion saturates.
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
    return fma(A[3 * i + 2], B[6 + j], fma(A[3 * i + 1], B[3 + j], __dmul_rn(A[3 * i], B[j])));
}

struct CloudArgs {
    const double* hi_cloud;     // [H][3]
    int H;
    const double* lo_sorted;    // [L][3] cell-sorted lo cloud
    const int32_t* cell_start;  // [ncell + 1]
    const uint32_t* near_bits;  // [ceil(ncell / 32)]: some lo point in the 27-cell neighbourhood
    double org[3];
    int dims[3];
    double cell;                // = mad_repeat_grid_cell(dist)
    double dist;
};

// Hits of pair pi: the CTA's threads share the hi cloud; the total is valid in thread 0.  The one body of the per-point
// arithmetic, for the single-structure and the batched kernel alike.
__device__ __forceinline__ int count_pair(const RepeatArgs& a, const CloudArgs& g, long long pi) {
    __shared__ double sR[9], shi[3], slo[3];
    __shared__ int s_count;
    const int tid = threadIdx.x;
    const int h = a.pair_hi[pi], l = a.pair_lo[pi];
    if (tid < 9) sR[tid] = pair_rotation(a, h, l, tid);
    if (tid < 3) { shi[tid] = a.hi_subv[3 * (long long)h + tid]; slo[tid] = a.lo_subv[3 * (long long)l + tid]; }
    if (tid == 0) s_count = 0;
    __syncthreads();
    int cnt = 0;
    for (int p = tid; p < g.H; p += blockDim.x) {
        const double dx = g.hi_cloud[3 * p] - shi[0], dy = g.hi_cloud[3 * p + 1] - shi[1], dz = g.hi_cloud[3 * p + 2] - shi[2];
        const double qx = __dadd_rn(fma(dz, sR[2], fma(dy, sR[1], __dmul_rn(dx, sR[0]))), slo[0]);
        const double qy = __dadd_rn(fma(dz, sR[5], fma(dy, sR[4], __dmul_rn(dx, sR[3]))), slo[1]);
        const double qz = __dadd_rn(fma(dz, sR[8], fma(dy, sR[7], __dmul_rn(dx, sR[6]))), slo[2]);
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
                    if (sqrt(fma(ez, ez, fma(ey, ey, __dmul_rn(ex, ex)))) < g.dist) { found = true; break; }
                }
            }
        cnt += found ? 1 : 0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xFFFFFFFFu, cnt, o);
    if ((tid & 31) == 0 && cnt) atomicAdd(&s_count, cnt);
    __syncthreads();
    return s_count;
}

// counts == nullptr: the count of pair p goes to results[p][1] as a double (mad_repeatability's in-place form)
__global__ void __launch_bounds__(128)
repeat_counts_kernel(RepeatArgs a, CloudArgs g, long long p0, int32_t* __restrict__ counts, double* __restrict__ results) {
    const long long pi = p0 + blockIdx.x;
    const int n = count_pair(a, g, pi);
    if (threadIdx.x == 0) {
        if (counts) counts[blockIdx.x] = n;
        else results[pi * 23 + 1] = (double)n;
    }
}

// The pairs [p0, p0 + gridDim.x) of a batch: each CTA counts its pair against the hi cloud and lo grid of the pair's
// structure (mad_repeat_counts_many).  lo_sorted and cell_start are those of the whole batch: cell_start holds indices
// into the concatenated cell-sorted clouds, so only the structure's cell and word offsets apply.  The structure's grid
// arguments sit in registers, not in the constant bank as in repeat_counts_kernel: left alone ptxas gives the kernel 72
// registers (7 CTAs per SM instead of 8) and it ran 13 % slower per pair on B200; capped at 64 registers (8 CTAs) it
// spills 52 bytes and runs 8 % slower (DESIGN.md section 6).
__global__ void __launch_bounds__(128, 8)
repeat_counts_many_kernel(RepeatArgs a, const long long* __restrict__ pair_off, int G, const MadCloudSeg* __restrict__ segs,
                          const double* __restrict__ hi_clouds, const double* __restrict__ lo_sorted,
                          const int32_t* __restrict__ cell_start, const uint32_t* __restrict__ near_bits, double cell,
                          double dist, long long p0, int32_t* __restrict__ counts) {
    const long long pi = p0 + blockIdx.x;
    const MadCloudSeg& s = segs[mad_segment_of([&](int k) { return pair_off[k]; }, G, pi)];
    CloudArgs g;
    g.hi_cloud = hi_clouds + 3 * s.hi_off; g.H = s.hi_n;
    g.lo_sorted = lo_sorted; g.cell_start = cell_start + s.cell_off; g.near_bits = near_bits + s.word_off;
    for (int q = 0; q < 3; ++q) { g.org[q] = s.org[q]; g.dims[q] = s.dims[q]; }
    g.cell = cell; g.dist = dist;
    const int n = count_pair(a, g, pi);
    if (threadIdx.x == 0) counts[blockIdx.x] = n;
}

// Element e = 23 pi + col of the rows; counts == nullptr: the count is read from results[e] (where repeat_counts_kernel
// left it), by the thread that then overwrites it.
__device__ __forceinline__ double row_value(const RepeatArgs& a, const double* __restrict__ pair_score,
                                            const int32_t* __restrict__ counts, const double* results, long long e, int H) {
    const long long pi = e / 23;
    const int col = (int)(e - pi * 23);
    const int h = a.pair_hi[pi], l = a.pair_lo[pi];
    if (col == 0) return pair_score[pi];
    if (col == 1) {
        const long long cnt = counts ? counts[pi] : (long long)results[e];
        return (double)(100LL * cnt) / (double)H;                          // 100 * count / l
    }
    if (col < 5) return a.lo_meta[4 * l + (col - 2)];                       // lo index, oct, main
    if (col < 8) return a.hi_meta[4 * h + (col - 5)];                       // hi index, oct, main
    if (col < 11) return a.hi_subv[3 * (long long)h + (col - 8)];
    if (col < 14) return a.lo_subv[3 * (long long)l + (col - 11)];
    return pair_rotation(a, h, l, col - 14);
}

__global__ void repeat_rows_kernel(RepeatArgs a, const double* __restrict__ pair_score, long long n_pairs,
                                   const int32_t* __restrict__ counts, int H, double* __restrict__ results) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n_pairs * 23; e += (long long)gridDim.x * blockDim.x)
        results[e] = row_value(a, pair_score, counts, results, e, H);
}

// H of each pair: the hi cloud size of the pair's structure
__global__ void repeat_rows_many_kernel(RepeatArgs a, const double* __restrict__ pair_score, long long n_pairs,
                                        const long long* __restrict__ pair_off, int G, const MadCloudSeg* __restrict__ segs,
                                        const int32_t* __restrict__ counts, double* __restrict__ results) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n_pairs * 23; e += (long long)gridDim.x * blockDim.x) {
        const int H = segs[mad_segment_of([&](int k) { return pair_off[k]; }, G, e / 23)].hi_n;
        results[e] = row_value(a, pair_score, counts, results, e, H);
    }
}

__global__ void mark_used_kernel(const int32_t* __restrict__ idx, long long n, uint8_t* __restrict__ used) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        used[idx[i]] = 1;
}

}  // namespace

// The cell of the lo grid: a little more than dist, so that no lo point within dist lies outside the 27 cells searched
// (the argument at the top of this file).
extern "C" double mad_repeat_grid_cell(double dist) { return dist * (1.0 + 0x1p-16); }

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
    g.cell = mad_repeat_grid_cell(dist); g.dist = dist;
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

namespace {

// Pair p of a batch marks its hi row and, in its structure's row of used_lo, its lo row; threads 0..G write the lower
// bounds of hi_row_off in pair_hi (pairs are hi-row-major), i.e. pair_off.
__global__ void mark_used_many_kernel(const int32_t* __restrict__ pair_hi, const int32_t* __restrict__ pair_lo, long long n,
                                      const long long* __restrict__ hi_row_off, int G, int n_lo, uint8_t* __restrict__ used_hi,
                                      uint8_t* __restrict__ used_lo, long long* __restrict__ pair_off) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n || i <= G; i += (long long)gridDim.x * blockDim.x) {
        if (i <= G) {
            long long lo = 0, hi = n;
            const long long r = hi_row_off[i];
            while (lo < hi) {
                const long long mid = (lo + hi) >> 1;
                if (pair_hi[mid] < r) lo = mid + 1; else hi = mid;
            }
            pair_off[i] = lo;
        }
        if (i < n) {
            const int h = pair_hi[i];
            const int g = mad_segment_of([&](int k) { return hi_row_off[k]; }, G, h);
            used_hi[h] = 1;
            used_lo[(long long)g * n_lo + pair_lo[i]] = 1;
        }
    }
}

int launch_counts_many(const RepeatArgs& a, const long long* pair_off, int G, const MadCloudSeg* segs, const double* hi_clouds,
                       const double* lo_sorted, const int32_t* cell_start, const uint32_t* near_bits, double dist, long long p0,
                       long long p1, int32_t* counts, void* stream) {
    MAD_CHECK_ARG(pair_off && G >= 1 && segs && hi_clouds && lo_sorted && cell_start && near_bits && dist > 0.0 && counts);
    MAD_PROF("repeat_counts_many_kernel", stream);
    repeat_counts_many_kernel<<<(unsigned)(p1 - p0), 128, 0, (cudaStream_t)stream>>>(a, pair_off, G, segs, hi_clouds, lo_sorted,
                                                                                    cell_start, near_bits,
                                                                                    mad_repeat_grid_cell(dist), dist, p0, counts);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

}  // namespace

extern "C" int mad_mark_used_many(const int32_t* pair_hi, const int32_t* pair_lo, long long n_pairs, const long long* hi_row_off,
                                  int G, int n_lo, uint8_t* used_hi, uint8_t* used_lo, long long* pair_off, void* stream) {
    MAD_CHECK_ARG(n_pairs >= 0 && G >= 1 && n_lo >= 0 && hi_row_off && pair_off);
    MAD_CHECK_ARG(n_pairs == 0 || (pair_hi && pair_lo && used_hi && used_lo));
    const long long work = std::max<long long>(n_pairs, G + 1);
    const int blocks = (int)std::min<long long>(mad_ceil_div(work, 256), (long long)mad_sm_count() * 8);
    MAD_PROF("mark_used_many_kernel", stream);
    mark_used_many_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(pair_hi, pair_lo, n_pairs, hi_row_off, G, n_lo, used_hi,
                                                                    used_lo, pair_off);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" int mad_repeat_counts_many(const int32_t* pair_hi, const int32_t* pair_lo, long long p0, long long p1,
                                      const long long* pair_off, int G, const double* hi_subv, const double* lo_subv,
                                      const int32_t* hi_meta, const int32_t* lo_meta, const double* rf_table,
                                      const double* rf_inv_table, int rf_zones, const double* hi_clouds, const double* lo_sorted,
                                      const int32_t* cell_start, const uint32_t* near_bits, const MadCloudSeg* segs, double dist,
                                      int32_t* counts, void* stream) {
    MAD_CHECK_ARG(p0 >= 0 && p0 <= p1 && p1 - p0 < (1LL << 31));
    if (p1 == p0) return MAD_OK;
    RepeatArgs a;
    int rc = fill_args(a, pair_hi, pair_lo, hi_subv, lo_subv, hi_meta, lo_meta, rf_table, rf_inv_table, rf_zones);
    if (rc != MAD_OK) return rc;
    return launch_counts_many(a, pair_off, G, segs, hi_clouds, lo_sorted, cell_start, near_bits, dist, p0, p1, counts, stream);
}

extern "C" int mad_repeat_rows_many(const int32_t* pair_hi, const int32_t* pair_lo, const double* pair_score, long long n_pairs,
                                    const long long* pair_off, int G, const double* hi_subv, const double* lo_subv,
                                    const int32_t* hi_meta, const int32_t* lo_meta, const double* rf_table,
                                    const double* rf_inv_table, int rf_zones, const int32_t* counts, const MadCloudSeg* segs,
                                    double* results, void* stream) {
    MAD_CHECK_ARG(n_pairs >= 0 && n_pairs < (1LL << 31));
    if (n_pairs == 0) return MAD_OK;
    MAD_CHECK_ARG(pair_score && pair_off && G >= 1 && counts && segs && results);
    RepeatArgs a;
    int rc = fill_args(a, pair_hi, pair_lo, hi_subv, lo_subv, hi_meta, lo_meta, rf_table, rf_inv_table, rf_zones);
    if (rc != MAD_OK) return rc;
    const int blocks = (int)std::min<long long>(mad_ceil_div(n_pairs * 23, 256), (long long)mad_sm_count() * 16);
    MAD_PROF("repeat_rows_many_kernel", stream);
    repeat_rows_many_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(a, pair_score, n_pairs, pair_off, G, segs, counts, results);
    MAD_LAUNCH_OK();
    return MAD_OK;
}
