// Keypoint detection for the MaD hot path on B200 (sm_100a):
//   a5  3x3x3 maxima of the LoG grid above a threshold, away from the borders
//       (skimage.feature.peak_local_max as called at mad/Detector.py:29)
//   a6  iterative sub-voxel Newton localisation + Hessian definiteness test
//       (Detector.check_localize, mad/Detector.py:53-123)
// One thread per interior voxel; the (rare) maxima are refined in place and appended to a
// candidate list with one atomicAdd per keypoint.  Canonical ordering (octave, value desc,
// raster index asc) and compaction of the accepted keypoints are done with CUB primitives.
#include <cub/cub.cuh>

#include "common.cuh"

namespace {

// float32 LU with partial pivoting (the algorithm of LAPACK sgetrf/sgetri behind
// np.linalg.inv on a float32 3x3), then offset = -(Hinv . G) in float32.
// Returns false when a pivot is exactly zero (numpy raises LinAlgError -> keypoint rejected).
__device__ bool newton_offset_f32(const float H[3][3], const float G[3], float off[3]) {
    float a[3][3];
    int perm[3] = {0, 1, 2};
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) a[i][j] = H[i][j];
    // LU, row pivoting
    for (int k = 0; k < 3; ++k) {
        int p = k;
        float best = fabsf(a[k][k]);
        for (int i = k + 1; i < 3; ++i) {
            const float v = fabsf(a[i][k]);
            if (v > best) { best = v; p = i; }
        }
        if (a[p][k] == 0.f) return false;
        if (p != k) {
            for (int j = 0; j < 3; ++j) { const float t = a[k][j]; a[k][j] = a[p][j]; a[p][j] = t; }
            const int t = perm[k]; perm[k] = perm[p]; perm[p] = t;
        }
        const float inv = __fdiv_rn(1.0f, a[k][k]);
        for (int i = k + 1; i < 3; ++i) {
            a[i][k] = __fmul_rn(a[i][k], inv);
            for (int j = k + 1; j < 3; ++j) a[i][j] = __fsub_rn(a[i][j], __fmul_rn(a[i][k], a[k][j]));
        }
    }
    // Hinv columns: solve L U x = P e_c
    float inv_m[3][3];
    for (int c = 0; c < 3; ++c) {
        float y[3];
        for (int i = 0; i < 3; ++i) {
            float s = (perm[i] == c) ? 1.f : 0.f;
            for (int j = 0; j < i; ++j) s = __fsub_rn(s, __fmul_rn(a[i][j], y[j]));
            y[i] = s;
        }
        for (int i = 2; i >= 0; --i) {
            float s = y[i];
            for (int j = i + 1; j < 3; ++j) s = __fsub_rn(s, __fmul_rn(a[i][j], inv_m[j][c]));
            inv_m[i][c] = __fdiv_rn(s, a[i][i]);
        }
    }
    for (int i = 0; i < 3; ++i) {
        float s = __fmul_rn(inv_m[i][0], G[0]);
        s = __fadd_rn(s, __fmul_rn(inv_m[i][1], G[1]));
        s = __fadd_rn(s, __fmul_rn(inv_m[i][2], G[2]));
        off[i] = -s;
    }
    return true;
}

// Largest eigenvalue of the symmetric 3x3 H (float64, trigonometric closed form).
__device__ double sym3_max_eig(const float Hf[3][3]) {
    const double a00 = Hf[0][0], a11 = Hf[1][1], a22 = Hf[2][2];
    const double a01 = Hf[0][1], a02 = Hf[0][2], a12 = Hf[1][2];
    const double p1 = a01 * a01 + a02 * a02 + a12 * a12;
    const double q = (a00 + a11 + a22) / 3.0;
    if (p1 == 0.0) return fmax(a00, fmax(a11, a22));
    const double p2 = (a00 - q) * (a00 - q) + (a11 - q) * (a11 - q) + (a22 - q) * (a22 - q) + 2.0 * p1;
    const double p = sqrt(p2 / 6.0);
    const double b00 = (a00 - q) / p, b11 = (a11 - q) / p, b22 = (a22 - q) / p;
    const double b01 = a01 / p, b02 = a02 / p, b12 = a12 / p;
    double r = 0.5 * (b00 * (b11 * b22 - b12 * b12) - b01 * (b01 * b22 - b12 * b02) + b02 * (b01 * b12 - b11 * b02));
    r = fmin(1.0, fmax(-1.0, r));
    const double phi = acos(r) / 3.0;
    return q + 2.0 * p * cos(phi);
}

// Phase 1: a thread owns one interior (y, z) column and walks over XS consecutive x planes
// (blockIdx.y = slab; one 32-bit divide per thread, all loads of a warp coalesced rows).
// Voxels above the threshold that equal their 3x3x3 maximum are appended as RAW candidates
// (accepted = -1) with one atomicAdd each -- they are rare (thousands per map).
constexpr int kDetectSlab = 8;
__global__ void __launch_bounds__(256)
detect_peaks_kernel(const float* __restrict__ L, int nx, int ny, int nz, int oct, int border, float thr,
                    MadKeypoint* __restrict__ cand, int cap, int* __restrict__ count) {
    const int iy = ny - 2 * border, iz = nz - 2 * border;
    const unsigned plane = (unsigned)iy * (unsigned)iz;
    const unsigned p = blockIdx.x * 256u + threadIdx.x;
    if (p >= plane) return;
    const int yy = (int)(p / (unsigned)iz);
    const int y = yy + border, z = (int)(p - (unsigned)yy * (unsigned)iz) + border;
    const long long sy = nz, sx = (long long)ny * nz;
    const int x0 = (int)blockIdx.y * kDetectSlab + border;
    const int x1 = min(nx - border, x0 + kDetectSlab);
    float vals[kDetectSlab];
#pragma unroll
    for (int q = 0; q < kDetectSlab; ++q) vals[q] = (x0 + q < x1) ? __ldg(L + (x0 + q) * sx + y * sy + z) : 0.f;
#pragma unroll
    for (int q = 0; q < kDetectSlab; ++q) {
        const float v = vals[q];
        if (!(v > thr)) continue;                      // also skips the padding of the last slab (0 <= thr)
        const int x = x0 + q;
        const long long c = x * sx + y * sy + z;
        bool is_max = true;
        for (int dx = -1; dx <= 1 && is_max; ++dx)
            for (int dy = -1; dy <= 1 && is_max; ++dy) {
                const float* row = L + c + dx * sx + dy * sy;
                if (__ldg(row - 1) > v || __ldg(row) > v || __ldg(row + 1) > v) is_max = false;
            }
        if (!is_max) continue;
        const int slot = atomicAdd(count, 1);
        if (slot < cap) {
            MadKeypoint k;
            k.vox[0] = x; k.vox[1] = y; k.vox[2] = z;
            k.oct = oct;
            k.off[0] = k.off[1] = k.off[2] = 0.f;
            k.val = v;
            k.peak[0] = x; k.peak[1] = y; k.peak[2] = z;
            k.accepted = -1;
            cand[slot] = k;
        }
    }
}

// Phase 2: one thread per raw candidate of this octave: check_localize (float32 arithmetic as
// NumPy 2 performs it, mad/Detector.py:53-123).
__global__ void __launch_bounds__(128)
detect_refine_kernel(const float* __restrict__ L, int nx, int ny, int nz, int oct,
                     MadKeypoint* __restrict__ cand, int cap, const int* __restrict__ count) {
    const long long sy = nz, sx = (long long)ny * nz;
    const int n = min(*count, cap);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        MadKeypoint k = cand[i];
        if (k.accepted != -1 || k.oct != oct) continue;
        const int x = k.peak[0], y = k.peak[1], z = k.peak[2];
        int px = x, py = y, pz = z;
        float off[3] = {0.f, 0.f, 0.f};
        float H[3][3];
        bool converged = false, singular = false;
        for (int it = 0; it < 5; ++it) {
            const float* q = L + px * sx + py * sy + pz;
            const float c2 = __fmul_rn(2.f, __ldg(q));
            const float xm = __ldg(q - sx), xp = __ldg(q + sx);
            const float ym = __ldg(q - sy), yp = __ldg(q + sy);
            const float zm = __ldg(q - 1), zp = __ldg(q + 1);
            const float xx = __fsub_rn(__fadd_rn(xm, xp), c2);
            const float yy = __fsub_rn(__fadd_rn(ym, yp), c2);
            const float zz = __fsub_rn(__fadd_rn(zm, zp), c2);
            const float xy = __fmul_rn(0.25f, __fsub_rn(__fsub_rn(__ldg(q + sx + sy), __ldg(q + sx - sy)),
                                                        __fsub_rn(__ldg(q - sx + sy), __ldg(q - sx - sy))));
            const float xz = __fmul_rn(0.25f, __fsub_rn(__fsub_rn(__ldg(q + sx + 1), __ldg(q + sx - 1)),
                                                        __fsub_rn(__ldg(q - sx + 1), __ldg(q - sx - 1))));
            const float yz = __fmul_rn(0.25f, __fsub_rn(__fsub_rn(__ldg(q + sy + 1), __ldg(q + sy - 1)),
                                                        __fsub_rn(__ldg(q - sy + 1), __ldg(q - sy - 1))));
            H[0][0] = xx; H[0][1] = xy; H[0][2] = xz;
            H[1][0] = xy; H[1][1] = yy; H[1][2] = yz;
            H[2][0] = xz; H[2][1] = yz; H[2][2] = zz;
            const float G[3] = {__fmul_rn(0.5f, __fsub_rn(xp, xm)), __fmul_rn(0.5f, __fsub_rn(yp, ym)),
                                __fmul_rn(0.5f, __fsub_rn(zp, zm))};
            if (!newton_offset_f32(H, G, off)) { singular = true; break; }
            if (fabsf(off[0]) < 0.6f && fabsf(off[1]) < 0.6f && fabsf(off[2]) < 0.6f) { converged = true; break; }
            if (off[0] < -0.6f && px - 1 > 0) px -= 1; else if (off[0] > 0.6f && px + 1 < nx - 1) px += 1;
            if (off[1] < -0.6f && py - 1 > 0) py -= 1; else if (off[1] > 0.6f && py + 1 < ny - 1) py += 1;
            if (off[2] < -0.6f && pz - 1 > 0) pz -= 1; else if (off[2] > 0.6f && pz + 1 < nz - 1) pz += 1;
        }
        bool ok = converged && !singular;
        if (ok && sym3_max_eig(H) > 0.0) ok = false;
        k.vox[0] = ok ? px : x; k.vox[1] = ok ? py : y; k.vox[2] = ok ? pz : z;
        k.off[0] = ok ? off[0] : 0.f; k.off[1] = ok ? off[1] : 0.f; k.off[2] = ok ? off[2] : 0.f;
        k.accepted = ok ? 1 : 0;
        cand[i] = k;
    }
}

__global__ void build_keys_kernel(const MadKeypoint* __restrict__ cand, int n, int ny0, int nz0, int ny1, int nz1,
                                  unsigned long long* __restrict__ keys, int* __restrict__ idx) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const MadKeypoint k = cand[i];
    const int ny = k.oct ? ny1 : ny0, nz = k.oct ? nz1 : nz0;
    const unsigned long long raster = ((unsigned long long)k.peak[0] * ny + k.peak[1]) * nz + k.peak[2];
    const unsigned int vb = 0x7FFFFFFFu - (__float_as_uint(k.val) & 0x7FFFFFFFu);  // value descending
    keys[i] = ((unsigned long long)(k.oct & 1) << 63) | ((unsigned long long)vb << 32) | (raster & 0xFFFFFFFFull);
    idx[i] = i;
}

__global__ void flags_kernel(const MadKeypoint* __restrict__ cand, const int* __restrict__ order, int n,
                             int* __restrict__ flags) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flags[i] = cand[order[i]].accepted;
}

__global__ void scatter_kernel(const MadKeypoint* __restrict__ cand, const int* __restrict__ order,
                               const int* __restrict__ flags, const int* __restrict__ pos, int n,
                               MadKeypoint* __restrict__ out, int* __restrict__ out_count) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (flags[i]) out[pos[i]] = cand[order[i]];
    if (i == n - 1) *out_count = pos[i] + flags[i];
}

struct KeyLess {
    __device__ __forceinline__ bool operator()(unsigned long long a, unsigned long long b) const { return a < b; }
};

// Candidate lists are small (10^3 - 10^5 entries): an 8-pass radix sort of 64-bit keys is eight launch-bound passes
// (~90 us at C2); a merge sort is one block sort plus log2(n / tile) merge passes.
constexpr int kMergeSortMax = 1 << 20;

struct SortLayout {
    size_t keys_in, keys_out, idx_in, idx_out, flags, pos, cub, total;
};

SortLayout sort_layout(int n) {
    SortLayout l;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o += mad_align_up(bytes, 256); return r; };
    const size_t nn = (size_t)(n > 0 ? n : 1);
    l.keys_in = take(nn * 8); l.keys_out = take(nn * 8);
    l.idx_in = take(nn * 4); l.idx_out = take(nn * 4);
    l.flags = take(nn * 4); l.pos = take(nn * 4);
    size_t a = 0, b = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, a, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                    (const int*)nullptr, (int*)nullptr, (int)nn);
    cub::DeviceScan::ExclusiveSum(nullptr, b, (const int*)nullptr, (int*)nullptr, (int)nn);
    size_t c = 0;
    cub::DeviceMergeSort::SortPairs(nullptr, c, (unsigned long long*)nullptr, (int*)nullptr, (int)nn, KeyLess());
    a = a > c ? a : c;
    l.cub = take(a > b ? a : b);
    l.total = o;
    return l;
}

}  // namespace

extern "C" int mad_detect(const float* log_grid, int nx, int ny, int nz, int oct, int border, float threshold,
                          MadKeypoint* cand, int cap, int* count, void* stream) {
    MAD_CHECK_ARG(log_grid && cand && count && cap > 0 && border >= 1);
    MAD_CHECK_ARG((long long)nx * ny * nz < (1ll << 32));
    if (nx <= 2 * border || ny <= 2 * border || nz <= 2 * border) return MAD_OK;  // nothing can be detected
    const int ix = nx - 2 * border, iy = ny - 2 * border, iz = nz - 2 * border;
    MAD_CHECK_ARG(ix <= 65535);
    cudaStream_t st = (cudaStream_t)stream;
    {
        dim3 grid_dim((unsigned)mad_ceil_div((long long)iy * iz, 256), (unsigned)mad_ceil_div(ix, kDetectSlab));
        MAD_PROF("detect_peaks_kernel", st);
        detect_peaks_kernel<<<grid_dim, 256, 0, st>>>(log_grid, nx, ny, nz, oct, border, threshold, cand, cap, count);
        MAD_LAUNCH_OK();
    }
    MAD_PROF("detect_refine_kernel", st);
    detect_refine_kernel<<<mad_sm_count(), 128, 0, st>>>(log_grid, nx, ny, nz, oct, cand, cap, count);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" size_t mad_sort_keypoints_workspace_bytes(int n) { return sort_layout(n).total; }

extern "C" int mad_sort_keypoints(const MadKeypoint* cand, int n, const int* dims_oct_host, MadKeypoint* out,
                                  int* out_count, void* workspace, size_t workspace_bytes, void* stream) {
    MAD_CHECK_ARG(out_count && dims_oct_host && n >= 0);
    cudaStream_t st = (cudaStream_t)stream;
    if (n == 0) {
        MAD_CUDA(cudaMemsetAsync(out_count, 0, sizeof(int), st));
        return MAD_OK;
    }
    MAD_CHECK_ARG(cand && out && workspace);
    const SortLayout l = sort_layout(n);
    MAD_CHECK_ARG(workspace_bytes >= l.total);
    char* ws = reinterpret_cast<char*>(workspace);
    auto* keys_in = reinterpret_cast<unsigned long long*>(ws + l.keys_in);
    auto* keys_out = reinterpret_cast<unsigned long long*>(ws + l.keys_out);
    int* idx_in = reinterpret_cast<int*>(ws + l.idx_in);
    int* idx_out = reinterpret_cast<int*>(ws + l.idx_out);
    int* flags = reinterpret_cast<int*>(ws + l.flags);
    int* pos = reinterpret_cast<int*>(ws + l.pos);
    const int tb = 256, nb = (int)mad_ceil_div(n, tb);
    {
        MAD_PROF("build_keys_kernel", st);
        build_keys_kernel<<<nb, tb, 0, st>>>(cand, n, dims_oct_host[1], dims_oct_host[2], dims_oct_host[4], dims_oct_host[5], keys_in, idx_in);
        MAD_LAUNCH_OK();
    }
    size_t cub_bytes = l.total - l.cub;
    if (n <= kMergeSortMax) {                                        // in place: the order ends up in idx_in
        MAD_PROF("cub_merge_sort_pairs", st);
        MAD_CUDA(cub::DeviceMergeSort::SortPairs(ws + l.cub, cub_bytes, keys_in, idx_in, n, KeyLess(), st));
        idx_out = idx_in;
    } else {
        MAD_PROF("cub_radix_sort_pairs", st);
        MAD_CUDA(cub::DeviceRadixSort::SortPairs(ws + l.cub, cub_bytes, keys_in, keys_out, idx_in, idx_out, n, 0, 64, st));
    }
    {
        MAD_PROF("flags_kernel", st);
        flags_kernel<<<nb, tb, 0, st>>>(cand, idx_out, n, flags);
        MAD_LAUNCH_OK();
    }
    cub_bytes = l.total - l.cub;
    {
        MAD_PROF("cub_exclusive_sum", st);
        MAD_CUDA(cub::DeviceScan::ExclusiveSum(ws + l.cub, cub_bytes, flags, pos, n, st));
    }
    MAD_PROF("scatter_kernel", st);
    scatter_kernel<<<nb, tb, 0, st>>>(cand, idx_out, flags, pos, n, out, out_count);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

// ---- a batch of G maps (mad_b200.pipeline.describe_many) ------------------------------------------------------------
namespace {

// cand_off[g] = candidates of the maps before g (each count clamped to cap), g = 0..G: one CTA.
__global__ void __launch_bounds__(256) cand_offsets_kernel(const int* __restrict__ counts, int G, int cap,
                                                           int* __restrict__ cand_off) {
    typedef cub::BlockScan<int, 256> Scan;
    __shared__ typename Scan::TempStorage tmp;
    int carry = 0;
    for (int g0 = 0; g0 < G; g0 += 256) {
        const int g = g0 + threadIdx.x;
        const int v = g < G ? min(counts[g], cap) : 0;
        int ex, total;
        Scan(tmp).ExclusiveSum(v, ex, total);
        if (g < G) cand_off[g] = carry + ex;
        carry += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) cand_off[G] = carry;
}

// The key of mad_sort_keypoints (build_keys_kernel) for candidate j of the packed batch, with its map's dims; the map
// order comes from the segments of the sort.  idx = the candidate's row in cand (map g's region starts at g cap).
__global__ void build_keys_many_kernel(const MadKeypoint* __restrict__ cand, int cap, const int* __restrict__ cand_off, int G,
                                       const int* __restrict__ dims, unsigned long long* __restrict__ keys,
                                       int* __restrict__ idx) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= cand_off[G]) return;
    const int g = mad_segment_of([&](int k) { return cand_off[k]; }, G, j);
    const int row = g * cap + (j - cand_off[g]);
    const MadKeypoint k = cand[row];
    const int* d = dims + 6 * g;
    const int ny = k.oct ? d[4] : d[1], nz = k.oct ? d[5] : d[2];
    const unsigned long long raster = ((unsigned long long)k.peak[0] * ny + k.peak[1]) * nz + k.peak[2];
    const unsigned int vb = 0x7FFFFFFFu - (__float_as_uint(k.val) & 0x7FFFFFFFu);  // value descending
    keys[j] = ((unsigned long long)(k.oct & 1) << 63) | ((unsigned long long)vb << 32) | (raster & 0xFFFFFFFFull);
    idx[j] = row;
}

__global__ void flags_many_kernel(const MadKeypoint* __restrict__ cand, const int* __restrict__ order, int n,
                                  int* __restrict__ flags) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= n) flags[i] = i < n ? cand[order[i]].accepted : 0;
}

__global__ void scatter_many_kernel(const MadKeypoint* __restrict__ cand, const int* __restrict__ order,
                                    const int* __restrict__ flags, const int* __restrict__ pos, int n,
                                    const int* __restrict__ cand_off, int G, MadKeypoint* __restrict__ out,
                                    int* __restrict__ kp_off) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= G) kp_off[i] = pos[cand_off[i]];
    if (i < n && flags[i]) out[pos[i]] = cand[order[i]];
}

struct SortManyLayout {
    size_t keys_in, keys_out, idx_in, idx_out, flags, pos, cand_off, cub, total;
};

SortManyLayout sort_many_layout(int n, int G) {
    SortManyLayout l;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o += mad_align_up(bytes, 256); return r; };
    const size_t nn = (size_t)(n > 0 ? n : 1);
    l.keys_in = take(nn * 8); l.keys_out = take(nn * 8);
    l.idx_in = take(nn * 4); l.idx_out = take(nn * 4);
    l.flags = take((nn + 1) * 4); l.pos = take((nn + 1) * 4);
    l.cand_off = take((size_t)(G + 1) * 4);
    size_t a = 0, b = 0;
    cub::DeviceSegmentedSort::StableSortPairs(nullptr, a, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                              (const int*)nullptr, (int*)nullptr, (int)nn, G, (const int*)nullptr,
                                              (const int*)nullptr);
    cub::DeviceScan::ExclusiveSum(nullptr, b, (const int*)nullptr, (int*)nullptr, (int)nn + 1);
    l.cub = take(a > b ? a : b);
    l.total = o;
    return l;
}

// subv of mad_feature_meta, the float64 operations of Detector.find_anchors one by one (no contraction).
__global__ void feature_meta_kernel(const MadKeypoint* __restrict__ kp, const MadOriented* __restrict__ oriented, int n,
                                    const int* __restrict__ kp_off, const int* __restrict__ ori_off, int G,
                                    const double* __restrict__ geo, int32_t* __restrict__ meta, double* __restrict__ subv) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n) return;
    const int g = mad_segment_of([&](int k) { return ori_off[k]; }, G, f);
    const MadOriented of = oriented[f];
    const MadKeypoint K = kp[kp_off[g] + of.kp];
    const double* q = geo + 5 * g;
    const double vs = q[K.oct ? 1 : 0];
    meta[4 * (long long)f + 0] = of.kp;
    meta[4 * (long long)f + 1] = K.oct;
    meta[4 * (long long)f + 2] = of.main_bin;
    meta[4 * (long long)f + 3] = of.sec_bin;
#pragma unroll
    for (int a = 0; a < 3; ++a)
        subv[3 * (long long)f + a] = __dadd_rn(__dmul_rn(__dadd_rn((double)K.vox[a], (double)K.off[a]), vs), q[2 + a]);
}

}  // namespace

extern "C" size_t mad_sort_keypoints_many_workspace_bytes(int n, int G) { return sort_many_layout(n, G).total; }

extern "C" int mad_sort_keypoints_many(const MadKeypoint* cand, int cap, const int* counts, int G, int n, const int* dims,
                                       MadKeypoint* out, int* kp_off, void* workspace, size_t workspace_bytes, void* stream) {
    MAD_CHECK_ARG(cand && counts && dims && kp_off && workspace && G >= 1 && cap >= 1 && n >= 0);
    MAD_CHECK_ARG((long long)G * cap < (1LL << 31) && n <= (long long)G * cap);
    MAD_CHECK_ARG(n == 0 || out);
    const SortManyLayout l = sort_many_layout(n, G);
    MAD_CHECK_ARG(workspace_bytes >= l.total);
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = reinterpret_cast<char*>(workspace);
    auto* keys_in = reinterpret_cast<unsigned long long*>(ws + l.keys_in);
    auto* keys_out = reinterpret_cast<unsigned long long*>(ws + l.keys_out);
    int* idx_in = reinterpret_cast<int*>(ws + l.idx_in);
    int* idx_out = reinterpret_cast<int*>(ws + l.idx_out);
    int* flags = reinterpret_cast<int*>(ws + l.flags);
    int* pos = reinterpret_cast<int*>(ws + l.pos);
    int* cand_off = reinterpret_cast<int*>(ws + l.cand_off);
    {
        MAD_PROF("cand_offsets_kernel", st);
        cand_offsets_kernel<<<1, 256, 0, st>>>(counts, G, cap, cand_off);
        MAD_LAUNCH_OK();
    }
    const int tb = 256, nb = (int)mad_ceil_div(n + 1, tb);
    if (n > 0) {
        {
            MAD_PROF("build_keys_many_kernel", st);
            build_keys_many_kernel<<<nb, tb, 0, st>>>(cand, cap, cand_off, G, dims, keys_in, idx_in);
            MAD_LAUNCH_OK();
        }
        size_t cub_bytes = l.total - l.cub;
        MAD_PROF("cub_segmented_sort_pairs", st);
        MAD_CUDA(cub::DeviceSegmentedSort::StableSortPairs(ws + l.cub, cub_bytes, keys_in, keys_out, idx_in, idx_out, n, G,
                                                           cand_off, cand_off + 1, st));
    }
    {
        MAD_PROF("flags_many_kernel", st);
        flags_many_kernel<<<nb, tb, 0, st>>>(cand, idx_out, n, flags);
        MAD_LAUNCH_OK();
    }
    {
        size_t cub_bytes = l.total - l.cub;
        MAD_PROF("cub_exclusive_sum", st);
        MAD_CUDA(cub::DeviceScan::ExclusiveSum(ws + l.cub, cub_bytes, flags, pos, n + 1, st));
    }
    MAD_PROF("scatter_many_kernel", st);
    scatter_many_kernel<<<(int)mad_ceil_div(std::max(n, G + 1), tb), tb, 0, st>>>(cand, idx_out, flags, pos, n, cand_off, G, out,
                                                                                 kp_off);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" int mad_feature_meta(const MadKeypoint* kp, const MadOriented* oriented, int n, const int* kp_off,
                                const int* ori_off, int G, const double* geo, int32_t* meta, double* subv, void* stream) {
    MAD_CHECK_ARG(kp_off && ori_off && geo && G >= 1 && n >= 0);
    if (n == 0) return MAD_OK;
    MAD_CHECK_ARG(kp && oriented && meta && subv);
    MAD_PROF("feature_meta_kernel", stream);
    feature_meta_kernel<<<(int)mad_ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(kp, oriented, n, kp_off, ori_off, G, geo,
                                                                                  meta, subv);
    MAD_LAUNCH_OK();
    return MAD_OK;
}
