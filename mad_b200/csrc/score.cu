// SURVEY.md 8f rank 4: the numeric work of get_solutions / build_assembly on HBM-resident grids.
//   * common-box reductions behind Dmap.get_CCC_with_grid (mad/Dmap.py:153-258), Dmap.get_CCC_with_dmap
//     (:260-372) and structure_utils.get_overlap (mad/structure_utils.py:163-259): ONE streaming pass over the
//     common box of two grids (8 B per voxel) yields every sum and count the three scores need;
//   * Dmap.mask_with (mad/Dmap.py:99-151);
//   * structure_utils.refine_pdb (mad/structure_utils.py:58-161): rigid-body steepest ascent of the atoms on the
//     map's gradient field, one CTA per candidate pose, the whole 500-step loop inside one launch.
// Sums are float64 and reduced in a fixed order (per-thread -> warp shuffle -> CTA -> a one-CTA finish kernel), so a
// result is reproducible from run to run.
#include <math.h>

#include <vector>

#include "common.cuh"

namespace {

constexpr int kBoxThreads = 256;
constexpr int kBoxSlots = 8;   // dot, s11, s22, s11 where b > 0, s22 where a > 0, #(a > iso & b > iso), #(a > 0 & b > 0), spare

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    return v;
}

// One thread per (y, z) column position of the common box, marching over a slab of x; z is the fastest axis of both
// grids, so a warp reads two contiguous 128 B rows per step.
__global__ void __launch_bounds__(kBoxThreads)
box_scores_kernel(const float* __restrict__ g1, int ny1, int nz1, const float* __restrict__ g2, int ny2, int nz2,
                  int x1, int y1, int z1, int x2, int y2, int z2, int ex, int ey, int ez, float iso,
                  double* __restrict__ partial) {
    const unsigned plane = (unsigned)ey * (unsigned)ez;
    const unsigned p = blockIdx.x * (unsigned)kBoxThreads + threadIdx.x;
    double acc[kBoxSlots];
#pragma unroll
    for (int k = 0; k < kBoxSlots; ++k) acc[k] = 0.0;
    if (p < plane) {
        const int j = (int)(p / (unsigned)ez), k = (int)(p - (unsigned)j * (unsigned)ez);
        const float* a_ptr = g1 + ((long long)x1 * ny1 + (y1 + j)) * nz1 + (z1 + k);
        const float* b_ptr = g2 + ((long long)x2 * ny2 + (y2 + j)) * nz2 + (z2 + k);
        const long long sa = (long long)ny1 * nz1, sb = (long long)ny2 * nz2;
        unsigned n_iso = 0, n_pos = 0;
        for (int i = blockIdx.y; i < ex; i += gridDim.y) {
            const double a = (double)__ldg(a_ptr + i * sa), b = (double)__ldg(b_ptr + i * sb);
            acc[0] += a * b;
            acc[1] += a * a;
            acc[2] += b * b;
            if (b > 0.0) acc[3] += a * a;
            if (a > 0.0) acc[4] += b * b;
            n_iso += (a > (double)iso && b > (double)iso);
            n_pos += (a > 0.0 && b > 0.0);
        }
        acc[5] = (double)n_iso;
        acc[6] = (double)n_pos;
    }
    __shared__ double red[kBoxThreads / 32][kBoxSlots];
#pragma unroll
    for (int k = 0; k < kBoxSlots; ++k) {
        const double s = warp_sum(acc[k]);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][k] = s;
    }
    __syncthreads();
    if (threadIdx.x < kBoxSlots) {
        double s = 0.0;
        for (int w = 0; w < kBoxThreads / 32; ++w) s += red[w][threadIdx.x];
        partial[((size_t)blockIdx.y * gridDim.x + blockIdx.x) * kBoxSlots + threadIdx.x] = s;
    }
}

// sum of the n_partial partials in a fixed order (per thread, warp shuffle, then the 8 warps)
__device__ __forceinline__ void box_scores_finish_cta(const double* __restrict__ partial, int n_partial, double* __restrict__ out) {
    __shared__ double red[8][kBoxSlots];
    double acc[kBoxSlots];
#pragma unroll
    for (int k = 0; k < kBoxSlots; ++k) acc[k] = 0.0;
    for (int i = threadIdx.x; i < n_partial; i += 256)
#pragma unroll
        for (int k = 0; k < kBoxSlots; ++k) acc[k] += partial[(size_t)i * kBoxSlots + k];
#pragma unroll
    for (int k = 0; k < kBoxSlots; ++k) {
        const double s = warp_sum(acc[k]);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][k] = s;
    }
    __syncthreads();
    if (threadIdx.x < kBoxSlots) {
        double s = 0.0;
        for (int w = 0; w < 8; ++w) s += red[w][threadIdx.x];
        out[threadIdx.x] = s;
    }
}

__global__ void __launch_bounds__(256)
box_scores_finish_kernel(const double* __restrict__ partial, int n_partial, double* __restrict__ out) {
    box_scores_finish_cta(partial, n_partial, out);
}

// ---- G grids against one target (mad_box_scores_many): a 1-D grid over the CTAs of every structure's partition --------
// CTA (bxi, byi) of structure g's (bx, by) partition does what CTA (bxi, byi) of box_scores_kernel's grid does for that
// box: the same columns, slabs, sums and partial slot.  (A device function shared with box_scores_kernel changed that
// kernel's instruction schedule, so its loop is restated here rather than shared.)
__global__ void __launch_bounds__(kBoxThreads)
box_scores_many_kernel(const float* __restrict__ g1, int ny1, int nz1, const MadScoreBox* __restrict__ boxes, int G, float iso,
                       double* __restrict__ partial_all) {
    const int g = mad_segment_of([&](int s) { return boxes[s].part0; }, G, (long long)blockIdx.x);
    const MadScoreBox& bx_ = boxes[g];
    const unsigned local = blockIdx.x - (unsigned)bx_.part0, gbx = (unsigned)bx_.bx, gby = (unsigned)bx_.by;
    const unsigned bxi = local % gbx, byi = local / gbx;
    const float* __restrict__ g2 = bx_.grid;
    const int ny2 = bx_.dims[1], nz2 = bx_.dims[2];
    const int x1 = bx_.box[0], y1 = bx_.box[1], z1 = bx_.box[2], x2 = bx_.box[3], y2 = bx_.box[4], z2 = bx_.box[5];
    const int ex = bx_.box[6], ey = bx_.box[7], ez = bx_.box[8];
    double* partial = partial_all + (size_t)bx_.part0 * kBoxSlots;
    const unsigned plane = (unsigned)ey * (unsigned)ez;
    const unsigned p = bxi * (unsigned)kBoxThreads + threadIdx.x;
    double acc[kBoxSlots];
#pragma unroll
    for (int k = 0; k < kBoxSlots; ++k) acc[k] = 0.0;
    if (p < plane) {
        const int j = (int)(p / (unsigned)ez), k = (int)(p - (unsigned)j * (unsigned)ez);
        const float* a_ptr = g1 + ((long long)x1 * ny1 + (y1 + j)) * nz1 + (z1 + k);
        const float* b_ptr = g2 + ((long long)x2 * ny2 + (y2 + j)) * nz2 + (z2 + k);
        const long long sa = (long long)ny1 * nz1, sb = (long long)ny2 * nz2;
        unsigned n_iso = 0, n_pos = 0;
        for (int i = byi; i < ex; i += gby) {
            const double a = (double)__ldg(a_ptr + i * sa), b = (double)__ldg(b_ptr + i * sb);
            acc[0] += a * b;
            acc[1] += a * a;
            acc[2] += b * b;
            if (b > 0.0) acc[3] += a * a;
            if (a > 0.0) acc[4] += b * b;
            n_iso += (a > (double)iso && b > (double)iso);
            n_pos += (a > 0.0 && b > 0.0);
        }
        acc[5] = (double)n_iso;
        acc[6] = (double)n_pos;
    }
    __shared__ double red[kBoxThreads / 32][kBoxSlots];
#pragma unroll
    for (int k = 0; k < kBoxSlots; ++k) {
        const double s = warp_sum(acc[k]);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][k] = s;
    }
    __syncthreads();
    if (threadIdx.x < kBoxSlots) {
        double s = 0.0;
        for (int w = 0; w < kBoxThreads / 32; ++w) s += red[w][threadIdx.x];
        partial[((size_t)byi * gbx + bxi) * kBoxSlots + threadIdx.x] = s;
    }
}

__global__ void __launch_bounds__(256)
box_scores_finish_many_kernel(const MadScoreBox* __restrict__ boxes, const double* __restrict__ partial, double* __restrict__ out) {
    const MadScoreBox& b = boxes[blockIdx.x];
    box_scores_finish_cta(partial + (size_t)b.part0 * kBoxSlots, b.bx * b.by, out + (size_t)blockIdx.x * kBoxSlots);
}

// every grid of the table cut at the isovalue in place (threshold_normalise_kernel without the division)
__global__ void __launch_bounds__(256)
threshold_many_kernel(const MadScoreBox* __restrict__ boxes, float isovalue) {
    const MadScoreBox& b = boxes[blockIdx.y];
    float* g = const_cast<float*>(b.grid);
    const long long n = (long long)b.dims[0] * b.dims[1] * b.dims[2];
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        g[i] = mad_threshold_normalise_one(g[i], isovalue, 1.f, 0);
}

__global__ void __launch_bounds__(256)
count_gt_kernel(const float* __restrict__ g, long long n, float thr, unsigned long long* __restrict__ out) {
    unsigned c = 0;
    for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += (long long)gridDim.x * 256) c += (__ldg(g + i) > thr);
    c = __reduce_add_sync(0xFFFFFFFFu, c);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, (unsigned long long)c);
}

// mad/Dmap.py:138-151: zero outside [lo, hi) on any axis, and inside wherever the mask grid is < 1e-8.
__global__ void __launch_bounds__(256)
mask_with_kernel(float* __restrict__ g1, int nx1, int ny1, int nz1, const float* __restrict__ g2, int ny2, int nz2,
                 int sx, int sy, int sz, int lx, int ly, int lz, int hx, int hy, int hz) {
    const unsigned plane = (unsigned)ny1 * (unsigned)nz1;
    const unsigned p = blockIdx.x * 256u + threadIdx.x;
    if (p >= plane) return;
    const int y = (int)(p / (unsigned)nz1), z = (int)(p - (unsigned)y * (unsigned)nz1);
    const bool in_yz = y >= ly && y < hy && z >= lz && z < hz;
    for (int x = blockIdx.y; x < nx1; x += gridDim.y) {
        const long long c = (long long)x * plane + p;
        bool keep = in_yz && x >= lx && x < hx;
        if (keep) keep = !(__ldg(g2 + ((long long)(x - sx) * ny2 + (y - sy)) * nz2 + (z - sz)) < 1e-8f);
        if (!keep) g1[c] = 0.f;
    }
}

// ---- rigid refinement ---------------------------------------------------------------------------------------
constexpr int kRefThreads = 1024;

struct RefineShared {
    double rot[9], trans[3], ct[3], m[9], stepv[3];
    double red[kRefThreads / 32][3];
    double total[3];
    double step_size;
    int batch, stop;
};

// interval i with p[i] <= x < p[i+1] (clamped to [0, n-2]) as scipy's find_indices does, from an arithmetic guess
__device__ __forceinline__ int find_interval(const double* __restrict__ p, int n, double x, double inv_h) {
    int i = (int)floor((x - p[0]) * inv_h);
    i = max(0, min(i, n - 2));
    while (i < n - 2 && x >= p[i + 1]) ++i;
    while (i > 0 && x < p[i]) --i;
    return i;
}

__device__ __forceinline__ void block_sum3(RefineShared& s, double v[3]) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const double w = warp_sum(v[k]);
        if ((threadIdx.x & 31) == 0) s.red[threadIdx.x >> 5][k] = w;
    }
    __syncthreads();
    if (threadIdx.x < 3) {
        double t = 0.0;
        for (int w = 0; w < kRefThreads / 32; ++w) t += s.red[w][threadIdx.x];
        s.total[threadIdx.x] = t;
    }
    __syncthreads();
}

// coords after "translate(-center); rotate(rot); translate(center + trans)" (mad/structure_utils.py:94-96)
__device__ __forceinline__ void pose(const double* __restrict__ init, int i, const double c[3], const RefineShared& s,
                                     double out[3]) {
    const double a0 = init[3 * i] + (-c[0]), a1 = init[3 * i + 1] + (-c[1]), a2 = init[3 * i + 2] + (-c[2]);
#pragma unroll
    for (int j = 0; j < 3; ++j)
        out[j] = fma(a2, s.rot[6 + j], fma(a1, s.rot[3 + j], a0 * s.rot[j])) + s.ct[j];
}

__global__ void __launch_bounds__(kRefThreads)
refine_kernel(const float4* __restrict__ grad, int nx, int ny, int nz, const double* __restrict__ px,
              const double* __restrict__ py, const double* __restrict__ pz, double voxsp,
              const double* __restrict__ init_all, const double* __restrict__ center_all,
              const double* __restrict__ max_dist_all, int n_atoms, int n_steps, double max_step, double min_step,
              double* __restrict__ coords_all, double* __restrict__ meta_all) {
    __shared__ RefineShared s;
    const int b = blockIdx.x, tid = threadIdx.x;
    const double* init = init_all + (size_t)b * n_atoms * 3;
    double* cur_out = coords_all + (size_t)b * n_atoms * 3;       // doubles as prev_atom_transf between batches
    const double c[3] = {center_all[3 * b], center_all[3 * b + 1], center_all[3 * b + 2]};
    const double max_dist = max_dist_all[b];
    const double ox = px[0], oy = py[0], oz = pz[0];
    // strict bounds of mad/structure_utils.py:101-103: o < x < o + n * voxsp - voxsp
    const double bx = ox + nx * voxsp - voxsp, by = oy + ny * voxsp - voxsp, bz = oz + nz * voxsp - voxsp;
    const double inv_h = 1.0 / voxsp;
    if (tid == 0) {
        for (int k = 0; k < 9; ++k) s.rot[k] = (k % 4 == 0) ? 1.0 : 0.0;
        s.trans[0] = s.trans[1] = s.trans[2] = 0.0;
        s.step_size = max_step;
        s.batch = 0;
        s.stop = 0;
    }
    for (int i = tid; i < 3 * n_atoms; i += kRefThreads) cur_out[i] = init[i];
    __syncthreads();
    int step = 0, converged = 0;
    for (; step < n_steps; ++step) {
        if (tid < 3) s.ct[tid] = c[tid] + s.trans[tid];
        __syncthreads();
        const bool translate = !(step & 1);
        double acc[3] = {0.0, 0.0, 0.0};
        int bad = 0;
        for (int i = tid; i < n_atoms; i += kRefThreads) {
            double q[3];
            pose(init, i, c, s, q);
            bad |= (isnan(q[0]) || isnan(q[1]) || isnan(q[2]));
            if (q[0] > ox && q[0] < bx && q[1] > oy && q[1] < by && q[2] > oz && q[2] < bz) {
                const int ix = find_interval(px, nx, q[0], inv_h), iy = find_interval(py, ny, q[1], inv_h),
                          iz = find_interval(pz, nz, q[2], inv_h);
                const double dx = (q[0] - px[ix]) / (px[ix + 1] - px[ix]), dy = (q[1] - py[iy]) / (py[iy + 1] - py[iy]),
                             dz = (q[2] - pz[iz]) / (pz[iz + 1] - pz[iz]);
                const double wx[2] = {1.0 - dx, dx}, wy[2] = {1.0 - dy, dy}, wz[2] = {1.0 - dz, dz};
                double g[3] = {0.0, 0.0, 0.0};
                // corner order and weight product of scipy's _evaluate_linear: ((1 * w0) * w1) * w2, value += v * w
#pragma unroll
                for (int cx = 0; cx < 2; ++cx)
#pragma unroll
                    for (int cy = 0; cy < 2; ++cy)
#pragma unroll
                        for (int cz = 0; cz < 2; ++cz) {
                            const float4 v = __ldg(grad + ((long long)(ix + cx) * ny + (iy + cy)) * nz + (iz + cz));
                            const double w = __dmul_rn(__dmul_rn(wx[cx], wy[cy]), wz[cz]);
                            g[0] = __dadd_rn(g[0], __dmul_rn((double)v.x, w));
                            g[1] = __dadd_rn(g[1], __dmul_rn((double)v.y, w));
                            g[2] = __dadd_rn(g[2], __dmul_rn((double)v.z, w));
                        }
                if (translate) {
                    acc[0] += g[0]; acc[1] += g[1]; acc[2] += g[2];
                } else {                                             // torque: cross(gradient, coords - center)
                    const double r0 = q[0] - c[0], r1 = q[1] - c[1], r2 = q[2] - c[2];
                    acc[0] += __dsub_rn(__dmul_rn(g[1], r2), __dmul_rn(g[2], r1));
                    acc[1] += __dsub_rn(__dmul_rn(g[2], r0), __dmul_rn(g[0], r2));
                    acc[2] += __dsub_rn(__dmul_rn(g[0], r1), __dmul_rn(g[1], r0));
                }
            }
        }
        if (__syncthreads_or(bad)) {                                // mad/structure_utils.py:97-98: return nan, False, step
            for (int i = tid; i < n_atoms; i += kRefThreads) {
                double q[3];
                pose(init, i, c, s, q);
                cur_out[3 * i] = q[0]; cur_out[3 * i + 1] = q[1]; cur_out[3 * i + 2] = q[2];
            }
            if (tid == 0) { meta_all[4 * b] = 0.0; meta_all[4 * b + 1] = (double)step; meta_all[4 * b + 2] = 1.0; meta_all[4 * b + 3] = s.step_size; }
            return;
        }
        block_sum3(s, acc);
        if (tid == 0) {
            const double t0 = s.total[0], t1 = s.total[1], t2 = s.total[2];
            const double inv = sqrt(t0 * t0 + t1 * t1 + t2 * t2);
            const double u0 = t0 / inv, u1 = t1 / inv, u2 = t2 / inv;       // unit_vector, mad/math_utils.py:5-13
            if (translate) {
                s.stepv[0] = u0 * s.step_size; s.stepv[1] = u1 * s.step_size; s.stepv[2] = u2 * s.step_size;
            } else {                                                         // euler_rod_mat, mad/math_utils.py:15-27
                const double angle = s.step_size / max_dist;
                const double a = cos(angle / 2.0), sn = sin(angle / 2.0);
                const double bb_ = -u0 * sn, cc_ = -u1 * sn, dd_ = -u2 * sn;
                const double aa = a * a, bb = bb_ * bb_, cc = cc_ * cc_, dd = dd_ * dd_;
                const double bc = bb_ * cc_, ad = a * dd_, ac = a * cc_, ab = a * bb_, bd = bb_ * dd_, cd = cc_ * dd_;
                s.m[0] = aa + bb - cc - dd; s.m[1] = 2 * (bc + ad);     s.m[2] = 2 * (bd - ac);
                s.m[3] = 2 * (bc - ad);     s.m[4] = aa + cc - bb - dd; s.m[5] = 2 * (cd + ab);
                s.m[6] = 2 * (bd + ac);     s.m[7] = 2 * (cd - ab);     s.m[8] = aa + dd - bb - cc;
            }
        }
        __syncthreads();
        const bool boundary = (s.batch + 1 == 4), last = (step == n_steps - 1);
        double maxn = 0.0;
        if (boundary || last) {                                     // coordinates after this step are needed
            for (int i = tid; i < n_atoms; i += kRefThreads) {
                double q[3], r[3];
                pose(init, i, c, s, q);
                if (translate) {
                    r[0] = q[0] + s.stepv[0]; r[1] = q[1] + s.stepv[1]; r[2] = q[2] + s.stepv[2];
                } else {
                    const double t0 = q[0] + (-1.0 * c[0] - s.trans[0]), t1 = q[1] + (-1.0 * c[1] - s.trans[1]),
                                 t2 = q[2] + (-1.0 * c[2] - s.trans[2]);
#pragma unroll
                    for (int j = 0; j < 3; ++j) r[j] = fma(t2, s.m[6 + j], fma(t1, s.m[3 + j], t0 * s.m[j])) + s.ct[j];
                }
                const double d0 = cur_out[3 * i] - r[0], d1 = cur_out[3 * i + 1] - r[1], d2 = cur_out[3 * i + 2] - r[2];
                maxn = fmax(maxn, sqrt(d0 * d0 + d1 * d1 + d2 * d2));
                cur_out[3 * i] = r[0]; cur_out[3 * i + 1] = r[1]; cur_out[3 * i + 2] = r[2];
            }
        }
        if (boundary) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) maxn = fmax(maxn, __shfl_xor_sync(0xFFFFFFFFu, maxn, o));
            if ((tid & 31) == 0) s.red[tid >> 5][0] = maxn;
        }
        __syncthreads();
        if (tid == 0) {
            if (translate) {
                s.trans[0] += s.stepv[0]; s.trans[1] += s.stepv[1]; s.trans[2] += s.stepv[2];
            } else {                                                 // rot_mat = rot_mat.dot(step_rot_mat)
                double n[9];
                for (int r = 0; r < 3; ++r)
                    for (int j = 0; j < 3; ++j)
                        n[3 * r + j] = fma(s.rot[3 * r + 2], s.m[6 + j], fma(s.rot[3 * r + 1], s.m[3 + j], s.rot[3 * r] * s.m[j]));
                for (int k = 0; k < 9; ++k) s.rot[k] = n[k];
            }
            s.batch += 1;
            if (s.batch == 4) {                                      // mad/structure_utils.py:141-147
                double mx = 0.0;
                for (int w = 0; w < kRefThreads / 32; ++w) mx = fmax(mx, s.red[w][0]);
                if (mx < s.step_size) s.step_size *= 0.5;
                s.batch = 0;
            }
            s.stop = (s.step_size < min_step);
        }
        __syncthreads();
        if (s.stop) { converged = 1; break; }
    }
    if (tid == 0) {
        meta_all[4 * b] = (double)converged;
        meta_all[4 * b + 1] = (double)(converged ? step : n_steps - 1);
        meta_all[4 * b + 2] = 0.0;
        meta_all[4 * b + 3] = s.step_size;
    }
}

}  // namespace

namespace {

// the (bx, by) partition of a non-empty common box: one CTA per 256 (y, z) columns, x split into slabs up to 8 CTAs per SM
void box_partition(int ex, int ey, int ez, long long* bx, long long* by) {
    *bx = mad_ceil_div((long long)ey * ez, kBoxThreads);
    *by = std::min<long long>(ex, std::max<long long>(1, (long long)mad_sm_count() * 8 / *bx));
}

}  // namespace

extern "C" size_t mad_box_scores_workspace_bytes(int ex, int ey, int ez) {
    if (ex <= 0 || ey <= 0 || ez <= 0) return 8 * sizeof(double);
    long long bx, by;
    box_partition(ex, ey, ez, &bx, &by);
    return (size_t)(bx * by) * kBoxSlots * sizeof(double);
}

extern "C" int mad_box_scores(const float* g1, int nx1, int ny1, int nz1, const float* g2, int nx2, int ny2, int nz2,
                              const int* box_host, float isovalue, double* out8, void* workspace, size_t workspace_bytes,
                              void* stream) {
    MAD_CHECK_ARG(g1 && g2 && box_host && out8 && workspace);
    const int x1 = box_host[0], y1 = box_host[1], z1 = box_host[2], x2 = box_host[3], y2 = box_host[4], z2 = box_host[5];
    const int ex = box_host[6], ey = box_host[7], ez = box_host[8];
    cudaStream_t st = (cudaStream_t)stream;
    if (ex <= 0 || ey <= 0 || ez <= 0) {                          // empty common box: every sum is zero
        MAD_CUDA(cudaMemsetAsync(out8, 0, kBoxSlots * sizeof(double), st));
        return MAD_OK;
    }
    MAD_CHECK_ARG(x1 >= 0 && y1 >= 0 && z1 >= 0 && x1 + ex <= nx1 && y1 + ey <= ny1 && z1 + ez <= nz1);
    MAD_CHECK_ARG(x2 >= 0 && y2 >= 0 && z2 >= 0 && x2 + ex <= nx2 && y2 + ey <= ny2 && z2 + ez <= nz2);
    MAD_CHECK_ARG(workspace_bytes >= mad_box_scores_workspace_bytes(ex, ey, ez));
    long long bx, by;
    box_partition(ex, ey, ez, &bx, &by);
    MAD_CHECK_ARG(bx < (1LL << 31) && by <= 65535);
    {
        MAD_PROF("box_scores_kernel", st);
        box_scores_kernel<<<dim3((unsigned)bx, (unsigned)by), kBoxThreads, 0, st>>>(
            g1, ny1, nz1, g2, ny2, nz2, x1, y1, z1, x2, y2, z2, ex, ey, ez, isovalue, static_cast<double*>(workspace));
        MAD_LAUNCH_OK();
    }
    {
        MAD_PROF("box_scores_finish_kernel", st);
        box_scores_finish_kernel<<<1, 256, 0, st>>>(static_cast<const double*>(workspace), (int)(bx * by), out8);
        MAD_LAUNCH_OK();
    }
    return MAD_OK;
}

namespace {

// bx, by and part0 of every record from its box; *n_partial = the partials of the whole batch
int score_layout(MadScoreBox* boxes, int G, long long* n_partial) {
    MAD_CHECK_ARG(boxes && n_partial && G >= 1);
    long long n = 0;
    for (int g = 0; g < G; ++g) {
        MadScoreBox& b = boxes[g];
        long long bx = 0, by = 0;
        if (b.box[6] > 0 && b.box[7] > 0 && b.box[8] > 0) box_partition(b.box[6], b.box[7], b.box[8], &bx, &by);
        MAD_CHECK_ARG(bx * by < (1LL << 31));
        b.part0 = n;
        b.bx = (int)bx;
        b.by = (int)by;
        n += bx * by;
    }
    MAD_CHECK_ARG(n < (1LL << 31));
    *n_partial = n;
    return MAD_OK;
}

// boxes_host must be the table mad_box_scores_layout laid out, every grid non-null with positive dims
int check_score_layout(const MadScoreBox* boxes_host, int G, long long* n_partial) {
    MAD_CHECK_ARG(boxes_host && G >= 1 && G <= 65535);
    std::vector<MadScoreBox> laid(boxes_host, boxes_host + G);
    const int rc = score_layout(laid.data(), G, n_partial);
    if (rc != MAD_OK) return rc;
    for (int g = 0; g < G; ++g) {
        const MadScoreBox& b = boxes_host[g];
        MAD_CHECK_ARG(laid[g].part0 == b.part0 && laid[g].bx == b.bx && laid[g].by == b.by);
        MAD_CHECK_ARG(b.grid && b.dims[0] > 0 && b.dims[1] > 0 && b.dims[2] > 0);
    }
    return MAD_OK;
}

}  // namespace

extern "C" int mad_box_scores_layout(MadScoreBox* boxes, int G, long long* n_partial) { return score_layout(boxes, G, n_partial); }

extern "C" int mad_box_scores_many(const float* g1, int nx1, int ny1, int nz1, const MadScoreBox* boxes_host, int G,
                                   const MadScoreBox* boxes, float isovalue, double* out, void* workspace,
                                   size_t workspace_bytes, void* stream) {
    MAD_CHECK_ARG(g1 && boxes && out && workspace);
    long long n_partial;
    const int rc = check_score_layout(boxes_host, G, &n_partial);
    if (rc != MAD_OK) return rc;
    for (int g = 0; g < G; ++g) {
        const MadScoreBox& b = boxes_host[g];
        const int* x = b.box;
        if (x[6] <= 0 || x[7] <= 0 || x[8] <= 0) continue;              // empty common box: its row is zero
        MAD_CHECK_ARG(x[0] >= 0 && x[1] >= 0 && x[2] >= 0 && x[0] + x[6] <= nx1 && x[1] + x[7] <= ny1 && x[2] + x[8] <= nz1);
        MAD_CHECK_ARG(x[3] >= 0 && x[4] >= 0 && x[5] >= 0 && x[3] + x[6] <= b.dims[0] && x[4] + x[7] <= b.dims[1] &&
                      x[5] + x[8] <= b.dims[2]);
        MAD_CHECK_ARG(b.by <= 65535);
    }
    MAD_CHECK_ARG(workspace_bytes >= (size_t)std::max<long long>(n_partial, 1) * kBoxSlots * sizeof(double));
    cudaStream_t st = (cudaStream_t)stream;
    if (n_partial > 0) {
        MAD_PROF("box_scores_many_kernel", st);
        box_scores_many_kernel<<<(unsigned)n_partial, kBoxThreads, 0, st>>>(g1, ny1, nz1, boxes, G, isovalue,
                                                                           static_cast<double*>(workspace));
        MAD_LAUNCH_OK();
    }
    MAD_PROF("box_scores_finish_many_kernel", st);
    box_scores_finish_many_kernel<<<G, 256, 0, st>>>(boxes, static_cast<const double*>(workspace), out);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" int mad_threshold_many(const MadScoreBox* boxes_host, int G, const MadScoreBox* boxes, float isovalue, void* stream) {
    MAD_CHECK_ARG(boxes);
    long long n_partial;
    const int rc = check_score_layout(boxes_host, G, &n_partial);
    if (rc != MAD_OK) return rc;
    long long max_n = 0;
    for (int g = 0; g < G; ++g)
        max_n = std::max(max_n, (long long)boxes_host[g].dims[0] * boxes_host[g].dims[1] * boxes_host[g].dims[2]);
    const long long cap = std::max<long long>(1, (long long)mad_sm_count() * 16 / G);
    const unsigned bx = (unsigned)std::max<long long>(1, std::min<long long>(mad_ceil_div(max_n, 256 * 4), cap));
    MAD_PROF("threshold_many_kernel", stream);
    threshold_many_kernel<<<dim3(bx, (unsigned)G), 256, 0, (cudaStream_t)stream>>>(boxes, isovalue);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" int mad_grid_count_gt(const float* grid, long long n, float thr, unsigned long long* out, void* stream) {
    MAD_CHECK_ARG(grid && out && n > 0);
    cudaStream_t st = (cudaStream_t)stream;
    MAD_CUDA(cudaMemsetAsync(out, 0, sizeof(unsigned long long), st));
    const int blocks = (int)std::min<long long>(mad_ceil_div(n, 256 * 8), (long long)mad_sm_count() * 8);
    MAD_PROF("count_gt_kernel", st);
    count_gt_kernel<<<std::max(blocks, 1), 256, 0, st>>>(grid, n, thr, out);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" int mad_mask_with(float* g1, int nx1, int ny1, int nz1, const float* g2, int nx2, int ny2, int nz2,
                             const int* shift_host, const int* lo_host, const int* hi_host, void* stream) {
    MAD_CHECK_ARG(g1 && g2 && shift_host && lo_host && hi_host && nx1 > 0 && ny1 > 0 && nz1 > 0);
    const int dims1[3] = {nx1, ny1, nz1}, dims2[3] = {nx2, ny2, nz2};
    for (int a = 0; a < 3; ++a) {
        MAD_CHECK_ARG(lo_host[a] >= 0 && hi_host[a] <= dims1[a]);
        if (hi_host[a] > lo_host[a])                                 // the kept range must lie inside the mask grid
            MAD_CHECK_ARG(lo_host[a] - shift_host[a] >= 0 && hi_host[a] - shift_host[a] <= dims2[a]);
    }
    dim3 grid_dim((unsigned)mad_ceil_div((long long)ny1 * nz1, 256), (unsigned)std::min(nx1, 64));
    MAD_PROF("mask_with_kernel", stream);
    mask_with_kernel<<<grid_dim, 256, 0, (cudaStream_t)stream>>>(g1, nx1, ny1, nz1, g2, ny2, nz2, shift_host[0], shift_host[1],
                                                                 shift_host[2], lo_host[0], lo_host[1], lo_host[2],
                                                                 hi_host[0], hi_host[1], hi_host[2]);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" int mad_refine_rigid(const float* grad4, int nx, int ny, int nz, const double* px, const double* py,
                                const double* pz, double voxsp, const double* init, const double* center,
                                const double* max_dist, int n_problems, int n_atoms, int n_steps, double max_step,
                                double min_step, double* coords_out, double* meta_out, void* stream) {
    MAD_CHECK_ARG(grad4 && px && py && pz && init && center && max_dist && coords_out && meta_out);
    MAD_CHECK_ARG(nx >= 2 && ny >= 2 && nz >= 2 && n_problems > 0 && n_atoms > 0 && n_steps > 0 && voxsp > 0.0);
    MAD_CHECK_ARG((reinterpret_cast<uintptr_t>(grad4) & 15) == 0);
    MAD_PROF("refine_kernel", stream);
    refine_kernel<<<n_problems, kRefThreads, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const float4*>(grad4), nx, ny, nz, px, py, pz, voxsp, init, center, max_dist, n_atoms, n_steps,
        max_step, min_step, coords_out, meta_out);
    MAD_LAUNCH_OK();
    return MAD_OK;
}
