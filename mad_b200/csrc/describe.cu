// a11/a12: 1024-bin descriptors (Descriptor.step06_distribute_subeqsp, mad/Descriptor.py:123-202)
// for B200 (sm_100a).
//
// One CTA per oriented feature.  The (2r)^3 sample lattice is rotated by inv(Rfinal) about the
// integer keypoint voxel in float64, the gradient is fetched with SciPy's nearest rule
// (half rounds DOWN) as one 16-byte load per sample, normalised in float32, rotated by Rfinal in
// float64, classified into the 16 EQSP zones (highest passing index wins, unassigned -> zone 0)
// and counted per 4x4x4 sub-block in a shared-memory histogram; the int16[1024] row is written
// with coalesced stores.  Any sample outside the grid zeroes the whole descriptor (:140-149).
#include <algorithm>

#include "common.cuh"
#include "eqsp_zones.cuh"

namespace {

struct OctDims { int n[2][3]; };

// The batch form of describe_kernel (mad_describe_many) takes its per-map arguments from a MadBatchMaps table, passed as
// the last parameter; the single-map form passes NoBatch there and reads its own grad / dims parameters.  Both forms
// run one body.
struct NoBatch { static constexpr bool kMaps = false; };

// scipy _rgi nearest rule: i = clip(floor(p), 0, n-2); idx = (p - i <= .5) ? i : i + 1 -- a half rounds
// DOWN.  For p in [0, n-1] (guaranteed by the bounds vote) this is exactly ceil(p - 0.5): p - 0.5 is
// exact for p >= 0.5 and stays in [-0.5, 0) below.
// ceil without the conversion unit: adding 1.5 * 2^52 with round-up leaves ceil(p - 0.5) in the low word (0 <= p < 2^31).
__device__ __forceinline__ int nearest_idx(double p) { return __double2loint(__dadd_ru(p - 0.5, 6755399441055744.0)); }

// Exact (reference-arithmetic) classification of one direction: float64 rotation, atan2, acos and
// the strict-inequality zone test.  Kept out of line: it runs for ~0.1 % of the samples and must
// not set the register budget of the main loop.
__device__ __noinline__ int zone_exact_dsc(ZoneTab T, const double* __restrict__ Rm, float gx, float gy, float gz) {
    const double vx0 = gx, vy0 = gy, vz0 = gz;
    const double vx = (vx0 * Rm[0] + vy0 * Rm[1]) + vz0 * Rm[2];
    const double vy = (vx0 * Rm[3] + vy0 * Rm[4]) + vz0 * Rm[5];
    const double vz = (vx0 * Rm[6] + vy0 * Rm[7]) + vz0 * Rm[8];
    double th = atan2(vy, vx);
    if (th < 0.0) th += MAD_TWO_PI;
    const double sth = th + MAD_TWO_PI;
    const double ph = acos(fmin(1.0, fmax(-1.0, vz)));
    int z[2];
    const int nzn = zones_of(T, th, sth, ph, z);
    if (nzn == 1) return z[0];
    if (nzn >= 2) return max(z[0], z[1]);           // ascending assignment: the higher index wins
    return 0;                                       // unassigned directions stay in zone 0 (:173)
}

// SIDE = 2 r known at compile time (16 for the default patch: one lattice column per thread, no tail tests) or 0 for
// any other radius.
template <int NB, int SIDE, int THREADS, class Batch>
__global__ void __launch_bounds__(THREADS, 768 / THREADS)
describe_kernel(const float4* __restrict__ grad0, const float4* __restrict__ grad1, OctDims dims,
                const MadKeypoint* __restrict__ kp, const MadOriented* __restrict__ oriented, int r,
                ZoneTab T, const double* __restrict__ rf_table, const double* __restrict__ rf_inv_table,
                int rf_zones, int16_t* __restrict__ dsc, const __grid_constant__ Batch batch) {
    __shared__ int cnt[MAD_DSC_LEN];
    __shared__ ZoneFast F;
    __shared__ double xt[32][3];           // lx * Ri[0], lx * Ri[3], lx * Ri[6] for the 2 r values of lx
    const int tid = threadIdx.x;
    if (SIDE) r = SIDE / 2;
    const MadOriented of = oriented[blockIdx.x];
    int row = of.kp, g = 0;
    if constexpr (Batch::kMaps) {          // feature b of the launch is in the map g with row0 <= b; kp counts from kp0
        g = mad_segment_of([&](int k) { return batch.m[k].row0; }, batch.G, blockIdx.x);
        row += batch.m[g].kp0;
    }
    const MadKeypoint K = kp[row];
    const int o = K.oct ? 1 : 0;
    const float4* __restrict__ grad = o ? grad1 : grad0;
    int nx = dims.n[o][0], ny = dims.n[o][1], nz = dims.n[o][2];
    if constexpr (Batch::kMaps) {
        grad = batch.m[g].grad[o];
        nx = batch.m[g].n[o][0]; ny = batch.m[g].n[o][1]; nz = batch.m[g].n[o][2];
    }
    const long long tab = ((long long)of.main_bin * rf_zones + of.sec_bin) * 9;
    double Ri[9];
    float Rmf[9];
#pragma unroll
    for (int q = 0; q < 9; ++q) { Ri[q] = rf_inv_table[tab + q]; Rmf[q] = (float)rf_table[tab + q]; }
    const int side = SIDE ? SIDE : 2 * r;
    const int c1 = r / 2, c2 = r, c3 = (3 * r) / 2;
    const double cx = K.vox[0], cy = K.vox[1], cz = K.vox[2];
    const double u0 = o ? (-(double)r + 0.5) : (double)(-2 * r + 1);
    const double du = o ? 1.0 : 2.0;

    for (int q = tid; q < MAD_DSC_LEN; q += blockDim.x) cnt[q] = 0;
    zone_fast_init(&F, T);
    if (tid < side) {
        const double lx = u0 + du * tid;
        xt[tid][0] = lx * Ri[0]; xt[tid][1] = lx * Ri[3]; xt[tid][2] = lx * Ri[6];
    }

    // Whole-patch bounds vote (RegularGridInterpolator bounds_error, mad/Descriptor.py:140-149).
    // Each coordinate ((lx*a + ly*b) + lz*c) + centre is a monotone function of lx, ly and lz in
    // IEEE arithmetic (rounding is monotone), so its extremes over the lattice are taken at the 8
    // corners: testing them is exactly equivalent to testing all (2r)^3 samples.
    int bad = 0;
    if (tid < 8) {
        const double lx = u0 + du * ((tid & 1) ? side - 1 : 0);
        const double ly = u0 + du * ((tid & 2) ? side - 1 : 0);
        const double lz = u0 + du * ((tid & 4) ? side - 1 : 0);
        const double px = ((lx * Ri[0] + ly * Ri[1]) + lz * Ri[2]) + cx;
        const double py = ((lx * Ri[3] + ly * Ri[4]) + lz * Ri[5]) + cy;
        const double pz = ((lx * Ri[6] + ly * Ri[7]) + lz * Ri[8]) + cz;
        bad = (px < 0.0 || px > (double)(nx - 1) || py < 0.0 || py > (double)(ny - 1) || pz < 0.0 || pz > (double)(nz - 1));
    }
    const int s_bad = __syncthreads_or(bad);       // also publishes cnt = 0, the zone tables and xt
    float vz_hi[NB];
    zone_fast_hi<NB>(F, vz_hi);
    int16_t* out = dsc + (long long)blockIdx.x * MAD_DSC_LEN;
    if (s_bad) {
        for (int q = tid; q < MAD_DSC_LEN; q += blockDim.x) out[q] = 0;
        return;
    }

    // A thread owns one (j, k) column of the lattice and walks along i (blockDim = side^2 when
    // side = 16): the j / k terms of the coordinate sums and the y / z sub-block are per-thread
    // constants.  Samples are handled in batches of GB: all gathers of a batch are issued before any
    // is consumed, and every phase is a separate branch-free loop over the batch so that the GB
    // dependency chains (normalise, rotate, atan2f, zone) interleave in the pipeline.
    constexpr int GB = 4;
    const int plane = side * side;
    for (int c = tid; c < plane; c += blockDim.x) {
        const int k = c % side, j = c / side;
        const double ly = u0 + du * j, lz = u0 + du * k;
        const double ay0 = ly * Ri[1], ay1 = ly * Ri[4], ay2 = ly * Ri[7];
        const double az0 = lz * Ri[2], az1 = lz * Ri[5], az2 = lz * Ri[8];
        const int by = (j >= c1) + (j >= c2) + (j >= c3);
        const int bz = (k >= c1) + (k >= c2) + (k >= c3);
        const int bin_jk = (16 * by + bz) * T.n_zones;
#pragma unroll 1                                                  // the unrolled walk (4096 SASS lines) misses the instruction cache
        for (int i0 = 0; i0 < (SIDE ? SIDE : side); i0 += GB) {
            float4 gv[GB];
#pragma unroll
            for (int u = 0; u < GB; ++u) {
                const int i = SIDE ? i0 + u : min(i0 + u, side - 1);
                const double px = ((xt[i][0] + ay0) + az0) + cx;
                const double py = ((xt[i][1] + ay1) + az1) + cy;
                const double pz = ((xt[i][2] + ay2) + az2) + cz;
                const int ix = nearest_idx(px), iy = nearest_idx(py), iz = nearest_idx(pz);
                gv[u] = __ldg(grad + (unsigned)((ix * ny + iy) * nz + iz));     // < 2^31 voxels (checked at launch)
            }
            float vx[GB], vy[GB], vz[GB];
            bool valid[GB];
#pragma unroll
            for (int u = 0; u < GB; ++u) {
                const float4 g = gv[u];
                // squared magnitude with the reference's float32 rounding; m < 1e-5 (zone -1, never counted,
                // :190) is decided exactly on m2; the fast path normalises with rsqrt (margin-covered)
                const float m2 = __fadd_rn(__fadd_rn(__fmul_rn(g.x, g.x), __fmul_rn(g.y, g.y)), __fmul_rn(g.z, g.z));
                valid[u] = (SIDE || i0 + u < side) && !(m2 < MAD_M2_LT);
                const float rinv = mad_rsqrt_approx(fmaxf(m2, 1e-30f));
                vx[u] = ((g.x * Rmf[0] + g.y * Rmf[1]) + g.z * Rmf[2]) * rinv;
                vy[u] = ((g.x * Rmf[3] + g.y * Rmf[4]) + g.z * Rmf[5]) * rinv;
                vz[u] = ((g.x * Rmf[6] + g.y * Rmf[7]) + g.z * Rmf[8]) * rinv;
            }
            int zone[GB];
#pragma unroll
            for (int u = 0; u < GB; ++u) zone[u] = zone_fast<NB>(F, vz_hi, vx[u], vy[u], vz[u]);
#pragma unroll
            for (int u = 0; u < GB; ++u) {
                if (valid[u]) {
                    // directions within 2e-5 rad of a zone edge take the exact path: float32 sqrt and
                    // divisions as NumPy does them (m > 1e-12 holds since m >= 1e-5), float64 rotation
                    if (zone[u] < 0) {
                        const float4 g = gv[u];
                        const float m = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(g.x, g.x), __fmul_rn(g.y, g.y)), __fmul_rn(g.z, g.z)));
                        zone[u] = zone_exact_dsc(T, rf_table + tab, __fdiv_rn(g.x, m), __fdiv_rn(g.y, m), __fdiv_rn(g.z, m));
                    }
                    const int i = i0 + u;
                    const int bx = (i >= c1) + (i >= c2) + (i >= c3);
                    atomicAdd(&cnt[bin_jk + 4 * bx * T.n_zones + zone[u]], 1);
                }
            }
        }
    }
    __syncthreads();
    for (int q = tid; q < MAD_DSC_LEN; q += blockDim.x) out[q] = (int16_t)cnt[q];
}

}  // namespace

// mad_describe's own per-map arguments (unused by the batch form).
struct OneMapArgs {
    const float4* grad0 = nullptr;
    const float4* grad1 = nullptr;
    OctDims dims = {};
};

// One describe_kernel launch of `ctas` CTAs: the checks and the kernel choice of mad_describe, shared by
// mad_describe_many.
template <class Batch>
static int launch_describe(const OneMapArgs& d, const Batch& batch, unsigned ctas, const MadKeypoint* kp, const MadOriented* oriented, int r,
                           const MadZoneTable* zones_host, const double* rf_table, const double* rf_inv_table, int rf_zones,
                           int16_t* dsc, void* stream) {
    MAD_CHECK_ARG(zones_host->n_zones * 64 == MAD_DSC_LEN);   // 64 sub-blocks x 16 zones
    MAD_CHECK_ARG(r >= 2 && r <= 16 && rf_zones > 0);
    ZoneTab T;
    T.bounds = zones_host->bounds; T.belt_first = zones_host->belt_first; T.belt_phi = zones_host->belt_phi;
    T.n_zones = zones_host->n_zones; T.n_belts = zones_host->n_belts; T.fast = zones_host->fast;
    MAD_CHECK_ARG(T.n_belts >= 1 && T.n_belts <= MAD_BELT_MAX && T.n_zones <= MAD_ZONE_MAX);
    MAD_PROF("describe_kernel", stream);
    auto launch = [&](auto kernel, int threads) {
        kernel<<<ctas, threads, 0, (cudaStream_t)stream>>>(d.grad0, d.grad1, d.dims, kp, oriented, r, T, rf_table, rf_inv_table,
                                                           rf_zones, dsc, batch);
    };
    // 128-thread CTAs (two lattice columns per thread, 6 CTAs per SM) measured 0.93 ms at C2 against 1.04 ms with 256
    // threads and 1.01 ms with 64: smaller CTAs lose less time at the two barriers of a feature
    if (T.n_belts <= 4 && r == 8) launch(describe_kernel<4, 16, 128, Batch>, 128);  // default: 16 zones (caps + 2 belts), patch 16
    else if (T.n_belts <= 4) launch(describe_kernel<4, 0, 256, Batch>, 256);
    else launch(describe_kernel<MAD_BELT_MAX, 0, 256, Batch>, 256);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" int mad_describe(const float* grad4_oct0, const float* grad4_oct1, const int* dims_oct_host,
                            const MadKeypoint* kp, const MadOriented* oriented, int n_oriented, int r,
                            const MadZoneTable* zones_host, const double* rf_table, const double* rf_inv_table,
                            int rf_zones, int16_t* dsc, void* stream) {
    MAD_CHECK_ARG(dims_oct_host && zones_host && n_oriented >= 0);
    if (n_oriented == 0) return MAD_OK;
    MAD_CHECK_ARG(grad4_oct0 && grad4_oct1 && kp && oriented && rf_table && rf_inv_table && dsc);
    OneMapArgs d;
    d.grad0 = reinterpret_cast<const float4*>(grad4_oct0);
    d.grad1 = reinterpret_cast<const float4*>(grad4_oct1);
    for (int o = 0; o < 2; ++o) for (int a = 0; a < 3; ++a) d.dims.n[o][a] = dims_oct_host[3 * o + a];
    for (int o = 0; o < 2; ++o)                                  // 32-bit voxel indices in the gather
        MAD_CHECK_ARG((long long)d.dims.n[o][0] * d.dims.n[o][1] * d.dims.n[o][2] < (1LL << 31));
    return launch_describe(d, NoBatch(), (unsigned)n_oriented, kp, oriented, r, zones_host, rf_table, rf_inv_table, rf_zones, dsc, stream);
}

extern "C" int mad_describe_many(const uint64_t* grads_host, const int* dims_host, const int* kp_off_host,
                                 const int* ori_off_host, int G, const MadKeypoint* kp, const MadOriented* oriented, int r,
                                 const MadZoneTable* zones_host, const double* rf_table, const double* rf_inv_table,
                                 int rf_zones, int16_t* dsc, void* stream) {
    MAD_CHECK_ARG(grads_host && dims_host && kp_off_host && ori_off_host && zones_host && G >= 1);
    MAD_CHECK_ARG(ori_off_host[0] == 0);
    for (int g = 0; g < G; ++g) {
        MAD_CHECK_ARG(ori_off_host[g + 1] >= ori_off_host[g] && kp_off_host[g + 1] >= kp_off_host[g]);
        for (int o = 0; o < 2; ++o)                              // 32-bit voxel indices in the gather
            MAD_CHECK_ARG((long long)dims_host[6 * g + 3 * o] * dims_host[6 * g + 3 * o + 1] * dims_host[6 * g + 3 * o + 2] < (1LL << 31));
    }
    if (ori_off_host[G] == 0) return MAD_OK;
    MAD_CHECK_ARG(kp && oriented && rf_table && rf_inv_table && dsc);
    for (int g0 = 0; g0 < G; g0 += kMadBatchMaps) {
        const int cnt = std::min(kMadBatchMaps, G - g0);
        const int d0 = ori_off_host[g0], d = ori_off_host[g0 + cnt] - d0;
        if (d == 0) continue;
        MadBatchMaps t;
        mad_batch_maps(t, g0, cnt, grads_host, dims_host, kp_off_host, ori_off_host);
        t.kp_off = nullptr;
        const int rc = launch_describe(OneMapArgs(), t, (unsigned)d, kp, oriented + d0, r, zones_host, rf_table, rf_inv_table, rf_zones,
                                       dsc + (long long)d0 * MAD_DSC_LEN, stream);
        if (rc != MAD_OK) return rc;
    }
    return MAD_OK;
}
