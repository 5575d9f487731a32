// a7-a10: dominant orientations (Orientator.assign_orientations, mad/Orientator.py:68-110,
// step01..step05 and process_df_gradient :116-343) for B200 (sm_100a).
//
// One CTA per keypoint.  The (2r+1)^3 gradient patch is gathered once (float4 per voxel, stride
// 2 in the upsampled octave), normalised in float32 exactly as NumPy does, and kept in shared
// memory; the spherical-mask voxels vote into a shared-memory histogram over the 112 EQSP
// zones (float32 angles for the unrotated patch, float64 after a rotation, as in the reference).
// Candidate selection (80 % rule, <= 6 main / <= 6 secondary) is done in the same kernel and
// the (main, sec) pairs land in a fixed 36-slot row per keypoint: no host round trip.
#include <cub/cub.cuh>

#include "common.cuh"
#include "eqsp_zones.cuh"

namespace {

struct OctDims { int n[2][3]; };

// The batch form of the kernels below (mad_orient_many) takes its per-map arguments from a MadBatchMaps table, passed as
// the last parameter; the single-map form passes NoBatch there and reads its own grad / dims parameters.  Both forms
// run one body.
struct NoBatch { static constexpr bool kMaps = false; };

__device__ __forceinline__ int norm50(int h, int hmax) {
    return (int)((double)h / (double)hmax * 50.0);   // np.array(h / max * 50, dtype=int32)
}

// Exact (reference-arithmetic) votes of one direction; out of line, they run for the ~0.1 % of
// directions within 2e-5 rad of a zone edge (zone_fast returned -1).  They start from the RAW
// gradient and normalise it as NumPy does (float32 sqrt and divisions where magn > 1e-5,
// mad/Orientator.py:160-163).
__device__ __forceinline__ void normalise_exact(float& gx, float& gy, float& gz) {
    const float m = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(gx, gx), __fmul_rn(gy, gy)), __fmul_rn(gz, gz)));
    if (m > 1e-5f) {
        gx = __fdiv_rn(gx, m);
        gy = __fdiv_rn(gy, m);
        gz = __fdiv_rn(gz, m);
    }
}
// Unrotated patch: float32 angles against float64 bounds (mad/Orientator.py:305-334 under NumPy 2).
__device__ __noinline__ void vote_exact_f32(ZoneTab T, float gx, float gy, float gz, int* hist) {
    normalise_exact(gx, gy, gz);
    float th = (float)atan2((double)gy, (double)gx);
    if (th < 0.f) th = __fadd_rn(th, 6.2831855f);
    const float sth = __fadd_rn(th, 6.2831855f);
    const float zc = fminf(1.f, fmaxf(-1.f, gz));
    const float ph = (float)acos((double)zc);
    int z[2];
    const int nzn = zones_of(T, (double)th, (double)sth, (double)ph, z);
    if (nzn > 0) atomicAdd(&hist[z[0]], 1);
    if (nzn > 1) atomicAdd(&hist[z[1]], 1);
}
// Rotated patch: float64 throughout (the rotation matrix is float64).
__device__ __noinline__ void vote_exact_f64(ZoneTab T, const double* __restrict__ R, float gx, float gy, float gz, int* hist) {
    normalise_exact(gx, gy, gz);
    const double px = gx, py = gy, pz = gz;
    const double vx = fma(pz, R[2], fma(py, R[1], px * R[0]));
    const double vy = fma(pz, R[5], fma(py, R[4], px * R[3]));
    const double vz = fma(pz, R[8], fma(py, R[7], px * R[6]));
    double th = atan2(vy, vx);
    if (th < 0.0) th += MAD_TWO_PI;
    const double sth = th + MAD_TWO_PI;
    const double ph = acos(fmin(1.0, fmax(-1.0, vz)));
    int z[2];
    const int nzn = zones_of(T, th, sth, ph, z);
    if (nzn > 0) atomicAdd(&hist[z[0]], 1);
    if (nzn > 1) atomicAdd(&hist[z[1]], 1);
}

// Ordered compaction of the zones [lo, hi) whose flag is set into out[0..8) (ascending zone index, as
// the reference's np.where); returns the total count.  Called by every thread of the CTA (<= 8 warps).
__device__ __forceinline__ int select_zones(bool flag, int zone, int* out, int* warp_cnt) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned m = __ballot_sync(0xFFFFFFFFu, flag);
    if (lane == 0) warp_cnt[warp] = __popc(m);
    __syncthreads();
    int base = 0, total = 0;
    const int nw = blockDim.x >> 5;
    for (int w = 0; w < nw; ++w) { const int c = warp_cnt[w]; if (w < warp) base += c; total += c; }
    if (flag) {
        const int p = base + __popc(m & ((1u << lane) - 1u));
        if (p < 8) out[p] = zone;
    }
    __syncthreads();
    return total;
}

template <int NB, class Batch>
__global__ void __launch_bounds__(128)
orient_kernel(const float4* __restrict__ grad0, const float4* __restrict__ grad1, OctDims dims,
              const MadKeypoint* __restrict__ kp, int r, const char4* __restrict__ mask_off, int n_mask,
              ZoneTab T, const double* __restrict__ r1_table, int lim_main, int lim_sec,
              int32_t* __restrict__ n_ori, int32_t* __restrict__ slots, const __grid_constant__ Batch batch) {
    extern __shared__ float4 pv[];     // [n_mask] RAW gradient (x, y, z) + w: 1/|g| (fast normalisation),
                                       //          0 = no vote (|g| < 1e-5), -1 = |g| == 1e-5 exactly (exact path only)
    __shared__ int hist[128];
    __shared__ int hn0[128];
    __shared__ int cur[128];
    __shared__ int s_main[8], s_sec[8], s_wcnt[8];
    __shared__ int s_hmax, s_count;
    __shared__ ZoneFast F;

    const int tid = threadIdx.x;
    int ki = blockIdx.x, g = 0;
    if constexpr (Batch::kMaps) {          // keypoint kp_off[0] + b of the batch; none at or beyond kp_off[G]
        ki += batch.kp_off[0];
        if (ki >= batch.kp_off[batch.G]) return;
        g = mad_segment_of([&](int k) { return batch.kp_off[k]; }, batch.G, ki);
    }
    const MadKeypoint K = kp[ki];
    const int o = K.oct ? 1 : 0;
    const float4* __restrict__ grad = o ? grad1 : grad0;
    int nx = dims.n[o][0], ny = dims.n[o][1], nz = dims.n[o][2];
    if constexpr (Batch::kMaps) {
        grad = batch.m[g].grad[o];
        nx = batch.m[g].n[o][0]; ny = batch.m[g].n[o][1]; nz = batch.m[g].n[o][2];
    }
    const int s = o ? 1 : 2;
    const int cx = K.vox[0], cy = K.vox[1], cz = K.vox[2];
    // border rejection of mad/Orientator.py:129-135,149-155 (uniform over the CTA)
    if (cx - s * r < 0 || cy - s * r < 0 || cz - s * r < 0 ||
        cx + s * r + 1 > nx - 1 || cy + s * r + 1 > ny - 1 || cz + s * r + 1 > nz - 1) {
        if (tid == 0) n_ori[ki] = 0;
        return;
    }
    if (tid < 128) { hist[tid] = 0; }
    if (tid == 0) { s_hmax = 0; s_count = 0; }
    zone_fast_init(&F, T);
    __syncthreads();
    float vz_hi[NB];
    zone_fast_hi<NB>(F, vz_hi);

    // ---- step01 + first histogram (float32 angles against float64 bounds) ----
    constexpr int GB = 4;                  // gathers issued per thread before the first one is consumed
    for (int i0 = tid; i0 < n_mask; i0 += GB * blockDim.x) {
        float4 gv[GB];
#pragma unroll
        for (int u = 0; u < GB; ++u) {
            const int i = i0 + u * blockDim.x;
            gv[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i < n_mask) {
                const char4 d = mask_off[i];
                const long long idx = ((long long)(cx + s * d.x) * ny + (cy + s * d.y)) * nz + (cz + s * d.z);
                gv[u] = __ldg(grad + idx);
            }
        }
        int zf[GB];
#pragma unroll
        for (int u = 0; u < GB; ++u) {                 // branch-free: the GB chains interleave
            float4 g = gv[u];
            // squared magnitude with NumPy's float32 rounding; the 1e-5 cut-offs are decided exactly on it
            const float m2 = __fadd_rn(__fadd_rn(__fmul_rn(g.x, g.x), __fmul_rn(g.y, g.y)), __fmul_rn(g.z, g.z));
            const float rinv = mad_rsqrt_approx(fmaxf(m2, 1e-30f));
            g.w = (m2 < MAD_M2_LT) ? 0.f : ((m2 >= MAD_M2_GT) ? rinv : -1.f);
            gv[u] = g;
            zf[u] = (g.w > 0.f) ? zone_fast<NB>(F, vz_hi, g.x * rinv, g.y * rinv, g.z * rinv) : -1;
        }
#pragma unroll
        for (int u = 0; u < GB; ++u) {
            const int i = i0 + u * blockDim.x;
            if (i < n_mask) {
                pv[i] = gv[u];
                if (gv[u].w != 0.f) {
                    if (zf[u] >= 0) atomicAdd(&hist[zf[u]], 1);
                    else vote_exact_f32(T, gv[u].x, gv[u].y, gv[u].z, hist);
                }
            }
        }
    }
    __syncthreads();
    if (tid < T.n_zones) atomicMax(&s_hmax, hist[tid]);
    __syncthreads();
    const int hmax0 = s_hmax;
    if (hmax0 == 0) {                      // no votes at all: no candidates (mad/Orientator.py:336-337,181)
        if (tid == 0) n_ori[ki] = 0;
        return;
    }
    if (tid < T.n_zones) hn0[tid] = norm50(hist[tid], hmax0);
    __syncthreads();
    // main candidates: zones with > max(hn) * 0.8 where max(hn) == 50, in ascending order
    const int nmain = select_zones(tid < T.n_zones && hn0[tid] > 40, tid, s_main, s_wcnt);
    if (nmain > lim_main) {
        if (tid == 0) n_ori[ki] = 0;
        return;
    }

    for (int mi = 0; mi < nmain; ++mi) {
        const int a = s_main[mi];
        bool have = true;
        if (a != 0) {
            // ---- step03: rotate the patch so that the centre of zone a goes to +z, re-histogram (float64) ----
            if (tid < 128) hist[tid] = 0;
            if (tid == 0) s_hmax = 0;
            __syncthreads();
            const double* R = r1_table + 9 * a;
            float rf[9];
#pragma unroll
            for (int q = 0; q < 9; ++q) rf[q] = (float)R[q];
            for (int i0 = tid; i0 < n_mask; i0 += GB * blockDim.x) {
                float4 gq[GB];
                int zq[GB];
#pragma unroll
                for (int u = 0; u < GB; ++u) {
                    const int i = min(i0 + u * (int)blockDim.x, n_mask - 1);
                    const float4 g = pv[i];
                    gq[u] = g;
                    const float vx = fmaf(g.z, rf[2], fmaf(g.y, rf[1], g.x * rf[0])) * g.w;
                    const float vy = fmaf(g.z, rf[5], fmaf(g.y, rf[4], g.x * rf[3])) * g.w;
                    const float vz = fmaf(g.z, rf[8], fmaf(g.y, rf[7], g.x * rf[6])) * g.w;
                    zq[u] = (g.w > 0.f) ? zone_fast<NB>(F, vz_hi, vx, vy, vz) : -1;
                }
#pragma unroll
                for (int u = 0; u < GB; ++u) {
                    if (i0 + u * (int)blockDim.x < n_mask && gq[u].w != 0.f) {
                        if (zq[u] >= 0) atomicAdd(&hist[zq[u]], 1);
                        else vote_exact_f64(T, R, gq[u].x, gq[u].y, gq[u].z, hist);
                    }
                }
            }
            __syncthreads();
            if (tid < T.n_zones) atomicMax(&s_hmax, hist[tid]);
            __syncthreads();
            const int hm = s_hmax;
            if (hm == 0) have = false;
            else if (tid < T.n_zones) cur[tid] = norm50(hist[tid], hm);
        } else {
            if (tid < T.n_zones) cur[tid] = hn0[tid];
        }
        __syncthreads();                    // every thread has read s_hmax / written cur
        if (tid == 0) s_hmax = 0;
        __syncthreads();
        // ---- step04/05: secondary zones among 1..n_zones-2, re-normalised to their own maximum ----
        const bool inner = tid >= 1 && tid < T.n_zones - 1;
        if (have && inner) atomicMax(&s_hmax, cur[tid]);
        __syncthreads();
        const int qmax = s_hmax;
        const int ns = select_zones(have && inner && qmax > 0 && norm50(cur[tid], max(qmax, 1)) > 40, tid, s_sec, s_wcnt);
        if (tid == 0 && have && qmax > 0 && ns <= lim_sec) {
            int c = s_count;
            for (int q = 0; q < ns && c < MAD_MAX_ORI; ++q) slots[(long long)ki * MAD_MAX_ORI + c++] = a | (s_sec[q] << 16);
            s_count = c;
        }
        __syncthreads();
    }
    if (tid == 0) n_ori[ki] = s_count;
}

__global__ void compact_oriented_kernel(const int32_t* __restrict__ n_ori, const int32_t* __restrict__ slots,
                                        const int* __restrict__ pos, int n_kp, MadOriented* __restrict__ out,
                                        int cap, int* __restrict__ out_count) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_kp) return;
    const int n = n_ori[i], p = pos[i];
    for (int q = 0; q < n; ++q) {
        if (p + q < cap) {
            const int v = slots[(long long)i * MAD_MAX_ORI + q];
            MadOriented of;
            of.kp = i;
            of.main_bin = (int16_t)(v & 0xFFFF);
            of.sec_bin = (int16_t)(v >> 16);
            out[p + q] = of;
        }
    }
    if (i == n_kp - 1) *out_count = p + n;
}

}  // namespace

// Host-side cache of the spherical-mask offsets (mad/Orientator.py:38-47), one per radius.
static char4* g_mask_dev[32] = {nullptr};
static int g_mask_count[32] = {0};

static int ensure_mask(int r, const char4** dev, int* count) {
    if (r < 1 || r >= 32) return MAD_ERR_ARG;
    if (!g_mask_dev[r]) {
        const double lim = r * 1.05;
        const int side = 2 * r + 1;
        char4* host = (char4*)malloc(sizeof(char4) * side * side * side);
        int n = 0;
        for (int dx = -r; dx <= r; ++dx)
            for (int dy = -r; dy <= r; ++dy)
                for (int dz = -r; dz <= r; ++dz)
                    if (sqrt((double)(dx * dx + dy * dy + dz * dz)) <= lim) {
                        host[n].x = (signed char)dx; host[n].y = (signed char)dy; host[n].z = (signed char)dz; host[n].w = 0;
                        ++n;
                    }
        char4* d = nullptr;
        if (cudaMalloc(&d, sizeof(char4) * n) != cudaSuccess) { free(host); return MAD_ERR_CUDA; }
        if (cudaMemcpy(d, host, sizeof(char4) * n, cudaMemcpyHostToDevice) != cudaSuccess) { free(host); return MAD_ERR_CUDA; }
        free(host);
        g_mask_dev[r] = d;
        g_mask_count[r] = n;
    }
    *dev = g_mask_dev[r];
    *count = g_mask_count[r];
    return MAD_OK;
}

// mad_orient's own per-map arguments (unused by the batch form).
struct OneMapArgs {
    const float4* grad0 = nullptr;
    const float4* grad1 = nullptr;
    OctDims dims = {};
};

// One orient_kernel launch of `ctas` CTAs: the checks and the kernel choice of mad_orient, shared by mad_orient_many.
template <class Batch>
static int launch_orient(const char* what, const OneMapArgs& d, const Batch& batch, unsigned ctas, const MadKeypoint* kp, int r,
                         const MadZoneTable* zones_host, const double* r1_table, int lim_main, int lim_sec,
                         int32_t* n_ori, int32_t* slots, void* stream) {
    MAD_CHECK_ARG(zones_host->n_zones >= 3 && zones_host->n_zones <= 128 && zones_host->n_belts < 32);
    MAD_CHECK_ARG(lim_main >= 0 && lim_main <= 6 && lim_sec >= 0 && lim_sec <= 6);
    const char4* mask = nullptr;
    int n_mask = 0;
    int rc = ensure_mask(r, &mask, &n_mask);
    if (rc != MAD_OK) { mad_set_error("%s: cannot build the spherical mask for r=%d", what, r); return rc; }
    ZoneTab T;
    T.bounds = zones_host->bounds; T.belt_first = zones_host->belt_first; T.belt_phi = zones_host->belt_phi;
    T.n_zones = zones_host->n_zones; T.n_belts = zones_host->n_belts; T.fast = zones_host->fast;
    const size_t smem = (size_t)n_mask * sizeof(float4);
    if (smem > 200 * 1024) { mad_set_error("%s: patch radius %d too large", what, r); return MAD_ERR_ARG; }
    MAD_CHECK_ARG(T.n_belts >= 1 && T.n_belts <= MAD_BELT_MAX && T.n_zones <= MAD_ZONE_MAX);
    auto launch = [&](auto kernel) -> int {
        MAD_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 48 * 1024)));
        MAD_PROF("orient_kernel", stream);
        kernel<<<ctas, 128, smem, (cudaStream_t)stream>>>(      // 64 / 256 threads measured 0.75 / 0.53 ms against 0.50 at C2
            d.grad0, d.grad1, d.dims, kp, r, mask, n_mask, T, r1_table, lim_main, lim_sec, n_ori, slots, batch);
        return MAD_OK;
    };
    int lrc;
    if (T.n_belts <= 4) lrc = launch(orient_kernel<4, Batch>);
    else if (T.n_belts <= 12) lrc = launch(orient_kernel<12, Batch>);    // the 112-zone table has 10 belts
    else lrc = launch(orient_kernel<MAD_BELT_MAX, Batch>);
    if (lrc != MAD_OK) return lrc;
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" int mad_orient(const float* grad4_oct0, const float* grad4_oct1, const int* dims_oct_host,
                          const MadKeypoint* kp, int n_kp, int r, const MadZoneTable* zones_host,
                          const double* r1_table, int lim_main, int lim_sec, int32_t* n_ori, int32_t* slots,
                          void* stream) {
    MAD_CHECK_ARG(dims_oct_host && zones_host && r1_table && n_kp >= 0);
    if (n_kp == 0) return MAD_OK;
    MAD_CHECK_ARG(grad4_oct0 && grad4_oct1 && kp && n_ori && slots);
    OneMapArgs d;
    d.grad0 = reinterpret_cast<const float4*>(grad4_oct0);
    d.grad1 = reinterpret_cast<const float4*>(grad4_oct1);
    for (int o = 0; o < 2; ++o) for (int a = 0; a < 3; ++a) d.dims.n[o][a] = dims_oct_host[3 * o + a];
    return launch_orient("mad_orient", d, NoBatch(), (unsigned)n_kp, kp, r, zones_host, r1_table, lim_main, lim_sec, n_ori, slots, stream);
}

extern "C" int mad_orient_many(const uint64_t* grads_host, const int* dims_host, const int* n_cand_host, int G,
                               const MadKeypoint* kp, const int* kp_off, int r, const MadZoneTable* zones_host,
                               const double* r1_table, int lim_main, int lim_sec, int32_t* n_ori, int32_t* slots,
                               void* stream) {
    MAD_CHECK_ARG(grads_host && dims_host && n_cand_host && zones_host && r1_table && G >= 1);
    MAD_CHECK_ARG(kp && kp_off && n_ori && slots);
    for (int g0 = 0; g0 < G; g0 += kMadBatchMaps) {
        const int cnt = std::min(kMadBatchMaps, G - g0);
        long long ctas = 0;                              // the candidates of these maps bound their keypoints
        for (int i = 0; i < cnt; ++i) {
            MAD_CHECK_ARG(n_cand_host[g0 + i] >= 0);
            ctas += n_cand_host[g0 + i];
        }
        MAD_CHECK_ARG(ctas < (1LL << 31));
        if (ctas == 0) continue;
        MadBatchMaps t;
        mad_batch_maps(t, g0, cnt, grads_host, dims_host, nullptr, nullptr);
        t.kp_off = kp_off + g0;
        const int rc = launch_orient("mad_orient_many", OneMapArgs(), t, (unsigned)ctas, kp, r, zones_host, r1_table, lim_main, lim_sec,
                                     n_ori, slots, stream);
        if (rc != MAD_OK) return rc;
    }
    return MAD_OK;
}

__global__ void zone_fast_build_kernel(ZoneTab T, ZoneFast* out) {
    __shared__ ZoneFast F;
    zone_fast_init(&F, T);
    __syncthreads();
    const uint32_t* src = reinterpret_cast<const uint32_t*>(&F);
    uint32_t* dst = reinterpret_cast<uint32_t*>(out);
    for (int i = threadIdx.x; i < (int)(sizeof(ZoneFast) / 4); i += blockDim.x) dst[i] = src[i];
}

extern "C" int mad_zone_fast_build(const MadZoneTable* zones_host, void* fast_out, void* stream) {
    MAD_CHECK_ARG(zones_host && fast_out && zones_host->bounds && zones_host->belt_first && zones_host->belt_phi);
    MAD_CHECK_ARG(zones_host->n_zones >= 1 && zones_host->n_zones <= MAD_ZONE_MAX);
    MAD_CHECK_ARG(zones_host->n_belts >= 1 && zones_host->n_belts <= MAD_BELT_MAX);
    MAD_CHECK_ARG((reinterpret_cast<uintptr_t>(fast_out) & 15) == 0);
    ZoneTab T;
    T.bounds = zones_host->bounds; T.belt_first = zones_host->belt_first; T.belt_phi = zones_host->belt_phi;
    T.n_zones = zones_host->n_zones; T.n_belts = zones_host->n_belts; T.fast = nullptr;
    MAD_PROF("zone_fast_build_kernel", stream);
    zone_fast_build_kernel<<<1, 128, 0, (cudaStream_t)stream>>>(T, reinterpret_cast<ZoneFast*>(fast_out));
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" size_t mad_compact_oriented_workspace_bytes(int n_kp) {
    size_t b = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, b, (const int*)nullptr, (int*)nullptr, n_kp > 0 ? n_kp : 1);
    return mad_align_up((size_t)(n_kp > 0 ? n_kp : 1) * sizeof(int), 256) + mad_align_up(b, 256);
}

extern "C" int mad_compact_oriented(const int32_t* n_ori, const int32_t* slots, int n_kp, MadOriented* oriented,
                                    int cap, int* out_count, void* workspace, size_t workspace_bytes, void* stream) {
    MAD_CHECK_ARG(out_count && n_kp >= 0);
    cudaStream_t st = (cudaStream_t)stream;
    if (n_kp == 0) {
        MAD_CUDA(cudaMemsetAsync(out_count, 0, sizeof(int), st));
        return MAD_OK;
    }
    MAD_CHECK_ARG(n_ori && slots && oriented && workspace && cap >= 0);
    MAD_CHECK_ARG(workspace_bytes >= mad_compact_oriented_workspace_bytes(n_kp));
    int* pos = reinterpret_cast<int*>(workspace);
    char* cub_ws = reinterpret_cast<char*>(workspace) + mad_align_up((size_t)n_kp * sizeof(int), 256);
    size_t cub_bytes = workspace_bytes - mad_align_up((size_t)n_kp * sizeof(int), 256);
    {
        MAD_PROF("cub_exclusive_sum", st);
        MAD_CUDA(cub::DeviceScan::ExclusiveSum(cub_ws, cub_bytes, n_ori, pos, n_kp, st));
    }
    MAD_PROF("compact_oriented_kernel", st);
    compact_oriented_kernel<<<(int)mad_ceil_div(n_kp, 256), 256, 0, st>>>(n_ori, slots, pos, n_kp, oriented, cap, out_count);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

namespace {

// The scan input of mad_compact_oriented_many: n_ori of the batch's keypoints, 0 for the rows [kp_off[G], n_rows].
__global__ void ori_counts_many_kernel(const int32_t* __restrict__ n_ori, const int* __restrict__ kp_off, int G, int n_rows,
                                       int* __restrict__ cnt) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= n_rows) cnt[i] = i < kp_off[G] ? n_ori[i] : 0;
}

__global__ void compact_oriented_many_kernel(const int32_t* __restrict__ n_ori, const int32_t* __restrict__ slots,
                                             const int* __restrict__ pos, const int* __restrict__ kp_off, int G,
                                             MadOriented* __restrict__ out, int cap, int* __restrict__ ori_off) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= G) ori_off[i] = pos[kp_off[i]];
    if (i >= kp_off[G]) return;
    const int g = mad_segment_of([&](int k) { return kp_off[k]; }, G, i);
    const int n = n_ori[i], p = pos[i];
    for (int q = 0; q < n; ++q) {
        if (p + q < cap) {
            const int v = slots[(long long)i * MAD_MAX_ORI + q];
            MadOriented of;
            of.kp = i - kp_off[g];                       // map-local, as mad_compact_oriented writes it for the map alone
            of.main_bin = (int16_t)(v & 0xFFFF);
            of.sec_bin = (int16_t)(v >> 16);
            out[p + q] = of;
        }
    }
}

}  // namespace

extern "C" size_t mad_compact_oriented_many_workspace_bytes(int n_rows) {
    size_t b = 0;
    const int n = n_rows + 1;
    cub::DeviceScan::ExclusiveSum(nullptr, b, (const int*)nullptr, (int*)nullptr, n);
    return 2 * mad_align_up((size_t)n * sizeof(int), 256) + mad_align_up(b, 256);
}

extern "C" int mad_compact_oriented_many(const int32_t* n_ori, const int32_t* slots, int n_rows, const int* kp_off, int G,
                                         MadOriented* oriented, int cap, int* ori_off, void* workspace,
                                         size_t workspace_bytes, void* stream) {
    MAD_CHECK_ARG(kp_off && ori_off && G >= 1 && n_rows >= 0 && n_rows < (1 << 30) && cap >= 0);
    MAD_CHECK_ARG(workspace && workspace_bytes >= mad_compact_oriented_many_workspace_bytes(n_rows));
    MAD_CHECK_ARG(n_rows == 0 || (n_ori && slots && oriented));
    cudaStream_t st = (cudaStream_t)stream;
    const int n = n_rows + 1;
    const size_t arr = mad_align_up((size_t)n * sizeof(int), 256);
    int* cnt = reinterpret_cast<int*>(workspace);
    int* pos = reinterpret_cast<int*>(reinterpret_cast<char*>(workspace) + arr);
    char* cub_ws = reinterpret_cast<char*>(workspace) + 2 * arr;
    size_t cub_bytes = workspace_bytes - 2 * arr;
    {
        MAD_PROF("ori_counts_many_kernel", st);
        ori_counts_many_kernel<<<(int)mad_ceil_div(n, 256), 256, 0, st>>>(n_ori, kp_off, G, n_rows, cnt);
        MAD_LAUNCH_OK();
    }
    {
        MAD_PROF("cub_exclusive_sum", st);
        MAD_CUDA(cub::DeviceScan::ExclusiveSum(cub_ws, cub_bytes, cnt, pos, n, st));
    }
    MAD_PROF("compact_oriented_many_kernel", st);
    compact_oriented_many_kernel<<<(int)mad_ceil_div(std::max(n, G + 1), 256), 256, 0, st>>>(n_ori, slots, pos, kp_off, G,
                                                                                            oriented, cap, ori_off);
    MAD_LAUNCH_OK();
    return MAD_OK;
}
