// a15: descriptor matching on the 5th-generation tensor cores (tcgen05 + TMEM + TMA), sm_100a.
//
// Replaces  preds = np.dot(hi_unit, lo_unit.T); np.where(preds > cc)  (mad/MaD.py:416-424).
// Descriptor entries are small non-negative integers, so the raw dot product is computed EXACTLY
// by one fp16 x fp16 -> fp32 UMMA pass while entries are <= 2048 (products <= 2^22) and every dot product
// is <= 2^24 -- guaranteed by max |hi|^2 * max |lo|^2 <= 2^48, which the dispatch checks; the cosine
// dot / sqrt(n_i n_j) is then evaluated in float64 from exact integers, only for the pairs an
// fp32 pre-filter cannot rule out.  The M x N score matrix is never written.
//
// Kernel shape (one CTA = one 128-row hi tile x one contiguous range of 256-column lo tiles):
//   warp 0      TMA producer   : cp.async.bulk.tensor (128B swizzle) of the hi/lo k-blocks into a
//                                4-stage shared-memory ring, mbarrier complete_tx
//   warp 1      MMA issuer     : tcgen05.mma.cta_group::1.kind::f16, M=128 N=256 K=16, fp32
//                                accumulators in TMEM (2 x 256 columns, double buffered)
//   warp 2      TMEM allocator
//   warps 4..7  epilogue       : tcgen05.ld (32 lanes x 32 columns), thread = one hi row;
//                                count / fill / top-k with the row state kept in registers
// Rows of the output are produced in ascending lo order by construction (each thread sweeps
// its row left to right), so the pair list comes out in np.where's row-major order without a sort.
#include <cuda.h>
#include <cuda_fp16.h>

#include "common.cuh"
#include "match_common.cuh"

namespace {

constexpr int BM = 128;           // hi rows per CTA (UMMA M)
constexpr int BN = 256;           // lo rows per tile (UMMA N)
constexpr int BK = 64;            // fp16 elements per k-block = one 128-byte swizzle row
constexpr int UK = 16;            // UMMA K for 16-bit inputs
constexpr int STAGES = 4;
constexpr int KBLOCKS = MAD_DSC_LEN / BK;
constexpr uint32_t A_BYTES = BM * BK * 2;
constexpr uint32_t B_BYTES = BN * BK * 2;
constexpr uint32_t STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int THREADS = 256;
constexpr uint32_t TMEM_COLS = 512;
// dynamic smem: [1024 align slack][STAGES x (A|B)][barriers + tmem ptr][rb staging 2 x 256 floats]
constexpr size_t SMEM_BYTES = 1024 + (size_t)STAGES * STAGE_BYTES + 256 + 2 * BN * sizeof(float);

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
    } while (!done);
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major operand tile in shared memory, rows of 128 bytes, 128B swizzle (what TMA wrote):
// start address >> 4, LBO = 1 (unused for swizzled K-major), SBO = 8 rows x 128 B, version 1
// (Blackwell), layout type 2 = SWIZZLE_128B.
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024u >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// kind::f16 instruction descriptor: D = f32 (bits 4-5 = 1), A = B = f16 (0), both K-major,
// N >> 3 at bits 17-22, M >> 4 at bits 24-28.
constexpr uint32_t kIdesc = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);

struct MatchArgs {
    int M, N, S;                  // rows of hi / lo, number of lo segments
    int tiles_per_seg;            // 256-column tiles per segment
    const int32_t* hi_n2;
    const int32_t* lo_n2;
    double cc;
    int mode;                     // 0 count, 1 fill, 2 top-k
    int32_t* seg_count;           // [M][S]
    const int64_t* seg_offset;    // [M][S]
    int32_t* pair_hi;
    int32_t* pair_lo;
    double* pair_score;
    int k, lo_index_base;
    uint32_t stage_tx_bytes;      // bytes TMA delivers per stage (lo box may have < 256 rows)
    int32_t* topk_idx;            // [S][M][k]
    double* topk_score;
};

__global__ void __launch_bounds__(THREADS, 1)
match_tc_kernel(const __grid_constant__ CUtensorMap map_hi, const __grid_constant__ CUtensorMap map_lo, MatchArgs a) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;                 // SWIZZLE_128B tiles need 1024-byte alignment
    uint8_t* gen = smem_raw + (base - raw);
    const uint32_t bars = base + STAGES * STAGE_BYTES;
    auto full_bar = [&](int s) { return bars + 8u * s; };
    auto empty_bar = [&](int s) { return bars + 8u * (STAGES + s); };
    auto tfull_bar = [&](int q) { return bars + 8u * (2 * STAGES + q); };
    auto tempty_bar = [&](int q) { return bars + 8u * (2 * STAGES + 2 + q); };
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(gen + STAGES * STAGE_BYTES + 8 * (2 * STAGES + 4));
    float* s_rb = reinterpret_cast<float*>(gen + STAGES * STAGE_BYTES + 256);   // [2][BN]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = blockIdx.x * BM;
    const int seg = blockIdx.y;
    const int n_tiles_total = (a.N + BN - 1) / BN;
    const int t_begin = seg * a.tiles_per_seg;
    const int t_end = min(n_tiles_total, t_begin + a.tiles_per_seg);

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        for (int q = 0; q < 2; ++q) { mbar_init(tfull_bar(q), 1); mbar_init(tempty_bar(q), 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===================== TMA producer (one elected lane) =====================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int t = t_begin; t < t_end; ++t) {
                for (int kb = 0; kb < KBLOCKS; ++kb) {
                    mbar_wait(empty_bar(stage), phase ^ 1u);
                    mbar_expect_tx(full_bar(stage), a.stage_tx_bytes);
                    const uint32_t sa = base + stage * STAGE_BYTES;
                    tma_load_2d(sa, &map_hi, full_bar(stage), kb * BK, m0);
                    tma_load_2d(sa + A_BYTES, &map_lo, full_bar(stage), kb * BK, t * BN);
                    if (++stage == STAGES) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (one thread) =====================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            int it = 0;
            for (int t = t_begin; t < t_end; ++t, ++it) {
                const int acc = it & 1;
                const uint32_t acc_phase = (uint32_t)(it >> 1) & 1u;
                mbar_wait(tempty_bar(acc), acc_phase ^ 1u);          // epilogue has drained this accumulator
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
                for (int kb = 0; kb < KBLOCKS; ++kb) {
                    mbar_wait(full_bar(stage), phase);
                    tc_fence_after();
                    const uint32_t sa = base + stage * STAGE_BYTES;
                    const uint64_t da = umma_smem_desc(sa);
                    const uint64_t db = umma_smem_desc(sa + A_BYTES);
#pragma unroll
                    for (int kk = 0; kk < BK / UK; ++kk) {
                        // advance 16 fp16 = 32 bytes inside the 128-byte swizzle row: +2 in 16-byte units
                        umma_f16(d_tmem, da + (uint64_t)(2 * kk), db + (uint64_t)(2 * kk), kIdesc, (kb | kk) ? 1u : 0u);
                    }
                    umma_commit(empty_bar(stage));                   // smem slot free when these MMAs retire
                    if (++stage == STAGES) { stage = 0; phase ^= 1u; }
                }
                umma_commit(tfull_bar(acc));                         // accumulator complete
            }
        }
    } else if (warp >= 4) {
        // ===================== epilogue: thread = one hi row =====================
        const int q = warp & 3;                                      // TMEM lane quadrant of this warp
        const int et = threadIdx.x - 128;                            // 0..127
        const int row = m0 + q * 32 + lane;
        const bool row_ok = row < a.M;
        const int n2a_i = row_ok ? a.hi_n2[row] : 0;
        const double n2a = (double)n2a_i;
        const float ra = n2a_i > 0 ? (float)(1.0 / sqrt(n2a)) : 0.f;
        const float cc_lo = (float)a.cc - 4e-6f;                     // fp32 pre-filter bound (|approx - exact| < 1e-6)
        int cnt = 0;
        long long wpos = 0;
        if (a.mode == 1 && row_ok) wpos = a.seg_offset[(long long)row * a.S + seg];
        double bs[MAD_TOPK_MAX];
        int bi[MAD_TOPK_MAX];
        float thr = -1.f;                                            // fp32 bound of the current k-th best
        if (a.mode == 2) {
#pragma unroll
            for (int i = 0; i < MAD_TOPK_MAX; ++i) { bs[i] = -INFINITY; bi[i] = -1; }
        }
        int it = 0;
        for (int t = t_begin; t < t_end; ++t, ++it) {
            const int acc = it & 1;
            const uint32_t acc_phase = (uint32_t)(it >> 1) & 1u;
            const int n0 = t * BN;
            // 1/sqrt(n_j) of this tile's columns (0 beyond N or for zero descriptors)
            float* rb = s_rb + acc * BN;
            for (int c = et; c < BN; c += 128) {
                const int col = n0 + c;
                int n2 = 0;
                if (col < a.N) n2 = __ldg(a.lo_n2 + col);
                rb[c] = n2 > 0 ? (float)(1.0 / sqrt((double)n2)) : 0.f;
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");
            mbar_wait(tfull_bar(acc), acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BN);
#pragma unroll 1
            for (int c0 = 0; c0 < BN; c0 += 32) {
                uint32_t v[32];
                tmem_ld32(taddr + (uint32_t)c0, v);
                tmem_ld_wait();
                if (row_ok) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float dotf = __uint_as_float(v[j]);
                        const float approx = dotf * ra * rb[c0 + j];
                        if (a.mode == 2) {
                            if (approx >= thr) {
                                const int col = n0 + c0 + j;
                                if (col < a.N) {
                                    const double s = mad_score((int)dotf, n2a, (double)__ldg(a.lo_n2 + col));
                                    mad_topk_insert(bs, bi, a.k, s, a.lo_index_base + col);
                                    const double kth = bs[a.k - 1];
                                    thr = (bi[a.k - 1] < 0) ? -1.f : (float)kth - 4e-6f;
                                }
                            }
                        } else if (approx > cc_lo) {
                            const int col = n0 + c0 + j;
                            if (col < a.N) {
                                const double s = mad_score((int)dotf, n2a, (double)__ldg(a.lo_n2 + col));
                                if (s > a.cc) {
                                    if (a.mode == 1) {
                                        a.pair_hi[wpos] = row;
                                        a.pair_lo[wpos] = col;
                                        a.pair_score[wpos] = s;
                                        ++wpos;
                                    }
                                    ++cnt;
                                }
                            }
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty_bar(acc));             // 4 arrivals free the accumulator
        }
        if (row_ok) {
            if (a.mode == 0) a.seg_count[(long long)row * a.S + seg] = cnt;
            if (a.mode == 2) {
                const long long o = ((long long)seg * a.M + row) * a.k;
                for (int i = 0; i < a.k; ++i) { a.topk_idx[o + i] = bi[i]; a.topk_score[o + i] = bs[i]; }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// [rows_padded][1024] fp16 row-major; box = 64 (k) x box_rows, 128-byte swizzle, OOB rows read as zero.
int make_map(CUtensorMap* map, const void* ptr, int rows_padded, int box_rows) {
    EncodeTiledFn enc = get_encode();
    if (!enc) {
        mad_set_error("mad_match: cuTensorMapEncodeTiled is not available from the CUDA driver");
        return MAD_ERR_NODEVICE;
    }
    cuuint64_t dims[2] = {(cuuint64_t)MAD_DSC_LEN, (cuuint64_t)rows_padded};
    cuuint64_t strides[1] = {(cuuint64_t)MAD_DSC_LEN * 2};
    cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        mad_set_error("mad_match: cuTensorMapEncodeTiled failed (%d)", (int)r);
        return MAD_ERR_CUDA;
    }
    return MAD_OK;
}

}  // namespace

// Number of lo segments the tensor-core kernel splits the reference axis into so that a small
// number of hi tiles still fills the 148 SMs.  Deterministic in (M, N, sm_count).
int mad_match_tc_segments(int M, int N) {
    if (M <= 0 || N <= 0) return 1;
    const int m_tiles = (int)mad_ceil_div(M, BM);
    const int n_tiles = (int)mad_ceil_div(N, BN);
    const int sms = mad_sm_count();
    int s = (int)mad_ceil_div(sms, m_tiles);
    if (m_tiles >= sms) s = 1;
    s = std::max(1, std::min(s, n_tiles));
    const int per = (int)mad_ceil_div(n_tiles, s);
    return (int)mad_ceil_div(n_tiles, per);          // no empty segments
}

int mad_match_tc(const void* hi_half, int M, int M_pad, const void* lo_half, int N, int N_pad, const int32_t* hi_n2,
                 const int32_t* lo_n2, double cc, int mode, int S, int32_t* seg_count, const int64_t* seg_offset,
                 int32_t* pair_hi, int32_t* pair_lo, double* pair_score, int k, int lo_index_base, int32_t* topk_idx,
                 double* topk_score, cudaStream_t st) {
    int dev = 0, major = 0;
    MAD_CUDA(cudaGetDevice(&dev));
    MAD_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
    if (major != 10) {
        mad_set_error("mad_match: the tcgen05 kernel needs an sm_100 device (found compute capability %d.x)", major);
        return MAD_ERR_NODEVICE;
    }
    CUtensorMap map_hi, map_lo;
    int rc = make_map(&map_hi, hi_half, M_pad, BM);
    if (rc != MAD_OK) return rc;
    const int lo_box = std::min(BN, N_pad);
    rc = make_map(&map_lo, lo_half, N_pad, lo_box);
    if (rc != MAD_OK) return rc;
    MatchArgs a;
    a.stage_tx_bytes = A_BYTES + (uint32_t)lo_box * BK * 2;
    a.M = M; a.N = N; a.S = S;
    const int n_tiles = (int)mad_ceil_div(N, BN);
    a.tiles_per_seg = (int)mad_ceil_div(n_tiles, S);
    a.hi_n2 = hi_n2; a.lo_n2 = lo_n2; a.cc = cc; a.mode = mode;
    a.seg_count = seg_count; a.seg_offset = seg_offset;
    a.pair_hi = pair_hi; a.pair_lo = pair_lo; a.pair_score = pair_score;
    a.k = k; a.lo_index_base = lo_index_base; a.topk_idx = topk_idx; a.topk_score = topk_score;
    MAD_CUDA(cudaFuncSetAttribute(match_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
    dim3 grid((unsigned)mad_ceil_div(M, BM), (unsigned)S);
    MAD_PROF(mode == 0 ? "match_tc_count_kernel" : mode == 1 ? "match_tc_fill_kernel" : "match_tc_topk_kernel", st);
    match_tc_kernel<<<grid, THREADS, SMEM_BYTES, st>>>(map_hi, map_lo, a);
    MAD_LAUNCH_OK();
    return MAD_OK;
}
