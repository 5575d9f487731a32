// a15: descriptor matching on the 5th-generation tensor cores, 8-bit integer path (sm_100a).
//
// Replaces  preds = np.dot(hi_unit, lo_unit.T); np.where(preds > cc)  (mad/MaD.py:416-424).
// Descriptor entries are vote counts of one 4x4x4-sample sub-block, i.e. integers <= 255 for every
// patch size the reference uses (<= 24); as uint8 operands of tcgen05.mma.kind::i8 with int32
// accumulators the raw dot product is EXACT, at twice the fp16 rate and half the operand bytes.
// The cosine dot / sqrt(n_i n_j) is evaluated in float64 from exact integers for the pairs an
// fp32 pre-filter cannot rule out.  The M x N score matrix is never written.
//
// Why this shape.  With operands streamed from L2 the fp16 kernel (match_tc.cu) needs 48 KB per
// 4.2 MFLOP, more than the ~43 B/clk/SM the L2 can deliver: it is L2-bound at ~15 % of the tensor
// peak.  Here the 128-row hi tile (128 x 1024 B = 128 KB) stays RESIDENT in shared memory for the
// CTA's whole sweep over the lo axis and only lo tiles are streamed: 16 KB per 4.2 MOP.
//
//   warp 0      TMA producer : hi tile once (8 boxes of 128 rows x 128 B, 128B swizzle), then the
//                              lo k-blocks into a 5-stage ring (mbarrier complete_tx)
//   warp 1      MMA issuer   : tcgen05.mma.cta_group::1.kind::i8, M=128 N=128 K=32, int32
//                              accumulators in TMEM (4 x 128 columns, 4-deep)
//   warp 2      TMEM allocator; warps 2 and 3 DRAIN the pair list in PAIRS mode (float64 decision, output
//               reservation, copy-out of the half buffers the epilogue warps publish)
//   warps 4..11 epilogue     : two groups of 4 warps alternating tiles; tcgen05.ld (32 lanes x 32
//                              columns), thread = one hi row
//        PAIRS mode: hits (row, col, dot) are staged per warp in shared memory and appended to a
//                    global candidate list by the drain warps (one atomicAdd per half buffer); a radix sort by
//                    (row, col) afterwards restores np.where's row-major order (match_finish).
//        TOPK mode : per-row running top-k in the thread (k <= 8: a register list keyed by float32 score images, near-ties
//                    decided on the float64 score), one partial list per (lo segment, epilogue group), thresholds of the two groups
//                    shared through shared memory.
#include <cuda.h>
#include <stdlib.h>

#include <type_traits>

#include "common.cuh"
#include "match_common.cuh"

namespace {

constexpr int BM = 128;            // hi rows per CTA (UMMA M)
constexpr int BN = 128;            // lo rows per tile (UMMA N) of the one-CTA kernel; lo rows PER CTA of a pair's 256-wide tile
constexpr int BKB = 128;           // bytes (= uint8 elements) per k-block = one 128-byte swizzle row
constexpr int UKB = 32;            // UMMA K for 8-bit inputs
constexpr int KBLOCKS = MAD_DSC_LEN / BKB;          // 8
constexpr int STAGES = 5;          // one CTA: 5 stages of 128 lo rows (16 KB)
constexpr int STAGES2 = 10;        // CTA pair: each CTA holds 64 of the 128 lo rows of a stage (8 KB): 10 stages
constexpr int ACCS = 4;            // TMEM accumulator ring (4 x 128 columns)
constexpr uint32_t KB_BYTES = BM * BKB;             // 16 KB: one k-block of 128 rows
constexpr uint32_t A_BYTES = KBLOCKS * KB_BYTES;    // 128 KB resident hi tile
constexpr int EPI_WARPS = 8;       // two epilogue groups of 4 warps (one per TMEM lane quadrant), alternating tiles
constexpr int THREADS = 128 + 32 * EPI_WARPS + 64;     // + warps 12, 13: two more drain warps of the top-8 mode (idle otherwise)
constexpr uint32_t TMEM_COLS = 512;
// count value a hand-off time-out leaves behind: the host raises instead of returning a truncated pair list
constexpr unsigned long long MAD_MATCH_TIMEOUT_COUNT = 1ull << 62;
constexpr int STG = 96;            // staged candidates per epilogue warp
constexpr size_t STG_BYTES = (size_t)EPI_WARPS * STG * (sizeof(unsigned long long) + sizeof(int));
constexpr size_t RB_BYTES = (size_t)2 * 2 * 256 * sizeof(float);          // per epilogue group, double-buffered 1/|lo| of a tile
// dynamic smem: [1024 slack][A 128K][B ring 80K][staging 9K][rnorm 8K][barriers, tmem slot, counters 512]
constexpr size_t THR_BYTES = 512;   // TOP8: per-row list thresholds published by the drain warps
// TOP8 staging: per epilogue warp 2 halves x 32 lanes x TOP_SLOTS self-contained 8-byte entries (in the pairs staging area)
constexpr int TOP_SLOTS = 2;
// TOP8: the first TOP_LOCAL_TILES tiles of a sweep are handled by the epilogue threads themselves (thread-local list, fresh
// threshold): 60 % of a row's ~8 ln(N / 8) candidate events fall into them, and through the hand-off every one of those
// would cost a round trip to a drain warp whose threshold lags.  Lists per (segment, row): drain, local group 0, local group 1.
constexpr int TOP_LOCAL_TILES = 4;
constexpr unsigned long long TOP_INVALID = ~0ull;
static_assert((size_t)EPI_WARPS * 2 * 32 * TOP_SLOTS * sizeof(unsigned long long) <= STG_BYTES, "TOP8 slots fit the staging area");
constexpr size_t SMEM_BYTES = 1024 + A_BYTES + (size_t)STAGES * KB_BYTES + STG_BYTES + RB_BYTES + 512 + THR_BYTES;
static_assert(SMEM_BYTES <= 232448, "shared memory budget of one sm_100 CTA");

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
// ---- CTA-pair (cta_group::2) variants.  Addresses are the issuing CTA's shared::cta offsets, which are
// valid shared::cluster addresses of that CTA; clearing bit 24 addresses the same offset in the
// pair's leader (even) CTA.
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA load whose bytes are accounted on the LEADER CTA's mbarrier (issued by both CTAs of the pair)
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar & kPeerBitMask), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void mbar_arrive_leader(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bar & kPeerBitMask) : "memory");
}
// commit that arrives on the barrier at this offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void umma_i8_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void umma_i8(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
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
__device__ __forceinline__ uint32_t tmem_ld1(uint32_t taddr) {
    uint32_t x;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(x) : "r"(taddr) : "memory");
    return x;
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
// kind::i8 instruction descriptor: D = s32 (bits 4-5 = 2), A = B = unsigned 8-bit (format 0), both
// K-major, N >> 3 at bits 17-22, M >> 4 at bits 24-28.
constexpr uint32_t kIdesc = (2u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
constexpr uint32_t kIdescPair = (2u << 4) | ((uint32_t)((2 * BN) >> 3) << 17) | ((uint32_t)((2 * BM) >> 4) << 24);   // M = 256, N = 256 over the pair

struct U8Args {
    int M, N, S;                  // rows of hi / lo, number of lo segments
    int tiles_per_seg;            // 128-column tiles per segment
    const int32_t* hi_n2;
    const int32_t* lo_n2;
    const float* lo_rnorm;        // 1/sqrt(n2) as float, 0 for zero descriptors; padded to N_pad
    double cc;
    // PAIRS
    unsigned long long* cand_key; // row * N + col (row-major rank of the pair: few key bits for the radix sort)
    int32_t* cand_dot;
    unsigned long long cap;
    unsigned long long* count;    // device counter (hits found, may exceed cap)
    // TOPK
    int k, lo_index_base;
    int local_tiles;              // TOP8: tiles at the start of a sweep handled by the epilogue threads themselves
    int dbg;                      // MAD_TOPK_DBG (measurement only): 1 = drain consumes without inserting, 2 = epilogue stages nothing
    int32_t* topk_idx;            // [2 S][M][k]: one list per (segment, epilogue group)
    double* topk_score;
};

// measurement counters of the top-8 hand-off (MAD_TOPK_DBG & 32): epilogue round cycles, publish-wait cycles, publishes, rounds,
// drain passes, drain busy cycles, entries inserted, entries dropped as stale
__device__ unsigned long long g_top_dbg[8];

enum { MODE_PAIRS = 0, MODE_TOPK = 1, MODE_TOP8 = 2 };   // TOP8: k <= 8, list in registers

// NCTA = 1: one CTA per 128-row hi tile.  NCTA = 2: a CTA pair (cluster of 2, cta_group::2) owns a
// 256-row hi tile -- each CTA keeps its own 128 rows resident and loads HALF of every lo stage, the
// leader issues M=256 MMAs that read both halves: the lo bytes fetched per MMA halve (the one-CTA
// kernel saturates the L2 -> SM path at ~62 % tensor activity) and the ring holds twice the stages.
template <int MODE, int NCTA>
__global__ void __launch_bounds__(THREADS, 1)
match_u8_kernel(const __grid_constant__ CUtensorMap map_hi, const __grid_constant__ CUtensorMap map_lo, U8Args a) {
    // Tile width.  The tensor core re-reads the hi operand from shared memory for every MMA, so with
    // N = 128 the operand reads (A 4 KB + B 4 KB per 64 clk) plus the TMA writes exceed the 128 B/clk
    // of shared memory: both 128-wide variants measured 61-62 % tensor activity.  The pair uses
    // N = 256 (each CTA stages 128 of the 256 lo rows): A is amortised over twice the columns.
    constexpr int TN = (NCTA == 2) ? 2 * BN : BN;
    constexpr int NACC = (int)TMEM_COLS / TN;                      // accumulators in TMEM: 4 x 128 or 2 x 256 columns
    constexpr int NSTAGE = STAGES;
    constexpr uint32_t SB = KB_BYTES;                              // bytes of a lo stage held by this CTA (128 rows x 128 B)
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;                 // SWIZZLE_128B tiles need 1024-byte alignment
    uint8_t* gen = smem_raw + (base - raw);
    const uint32_t b_ring = base + A_BYTES;
    constexpr uint32_t STG_OFF = A_BYTES + STAGES * KB_BYTES;     // (NSTAGE * SB is the same 80 KB)
    unsigned long long* stg_key = reinterpret_cast<unsigned long long*>(gen + STG_OFF);        // [EPI_WARPS][STG]
    int* stg_dot = reinterpret_cast<int*>(gen + STG_OFF + EPI_WARPS * STG * sizeof(unsigned long long));   // [EPI_WARPS][STG]
    float* s_rb = reinterpret_cast<float*>(gen + STG_OFF + (uint32_t)STG_BYTES);                  // [2 groups][2][256]
    constexpr uint32_t BAR_OFF = STG_OFF + (uint32_t)(STG_BYTES + RB_BYTES);
    const uint32_t bars = base + BAR_OFF;
    auto full_bar = [&](int s) { return bars + 8u * s; };
    auto empty_bar = [&](int s) { return bars + 8u * (NSTAGE + s); };
    auto tfull_bar = [&](int q) { return bars + 8u * (2 * NSTAGE + q); };
    auto tempty_bar = [&](int q) { return bars + 8u * (2 * NSTAGE + ACCS + q); };   // (ACCS slots reserved, NACC used)
    const uint32_t a_bar = bars + 8u * (2 * NSTAGE + 2 * ACCS);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(gen + BAR_OFF + 8 * (2 * NSTAGE + 2 * ACCS + 1));
    // hand-off words between the epilogue warps and the two drain warps (PAIRS mode): [EPI_WARPS][2] half-buffer states
    // (0 = free, n > 0 = n staged entries ready) followed by [EPI_WARPS] "this epilogue warp has finished" flags
    volatile int* s_half = reinterpret_cast<volatile int*>(gen + BAR_OFF + 8 * (2 * NSTAGE + 2 * ACCS + 2));
    volatile int* s_done = s_half + 2 * EPI_WARPS;
    static_assert(8 * (2 * STAGES + 2 * ACCS + 2) + 3 * EPI_WARPS * sizeof(int) <= 512, "misc shared region");
    // TOP8 (k <= 8): the epilogue warps only STAGE candidates (lane l of epilogue warp e owns TOP_SLOTS slots per half), the
    // two drain warps keep the per-row lists in registers and publish each row's threshold here
    volatile unsigned long long* top_slots = reinterpret_cast<volatile unsigned long long*>(gen + STG_OFF);
    volatile float* s_thr8 = reinterpret_cast<volatile float*>(gen + BAR_OFF + 512);             // [BM]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = (NCTA == 2) ? cluster_ctarank() : 0u;    // 0 = leader of the pair
    const int m0 = blockIdx.x * BM;                                // pairs are consecutive blockIdx.x: rows follow
    const int seg = blockIdx.y;
    const int n_tiles_total = (a.N + TN - 1) / TN;
    const int t_begin = seg * a.tiles_per_seg;
    const int t_end = min(n_tiles_total, t_begin + a.tiles_per_seg);

    if (threadIdx.x == 0) {
        for (int s = 0; s < NSTAGE; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        // the leader's "accumulator drained" barrier collects the 4 epilogue warps of BOTH CTAs
        // one-CTA kernel: a tile is drained by ONE epilogue group (4 warps); pair kernel: by both groups
        // (each takes 128 of the 256 columns) of both CTAs
        for (int q = 0; q < NACC; ++q) { mbar_init(tfull_bar(q), 1); mbar_init(tempty_bar(q), NCTA == 2 ? 16 : 4); }
        mbar_init(a_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (threadIdx.x < 3 * EPI_WARPS) s_half[threadIdx.x] = 0;
    // top-k, pair kernel: the two epilogue groups keep separate lists for the two column halves of the SAME rows; each
    // publishes its list's threshold here (the staging area is unused in top-k mode) and pre-filters with the larger of
    // the two -- the merged k-th best is at least that good, so nothing that could reach the merged list is skipped
    volatile float* s_thr = reinterpret_cast<volatile float*>(gen + STG_OFF);                  // [2 groups][BM]
    if (MODE == MODE_TOPK && threadIdx.x < 2 * BM) s_thr[threadIdx.x] = -1.f;
    if (MODE == MODE_TOP8) {
        for (int i = threadIdx.x; i < EPI_WARPS * 2 * 32 * TOP_SLOTS; i += THREADS) top_slots[i] = TOP_INVALID;
        if (threadIdx.x < BM) s_thr8[threadIdx.x] = -1.f;
    }
    if (NCTA == 2) cluster_sync_all();                             // barriers of both CTAs exist before any remote arrive
    if (warp == 2) {
        if (NCTA == 2) {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===================== TMA producer (one elected lane) =====================
        if (lane == 0) {
            if (NCTA == 2) {
                // both hi tiles (2 x 128 KB) and both halves of every lo stage are accounted on the LEADER's barriers
                if (rank == 0) mbar_expect_tx(a_bar, 2 * A_BYTES);
                for (int kb = 0; kb < KBLOCKS; ++kb) tma_load_2d_2sm(base + kb * KB_BYTES, &map_hi, a_bar, kb * BKB, m0);
            } else {
                mbar_expect_tx(a_bar, A_BYTES);
                for (int kb = 0; kb < KBLOCKS; ++kb) tma_load_2d(base + kb * KB_BYTES, &map_hi, a_bar, kb * BKB, m0);
            }
            int stage = 0;
            uint32_t phase = 0;
            for (int t = t_begin; t < t_end; ++t) {
                for (int kb = 0; kb < KBLOCKS; ++kb) {
                    mbar_wait(empty_bar(stage), phase ^ 1u);       // own barrier: the pair's commit arrives in both CTAs
                    if (NCTA == 2) {
                        if (rank == 0) mbar_expect_tx(full_bar(stage), 2 * KB_BYTES);
                        tma_load_2d_2sm(b_ring + stage * SB, &map_lo, full_bar(stage), kb * BKB, t * TN + (int)rank * BN);
                    } else {
                        mbar_expect_tx(full_bar(stage), KB_BYTES);
                        tma_load_2d(b_ring + stage * SB, &map_lo, full_bar(stage), kb * BKB, t * BN);
                    }
                    if (++stage == NSTAGE) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (one thread) =====================
        if (lane == 0 && rank == 0) {                                // in a pair only the leader issues MMAs
            mbar_wait(a_bar, 0);
            tc_fence_after();
            int stage = 0;
            uint32_t phase = 0;
            int it = 0;
            for (int t = t_begin; t < t_end; ++t, ++it) {
                const int acc = it % NACC;
                const uint32_t acc_phase = (uint32_t)(it / NACC) & 1u;
                mbar_wait(tempty_bar(acc), acc_phase ^ 1u);          // epilogue has drained this accumulator
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * TN);
                for (int kb = 0; kb < KBLOCKS; ++kb) {
                    mbar_wait(full_bar(stage), phase);
                    tc_fence_after();
                    const uint64_t da = umma_smem_desc(base + kb * KB_BYTES);
                    const uint64_t db = umma_smem_desc(b_ring + stage * SB);
#pragma unroll
                    for (int kk = 0; kk < BKB / UKB; ++kk) {
                        // advance 32 bytes inside the 128-byte swizzle row: +2 in 16-byte units
                        if (NCTA == 2) umma_i8_pair(d_tmem, da + (uint64_t)(2 * kk), db + (uint64_t)(2 * kk), kIdescPair, (kb | kk) ? 1u : 0u);
                        else umma_i8(d_tmem, da + (uint64_t)(2 * kk), db + (uint64_t)(2 * kk), kIdesc, (kb | kk) ? 1u : 0u);
                    }
                    // smem slot free (in both CTAs of a pair) when these MMAs retire
                    if (NCTA == 2) umma_commit_pair(empty_bar(stage)); else umma_commit(empty_bar(stage));
                    if (++stage == NSTAGE) { stage = 0; phase ^= 1u; }
                }
                // accumulator complete (signalled to the epilogues of both CTAs of a pair)
                if (NCTA == 2) umma_commit_pair(tfull_bar(acc)); else umma_commit(tfull_bar(acc));
            }
        }
    } else if (warp >= 2 && warp < 4 && MODE == MODE_PAIRS) {
        // ===================== drain warps (PAIRS): warp 2 serves epilogue group 0, warp 3 group 1 =====================
        // The epilogue warps only STAGE the candidates that pass the fp32 pre-filter; when a half buffer is full they
        // publish it here and carry on in the other half.  These two otherwise idle warps take the float64 decision, reserve
        // the output range (one global atomicAdd per half buffer) and write the pairs.  All of that used to sit in the
        // epilogue warps, and with the tile's accumulator released only when the slowest of a pair's 16 epilogue warps is
        // done, every flush (~1500 cycles) delayed the tensor pipe: 0.32 ms of the 1.50 ms C2 launch.
        // A staged entry is self-contained: |lo|^2 in the high word, (column << 5 | owning lane) in the low word.  The
        // comparison dot / sqrt(p) > cc is decided on exact integers, dot^2 against cc^2 p, whenever the two differ by more
        // than 1e-13 relative (sqrt and division are correctly rounded: their 2.3e-16 cannot flip such a case); only closer
        // cases evaluate the quotient itself.
        constexpr int HALF = STG / 2;
        const int e0 = (warp - 2) * 4;                               // first epilogue warp served
        const double cc2 = a.cc * a.cc;
        int hi_n2_reg[4];                                            // |hi|^2 of the CTA's 128 rows: lane l holds rows q * 32 + l
#pragma unroll
        for (int qq = 0; qq < 4; ++qq) hi_n2_reg[qq] = (m0 + qq * 32 + lane < a.M) ? __ldg(a.hi_n2 + m0 + qq * 32 + lane) : 0;
        for (long long spins = 0; spins < (1LL << 27); ++spins) {    // (bounded: a protocol error must not hang the device)
            int done = 0;
            for (int e = e0; e < e0 + 4; ++e) done += mad_ld_acquire_cta(&s_done[e]);
            bool any = false;
            for (int e = e0; e < e0 + 4; ++e) {
                for (int h = 0; h < 2; ++h) {
                    const int n = mad_ld_acquire_cta(&s_half[2 * e + h]);      // (acquire: the entries were written before the state word)
                    if (n <= 0) continue;
                    any = true;
                    const unsigned long long* hk = stg_key + e * STG + h * HALF;
                    const int* hd = stg_dot + e * STG + h * HALF;
                    unsigned long long ent[2];
                    int dot[2];
                    bool ok[2];
#pragma unroll
                    for (int k = 0; k < 2; ++k) {
                        const int i = lane + 32 * k;
                        ent[k] = (i < n) ? hk[i] : 0ull;
                        dot[k] = (i < n) ? hd[i] : 0;
                    }
                    __syncwarp();
                    if (lane == 0) mad_st_release_cta(&s_half[2 * e + h], 0);   // the half may be refilled: its entries are in registers
                    int total = 0, pos[2];
                    const int qe = e & 3;
                    const int n2_q = qe == 0 ? hi_n2_reg[0] : (qe == 1 ? hi_n2_reg[1] : (qe == 2 ? hi_n2_reg[2] : hi_n2_reg[3]));
#pragma unroll
                    for (int k = 0; k < 2; ++k) {
                        ok[k] = false;
                        const unsigned low = (unsigned)ent[k];
                        const double n2r = (double)__shfl_sync(0xFFFFFFFFu, n2_q, (int)(low & 31u));
                        if (lane + 32 * k < n) {
                            const int row = m0 + qe * 32 + (int)(low & 31u);
                            const double n2c = (double)(unsigned)(ent[k] >> 32);
                            const double p = n2r * n2c, lhs = (double)dot[k] * (double)dot[k], rhs = cc2 * p;
                            if (p > 0.0 && a.cc > 0.0 && lhs > rhs * (1.0 + 1e-13)) ok[k] = true;
                            else if (p > 0.0 && a.cc > 0.0 && lhs < rhs * (1.0 - 1e-13)) ok[k] = false;
                            else ok[k] = mad_score(dot[k], n2r, n2c) > a.cc;     // a zero norm scores 0
                            ent[k] = (unsigned long long)row * (unsigned long long)a.N + (unsigned long long)(low >> 5);
                        }
                        const unsigned m = __ballot_sync(0xFFFFFFFFu, ok[k]);
                        pos[k] = total + __popc(m & ((1u << lane) - 1u));
                        total += __popc(m);
                    }
                    if (total > 0) {
                        unsigned long long gb = 0;
                        if (lane == 0) gb = atomicAdd(a.count, (unsigned long long)total);
                        gb = __shfl_sync(0xFFFFFFFFu, gb, 0);
#pragma unroll
                        for (int k = 0; k < 2; ++k)
                            if (ok[k] && gb + pos[k] < a.cap) { a.cand_key[gb + pos[k]] = ent[k]; a.cand_dot[gb + pos[k]] = dot[k]; }
                    }
                }
            }
            if (!any) {
                if (done == 4) break;                                // flags read BEFORE the scan that found nothing
                __nanosleep(200);
            }
            if (spins == (1LL << 27) - 1 && lane == 0) atomicExch(a.count, MAD_MATCH_TIMEOUT_COUNT);   // fail loudly on the host
        }
    } else if ((warp == 2 || warp == 3 || warp >= 4 + EPI_WARPS) && MODE == MODE_TOP8) {
        // ===================== drain warps (TOP8): warps 2, 3, 12, 13 own the lists of one 32-row quadrant each ==========
        // Lane l keeps the top-8 list of row 32 dq + l in registers: (float32 score image, dot, |lo|^2, index), ordered by the
        // float64 score and then the index wherever the images are closer than 4e-6.  The epilogue warps of BOTH groups stage
        // their candidates per lane (lane l of an epilogue warp of quadrant q owns row 32 q + l), so a published half is
        // consumed by all 32 lanes at once: every lane inserts its own row's (at most TOP_SLOTS) entries -- no routing, no
        // atomics, one list per row for both column halves of a tile.
        // With the lists in the epilogue threads a warp paid ~300 cycles per candidate of ANY of its 32 rows on the critical
        // path of its tile (140 candidate events per row at 100 000 columns: 1.3 M cycles against 1.6 M of MMA work).
        const int dq = warp < 4 ? warp - 2 : warp - (4 + EPI_WARPS) + 2;
        float ts[8];
        int td[8], tn[8], bi[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) { ts[i] = 0.f; td[i] = 0; tn[i] = 1; bi[i] = -1; }
        const int row = m0 + 32 * dq + lane;
        const int n2a_i = row < a.M ? __ldg(a.hi_n2 + row) : 0;
        const float ra = n2a_i > 0 ? (float)(1.0 / sqrt((double)n2a_i)) : 0.f;
        bool timeout = false;
        for (long long spins = 0;; ++spins) {
            if (spins >= (1LL << 26)) { timeout = true; break; }      // (bounded: a protocol error must not hang the device)
            const int done = mad_ld_acquire_cta(&s_done[dq]) + mad_ld_acquire_cta(&s_done[4 + dq]);
            bool any = false;
#pragma unroll 1
            for (int g = 0; g < 2; ++g) {
                const int e = g * 4 + dq;                             // epilogue warp of group g, quadrant dq
#pragma unroll 1
                for (int h = 0; h < 2; ++h) {
                    const int tt = mad_ld_acquire_cta(&s_half[2 * e + h]);      // (acquire: the entries were written before the state word)
                    if (tt <= 0) continue;
                    any = true;
                    const long long dc0 = (a.dbg & 32) ? clock64() : 0;
                    int n_ins = 0, n_stale = 0;
                    volatile unsigned long long* sl = top_slots + ((e * 2 + h) * 32 + lane) * TOP_SLOTS;
                    unsigned long long ent[TOP_SLOTS];
#pragma unroll
                    for (int u = 0; u < TOP_SLOTS; ++u) { ent[u] = sl[u]; sl[u] = TOP_INVALID; }
                    __syncwarp();
                    if (lane == 0) mad_st_release_cta(&s_half[2 * e + h], 0);                  // the half may be refilled
                    const int colbase = a.lo_index_base + (tt - 1) * TN;
                    bool changed = false;
#pragma unroll
                    for (int u = 0; u < TOP_SLOTS; ++u) {
                        const bool has = ent[u] != TOP_INVALID && !(a.dbg & 1);
                        if (!__any_sync(0xFFFFFFFFu, has)) continue;
                        const int dot = (int)(ent[u] >> 35), n2b = (int)((ent[u] >> 8) & 0x7FFFFFFull);
                        const int id = colbase + (int)(ent[u] & 0xFFull);
                        const bool nz = n2a_i > 0 && n2b > 0;           // a zero descriptor scores 0 whatever the dot product: key (0, 1)
                        const float s32 = nz ? (float)dot * rsqrtf((float)n2b) * ra : 0.f;
                        // stale candidates (staged under an older threshold) are dropped on the image of the 8th entry
                        const bool live = has && (bi[7] < 0 || s32 >= ts[7] * (1.f - 4e-6f));
                        if (!__any_sync(0xFFFFFFFFu, live)) { n_stale += has; continue; }
                        mad_top8f_insert(ts, td, tn, bi, live, s32, nz ? dot : 0, nz ? n2b : 1, id, (double)n2a_i);
                        changed |= live;
                        n_ins += live;
                        n_stale += has && !live;
                    }
                    if (a.dbg & 32) {
                        n_ins = __reduce_add_sync(0xFFFFFFFFu, n_ins);
                        n_stale = __reduce_add_sync(0xFFFFFFFFu, n_stale);
                        if (lane == 0) {
                            atomicAdd(&g_top_dbg[4], 1ull); atomicAdd(&g_top_dbg[5], (unsigned long long)(clock64() - dc0));
                            atomicAdd(&g_top_dbg[6], (unsigned long long)n_ins); atomicAdd(&g_top_dbg[7], (unsigned long long)n_stale);
                        }
                    }
                    // fp32 image of the 8th entry's score (error < 1e-6) minus the pre-filter margin
                    // (atomicMax on the int image: thresholds are >= 0 or the initial -1, and the epilogue threads seed the
                    //  same word with the 8th score of their local lists)
                    if (changed && bi[7] >= 0) atomicMax(reinterpret_cast<int*>(const_cast<float*>(&s_thr8[dq * 32 + lane])), __float_as_int(fmaxf(ts[7] - 4e-6f, 0.f)));
                }
            }
            if (!any) {
                if (done == 2) break;                                // flags read BEFORE the scan that found nothing
                // idle: poll a few times per tile only (a polling loop that spins every ~100 cycles in four warps took a
                // quarter of the SM's issue slots away from the epilogue warps: +25 % on the whole sweep)
                __nanosleep(a.dbg & 16 ? 32 : (a.dbg & 64 ? 1000 : 300));
            }
        }
        if (row < a.M) {                                             // list 0 of the 3 lists of (segment, row)
            const long long o = ((long long)(seg * 3) * a.M + row) * a.k;
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (i < a.k) {
                    a.topk_idx[o + i] = timeout ? MAD_TOPK_INCOMPLETE : bi[i];
                    a.topk_score[o + i] = bi[i] < 0 ? -INFINITY : (td[i] == 0 ? 0.0 : mad_score(td[i], (double)n2a_i, (double)tn[i]));
                }
        }
    } else if (warp >= 4 && warp < 4 + EPI_WARPS) {
        // ===================== epilogue: thread = one hi row =====================
        const int q = warp & 3;                                      // TMEM lane quadrant of this warp
        const int ew = warp - 4;                                     // epilogue warp 0..7
        const int grp = ew >> 2;                                     // group 0 takes even tiles of the sweep, group 1 odd
        const int row = m0 + q * 32 + lane;
        const bool row_ok = row < a.M;
        const int n2a_i = row_ok ? a.hi_n2[row] : 0;
        const double n2a = (double)n2a_i;
        const float ra = n2a_i > 0 ? (float)(1.0 / sqrt(n2a)) : 0.f;
        // fp32 pre-filter: dot * rb > (cc - 4e-6) / ra   (|approx - exact| < 1e-6).  A zero row scores 0 against every
        // column: all of them pass when cc < 0, none otherwise.
        const float thr_pairs = !row_ok ? INFINITY : (n2a_i > 0 ? ((float)a.cc - 4e-6f) / ra : (a.cc < 0.0 ? -INFINITY : INFINITY));
        unsigned long long* my_key = stg_key + ew * STG;
        int* my_dot = stg_dot + ew * STG;
        constexpr bool kTop = (MODE == MODE_TOPK || MODE == MODE_TOP8);
        constexpr int kList = (MODE == MODE_TOPK) ? MAD_TOPK_MAX : 1;
        double bs[kList];                                            // MODE_TOPK (k > 8): the list lives in the epilogue thread
        int bi[kList];
        float thr = -1.f;                                            // fp32 bound of the current worst list entry
        if (MODE == MODE_TOPK) {
#pragma unroll
            for (int i = 0; i < kList; ++i) { bs[i] = -INFINITY; bi[i] = -1; }
        }
        const int k_last = a.k - 1;
        int top_cnt = 0;                                             // TOP8: entries this lane has staged in the current half
        float ls[8];                                                 // TOP8: thread-local list of the first TOP_LOCAL_TILES tiles
        int ld[8], ln[8], li[8];
        if (MODE == MODE_TOP8) {
#pragma unroll
            for (int i = 0; i < 8; ++i) { ls[i] = 0.f; ld[i] = 0; ln[i] = 1; li[i] = -1; }
        }
        auto flush_local = [&]() {                                   // the local list becomes list 1 + grp of (segment, row); its
                                                                     // 8th score seeds the row's threshold for the staged phase
            if (li[7] >= 0) atomicMax(reinterpret_cast<int*>(const_cast<float*>(&s_thr8[q * 32 + lane])), __float_as_int(fmaxf(ls[7] - 4e-6f, 0.f)));
            if (row_ok) {
                const long long o = ((long long)(seg * 3 + 1 + grp) * a.M + row) * a.k;
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    if (i < a.k) {
                        a.topk_idx[o + i] = li[i];
                        a.topk_score[o + i] = li[i] < 0 ? -INFINITY : (ld[i] == 0 ? 0.0 : mad_score(ld[i], n2a, (double)ln[i]));
                    }
            }
        };
        // Candidates that pass the fp32 pre-filter are only STAGED here (two shared-memory stores); the drain warps take
        // the float64 decision and write the pairs.
        int stg_n = 0;                                               // candidates staged by this warp (warp-uniform register)
        constexpr int HALF = STG / 2;
        static_assert(HALF >= 32, "a half buffer must take one ballot round");
        int cur = 0;                                                 // half being filled
        auto publish = [&](int n) {                                  // hand the current half (n entries) to the drain warp
            __syncwarp();
            if (n > 0) {
                if (lane == 0) {
                    mad_st_release_cta(&s_half[2 * ew + cur], n);    // (release; MEMBAR.SC.CTA of __threadfence_block is far heavier)
                    long long spins = 0;
                    while (mad_ld_acquire_cta(&s_half[2 * ew + (cur ^ 1)]) != 0 && ++spins < (1LL << 27)) __nanosleep(64);   // other half still in use
                    if (spins >= (1LL << 27)) atomicExch(a.count, MAD_MATCH_TIMEOUT_COUNT);              // fail loudly on the host
                }
                cur ^= 1;
                __syncwarp();
            }
        };
        auto publish_top = [&](int t) {                              // TOP8: hand the current half (entries of tile t) to the drain warp
            __syncwarp();
            if (lane == 0) {
                mad_st_release_cta(&s_half[2 * ew + cur], t + 1);    // (the lanes' entries are ordered before it by the __syncwarp)
                long long spins = 0;
                const long long c0 = (a.dbg & 32) ? clock64() : 0;
                while (mad_ld_acquire_cta(&s_half[2 * ew + (cur ^ 1)]) != 0 && ++spins < (1LL << 26)) __nanosleep(32);   // other half still in use
                if (a.dbg & 32) { atomicAdd(&g_top_dbg[1], (unsigned long long)(clock64() - c0)); atomicAdd(&g_top_dbg[2], 1ull); }
            }
            cur ^= 1;
            top_cnt = 0;
            __syncwarp();
        };
        // Work split between the two epilogue groups.  One-CTA kernel (128-wide tiles, 4 accumulators): the
        // groups alternate tiles.  Pair kernel (256-wide tiles, only 2 accumulators fit TMEM): both groups
        // drain EVERY tile, each its own 128 columns, so an accumulator is free after half an epilogue.
        constexpr bool kSplitCols = (NCTA == 2);
        constexpr int kStep = kSplitCols ? 1 : 2;
        const int c_lo = kSplitCols ? grp * BN : 0;                  // this group's 128 columns of a tile
        float* my_rb = s_rb + grp * 2 * 256;                         // shared by the 4 warps of this group
        const int gt = threadIdx.x - 128 - grp * 128;                // thread index inside the group, 0..127
        auto stage_rb = [&](int t, int buf) {                        // 128 floats of this tile, one float4 per thread
            if (gt < BN / 4) {
                const float4 r4 = __ldg(reinterpret_cast<const float4*>(a.lo_rnorm + (long long)t * TN + c_lo) + gt);
                reinterpret_cast<float4*>(my_rb + buf * 256)[gt] = r4;
                {                                                    // |lo|^2 (exact integers) in the buffer's unused upper half
                    const int c = t * TN + c_lo + 4 * gt;
                    int4 n4;
                    n4.x = (c < a.N) ? __ldg(a.lo_n2 + c) : 0;
                    n4.y = (c + 1 < a.N) ? __ldg(a.lo_n2 + c + 1) : 0;
                    n4.z = (c + 2 < a.N) ? __ldg(a.lo_n2 + c + 2) : 0;
                    n4.w = (c + 3 < a.N) ? __ldg(a.lo_n2 + c + 3) : 0;
                    reinterpret_cast<int4*>(my_rb + buf * 256 + 128)[gt] = n4;
                }
            }
        };
        auto group_sync = [&]() { asm volatile("bar.sync %0, 128;" ::"r"(1 + grp) : "memory"); };
        const int t_first = t_begin + (kSplitCols ? 0 : grp);
        int it = kSplitCols ? 0 : grp;                               // position of the tile in this CTA's sweep
        int par = 0;                                                 // which rnorm buffer holds the current tile
        if (t_first < t_end) stage_rb(t_first, 0);
        // The tile loop exists twice: the first TOP_LOCAL_TILES tiles of a top-8 sweep run with the thread-local list
        // (top_local), all others without it -- as ONE loop the list stayed live for the whole sweep and was spilled and
        // reloaded around every tile.
        auto tile_body = [&](auto local_tag, const int t, const int it, const int par) {
            const int acc = it % NACC;
            const uint32_t acc_phase = (uint32_t)(it / NACC) & 1u;
            const int n0 = t * TN;
            constexpr bool top_local = decltype(local_tag)::value;   // (two instantiations: the local list's registers are dead in the second)
            group_sync();                                            // this tile's norms are staged; the other buffer is free
            if (t + kStep < t_end) stage_rb(t + kStep, par ^ 1);     // this group's next tile: latency hidden by this tile
            const float* rbt = my_rb + par * 256 - c_lo;             // indexed by the column inside the tile
            mbar_wait(tfull_bar(acc), acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * TN);
#pragma unroll 1
            for (int c0 = c_lo; c0 < c_lo + BN; c0 += 32) {
                uint32_t v[32];
                tmem_ld32(taddr + (uint32_t)c0, v);
                tmem_ld_wait();
                if (c0 == c_lo + BN - 32 && !(a.dbg & 4)) {
                    // the tile's last 32 columns are in registers: the accumulator goes back to the MMA warp NOW, so the
                    // processing of this chunk (a quarter of the epilogue) is off the tensor pipe's critical path
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) {                                 // 4 (x2 in a pair) arrivals free the accumulator
                        if (NCTA == 2) mbar_arrive_leader(tempty_bar(acc)); else mbar_arrive(tempty_bar(acc));
                    }
                }
                // Branch-free pre-filter over the 32 columns (the epilogue must stay small: an unrolled
                // branchy body overflowed the instruction cache and made the epilogue the bottleneck);
                // the rare candidates are then fetched again from TMEM one column at a time.
                float thr_eff = thr;
                if (MODE == MODE_TOPK && kSplitCols) thr_eff = fmaxf(thr, s_thr[(grp ^ 1) * BM + q * 32 + lane]);
                if (MODE == MODE_TOP8)                                // local phase: this thread's own 8th score; then the row's threshold
                    thr_eff = top_local ? (li[7] < 0 ? -1.f : ls[7] - 4e-6f) : s_thr8[q * 32 + lane];   // as published by its drain warp
                const float lim = kTop ? (row_ok && ra > 0.f ? thr_eff / ra : INFINITY) : thr_pairs;
                unsigned mask = 0;
#pragma unroll
                for (int j4 = 0; j4 < 8; ++j4) {                     // 1/|lo| of four columns at a time (not 32 registers held)
                    const float4 r4 = reinterpret_cast<const float4*>(rbt + c0)[j4];
                    const float rb[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const float sc = (float)(int)v[4 * j4 + u] * rb[u];
                        const bool pass = kTop ? (sc >= lim) : (sc > lim);
                        mask |= (pass ? 1u : 0u) << (4 * j4 + u);
                    }
                }
                // zero row: every score is 0 and ties go to the lowest index -- only the first k columns matter
                if (MODE == MODE_TOPK && row_ok && ra == 0.f) mask = (bi[k_last] < 0) ? 0xFFFFFFFFu : 0u;
                if (MODE == MODE_TOP8) {
                    // zero row: only the first 8 columns of the sweep can make its list (score 0, lowest indices)
                    if (row_ok && ra == 0.f) mask = (t == t_begin && c0 == 0) ? 0xFFu : 0u;
                    const int left = a.N - (n0 + c0);                // columns of this chunk that exist
                    if (left < 32) mask &= (left <= 0) ? 0u : ((1u << left) - 1u);
                    if (a.dbg & 2) mask = 0u;
                    if (top_local) {
                        // thread-local phase: one ballot per round, all lanes with a candidate run the (float32-image) insertion
                        // network together; a candidate is re-checked against the list as it is NOW
                        for (;;) {
                            if (__ballot_sync(0xFFFFFFFFu, mask != 0u) == 0u) break;
                            const bool has = mask != 0u;
                            const int j = has ? __ffs(mask) - 1 : 0;
                            mask &= mask - 1;
                            const int dot = (int)mad_select32(v, j);
                            const int n2b = __float_as_int(rbt[c0 + j + 128]);
                            const bool nz = n2a_i > 0 && n2b > 0;
                            const float s32 = nz ? (float)dot * rbt[c0 + j] * ra : 0.f;
                            const bool live = has && (li[7] < 0 || s32 >= ls[7] * (1.f - 4e-6f));
                            if (__any_sync(0xFFFFFFFFu, live))
                                mad_top8f_insert(ls, ld, ln, li, live, s32, nz ? dot : 0, nz ? n2b : 1, a.lo_index_base + n0 + c0 + j, n2a);
                        }
                        continue;
                    }
                    // Candidates are only STAGED (one 8-byte shared-memory store each, into this lane's own slots): one ballot
                    // per round, as in pairs mode; the drain warp that owns the row's list takes it from there.
                    const long long rc0 = (a.dbg & 32) ? clock64() : 0;
                    int n_rounds = 0;
                    for (;;) {
                        const unsigned b = __ballot_sync(0xFFFFFFFFu, mask != 0u);
                        if (b == 0u) break;
                        ++n_rounds;
                        if (__ballot_sync(0xFFFFFFFFu, mask != 0u && top_cnt == TOP_SLOTS) != 0u) publish_top(t);
                        if (mask) {
                            const int j = __ffs(mask) - 1;
                            mask &= mask - 1;
                            const unsigned long long dot = (unsigned long long)mad_select32(v, j);
                            const unsigned long long n2b = (unsigned long long)(unsigned)__float_as_int(rbt[c0 + j + 128]);
                            top_slots[((ew * 2 + cur) * 32 + lane) * TOP_SLOTS + top_cnt] = (dot << 35) | (n2b << 8) | (unsigned long long)(c0 + j);
                            ++top_cnt;
                        }
                    }
                    if ((a.dbg & 32) && lane == 0 && n_rounds) {
                        atomicAdd(&g_top_dbg[0], (unsigned long long)(clock64() - rc0));
                        atomicAdd(&g_top_dbg[3], (unsigned long long)n_rounds);
                    }
                } else if (kTop) {
                    // each lane walks its own (rare) candidates; the value comes out of the registers
                    // through a select tree, so lanes with candidates in different columns run together
                    while (mask) {
                        const int j = __ffs(mask) - 1;
                        mask &= mask - 1;
                        const int dot = (int)mad_select32(v, j);
                        const int col = n0 + c0 + j;
                        if (col < a.N) {
                            const int n2b = __float_as_int(rbt[c0 + j + 128]);                       // |lo|^2 from the tile buffer
                            {
                                const double s = mad_score(dot, n2a, (double)n2b);
                                mad_topk_insert(bs, bi, a.k, s, a.lo_index_base + col);
                                thr = (bi[k_last] < 0) ? -1.f : (float)bs[k_last] - 4e-6f;
                                if (kSplitCols) s_thr[grp * BM + q * 32 + lane] = thr;
                            }
                        }
                    }
                } else {
                    // Pairs: no atomics on the hot path; each lane writes its own (usually <= 1) candidates, reading the
                    // dot product out of its registers through the select tree.
                    const int left = a.N - (n0 + c0);                // columns of this chunk that exist (rnorm is 0 beyond N,
                    if (left < 32) mask &= (left <= 0) ? 0u : ((1u << left) - 1u);   // but cc <= 0 would let padding through)
                    // One ballot per round hands every lane that still has a candidate its staging slot (round r takes
                    // the r-th candidate of each lane; most lanes have none, a few one): ~100 cycles of latency per round
                    // instead of the five dependent shuffles of a prefix sum.  A chunk with a hit sits on the critical path
                    // of its tile (the accumulator is released when the slowest of the pair's 16 epilogue warps is done).
                    const unsigned lt = (1u << lane) - 1u;
                    for (;;) {
                        const unsigned b = __ballot_sync(0xFFFFFFFFu, mask != 0u);
                        if (b == 0u) break;
                        const int nb = __popc(b);
                        if (stg_n + nb > HALF) { publish(stg_n); stg_n = 0; }
                        if (mask) {
                            const int j = __ffs(mask) - 1;
                            mask &= mask - 1;
                            const int p = cur * HALF + stg_n + __popc(b & lt);
                            my_key[p] = ((unsigned long long)(unsigned)__float_as_int(rbt[c0 + j + 128]) << 32) |
                                        (unsigned long long)(((unsigned)(n0 + c0 + j) << 5) | (unsigned)lane);
                            my_dot[p] = (int)mad_select32(v, j);
                        }
                        stg_n += nb;
                    }
                }
            }
            if (a.dbg & 4) {                                         // (measurement: release at the end of the tile's epilogue)
                tc_fence_before();
                __syncwarp();
                if (lane == 0) { if (NCTA == 2) mbar_arrive_leader(tempty_bar(acc)); else mbar_arrive(tempty_bar(acc)); }
            }
            // TOP8: the tile's candidates go to the drain warp now (a half never mixes tiles: its state word names the tile),
            // so a row's threshold lags by at most one tile
            if (MODE == MODE_TOP8 && __ballot_sync(0xFFFFFFFFu, top_cnt > 0) != 0u) publish_top(t);
        };
        int t = t_first;
        if (MODE == MODE_TOP8) {
            for (int n = 0; n < a.local_tiles && t < t_end; ++n, t += kStep, it += kStep, par ^= 1) tile_body(std::true_type{}, t, it, par);
            flush_local();
        }
        for (; t < t_end; t += kStep, it += kStep, par ^= 1) tile_body(std::false_type{}, t, it, par);
        if (!kTop) {
            publish(stg_n);
            __syncwarp();
            if (lane == 0) mad_st_release_cta(&s_done[ew], 1);
        }
        if (MODE == MODE_TOP8) {
            __syncwarp();
            if (lane == 0) mad_st_release_cta(&s_done[ew], 1);
        }
        if (MODE == MODE_TOPK && row_ok) {
            // one partial list per (segment, epilogue group): the host merges 2 S lists
            const long long o = ((long long)(seg * 2 + grp) * a.M + row) * a.k;
            for (int i = 0; i < a.k; ++i) { a.topk_idx[o + i] = bi[i]; a.topk_score[o + i] = bs[i]; }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (NCTA == 2) cluster_sync_all();                             // both CTAs are done with TMEM and each other's barriers
    if (warp == 2) {
        tc_fence_after();
        if (NCTA == 2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
        else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
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

// [rows_padded][1024] uint8 row-major; box = 128 bytes (k) x 128 rows, 128-byte swizzle.
int make_map(CUtensorMap* map, const void* ptr, int rows_padded, int box_rows = BM) {
    EncodeTiledFn enc = get_encode();
    if (!enc) {
        mad_set_error("mad_match: cuTensorMapEncodeTiled is not available from the CUDA driver");
        return MAD_ERR_NODEVICE;
    }
    cuuint64_t dims[2] = {(cuuint64_t)MAD_DSC_LEN, (cuuint64_t)rows_padded};
    cuuint64_t strides[1] = {(cuuint64_t)MAD_DSC_LEN};
    cuuint32_t box[2] = {(cuuint32_t)BKB, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        mad_set_error("mad_match: cuTensorMapEncodeTiled failed (%d)", (int)r);
        return MAD_ERR_CUDA;
    }
    return MAD_OK;
}

int check_device() {
    int dev = 0, major = 0;
    MAD_CUDA(cudaGetDevice(&dev));
    MAD_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
    if (major != 10) {
        mad_set_error("mad_match: the tcgen05 kernel needs an sm_100 device (found compute capability %d.x)", major);
        return MAD_ERR_NODEVICE;
    }
    return MAD_OK;
}

}  // namespace

// Number of lo segments: minimises  waves x (tiles per segment + fixed)  -- one CTA per SM (224 KB of shared memory).
static int pick_ncta(int M, int N_pad);

// fixed_tiles: what a CTA costs besides its lo tiles, in tile-equivalents (~2.07 us): loading the hi tile (1) and, in top-8
// mode, the thread-local start-up tiles and the early staged phase (~110 us measured = 53).
// slack > 1: the SMALLEST number of segments whose cost is within that factor of the best.
static int u8_segments(int M, int N, double slack, int fixed_tiles) {
    if (M <= 0 || N <= 0) return 1;
    const int tn = pick_ncta(M, 256) == 2 ? 2 * BN : BN;           // tile width of the variant this M gets
    const long long m_tiles = mad_ceil_div(M, BM);
    const long long n_tiles = mad_ceil_div(N, tn);
    const long long sms = mad_sm_count();
    long long best_s = 1, best_cost = -1;
    auto cost_of = [&](long long s) -> long long {
        const long long per = mad_ceil_div(n_tiles, s);
        const long long segs = mad_ceil_div(n_tiles, per);      // no empty segments
        if (segs != s) return -1;
        return mad_ceil_div(m_tiles * s, sms) * (per + fixed_tiles);
    };
    for (long long s = 1; s <= n_tiles; ++s) {
        const long long cost = cost_of(s);
        if (cost < 0) continue;
        if (best_cost < 0 || cost < best_cost) { best_cost = cost; best_s = s; }
    }
    if (slack > 1.0)
        for (long long s = 1; s < best_s; ++s) {
            const long long cost = cost_of(s);
            if (cost >= 0 && (double)cost <= slack * (double)best_cost) return (int)s;
        }
    return (int)best_s;
}

int mad_match_u8_segments(int M, int N) { return u8_segments(M, N, 1.0, 1); }

// Top-8: every (segment, row) keeps its own lists and pays its own start-up (the first tiles of a sweep see 60 % of a
// row's candidate events), so a CTA's fixed cost is ~53 tile-equivalents; with that in the model the sweep of 100 000 x
// 100 000 rows stays in ONE segment, and the short launch over the rows of a poorly filled last wave (mad_match_topk)
// gets 3.
int mad_match_u8_segments_topk(int M, int N) {
    static const int fixed = getenv("MAD_TOPK_FIXED_TILES") ? atoi(getenv("MAD_TOPK_FIXED_TILES")) : 53;
    return u8_segments(M, N, 1.0, fixed);
}

// CTA pairs are used when there are at least two hi tiles (MAD_MATCH_ONE_CTA=1 forces the one-CTA kernel).
// (the pair's 256-wide tiles read 1/|lo| in 256-float blocks: the lo set must be padded to 256 rows)
static int pick_ncta(int M, int N_pad) {
    static const bool one = getenv("MAD_MATCH_ONE_CTA") != nullptr;
    return (!one && M > BM && N_pad % 256 == 0) ? 2 : 1;
}

static int launch_common(const void* hi_u8, int M_pad, const void* lo_u8, int N_pad, int ncta, CUtensorMap* map_hi,
                         CUtensorMap* map_lo) {
    int rc = check_device();
    if (rc != MAD_OK) return rc;
    rc = make_map(map_hi, hi_u8, M_pad);
    if (rc != MAD_OK) return rc;
    (void)ncta;
    return make_map(map_lo, lo_u8, N_pad, BN);                     // 128 lo rows per CTA and stage in both variants
}

template <int MODE>
static int launch_u8(int ncta, int M, int S, const CUtensorMap& map_hi, const CUtensorMap& map_lo, const U8Args& a,
                     cudaStream_t st) {
    if (ncta == 2) {
        auto kern = match_u8_kernel<MODE, 2>;
        MAD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(2u * (unsigned)mad_ceil_div(M, 2 * BM), (unsigned)S);
        cfg.blockDim = dim3(THREADS);
        cfg.dynamicSmemBytes = SMEM_BYTES;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        MAD_CUDA(cudaLaunchKernelEx(&cfg, kern, map_hi, map_lo, a));
    } else {
        auto kern = match_u8_kernel<MODE, 1>;
        MAD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
        dim3 grid((unsigned)mad_ceil_div(M, BM), (unsigned)S);
        kern<<<grid, THREADS, SMEM_BYTES, st>>>(map_hi, map_lo, a);
    }
    MAD_LAUNCH_OK();
    return MAD_OK;
}

int mad_match_u8_pairs(const void* hi_u8, int M, int M_pad, const void* lo_u8, int N, int N_pad, const int32_t* hi_n2,
                       const int32_t* lo_n2, const float* lo_rnorm, double cc, unsigned long long* cand_key,
                       int32_t* cand_dot, unsigned long long cap, unsigned long long* count, cudaStream_t st) {
    CUtensorMap map_hi, map_lo;
    const int ncta = pick_ncta(M, N_pad);
    int rc = launch_common(hi_u8, M_pad, lo_u8, N_pad, ncta, &map_hi, &map_lo);
    if (rc != MAD_OK) return rc;
    if (N_pad > (1 << 27)) { mad_set_error("mad_match_pairs: more than 2^27 lo rows"); return MAD_ERR_ARG; }   // staged entries hold column << 5
    U8Args a = {};
    a.M = M; a.N = N;
    a.S = mad_match_u8_segments(M, N);
    a.tiles_per_seg = (int)mad_ceil_div(mad_ceil_div(N, BN * ncta), a.S);
    a.hi_n2 = hi_n2; a.lo_n2 = lo_n2; a.lo_rnorm = lo_rnorm; a.cc = cc;
    a.cand_key = cand_key; a.cand_dot = cand_dot; a.cap = cap; a.count = count;
    a.dbg = getenv("MAD_TOPK_DBG") ? atoi(getenv("MAD_TOPK_DBG")) : 0;
    MAD_PROF("match_u8_pairs_kernel", st);
    return launch_u8<MODE_PAIRS>(ncta, M, a.S, map_hi, map_lo, a, st);
}

int mad_match_u8_topk(const void* hi_u8, int M, int M_pad, const void* lo_u8, int N, int N_pad, const int32_t* hi_n2,
                      const int32_t* lo_n2, const float* lo_rnorm, int S, int k, int lo_index_base, int32_t* topk_idx,
                      double* topk_score, cudaStream_t st) {
    CUtensorMap map_hi, map_lo;
    const int ncta = pick_ncta(M, N_pad);
    int rc = launch_common(hi_u8, M_pad, lo_u8, N_pad, ncta, &map_hi, &map_lo);
    if (rc != MAD_OK) return rc;
    U8Args a = {};
    a.M = M; a.N = N; a.S = S;
    a.tiles_per_seg = (int)mad_ceil_div(mad_ceil_div(N, BN * ncta), S);
    a.hi_n2 = hi_n2; a.lo_n2 = lo_n2; a.lo_rnorm = lo_rnorm; a.cc = 0.0;
    a.k = k; a.lo_index_base = lo_index_base; a.topk_idx = topk_idx; a.topk_score = topk_score;
    a.local_tiles = getenv("MAD_TOPK_LOCAL") ? atoi(getenv("MAD_TOPK_LOCAL")) : TOP_LOCAL_TILES;
    a.dbg = getenv("MAD_TOPK_DBG") ? atoi(getenv("MAD_TOPK_DBG")) : 0;
    if (a.dbg & 32) {
        unsigned long long z[8] = {0};
        cudaMemcpyToSymbolAsync(g_top_dbg, z, sizeof(z), 0, cudaMemcpyHostToDevice, st);
    }
    {
        MAD_PROF("match_u8_topk_kernel", st);
        rc = k <= 8 ? launch_u8<MODE_TOP8>(ncta, M, S, map_hi, map_lo, a, st) : launch_u8<MODE_TOPK>(ncta, M, S, map_hi, map_lo, a, st);
    }
    if (rc == MAD_OK && (a.dbg & 32)) {
        unsigned long long z[8];
        cudaStreamSynchronize(st);
        cudaMemcpyFromSymbol(z, g_top_dbg, sizeof(z));
        const double ctas = (double)(ncta == 2 ? 2 * mad_ceil_div(M, 2 * BM) : mad_ceil_div(M, BM)) * S;
        fprintf(stderr, "[top8 dbg] per CTA: round cycles %.0f (per epilogue warp %.0f), publish-wait cycles %.0f, publishes %.0f, rounds %.0f, "
                        "drain passes %.0f, drain busy cycles %.0f (per drain warp %.0f), inserted %.0f, stale %.0f\n",
                z[0] / ctas, z[0] / ctas / 8, z[1] / ctas, z[2] / ctas, z[3] / ctas, z[4] / ctas, z[5] / ctas, z[5] / ctas / 4, z[6] / ctas, z[7] / ctas);
    }
    return rc;
}
