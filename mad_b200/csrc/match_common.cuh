// Shared pieces of the descriptor-matching kernels (mad/MaD.py:416-424).
#pragma once
#include <math.h>
#include "common.cuh"

#define MAD_TOPK_MAX 32

// cosine similarity from the exact integer dot product and exact squared norms, in float64:
// one sqrt and one division, both correctly rounded (IEEE) on host and device alike.
__host__ __device__ __forceinline__ double mad_score(int dot, double n2a, double n2b) {
    const double p = n2a * n2b;
    return p > 0.0 ? (double)dot / sqrt(p) : 0.0;   // zero descriptors stay zero vectors (:416-417)
}

// Keeps (bs, bi)[0..k) sorted by (score descending, index ascending).
__host__ __device__ __forceinline__ void mad_topk_insert(double* bs, int* bi, int k, double s, int id) {
    const double ls = bs[k - 1];
    const int li = bi[k - 1];
    if (!(s > ls || (s == ls && (li < 0 || id < li)))) return;
    int q = k - 1;
    while (q > 0) {
        const double ps = bs[q - 1];
        const int pi = bi[q - 1];
        if (s > ps || (s == ps && (pi < 0 || id < pi))) { bs[q] = ps; bi[q] = pi; --q; }
        else break;
    }
    bs[q] = s;
    bi[q] = id;
}

// (s, id) ranks before (ps, pi) in the (score desc, index asc) order; empty slots (pi < 0) rank last.
__host__ __device__ __forceinline__ bool mad_topk_before(double s, int id, double ps, int pi) {
    return s > ps || (s == ps && (pi < 0 || id < pi));
}

// Register-resident list of exactly 8 entries (static indices only): new[q] = the old q-1 if the
// candidate ranks before it, else the candidate if it ranks before the old q, else the old q.
__device__ __forceinline__ void mad_top8_insert(double (&bs)[8], int (&bi)[8], double s, int id) {
    bool c[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) c[q] = mad_topk_before(s, id, bs[q], bi[q]);
#pragma unroll
    for (int q = 7; q >= 1; --q) {
        bs[q] = c[q - 1] ? bs[q - 1] : (c[q] ? s : bs[q]);
        bi[q] = c[q - 1] ? bi[q - 1] : (c[q] ? id : bi[q]);
    }
    bs[0] = c[0] ? s : bs[0];
    bi[0] = c[0] ? id : bi[0];
}

// Register list of 8 entries (float32 image of the score, dot, |lo|^2, index) for ONE hi row (|hi|^2 = n2a).  The images have
// a relative error < 1e-6, so two entries whose images differ by more than 4e-6 of the larger one are ordered by them; closer
// ones are ordered as every other path orders them: by the float64 mad_score, then by the index.  (Equal integer ratios
// dot^2 / |lo|^2 do not imply equal float64 scores: a lo row b and its multiple m b have the same cosine, yet their two
// roundings of d / sqrt(n_a n_b) and m d / sqrt(n_a m^2 n_b) differ by one ulp in about a third of the cases.)
// (out of line: it runs for near-ties only and must not bloat its callers -- the matcher's warps share one instruction cache)
static __device__ __noinline__ bool mad_score_before_nl(int d, int n, int id, int pd, int pn, int pi, double n2a) {
    return mad_topk_before(mad_score(d, n2a, (double)n), id, mad_score(pd, n2a, (double)pn), pi);
}
__device__ __forceinline__ bool mad_score32_before(float s, int d, int n, int id, float ps, int pd, int pn, int pi, double n2a) {
    if (pi < 0) return true;
    const float tol = 4e-6f * fmaxf(s, ps);
    if (s > ps + tol) return true;
    if (s < ps - tol) return false;
    return mad_score_before_nl(d, n, id, pd, pn, pi, n2a);
}

// Called by ALL lanes of a warp (`active` = this lane has a candidate).  The eight position decisions are taken on the
// images; only if some lane of the warp has an image within the tolerance of one of its entries does the warp redo the
// decisions on the float64 scores (one warp-uniform branch: square roots and divisions stay off the common path).
__device__ __forceinline__ void mad_top8f_insert(float (&ts)[8], int (&td)[8], int (&tn)[8], int (&bi)[8], bool active, float s,
                                                 int d, int n, int id, double n2a) {
    bool c[8];
    bool amb = false;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const float ps = ts[q];
        const bool empty = bi[q] < 0;
        const float tol = 4e-6f * fmaxf(s, ps);
        const bool gt = s > ps + tol, lt = s < ps - tol;
        c[q] = active && (empty || gt);
        amb |= active && !empty && !gt && !lt;
    }
    if (__any_sync(0xFFFFFFFFu, amb)) {
#pragma unroll
        for (int q = 0; q < 8; ++q) c[q] = active && mad_score32_before(s, d, n, id, ts[q], td[q], tn[q], bi[q], n2a);
    }
#pragma unroll
    for (int q = 7; q >= 1; --q) {
        ts[q] = c[q - 1] ? ts[q - 1] : (c[q] ? s : ts[q]);
        td[q] = c[q - 1] ? td[q - 1] : (c[q] ? d : td[q]);
        tn[q] = c[q - 1] ? tn[q - 1] : (c[q] ? n : tn[q]);
        bi[q] = c[q - 1] ? bi[q - 1] : (c[q] ? id : bi[q]);
    }
    ts[0] = c[0] ? s : ts[0];
    td[0] = c[0] ? d : td[0];
    tn[0] = c[0] ? n : tn[0];
    bi[0] = c[0] ? id : bi[0];
}

// Release / acquire accesses to a shared-memory state word (CTA scope): the hand-off protocols below order their data
// with these instead of __threadfence_block(), which compiles to the much heavier MEMBAR.SC.CTA.
__device__ __forceinline__ void mad_st_release_cta(volatile int* p, int v) {
    asm volatile("st.release.cta.shared::cta.s32 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared((const void*)p)), "r"(v) : "memory");
}
__device__ __forceinline__ int mad_ld_acquire_cta(volatile int* p) {
    int v;
    asm volatile("ld.acquire.cta.shared::cta.s32 %0, [%1];" : "=r"(v) : "r"((uint32_t)__cvta_generic_to_shared((const void*)p)) : "memory");
    return v;
}

// v[j] for a run-time j without spilling v to local memory: 5 levels of selects.
__device__ __forceinline__ uint32_t mad_select32(const uint32_t (&v)[32], int j) {
    uint32_t a[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) a[i] = (j & 1) ? v[2 * i + 1] : v[2 * i];
    uint32_t b[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) b[i] = (j & 2) ? a[2 * i + 1] : a[2 * i];
    uint32_t c[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) c[i] = (j & 4) ? b[2 * i + 1] : b[2 * i];
    const uint32_t d0 = (j & 8) ? c[1] : c[0], d1 = (j & 8) ? c[3] : c[2];
    return (j & 16) ? d1 : d0;
}

// Both kernels cut the lo axis into S segments of `tiles_per_seg` 256-column tiles.
#define MAD_MATCH_SEG_TILE 256

// MAD_ERR_ARG (with a message naming `who`) if either set is flagged as not a descriptor set (MAD_DSC_REFUSED).
int mad_check_descriptor_sets(const MadDscSet* hi, const MadDscSet* lo, const char* who);

int mad_match_simt(const int16_t* hi, int M, const int16_t* lo, int N, const int32_t* hi_n2, const int32_t* lo_n2,
                   double cc, int mode, int S, int32_t* seg_count, const int64_t* seg_offset, int32_t* pair_hi,
                   int32_t* pair_lo, double* pair_score, int k, int lo_index_base, int32_t* topk_idx,
                   double* topk_score, cudaStream_t st);

int mad_match_tc_segments(int M, int N);
int mad_match_tc(const void* hi_half, int M, int M_pad, const void* lo_half, int N, int N_pad,
                 const int32_t* hi_n2, const int32_t* lo_n2, double cc, int mode, int S, int32_t* seg_count,
                 const int64_t* seg_offset, int32_t* pair_hi, int32_t* pair_lo, double* pair_score, int k,
                 int lo_index_base, int32_t* topk_idx, double* topk_score, cudaStream_t st);
int mad_topk_merge_launch(const int32_t* idx_in, const double* score_in, int G, int M, int k, int32_t* idx_out,
                          double* score_out, cudaStream_t st);

// uint8 tcgen05 kernel (match_u8.cu): 128-column tiles, hi tile resident in shared memory.
int mad_match_u8_segments(int M, int N);
int mad_match_u8_segments_topk(int M, int N);
int mad_match_u8_pairs(const void* hi_u8, int M, int M_pad, const void* lo_u8, int N, int N_pad, const int32_t* hi_n2,
                       const int32_t* lo_n2, const float* lo_rnorm, double cc, unsigned long long* cand_key,
                       int32_t* cand_dot, unsigned long long cap, unsigned long long* count, cudaStream_t st);
int mad_match_u8_topk(const void* hi_u8, int M, int M_pad, const void* lo_u8, int N, int N_pad, const int32_t* hi_n2,
                      const int32_t* lo_n2, const float* lo_rnorm, int S, int k, int lo_index_base, int32_t* topk_idx,
                      double* topk_score, cudaStream_t st);
