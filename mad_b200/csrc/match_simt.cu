// a15: descriptor matching (mad/MaD.py:416-424) -- support kernels and the SIMT integer kernel.
//
// The production contraction is the tcgen05 kernel in match_tc.cu.  This file holds what is
// shared (norms, fp16 operand conversion, scans, top-k merge) plus a plain CUDA-core integer
// kernel with the SAME output contract; it exists so the tensor-core path can be checked on the
// device against an independent implementation (tests) and is never selected implicitly.
//
// Contract: score(i,j) = dot(hi_i, lo_j) / sqrt(n_i * n_j) in float64 with the integer dot and
// squared norms exact (entries are small non-negative integers); pairs with score > cc are
// emitted row-major with lo ascending, exactly the order of np.where(preds > cc).
#include <cub/cub.cuh>
#include <cub/iterator/transform_input_iterator.cuh>

#include "common.cuh"
#include "match_common.cuh"

namespace {

__global__ void norms_kernel(const int16_t* __restrict__ dsc, int rows, int32_t* __restrict__ norm2) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= rows) return;
    const int16_t* p = dsc + (long long)warp * MAD_DSC_LEN;
    int s = 0;
    for (int k = lane; k < MAD_DSC_LEN; k += 32) { const int v = p[k]; s += v * v; }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
    if (lane == 0) norm2[warp] = s;
}

__global__ void to_half_kernel(const int16_t* __restrict__ dsc, int rows, int rows_padded, __half* __restrict__ out) {
    const long long total = (long long)rows_padded * MAD_DSC_LEN;
    for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < total; g += (long long)gridDim.x * blockDim.x) {
        const long long row = g / MAD_DSC_LEN;
        out[g] = (row < rows) ? __int2half_rn((int)dsc[g]) : __float2half(0.f);
    }
}

constexpr int TM = 64, TN = 64, TK = 64;

// mode 0: count, 1: fill, 2: top-k
__global__ void __launch_bounds__(256)
match_simt_kernel(const int16_t* __restrict__ hi, int M, const int16_t* __restrict__ lo, int N,
                  const int32_t* __restrict__ hi_n2, const int32_t* __restrict__ lo_n2, double cc, int mode,
                  int S, int cols_per_seg, int32_t* __restrict__ row_count, const int64_t* __restrict__ row_offset,
                  int32_t* __restrict__ pair_hi, int32_t* __restrict__ pair_lo, double* __restrict__ pair_score,
                  int k, int lo_index_base, int32_t* __restrict__ topk_idx, double* __restrict__ topk_score) {
    __shared__ int16_t sa[TM][TK + 2];
    __shared__ int16_t sb[TN][TK + 2];
    __shared__ int dots[TM][TN + 1];
    const int tid = threadIdx.x;
    const int m0 = blockIdx.x * TM;
    const int seg = blockIdx.y;
    const int n_begin = seg * cols_per_seg;
    const int n_end = min(N, n_begin + cols_per_seg);
    const int ty = tid / 16, tx = tid % 16;   // 16x16 threads, 4x4 outputs each

    // per-row running state (threads 0..63 own one row each)
    const int my_row = m0 + tid;
    long long wpos = 0;
    int cnt = 0;
    double bs[MAD_TOPK_MAX];
    int bi[MAD_TOPK_MAX];
    if (mode == 2) for (int q = 0; q < MAD_TOPK_MAX; ++q) { bs[q] = -INFINITY; bi[q] = -1; }
    if (mode == 1 && tid < TM && my_row < M) wpos = row_offset[(long long)my_row * S + seg];
    const double my_n2 = (tid < TM && my_row < M) ? (double)hi_n2[my_row] : 0.0;

    for (int n0 = n_begin; n0 < n_end; n0 += TN) {
        int acc[4][4];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) acc[a][b] = 0;
        for (int k0 = 0; k0 < MAD_DSC_LEN; k0 += TK) {
            for (int q = tid; q < TM * TK; q += 256) {
                const int r = q / TK, c = q % TK;
                sa[r][c] = (m0 + r < M) ? hi[(long long)(m0 + r) * MAD_DSC_LEN + k0 + c] : (int16_t)0;
                sb[r][c] = (n0 + r < n_end) ? lo[(long long)(n0 + r) * MAD_DSC_LEN + k0 + c] : (int16_t)0;
            }
            __syncthreads();
#pragma unroll 8
            for (int kk = 0; kk < TK; ++kk) {
                int av[4], bv[4];
#pragma unroll
                for (int a = 0; a < 4; ++a) av[a] = sa[ty * 4 + a][kk];
#pragma unroll
                for (int b = 0; b < 4; ++b) bv[b] = sb[tx * 4 + b][kk];
#pragma unroll
                for (int a = 0; a < 4; ++a)
#pragma unroll
                    for (int b = 0; b < 4; ++b) acc[a][b] += av[a] * bv[b];
            }
            __syncthreads();
        }
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) dots[ty * 4 + a][tx * 4 + b] = acc[a][b];
        __syncthreads();
        if (tid < TM && my_row < M) {
            for (int j = 0; j < TN && n0 + j < n_end; ++j) {
                const double s = mad_score(dots[tid][j], my_n2, (double)lo_n2[n0 + j]);
                if (mode == 2) {
                    mad_topk_insert(bs, bi, k, s, lo_index_base + n0 + j);
                } else if (s > cc) {
                    if (mode == 1) { pair_hi[wpos] = my_row; pair_lo[wpos] = n0 + j; pair_score[wpos] = s; ++wpos; }
                    ++cnt;
                }
            }
        }
        __syncthreads();
    }
    if (tid < TM && my_row < M) {
        if (mode == 0) row_count[(long long)my_row * S + seg] = cnt;
        if (mode == 2)
            for (int q = 0; q < k; ++q) {
                const long long o = ((long long)seg * M + my_row) * k + q;
                topk_idx[o] = bi[q];
                topk_score[o] = bs[q];
            }
    }
}

__global__ void topk_merge_kernel(const int32_t* __restrict__ idx_in, const double* __restrict__ score_in, int G, int M,
                                  int k, int32_t* __restrict__ idx_out, double* __restrict__ score_out) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= M) return;
    double bs[MAD_TOPK_MAX];
    int bi[MAD_TOPK_MAX];
    for (int q = 0; q < MAD_TOPK_MAX; ++q) { bs[q] = -INFINITY; bi[q] = -1; }
    bool incomplete = false;                    // an input list of this row is incomplete (-2): so is the merged one
    for (int g = 0; g < G; ++g)
        for (int q = 0; q < k; ++q) {
            const long long p = ((long long)g * M + row) * k + q;
            const int id = idx_in[p];
            if (id >= 0) mad_topk_insert(bs, bi, k, score_in[p], id);
            incomplete |= id == MAD_TOPK_INCOMPLETE;
        }
    for (int q = 0; q < k; ++q) {
        idx_out[(long long)row * k + q] = incomplete ? MAD_TOPK_INCOMPLETE : bi[q];
        score_out[(long long)row * k + q] = incomplete ? -INFINITY : bs[q];
    }
}

struct CastI64 {
    __host__ __device__ int64_t operator()(const int32_t& v) const { return (int64_t)v; }
};

__global__ void scan_total_kernel(const int32_t* in, const int64_t* out, int n, int64_t* total) {
    *total = out[n - 1] + (int64_t)in[n - 1];
}

}  // namespace

extern "C" int mad_dsc_norms(const int16_t* dsc, int rows, int32_t* norm2, void* stream) {
    MAD_CHECK_ARG(rows >= 0);
    if (rows == 0) return MAD_OK;
    MAD_CHECK_ARG(dsc && norm2);
    MAD_PROF("norms_kernel", stream);
    norms_kernel<<<(int)mad_ceil_div((long long)rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(dsc, rows, norm2);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" int mad_dsc_to_half(const int16_t* dsc, int rows, int rows_padded, void* half_out, void* stream) {
    MAD_CHECK_ARG(rows >= 0 && rows_padded >= rows);
    if (rows_padded == 0) return MAD_OK;
    MAD_CHECK_ARG(dsc && half_out);
    const long long total = (long long)rows_padded * MAD_DSC_LEN;
    const int blocks = (int)std::min<long long>(mad_ceil_div(total, 256), (long long)mad_sm_count() * 16);
    MAD_PROF("to_half_kernel", stream);
    to_half_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(dsc, rows, rows_padded, reinterpret_cast<__half*>(half_out));
    MAD_LAUNCH_OK();
    return MAD_OK;
}

int mad_match_simt(const int16_t* hi, int M, const int16_t* lo, int N, const int32_t* hi_n2, const int32_t* lo_n2,
                   double cc, int mode, int S, int32_t* seg_count, const int64_t* seg_offset, int32_t* pair_hi,
                   int32_t* pair_lo, double* pair_score, int k, int lo_index_base, int32_t* topk_idx,
                   double* topk_score, cudaStream_t st) {
    const int n_tiles = (int)mad_ceil_div(N, MAD_MATCH_SEG_TILE);
    const int cols_per_seg = (int)mad_ceil_div(n_tiles, S) * MAD_MATCH_SEG_TILE;
    dim3 grid((unsigned)mad_ceil_div(M, TM), (unsigned)S);
    MAD_PROF("match_simt_kernel", st);
    match_simt_kernel<<<grid, 256, 0, st>>>(hi, M, lo, N, hi_n2, lo_n2, cc, mode, S, cols_per_seg, seg_count, seg_offset,
                                            pair_hi, pair_lo, pair_score, k, lo_index_base, topk_idx, topk_score);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" size_t mad_exclusive_scan_workspace_bytes(int n) {
    size_t b = 0;
    cub::TransformInputIterator<int64_t, CastI64, const int32_t*> it((const int32_t*)nullptr, CastI64());
    cub::DeviceScan::ExclusiveSum(nullptr, b, it, (int64_t*)nullptr, n > 0 ? n : 1);
    return mad_align_up(b, 256);
}

extern "C" int mad_exclusive_scan_i32_to_i64(const int32_t* in, int n, int64_t* out, int64_t* total, void* workspace,
                                             size_t workspace_bytes, void* stream) {
    MAD_CHECK_ARG(n >= 0 && total);
    cudaStream_t st = (cudaStream_t)stream;
    if (n == 0) {
        MAD_CUDA(cudaMemsetAsync(total, 0, sizeof(int64_t), st));
        return MAD_OK;
    }
    MAD_CHECK_ARG(in && out && workspace);
    cub::TransformInputIterator<int64_t, CastI64, const int32_t*> it(in, CastI64());
    size_t b = workspace_bytes;
    {
        MAD_PROF("cub_exclusive_sum", st);
        MAD_CUDA(cub::DeviceScan::ExclusiveSum(workspace, b, it, out, n, st));
    }
    MAD_PROF("scan_total_kernel", st);
    scan_total_kernel<<<1, 1, 0, st>>>(in, out, n, total);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

int mad_topk_merge_launch(const int32_t* idx_in, const double* score_in, int G, int M, int k, int32_t* idx_out,
                          double* score_out, cudaStream_t st) {
    MAD_PROF("topk_merge_kernel", st);
    topk_merge_kernel<<<(int)mad_ceil_div(M, 128), 128, 0, st>>>(idx_in, score_in, G, M, k, idx_out, score_out);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" int mad_topk_merge(const int32_t* idx_in, const double* score_in, int G, int M, int k, int32_t* idx_out,
                              double* score_out, void* stream) {
    MAD_CHECK_ARG(G >= 1 && M >= 0 && k >= 1 && k <= MAD_TOPK_MAX);
    if (M == 0) return MAD_OK;
    MAD_CHECK_ARG(idx_in && score_in && idx_out && score_out);
    return mad_topk_merge_launch(idx_in, score_in, G, M, k, idx_out, score_out, (cudaStream_t)stream);
}
