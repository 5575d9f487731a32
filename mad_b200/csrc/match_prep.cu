// a15 support kernels: descriptor-set preparation (exact norms, uint8 tensor-core operand) and the
// finish step of the one-pass threshold matcher (sort candidates into np.where's row-major order,
// evaluate the float64 cosine from exact integers).  mad/MaD.py:416-424.
#include <cub/cub.cuh>

#include "common.cuh"
#include "match_common.cuh"

namespace {

// One warp per (padded) row: squared norm, 1/sqrt(norm) as float, uint8 copy (values clamped to
// 255 -- max_entry tells the host whether the copy is exact), zero rows beyond `rows`; the set's largest
// squared norm (which kernels compute the dot products exactly) goes to max_norm2.
__global__ void __launch_bounds__(256)
dsc_prepare_kernel(const int16_t* __restrict__ dsc, int rows, int rows_padded, int32_t* __restrict__ norm2,
                   float* __restrict__ rnorm, uint8_t* __restrict__ u8, int32_t* __restrict__ max_entry,
                   int32_t* __restrict__ max_norm2) {
    const int row = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows_padded) return;
    long long acc = 0;
    int mx = 0;
    // lane handles 32 consecutive entries: 4 x (8 x int16 = 16 B) loads, 2 x 16 B stores
    uint32_t packed[8];
    if (row < rows) {
        const uint4* src = reinterpret_cast<const uint4*>(dsc + (long long)row * MAD_DSC_LEN + lane * 32);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const uint4 v = __ldg(src + q);
            const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int h = 0; h < 4; ++h) {
                const int e0 = (int)(int16_t)(w[h] & 0xFFFFu), e1 = (int)(int16_t)(w[h] >> 16);
                acc += (long long)e0 * e0 + (long long)e1 * e1;
                mx = max(mx, max(e0, e1));
                if (e0 < 0 || e1 < 0) mx = MAD_DSC_REFUSED;     // negative entries: not a descriptor
                const uint32_t b0 = (uint32_t)min(max(e0, 0), 255), b1 = (uint32_t)min(max(e1, 0), 255);
                const int slot = q * 8 + h * 2;                  // byte index within the lane's 32 bytes
                if ((slot & 3) == 0) packed[slot >> 2] = b0 | (b1 << 8);
                else packed[slot >> 2] |= (b0 << 16) | (b1 << 24);
            }
        }
    } else {
#pragma unroll
        for (int q = 0; q < 8; ++q) packed[q] = 0;
    }
    if (u8) {
        uint4* dst = reinterpret_cast<uint4*>(u8 + (long long)row * MAD_DSC_LEN + lane * 32);
        dst[0] = make_uint4(packed[0], packed[1], packed[2], packed[3]);
        dst[1] = make_uint4(packed[4], packed[5], packed[6], packed[7]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        acc += __shfl_xor_sync(0xFFFFFFFFu, acc, o);
        mx = max(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, o));
    }
    if (lane == 0) {
        if (acc > 0x7FFFFFFFLL) mx = MAD_DSC_REFUSED;           // norm does not fit int32: refuse the set
        if (row < rows) norm2[row] = (int32_t)acc;
        rnorm[row] = acc > 0 ? (float)(1.0 / sqrt((double)acc)) : 0.f;
        if (mx > 0) atomicMax(max_entry, mx);
        if (max_norm2 && acc > 0) atomicMax(max_norm2, (int32_t)min(acc, 0x7FFFFFFFLL));
    }
}

__global__ void pairs_finish_kernel(const unsigned long long* __restrict__ key, const int32_t* __restrict__ dot,
                                    long long n, unsigned long long lo_rows, const int32_t* __restrict__ hi_n2,
                                    const int32_t* __restrict__ lo_n2,
                                    int32_t* __restrict__ pair_hi, int32_t* __restrict__ pair_lo,
                                    double* __restrict__ score) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned long long k = key[i];
    const int row = (int)(k / lo_rows), col = (int)(k % lo_rows);      // key = row * lo_rows + col
    pair_hi[i] = row;
    pair_lo[i] = col;
    score[i] = mad_score(dot[i], (double)__ldg(hi_n2 + row), (double)__ldg(lo_n2 + col));
}

// Compact form: the exact integer dot product instead of the float64 score (12 instead of 16 bytes per pair on the way to
// the host, which recomputes dot / sqrt(|hi|^2 |lo|^2) from the norms with the same correctly rounded operations).
__global__ void pairs_finish_dot_kernel(const unsigned long long* __restrict__ key, const int32_t* __restrict__ dot, long long n,
                                        unsigned long long lo_rows, int32_t* __restrict__ pair_hi, int32_t* __restrict__ pair_lo,
                                        int32_t* __restrict__ pair_dot) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned long long k = key[i];
    pair_hi[i] = (int)(k / lo_rows);
    pair_lo[i] = (int)(k % lo_rows);
    pair_dot[i] = dot[i];
}

// The candidate counter is reset by a kernel, not cudaMemsetAsync: a memset may be routed through a
// copy engine and then queues behind a large device-to-host copy of another stream (observed: the
// matching kernel waited 1.4 ms for the descriptor table's copy-out).
__global__ void zero_u64_kernel(unsigned long long* p) { *p = 0ull; }

struct FinishLayout {
    size_t key_off, dot_off, cub_off, cub_bytes, total;
};

FinishLayout finish_layout(long long n) {
    FinishLayout L;
    const size_t nn = (size_t)(n > 0 ? n : 1);
    L.key_off = 0;
    L.dot_off = mad_align_up(nn * sizeof(unsigned long long), 256);
    L.cub_off = L.dot_off + mad_align_up(nn * sizeof(int32_t), 256);
    size_t b = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, b, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                    (const int32_t*)nullptr, (int32_t*)nullptr, (int)nn, 0, 64);
    L.cub_bytes = mad_align_up(b, 256);
    L.total = L.cub_off + L.cub_bytes;
    return L;
}

}  // namespace

extern "C" int mad_dsc_prepare(const int16_t* dsc, int rows, int rows_padded, int32_t* norm2, float* rnorm,
                               uint8_t* u8, int32_t* max_entry, int32_t* max_norm2, void* stream) {
    MAD_CHECK_ARG(rows >= 0 && rows_padded >= rows);
    if (rows_padded == 0) return MAD_OK;
    MAD_CHECK_ARG((rows == 0 || dsc) && norm2 && rnorm && max_entry);
    MAD_CHECK_ARG((reinterpret_cast<uintptr_t>(dsc) & 15) == 0 && (reinterpret_cast<uintptr_t>(u8) & 15) == 0);
    MAD_PROF("dsc_prepare_kernel", stream);
    dsc_prepare_kernel<<<(unsigned)mad_ceil_div((long long)rows_padded * 32, 256), 256, 0, (cudaStream_t)stream>>>(
        dsc, rows, rows_padded, norm2, rnorm, u8, max_entry, max_norm2);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" int mad_match_pairs(const MadDscSet* hi, const MadDscSet* lo, double cc, uint64_t* cand_key, int32_t* cand_dot,
                               uint64_t cap, uint64_t* count, void* stream) {
    MAD_CHECK_ARG(hi && lo && count && hi->rows >= 0 && lo->rows >= 0);
    cudaStream_t st = (cudaStream_t)stream;
    {
        MAD_PROF("zero_u64_kernel", st);
        zero_u64_kernel<<<1, 1, 0, st>>>(reinterpret_cast<unsigned long long*>(count));
        MAD_LAUNCH_OK();
    }
    if (hi->rows == 0 || lo->rows == 0) return MAD_OK;
    MAD_CHECK_ARG(hi->u8 && lo->u8 && hi->norm2 && lo->norm2 && lo->rnorm && cand_key && cand_dot);
    MAD_CHECK_ARG(hi->rows_padded >= hi->rows && hi->rows_padded % 128 == 0);
    MAD_CHECK_ARG(lo->rows_padded >= lo->rows && lo->rows_padded % 128 == 0);
    int rc = mad_check_descriptor_sets(hi, lo, "mad_match_pairs");
    if (rc != MAD_OK) return rc;
    if (hi->max_entry > 255 || lo->max_entry > 255) {
        mad_set_error("mad_match_pairs: descriptor entries up to %d do not fit the uint8 tensor-core operand "
                      "(use mad_match_count/mad_match_fill with impl = 2 or 1)",
                      hi->max_entry > lo->max_entry ? hi->max_entry : lo->max_entry);
        return MAD_ERR_ARG;
    }
    return mad_match_u8_pairs(hi->u8, hi->rows, hi->rows_padded, lo->u8, lo->rows, lo->rows_padded, hi->norm2, lo->norm2,
                              lo->rnorm, cc, reinterpret_cast<unsigned long long*>(cand_key), cand_dot,
                              (unsigned long long)cap, reinterpret_cast<unsigned long long*>(count), st);
}

extern "C" size_t mad_match_pairs_finish_workspace_bytes(long long n) { return finish_layout(n).total; }

static int pairs_finish_impl(const uint64_t* cand_key, const int32_t* cand_dot, long long n, int hi_rows, int lo_rows,
                             const int32_t* hi_n2, const int32_t* lo_n2, int32_t* pair_hi, int32_t* pair_lo, double* pair_score,
                             int32_t* pair_dot, void* workspace, size_t workspace_bytes, void* stream);

extern "C" int mad_match_pairs_finish(const uint64_t* cand_key, const int32_t* cand_dot, long long n, int hi_rows,
                                      int lo_rows, const int32_t* hi_n2, const int32_t* lo_n2, int32_t* pair_hi, int32_t* pair_lo,
                                      double* pair_score, void* workspace, size_t workspace_bytes, void* stream) {
    MAD_CHECK_ARG(n >= 0 && n < (1LL << 31));
    if (n == 0) return MAD_OK;
    MAD_CHECK_ARG(hi_n2 && lo_n2 && pair_score);
    return pairs_finish_impl(cand_key, cand_dot, n, hi_rows, lo_rows, hi_n2, lo_n2, pair_hi, pair_lo, pair_score, nullptr, workspace,
                             workspace_bytes, stream);
}

extern "C" int mad_match_pairs_finish_dot(const uint64_t* cand_key, const int32_t* cand_dot, long long n, int hi_rows, int lo_rows,
                                          int32_t* pair_hi, int32_t* pair_lo, int32_t* pair_dot, void* workspace,
                                          size_t workspace_bytes, void* stream) {
    MAD_CHECK_ARG(n >= 0 && n < (1LL << 31));
    if (n == 0) return MAD_OK;
    MAD_CHECK_ARG(pair_dot);
    return pairs_finish_impl(cand_key, cand_dot, n, hi_rows, lo_rows, nullptr, nullptr, pair_hi, pair_lo, nullptr, pair_dot, workspace,
                             workspace_bytes, stream);
}

static int pairs_finish_impl(const uint64_t* cand_key, const int32_t* cand_dot, long long n, int hi_rows, int lo_rows,
                             const int32_t* hi_n2, const int32_t* lo_n2, int32_t* pair_hi, int32_t* pair_lo, double* pair_score,
                             int32_t* pair_dot, void* workspace, size_t workspace_bytes, void* stream) {
    MAD_CHECK_ARG(cand_key && cand_dot && pair_hi && pair_lo && workspace && hi_rows > 0 && lo_rows > 0);
    const FinishLayout L = finish_layout(n);
    MAD_CHECK_ARG(workspace_bytes >= L.total);
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = reinterpret_cast<char*>(workspace);
    unsigned long long* key_sorted = reinterpret_cast<unsigned long long*>(ws + L.key_off);
    int32_t* dot_sorted = reinterpret_cast<int32_t*>(ws + L.dot_off);
    int key_bits = 1;                                               // keys are < hi_rows * lo_rows
    while (key_bits < 64 && (1ULL << key_bits) < (unsigned long long)hi_rows * (unsigned long long)lo_rows) ++key_bits;
    size_t b = L.cub_bytes;
    {
        MAD_PROF("cub_radix_sort_pairs", st);
        MAD_CUDA(cub::DeviceRadixSort::SortPairs(ws + L.cub_off, b, reinterpret_cast<const unsigned long long*>(cand_key),
                                                 key_sorted, cand_dot, dot_sorted, (int)n, 0, key_bits, st));
    }
    MAD_PROF("pairs_finish_kernel", st);
    if (pair_dot)
        pairs_finish_dot_kernel<<<(unsigned)mad_ceil_div(n, 256), 256, 0, st>>>(key_sorted, dot_sorted, n, (unsigned long long)lo_rows, pair_hi,
                                                                               pair_lo, pair_dot);
    else
        pairs_finish_kernel<<<(unsigned)mad_ceil_div(n, 256), 256, 0, st>>>(key_sorted, dot_sorted, n, (unsigned long long)lo_rows, hi_n2, lo_n2,
                                                                           pair_hi, pair_lo, pair_score);
    MAD_LAUNCH_OK();
    return MAD_OK;
}
