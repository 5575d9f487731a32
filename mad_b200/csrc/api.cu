// C-ABI glue of libmad_b200: error text, device info, matching entry points (dispatch between
// the tcgen05 kernel and the SIMT check kernel -- never implicit).
#include <stdarg.h>
#include <string.h>

#include "common.cuh"
#include "match_common.cuh"

static thread_local char g_err[512] = "";

void mad_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int mad_sm_count() {
    static int cached = 0;
    if (!cached) {
        int dev = 0, n = 0;
        if (cudaGetDevice(&dev) == cudaSuccess &&
            cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
            cached = n;
        else
            return 148;
    }
    return cached;
}

// ---- launch accounting + optional per-launch event timing ---------------------------------------
#include <atomic>
#include <mutex>
#include <vector>
namespace {
struct ProfRec { const char* name; cudaEvent_t a, b; };
std::atomic<long long> g_launches{0};
std::atomic<int> g_prof_on{0};
std::mutex g_prof_mu;
std::vector<ProfRec> g_prof;
}  // namespace

MadProfScope::MadProfScope(const char* name, cudaStream_t stream) : slot(-1), st(stream) {
    g_launches.fetch_add(1, std::memory_order_relaxed);
    if (!g_prof_on.load(std::memory_order_relaxed)) return;
    ProfRec r;
    r.name = name;
    if (cudaEventCreate(&r.a) != cudaSuccess || cudaEventCreate(&r.b) != cudaSuccess) return;
    cudaEventRecord(r.a, st);
    std::lock_guard<std::mutex> lk(g_prof_mu);
    g_prof.push_back(r);
    slot = (int)g_prof.size() - 1;
}
MadProfScope::~MadProfScope() {
    if (slot < 0) return;
    std::lock_guard<std::mutex> lk(g_prof_mu);
    cudaEventRecord(g_prof[slot].b, st);
}

extern "C" long long mad_launch_count(void) { return g_launches.load(); }
extern "C" int mad_profile_enable(int on) {
    g_prof_on.store(on ? 1 : 0);
    return MAD_OK;
}
extern "C" int mad_profile_count(void) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    return (int)g_prof.size();
}
extern "C" int mad_profile_get(int i, const char** name, float* ms) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    MAD_CHECK_ARG(name && ms && i >= 0 && i < (int)g_prof.size());
    MAD_CUDA(cudaEventSynchronize(g_prof[i].b));
    MAD_CUDA(cudaEventElapsedTime(ms, g_prof[i].a, g_prof[i].b));
    *name = g_prof[i].name;
    return MAD_OK;
}
extern "C" int mad_profile_reset(void) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    for (auto& r : g_prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    g_prof.clear();
    return MAD_OK;
}

extern "C" const char* mad_last_error_string(void) { return g_err; }
extern "C" int mad_version(void) { return 100; }

extern "C" int mad_device_info(int* sm_count, int* cc_major, int* cc_minor) {
    MAD_CHECK_ARG(sm_count && cc_major && cc_minor);
    int dev = 0;
    MAD_CUDA(cudaGetDevice(&dev));
    MAD_CUDA(cudaDeviceGetAttribute(sm_count, cudaDevAttrMultiProcessorCount, dev));
    MAD_CUDA(cudaDeviceGetAttribute(cc_major, cudaDevAttrComputeCapabilityMajor, dev));
    MAD_CUDA(cudaDeviceGetAttribute(cc_minor, cudaDevAttrComputeCapabilityMinor, dev));
    return MAD_OK;
}

int mad_check_descriptor_sets(const MadDscSet* hi, const MadDscSet* lo, const char* who) {
    if (hi->max_entry >= MAD_DSC_REFUSED || lo->max_entry >= MAD_DSC_REFUSED) {
        mad_set_error("%s: not a descriptor set (a negative entry, or a squared norm >= 2^31)", who);
        return MAD_ERR_ARG;
    }
    return MAD_OK;
}

// The fp16 kernel accumulates in fp32: exact while every partial sum of a dot product is <= 2^24.  Entries in [0, 2048]
// are exact in fp16, and with max |hi|^2 * max |lo|^2 <= 2^48 every dot product is <= 2^24 (Cauchy-Schwarz).
static bool fp16_exact(const MadDscSet* hi, const MadDscSet* lo) {
    return hi->max_entry >= 0 && lo->max_entry >= 0 && hi->max_entry <= 2048 && lo->max_entry <= 2048 &&
           hi->max_norm2 >= 0 && lo->max_norm2 >= 0 && (double)hi->max_norm2 * (double)lo->max_norm2 <= 281474976710656.0;
}

static int check_sets(const MadDscSet* hi, const MadDscSet* lo, int impl) {
    MAD_CHECK_ARG(hi && lo && hi->rows >= 0 && lo->rows >= 0);
    MAD_CHECK_ARG(impl == 0 || impl == 1 || impl == 2);
    if (hi->rows == 0 || lo->rows == 0) return MAD_OK;
    MAD_CHECK_ARG(hi->norm2 && lo->norm2);
    const int rc = mad_check_descriptor_sets(hi, lo, "mad_match");
    if (rc != MAD_OK) return rc;
    if (impl == 1) {
        MAD_CHECK_ARG(hi->dsc && lo->dsc);
    } else {
        if (impl == 2) MAD_CHECK_ARG(hi->half && lo->half);
        if (impl == 2 && !fp16_exact(hi, lo)) {
            mad_set_error("mad_match: the fp16 kernel (impl = 2) is exact only for entries in [0, 2048] and max |hi|^2 * max "
                          "|lo|^2 <= 2^48 (here max entry %d / %d, max |.|^2 %d / %d; -1 = not known): use impl = 1",
                          hi->max_entry, lo->max_entry, hi->max_norm2, lo->max_norm2);
            return MAD_ERR_ARG;
        }
        if (impl == 0) MAD_CHECK_ARG(hi->u8 && lo->u8 && lo->rnorm);
        MAD_CHECK_ARG(hi->rows_padded >= hi->rows && hi->rows_padded % 128 == 0);
        MAD_CHECK_ARG(lo->rows_padded >= lo->rows && lo->rows_padded % 128 == 0);
        if (impl == 0 && (hi->max_entry > 255 || lo->max_entry > 255)) {
            mad_set_error("mad_match: descriptor entries up to %d do not fit the uint8 kernel (use impl = 2)",
                          hi->max_entry > lo->max_entry ? hi->max_entry : lo->max_entry);
            return MAD_ERR_ARG;
        }
    }
    return MAD_OK;
}

static int run_match(const MadDscSet* hi, const MadDscSet* lo, double cc, int mode, int S, int32_t* seg_count,
                     const int64_t* seg_offset, int32_t* pair_hi, int32_t* pair_lo, double* pair_score, int k, int base,
                     int32_t* topk_idx, double* topk_score, int impl, cudaStream_t st) {
    if (impl == 1)
        return mad_match_simt(hi->dsc, hi->rows, lo->dsc, lo->rows, hi->norm2, lo->norm2, cc, mode, S, seg_count, seg_offset,
                              pair_hi, pair_lo, pair_score, k, base, topk_idx, topk_score, st);
    return mad_match_tc(hi->half, hi->rows, hi->rows_padded, lo->half, lo->rows, lo->rows_padded, hi->norm2, lo->norm2, cc,
                        mode, S, seg_count, seg_offset, pair_hi, pair_lo, pair_score, k, base, topk_idx, topk_score, st);
}

// Segment count of the two-pass count / fill kernels (impl 1 and 2 share the fp16 kernel's choice: 256-column tiles,
// same output layout).  impl 0 (one-pass uint8 kernel) has no count / fill form: mad_match_count / mad_match_fill reject
// it; the value returned for impl 0 only sizes the top-k workspace of that kernel.
extern "C" int mad_match_segments(int M, int N, int impl) {
    return impl == 0 ? mad_match_u8_segments(M, N) : mad_match_tc_segments(M, N);
}

static int check_segments(const MadDscSet* hi, const MadDscSet* lo, int n_seg) {
    const int n_tiles = (int)mad_ceil_div(lo->rows, 128);
    MAD_CHECK_ARG(n_seg >= 1 && n_seg <= (n_tiles > 0 ? n_tiles : 1));
    (void)hi;
    return MAD_OK;
}

extern "C" int mad_match_count(const MadDscSet* hi, const MadDscSet* lo, double cc, int n_seg, int32_t* seg_count,
                               int impl, void* stream) {
    if (impl == 0) {
        mad_set_error("%s: impl 0 (the one-pass uint8 tcgen05 kernel) has no count/fill form -- call mad_match_pairs + "
                      "mad_match_pairs_finish; count/fill serve impl 1 (SIMT check) and 2 (fp16 tcgen05)", "mad_match_count");
        return MAD_ERR_ARG;
    }
    int rc = check_sets(hi, lo, impl);
    if (rc != MAD_OK) return rc;
    if (hi->rows == 0) return MAD_OK;
    MAD_CHECK_ARG(seg_count && n_seg >= 1);
    if (lo->rows == 0) {
        MAD_CUDA(cudaMemsetAsync(seg_count, 0, sizeof(int32_t) * (size_t)hi->rows * n_seg, (cudaStream_t)stream));
        return MAD_OK;
    }
    rc = check_segments(hi, lo, n_seg);
    if (rc != MAD_OK) return rc;
    return run_match(hi, lo, cc, 0, n_seg, seg_count, nullptr, nullptr, nullptr, nullptr, 0, 0, nullptr, nullptr, impl,
                     (cudaStream_t)stream);
}

extern "C" int mad_match_fill(const MadDscSet* hi, const MadDscSet* lo, double cc, int n_seg, const int64_t* seg_offset,
                              int32_t* pair_hi, int32_t* pair_lo, double* pair_score, int impl, void* stream) {
    if (impl == 0) {
        mad_set_error("%s: impl 0 (the one-pass uint8 tcgen05 kernel) has no count/fill form -- call mad_match_pairs + "
                      "mad_match_pairs_finish; count/fill serve impl 1 (SIMT check) and 2 (fp16 tcgen05)", "mad_match_fill");
        return MAD_ERR_ARG;
    }
    int rc = check_sets(hi, lo, impl);
    if (rc != MAD_OK) return rc;
    if (hi->rows == 0 || lo->rows == 0) return MAD_OK;
    MAD_CHECK_ARG(seg_offset && pair_hi && pair_lo && pair_score);
    rc = check_segments(hi, lo, n_seg);
    if (rc != MAD_OK) return rc;
    return run_match(hi, lo, cc, 1, n_seg, nullptr, seg_offset, pair_hi, pair_lo, pair_score, 0, 0, nullptr, nullptr, impl,
                     (cudaStream_t)stream);
}

// Partial top-k lists a kernel writes per hi row: the uint8 kernel has two epilogue groups per
// segment, each with its own list.
// k <= 8: three lists per segment (the drain warps' list + the two epilogue groups' lists of the sweep's first tiles);
// k > 8: one per (segment, group)
static int u8_lists_per_segment(int k) { return k <= 8 ? 3 : 2; }
static int topk_lists(int M, int N, int k, int impl) {
    return impl == 0 ? u8_lists_per_segment(k) * mad_match_u8_segments_topk(M, N) : mad_match_segments(M, N, impl);
}

static size_t topk_part_workspace_bytes(int M, int N, int k, int impl) {
    const int S = topk_lists(M, N, k, impl);
    if (S <= 1 || M <= 0) return 256;
    return mad_align_up((size_t)S * M * k * sizeof(int32_t), 256) + mad_align_up((size_t)S * M * k * sizeof(double), 256);
}

// Rows of a poorly filled LAST WAVE of the uint8 top-8 kernel.  A CTA pair owns 256 hi rows and sweeps the whole lo set, so
// 100 000 rows are 391 pairs = 5.28 waves of 74 and the last wave keeps 28 % of the machine busy for a full sweep.  When the
// last wave is at most half full its rows get a launch of their own with the lo axis cut into segments (more, shorter CTAs):
// 5 full waves + a short tail launch instead of 6 waves.
static int topk_tail_rows(int M, int k, int impl) {
    if (impl != 0 || k > 8 || getenv("MAD_TOPK_NO_TAIL")) return 0;
    const int per_wave = mad_sm_count() / 2;
    const int pairs = (int)mad_ceil_div(M, 256);
    if (per_wave <= 0 || pairs <= per_wave) return 0;
    const int tail = pairs % per_wave;
    if (tail == 0 || 2 * tail > per_wave) return 0;
    return M - (pairs - tail) * 256;
}

extern "C" size_t mad_match_topk_workspace_bytes(int M, int N, int k, int impl) {
    const int tail = topk_tail_rows(M, k, impl);
    if (tail <= 0) return topk_part_workspace_bytes(M, N, k, impl);
    return std::max(topk_part_workspace_bytes(M - tail, N, k, impl), topk_part_workspace_bytes(tail, N, k, impl));
}

static int topk_part(const MadDscSet* hi, const MadDscSet* lo, int k, int lo_index_base, int32_t* topk_idx, double* topk_score,
                     void* workspace, size_t workspace_bytes, int impl, cudaStream_t st) {
    const int M = hi->rows;
    const int S = topk_lists(M, lo->rows, k, impl);                // lists to merge
    auto run_topk = [&](int lists, int32_t* oi, double* os) {
        const int segs = impl == 0 ? lists / u8_lists_per_segment(k) : lists;
        if (impl == 0)
            return mad_match_u8_topk(hi->u8, hi->rows, hi->rows_padded, lo->u8, lo->rows, lo->rows_padded, hi->norm2,
                                     lo->norm2, lo->rnorm, segs, k, lo_index_base, oi, os, st);
        return run_match(hi, lo, 0.0, 2, segs, nullptr, nullptr, nullptr, nullptr, nullptr, k, lo_index_base, oi, os, impl, st);
    };
    if (S == 1) return run_topk(1, topk_idx, topk_score);
    MAD_CHECK_ARG(workspace && workspace_bytes >= topk_part_workspace_bytes(M, lo->rows, k, impl));
    int32_t* pidx = reinterpret_cast<int32_t*>(workspace);
    double* pscore = reinterpret_cast<double*>(reinterpret_cast<char*>(workspace) +
                                               mad_align_up((size_t)S * M * k * sizeof(int32_t), 256));
    int rc = run_topk(S, pidx, pscore);
    if (rc != MAD_OK) return rc;
    return mad_topk_merge_launch(pidx, pscore, S, M, k, topk_idx, topk_score, st);
}

extern "C" int mad_match_topk(const MadDscSet* hi, const MadDscSet* lo, int k, int lo_index_base, int32_t* topk_idx,
                              double* topk_score, void* workspace, size_t workspace_bytes, int impl, void* stream) {
    int rc = check_sets(hi, lo, impl);
    if (rc != MAD_OK) return rc;
    MAD_CHECK_ARG(k >= 1 && k <= MAD_TOPK_MAX);
    if (hi->rows == 0) return MAD_OK;
    MAD_CHECK_ARG(topk_idx && topk_score);
    cudaStream_t st = (cudaStream_t)stream;
    const int M = hi->rows;
    if (lo->rows == 0) {            // nothing to match: -1 / -inf padding
        MAD_CUDA(cudaMemsetAsync(topk_idx, 0xFF, sizeof(int32_t) * (size_t)M * k, st));
        // -inf as float64 = 0xFFF0000000000000: written by the merge kernel over zero shards
        return mad_topk_merge_launch(topk_idx, topk_score, 0, M, k, topk_idx, topk_score, st);
    }
    const int tail = topk_tail_rows(M, k, impl);
    if (tail <= 0) return topk_part(hi, lo, k, lo_index_base, topk_idx, topk_score, workspace, workspace_bytes, impl, st);
    // two launches on the same stream (the workspace is reused in stream order): the full waves, then the tail rows
    const int M0 = M - tail;                                       // a multiple of 256
    MadDscSet a = *hi, b = *hi;
    a.rows = M0;
    a.rows_padded = M0;
    b.rows = tail;
    b.rows_padded = hi->rows_padded - M0;
    b.dsc = hi->dsc ? hi->dsc + (size_t)M0 * MAD_DSC_LEN : nullptr;
    b.u8 = hi->u8 ? hi->u8 + (size_t)M0 * MAD_DSC_LEN : nullptr;
    b.norm2 = hi->norm2 + M0;
    b.rnorm = hi->rnorm ? hi->rnorm + M0 : nullptr;
    rc = topk_part(&a, lo, k, lo_index_base, topk_idx, topk_score, workspace, workspace_bytes, impl, st);
    if (rc != MAD_OK) return rc;
    return topk_part(&b, lo, k, lo_index_base, topk_idx + (size_t)M0 * k, topk_score + (size_t)M0 * k, workspace, workspace_bytes,
                     impl, st);
}

// ---- small device -> host readbacks that do not use a copy engine -------------------------------------------------
// A cudaMemcpyAsync of a few bytes queues behind whatever large transfer the copy engine of that direction is busy with
// (observed: a 4-byte count waited 1.5 ms for the 82 MB descriptor table of the previous map).  This kernel stores the
// words straight into pinned, device-mapped host memory over PCIe instead.
namespace {
__global__ void publish_small_kernel(const unsigned int* __restrict__ src, volatile unsigned int* dst, int n_words) {
    for (int i = threadIdx.x; i < n_words; i += blockDim.x) dst[i] = src[i];
    __threadfence_system();
}
}  // namespace

extern "C" int mad_publish_small(const void* src_dev, void* dst_host_mapped, int bytes, void* stream) {
    MAD_CHECK_ARG(src_dev && dst_host_mapped && bytes > 0 && bytes <= 4096 && bytes % 4 == 0);
    MAD_CHECK_ARG((reinterpret_cast<uintptr_t>(src_dev) & 3) == 0 && (reinterpret_cast<uintptr_t>(dst_host_mapped) & 3) == 0);
    MAD_PROF("publish_small_kernel", stream);
    publish_small_kernel<<<1, 64, 0, (cudaStream_t)stream>>>(static_cast<const unsigned int*>(src_dev),
                                                             static_cast<volatile unsigned int*>(dst_host_mapped), bytes / 4);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

// ---- bulk device -> host copy by a kernel ---------------------------------------------------------------------------
// Results of map i travel home while map i+1 is computing.  A cudaMemcpyAsync would keep the device -> host copy engine
// busy for milliseconds, and every small operation of the next map that the driver routes through a copy engine (the
// cudaMemsetAsync calls inside CUB's radix sort, for one) queues behind it: the pipelined end-to-end time swung between
// 9.1 and 14 ms per map depending on how the two happened to align.  A handful of CTAs storing 16-byte words straight into
// pinned, device-mapped host memory move the same bytes over PCIe without touching a copy engine.
namespace {
__global__ void __launch_bounds__(256)
copy_to_host_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst, long long n16, const unsigned char* __restrict__ src_tail,
                    unsigned char* __restrict__ dst_tail, int n_tail) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n16; i += stride) {
        const uint4 v = __ldcs(src + i);
        __stcs(dst + i, v);
    }
    if (blockIdx.x == 0 && (int)threadIdx.x < n_tail) dst_tail[threadIdx.x] = src_tail[threadIdx.x];
}
}  // namespace

extern "C" int mad_copy_to_host(const void* src_dev, void* dst_host_mapped, long long bytes, int n_ctas, void* stream) {
    MAD_CHECK_ARG(src_dev && dst_host_mapped && bytes > 0 && n_ctas >= 1 && n_ctas <= 1024);
    MAD_CHECK_ARG((reinterpret_cast<uintptr_t>(src_dev) & 15) == 0 && (reinterpret_cast<uintptr_t>(dst_host_mapped) & 15) == 0);
    const long long n16 = bytes / 16;
    const int n_tail = (int)(bytes - n16 * 16);
    const unsigned char* s8 = static_cast<const unsigned char*>(src_dev);
    unsigned char* d8 = static_cast<unsigned char*>(dst_host_mapped);
    MAD_PROF("copy_to_host_kernel", stream);
    copy_to_host_kernel<<<n_ctas, 256, 0, (cudaStream_t)stream>>>(static_cast<const uint4*>(src_dev), static_cast<uint4*>(dst_host_mapped),
                                                                  n16, s8 + n16 * 16, d8 + n16 * 16, n_tail);
    MAD_LAUNCH_OK();
    return MAD_OK;
}
