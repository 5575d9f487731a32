// Atoms -> simulated density map (PDB.structure_to_density, mad/PDB.py:131-163 and
// interpolate_to_grid_massweighted :215-292), the step in front of the hot path (SURVEY.md 8f rank 2).
//   1. mass-weighted trilinear splat of the atoms into a float64 grid (margin 2 + pad voxels)
//   2. division by the grid maximum (float64)
//   3. "full" convolution with the Gaussian exp(-r^2 / 2 sigma^2) truncated at 3 sigma and normalised to
//      sum 1 (scipy.signal.convolve: zero extension, output grows by 2r per axis) -- done as three 1-D
//      float64 passes (the kernel is a product; the reference's FFT / direct sum differs by ~1e-16)
//   4. float32 cast; max normalisation and isovalue cut are mad_grid_max / mad_threshold_normalise.
#include <cub/cub.cuh>
#include <math.h>

#include <vector>

#include "common.cuh"

namespace {

__global__ void __launch_bounds__(256)
splat_kernel(const double* __restrict__ xyz, const double* __restrict__ mass, int n, double minx, double miny, double minz,
             double voxelsp, int margin, int py, int pz, double* __restrict__ grid) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double gx = margin + (xyz[3 * i] - minx) / voxelsp;          // mad/PDB.py:262-264
    const double gy = margin + (xyz[3 * i + 1] - miny) / voxelsp;
    const double gz = margin + (xyz[3 * i + 2] - minz) / voxelsp;
    const double fx = floor(gx), fy = floor(gy), fz = floor(gz);
    const int x0 = (int)fx, y0 = (int)fy, z0 = (int)fz;
    const double a = (fx + 1.0) - gx, b = (fy + 1.0) - gy, c = (fz + 1.0) - gz;   // :275-277
    const double m = mass[i];
    auto at = [&](int x, int y, int z) { return grid + ((long long)x * py + y) * pz + z; };
    atomicAdd(at(x0, y0, z0), m * a * b * c);                           // :278-285 (same products, atomics reorder the sums)
    atomicAdd(at(x0, y0, z0 + 1), m * a * b * (1 - c));
    atomicAdd(at(x0, y0 + 1, z0), m * a * (1 - b) * c);
    atomicAdd(at(x0 + 1, y0, z0), m * (1 - a) * b * c);
    atomicAdd(at(x0, y0 + 1, z0 + 1), m * a * (1 - b) * (1 - c));
    atomicAdd(at(x0 + 1, y0 + 1, z0), m * (1 - a) * (1 - b) * c);
    atomicAdd(at(x0 + 1, y0, z0 + 1), m * (1 - a) * b * (1 - c));
    atomicAdd(at(x0 + 1, y0 + 1, z0 + 1), m * (1 - a) * (1 - b) * (1 - c));
}

__global__ void __launch_bounds__(256)
max_f64_kernel(const double* __restrict__ g, long long n, unsigned long long* __restrict__ out_bits) {
    double m = 0.0;                                                     // the grid is non-negative
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        m = fmax(m, g[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(out_bits, (unsigned long long)__double_as_longlong(m));   // order-preserving for m >= 0
}

__global__ void __launch_bounds__(256)
divide_f64_kernel(double* __restrict__ g, long long n, const unsigned long long* __restrict__ max_bits) {
    const double m = __longlong_as_double((long long)*max_bits);
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        g[i] = g[i] / m;
}

// "full" 1-D convolution along one axis with zero extension: out extent = n + 2r.
// in: [outer][n][inner] -> out: [outer][n + 2r][inner];  out[i] = sum_j w[j] * in[i - j]  (j = 0..2r, symmetric w)
// Output element gidx of the convolution; the single-grid and the batched kernels both compute a voxel with it.
__device__ __forceinline__ double conv_full_voxel(const double* __restrict__ in, int n, long long inner, int r,
                                                  const double* __restrict__ w, long long gidx) {
    const long long j = gidx % inner;
    const long long t = gidx / inner;
    const int i = (int)(t % (n + 2 * r));
    const long long o = t / (n + 2 * r);
    const double* line = in + o * (long long)n * inner + j;
    double acc = 0.0;
    for (int q = 0; q <= 2 * r; ++q) {
        const int src = i - q;
        if (src >= 0 && src < n) acc = fma(w[q], line[(long long)src * inner], acc);
    }
    return acc;
}

template <typename TOut>
__global__ void __launch_bounds__(256)
conv_full_kernel(const double* __restrict__ in, long long outer, int n, long long inner, int r, const double* __restrict__ w,
                 TOut* __restrict__ out) {
    const long long total = outer * (long long)(n + 2 * r) * inner;
    for (long long gidx = blockIdx.x * (long long)blockDim.x + threadIdx.x; gidx < total; gidx += (long long)gridDim.x * blockDim.x)
        out[gidx] = (TOut)conv_full_voxel(in, n, inner, r, w, gidx);
}

// ---- batches of G structures (mad_density_*_many) ------------------------------------------------------------------
// Every batched kernel runs on a grid of (x blocks, G): blockIdx.y is the structure, whose record in the device copy of
// the MadDensityBox table gives its atoms, its box and where each stage of it lives.

// dims of a structure's box at stage s: the splat box grown by 2r along the axes the first s passes have convolved
__host__ __device__ __forceinline__ void stage_dims(const MadDensityBox& b, int r, int s, long long d[3]) {
    for (int a = 0; a < 3; ++a) d[a] = b.dims[a] + (a < s ? 2 * r : 0);
}

__host__ __device__ __forceinline__ long long stage_size(const MadDensityBox& b, int r, int s) {
    long long d[3];
    stage_dims(b, r, s, d);
    return d[0] * d[1] * d[2];
}

// The 8 corner contributions of every atom, atom-major and corner-minor, keyed by their global voxel (box offset + local
// voxel).  Statement order and products of interpolate_to_grid_massweighted (mad/PDB.py:262-285), each operation
// rounded once, as Python evaluates them.
__global__ void __launch_bounds__(256)
splat_emit_kernel(const double* __restrict__ xyz, const double* __restrict__ mass, const MadDensityBox* __restrict__ boxes,
                  double voxelsp, unsigned long long* __restrict__ keys, double* __restrict__ vals) {
    const MadDensityBox& b = boxes[blockIdx.y];
    const int n = b.n_atoms, py = b.dims[1], pz = b.dims[2];
    const double margin = (double)b.margin;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const long long at = b.atom0 + i;
        const double gx = __dadd_rn(margin, __ddiv_rn(__dsub_rn(xyz[3 * at], b.min[0]), voxelsp));
        const double gy = __dadd_rn(margin, __ddiv_rn(__dsub_rn(xyz[3 * at + 1], b.min[1]), voxelsp));
        const double gz = __dadd_rn(margin, __ddiv_rn(__dsub_rn(xyz[3 * at + 2], b.min[2]), voxelsp));
        const double fx = floor(gx), fy = floor(gy), fz = floor(gz);
        const int x0 = (int)fx, y0 = (int)fy, z0 = (int)fz;
        const double a = __dsub_rn(fx + 1.0, gx), c_b = __dsub_rn(fy + 1.0, gy), c = __dsub_rn(fz + 1.0, gz);
        const double a1 = __dsub_rn(1.0, a), b1 = __dsub_rn(1.0, c_b), c1 = __dsub_rn(1.0, c);
        const double m = mass[at];
        const double ma = __dmul_rn(m, a), ma1 = __dmul_rn(m, a1);
        const double v[8] = {__dmul_rn(__dmul_rn(ma, c_b), c),  __dmul_rn(__dmul_rn(ma, c_b), c1),
                             __dmul_rn(__dmul_rn(ma, b1), c),   __dmul_rn(__dmul_rn(ma1, c_b), c),
                             __dmul_rn(__dmul_rn(ma, b1), c1),  __dmul_rn(__dmul_rn(ma1, b1), c),
                             __dmul_rn(__dmul_rn(ma1, c_b), c1), __dmul_rn(__dmul_rn(ma1, b1), c1)};
        const int dx[8] = {0, 0, 0, 1, 0, 1, 1, 1}, dy[8] = {0, 0, 1, 0, 1, 1, 0, 1}, dz[8] = {0, 1, 0, 0, 1, 0, 1, 1};
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            keys[8 * at + k] = (unsigned long long)(b.off[0] + ((long long)(x0 + dx[k]) * py + (y0 + dy[k])) * pz + (z0 + dz[k]));
            vals[8 * at + k] = v[k];
        }
    }
}

// One thread per run of equal keys in the stably sorted contributions: the voxel's sum in emission order, from 0.0, as the
// reference's loop forms it.
__global__ void __launch_bounds__(256)
splat_fold_kernel(const unsigned long long* __restrict__ keys, const double* __restrict__ vals, int n, double* __restrict__ grid) {
    for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
        const unsigned long long key = keys[k];
        if (k > 0 && keys[k - 1] == key) continue;
        double s = 0.0;
        for (long long j = k; j < n && keys[j] == key; ++j) s = __dadd_rn(s, vals[j]);
        grid[key] = s;
    }
}

__global__ void __launch_bounds__(256)
max_f64_many_kernel(const double* __restrict__ g, const MadDensityBox* __restrict__ boxes, unsigned long long* __restrict__ out_bits) {
    const MadDensityBox& b = boxes[blockIdx.y];
    const long long n = (long long)b.dims[0] * b.dims[1] * b.dims[2];
    const double* s = g + b.off[0];
    double m = 0.0;                                                     // the grid is non-negative
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        m = fmax(m, s[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(out_bits + blockIdx.y, (unsigned long long)__double_as_longlong(m));
}

__global__ void __launch_bounds__(256)
divide_f64_many_kernel(double* __restrict__ g, const MadDensityBox* __restrict__ boxes, const unsigned long long* __restrict__ max_bits) {
    const MadDensityBox& b = boxes[blockIdx.y];
    const long long n = (long long)b.dims[0] * b.dims[1] * b.dims[2];
    double* s = g + b.off[0];
    const double m = __longlong_as_double((long long)max_bits[blockIdx.y]);
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        s[i] = s[i] / m;
}

// Pass p of the three: stage p (float64) -> stage p + 1, along axis p.
template <typename TOut>
__global__ void __launch_bounds__(256)
conv_full_many_kernel(const double* __restrict__ in, const MadDensityBox* __restrict__ boxes, int pass, int r,
                      const double* __restrict__ w, TOut* __restrict__ out) {
    const MadDensityBox& b = boxes[blockIdx.y];
    const long long dx = b.dims[0] + (pass > 0 ? 2 * r : 0), dy = b.dims[1] + (pass > 1 ? 2 * r : 0), dz = b.dims[2];
    const long long outer = pass == 0 ? 1 : (pass == 1 ? dx : dx * dy);
    const int n = (int)(pass == 0 ? dx : (pass == 1 ? dy : dz));
    const long long inner = pass == 0 ? dy * dz : (pass == 1 ? dz : 1);
    const double* src = in + b.off[pass];
    TOut* dst = out + b.off[pass + 1];
    const long long total = outer * (long long)(n + 2 * r) * inner;
    for (long long gidx = blockIdx.x * (long long)blockDim.x + threadIdx.x; gidx < total; gidx += (long long)gridDim.x * blockDim.x)
        dst[gidx] = (TOut)conv_full_voxel(src, n, inner, r, w, gidx);
}

// grid_max_kernel's ordered-image maximum, one per structure map
__global__ void __launch_bounds__(256)
map_max_many_kernel(const float* __restrict__ maps, const MadDensityBox* __restrict__ boxes, int r, unsigned int* __restrict__ out_ord) {
    const MadDensityBox& b = boxes[blockIdx.y];
    const long long n = stage_size(b, r, 3);
    const float* g = maps + b.off[3];
    unsigned int m = 0u;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        m = max(m, mad_f2ord(__ldg(g + i)));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
    if ((threadIdx.x & 31) == 0 && m) atomicMax(out_ord + blockIdx.y, m);
}

// what structure_to_density_device does after reading the maximum back: mad_threshold_normalise(-inf, vmax, divide), then,
// for a non-zero isovalue, mad_threshold_normalise(isovalue, 1, no divide)
__global__ void __launch_bounds__(256)
map_normalise_many_kernel(float* __restrict__ maps, const MadDensityBox* __restrict__ boxes, int r, const unsigned int* __restrict__ ord,
                          float isovalue, int cut) {
    const MadDensityBox& b = boxes[blockIdx.y];
    const long long n = stage_size(b, r, 3);
    float* g = maps + b.off[3];
    const float vmax = __uint_as_float(mad_ord2bits(ord[blockIdx.y]));
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        float v = mad_threshold_normalise_one(g[i], -INFINITY, vmax, 1);
        if (cut) v = mad_threshold_normalise_one(v, isovalue, 1.f, 0);
        g[i] = v;
    }
}

}  // namespace

extern "C" int mad_density_splat(const double* xyz, const double* mass, int n_atoms, const double* min_host, double voxelsp,
                                 int margin, int px, int py, int pz, double* grid, void* stream) {
    MAD_CHECK_ARG(xyz && mass && min_host && grid && n_atoms > 0 && voxelsp > 0 && margin >= 1 && px > 0 && py > 0 && pz > 0);
    cudaStream_t st = (cudaStream_t)stream;
    MAD_CUDA(cudaMemsetAsync(grid, 0, sizeof(double) * (size_t)px * py * pz, st));
    MAD_PROF("splat_kernel", st);
    splat_kernel<<<(unsigned)mad_ceil_div(n_atoms, 256), 256, 0, st>>>(xyz, mass, n_atoms, min_host[0], min_host[1], min_host[2],
                                                                       voxelsp, margin, py, pz, grid);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" int mad_normalise_f64(double* grid, long long n, void* scratch8, void* stream) {
    MAD_CHECK_ARG(grid && scratch8 && n > 0);
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long* bits = reinterpret_cast<unsigned long long*>(scratch8);
    MAD_CUDA(cudaMemsetAsync(bits, 0, 8, st));
    const int blocks = (int)std::max<long long>(1, std::min<long long>(mad_ceil_div(n, 1024), (long long)mad_sm_count() * 8));
    {
        MAD_PROF("max_f64_kernel", st);
        max_f64_kernel<<<blocks, 256, 0, st>>>(grid, n, bits);
        MAD_LAUNCH_OK();
    }
    MAD_PROF("divide_f64_kernel", st);
    divide_f64_kernel<<<blocks, 256, 0, st>>>(grid, n, bits);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" int mad_conv_full_f64(const double* in, long long outer, int n, long long inner, const double* w_dev, int radius,
                                 void* out, int out_is_f32, void* stream) {
    MAD_CHECK_ARG(in && w_dev && out && outer > 0 && n > 0 && inner > 0 && radius >= 0);
    const long long total = outer * (long long)(n + 2 * radius) * inner;
    const int blocks = (int)std::max<long long>(1, std::min<long long>(mad_ceil_div(total, 256), (long long)mad_sm_count() * 16));
    MAD_PROF("conv_full_kernel", stream);
    if (out_is_f32)
        conv_full_kernel<float><<<blocks, 256, 0, (cudaStream_t)stream>>>(in, outer, n, inner, radius, w_dev, reinterpret_cast<float*>(out));
    else
        conv_full_kernel<double><<<blocks, 256, 0, (cudaStream_t)stream>>>(in, outer, n, inner, radius, w_dev, reinterpret_cast<double*>(out));
    MAD_LAUNCH_OK();
    return MAD_OK;
}

// ---- batches of G structures ----------------------------------------------------------------------------------------
namespace {

constexpr long long kMaxContrib = (1LL << 31) - 1;

// atom0 and off[4] of every record from n_atoms, dims and r; totals[5] = (atoms, elements of the four stages)
int density_layout(MadDensityBox* boxes, int G, int radius, long long* totals) {
    MAD_CHECK_ARG(boxes && totals && G >= 1 && G <= 65535 && radius >= 0 && radius < (1 << 20));
    long long atoms = 0, t[4] = {0, 0, 0, 0};
    for (int g = 0; g < G; ++g) {
        MadDensityBox& b = boxes[g];
        MAD_CHECK_ARG(b.n_atoms > 0 && b.margin >= 1);
        MAD_CHECK_ARG(b.dims[0] > 0 && b.dims[1] > 0 && b.dims[2] > 0);
        for (int a = 0; a < 3; ++a) MAD_CHECK_ARG(b.dims[a] + 2LL * radius < (1LL << 30));
        b.atom0 = atoms;
        atoms += b.n_atoms;
        MAD_CHECK_ARG(8 * atoms <= kMaxContrib);
        for (int s = 0; s < 4; ++s) {
            b.off[s] = t[s];
            const long long n = stage_size(b, radius, s);
            MAD_CHECK_ARG(n > 0 && n < (1LL << 50) && t[s] + n < (1LL << 52));
            t[s] += n;
        }
    }
    totals[0] = atoms;
    for (int s = 0; s < 4; ++s) totals[1 + s] = t[s];
    return MAD_OK;
}

// boxes_host must be the table mad_density_layout laid out (for this radius when stages > 1): atom0 and off[0, stages)
int check_layout(const MadDensityBox* boxes_host, int G, int radius, int stages, long long* totals) {
    MAD_CHECK_ARG(boxes_host && G >= 1 && G <= 65535);
    std::vector<MadDensityBox> laid(boxes_host, boxes_host + G);
    const int rc = density_layout(laid.data(), G, radius, totals);
    if (rc != MAD_OK) return rc;
    for (int g = 0; g < G; ++g) {
        MAD_CHECK_ARG(laid[g].atom0 == boxes_host[g].atom0);
        for (int s = 0; s < stages; ++s) MAD_CHECK_ARG(laid[g].off[s] == boxes_host[g].off[s]);
    }
    return MAD_OK;
}

// x blocks per structure of a (x, G) grid: enough for the largest structure's `n` elements at `per_block` each, no more
// than `waves` blocks per SM over the whole batch (but at least one per structure)
unsigned per_structure_blocks(long long max_n, long long per_block, int G, int waves) {
    const long long cap = std::max<long long>(1, (long long)mad_sm_count() * waves / G);
    return (unsigned)std::max<long long>(1, std::min<long long>(mad_ceil_div(max_n, per_block), cap));
}

long long max_stage_size(const MadDensityBox* boxes_host, int G, int radius, int s) {
    long long m = 0;
    for (int g = 0; g < G; ++g) m = std::max(m, stage_size(boxes_host[g], radius, s));
    return m;
}

struct SplatLayout {
    size_t keys_in, keys_out, vals_in, vals_out, cub, cub_bytes, total;
};

SplatLayout splat_layout(long long n_contrib, int end_bit) {
    SplatLayout l;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o += mad_align_up(bytes, 256); return r; };
    const size_t nn = (size_t)std::max<long long>(n_contrib, 1);
    l.keys_in = take(nn * 8); l.keys_out = take(nn * 8);
    l.vals_in = take(nn * 8); l.vals_out = take(nn * 8);
    size_t a = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, a, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                    (const double*)nullptr, (double*)nullptr, (int)nn, 0, end_bit);
    l.cub_bytes = a;
    l.cub = take(a);
    l.total = o;
    return l;
}

}  // namespace

extern "C" int mad_density_layout(MadDensityBox* boxes, int G, int radius, long long* totals) {
    return density_layout(boxes, G, radius, totals);
}

extern "C" size_t mad_density_splat_many_workspace_bytes(int n_atoms) {
    if (n_atoms < 0 || 8LL * n_atoms > kMaxContrib) return 0;
    return splat_layout(8LL * std::max(n_atoms, 0), 64).total;
}

extern "C" int mad_density_splat_many(const double* xyz, const double* mass, const MadDensityBox* boxes_host, int G,
                                      const MadDensityBox* boxes, double voxelsp, double* grid, void* workspace,
                                      size_t workspace_bytes, void* stream) {
    MAD_CHECK_ARG(xyz && mass && boxes && grid && workspace && voxelsp > 0);
    long long totals[5];
    const int rc = check_layout(boxes_host, G, 0, 1, totals);
    if (rc != MAD_OK) return rc;
    const long long n = 8 * totals[0];
    int end_bit = 1;
    while (end_bit < 64 && ((unsigned long long)(totals[1] - 1) >> end_bit)) ++end_bit;
    const SplatLayout l = splat_layout(n, end_bit);
    MAD_CHECK_ARG(workspace_bytes >= l.total && l.total <= mad_density_splat_many_workspace_bytes((int)totals[0]));
    char* ws = static_cast<char*>(workspace);
    auto* keys_in = reinterpret_cast<unsigned long long*>(ws + l.keys_in);
    auto* keys_out = reinterpret_cast<unsigned long long*>(ws + l.keys_out);
    auto* vals_in = reinterpret_cast<double*>(ws + l.vals_in);
    auto* vals_out = reinterpret_cast<double*>(ws + l.vals_out);
    cudaStream_t st = (cudaStream_t)stream;
    MAD_CUDA(cudaMemsetAsync(grid, 0, sizeof(double) * (size_t)totals[1], st));
    long long max_atoms = 0;
    for (int g = 0; g < G; ++g) max_atoms = std::max<long long>(max_atoms, boxes_host[g].n_atoms);
    {
        MAD_PROF("splat_emit_kernel", st);
        splat_emit_kernel<<<dim3(per_structure_blocks(max_atoms, 256, G, 8), (unsigned)G), 256, 0, st>>>(
            xyz, mass, boxes, voxelsp, keys_in, vals_in);
        MAD_LAUNCH_OK();
    }
    {
        MAD_PROF("splat_sort", st);
        size_t cub_bytes = l.cub_bytes;
        MAD_CUDA(cub::DeviceRadixSort::SortPairs(ws + l.cub, cub_bytes, keys_in, keys_out, vals_in, vals_out, (int)n, 0, end_bit, st));
    }
    MAD_PROF("splat_fold_kernel", st);
    const int blocks = (int)std::max<long long>(1, std::min<long long>(mad_ceil_div(n, 256), (long long)mad_sm_count() * 16));
    splat_fold_kernel<<<blocks, 256, 0, st>>>(keys_out, vals_out, (int)n, grid);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" int mad_normalise_f64_many(double* grid, const MadDensityBox* boxes_host, int G, const MadDensityBox* boxes,
                                      void* scratch, void* stream) {
    MAD_CHECK_ARG(grid && boxes && scratch);
    long long totals[5];
    const int rc = check_layout(boxes_host, G, 0, 1, totals);
    if (rc != MAD_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long* bits = reinterpret_cast<unsigned long long*>(scratch);
    MAD_CUDA(cudaMemsetAsync(bits, 0, 8 * (size_t)G, st));
    const dim3 grid_dim(per_structure_blocks(max_stage_size(boxes_host, G, 0, 0), 1024, G, 8), (unsigned)G);
    {
        MAD_PROF("max_f64_many_kernel", st);
        max_f64_many_kernel<<<grid_dim, 256, 0, st>>>(grid, boxes, bits);
        MAD_LAUNCH_OK();
    }
    MAD_PROF("divide_f64_many_kernel", st);
    divide_f64_many_kernel<<<grid_dim, 256, 0, st>>>(grid, boxes, bits);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" int mad_conv_full_f64_many(const double* in, const MadDensityBox* boxes_host, int G, const MadDensityBox* boxes,
                                      int pass, const double* w_dev, int radius, void* out, void* stream) {
    MAD_CHECK_ARG(in && boxes && w_dev && out && pass >= 0 && pass <= 2);
    long long totals[5];
    const int rc = check_layout(boxes_host, G, radius, 4, totals);
    if (rc != MAD_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const dim3 grid_dim(per_structure_blocks(max_stage_size(boxes_host, G, radius, pass + 1), 256, G, 16), (unsigned)G);
    MAD_PROF("conv_full_many_kernel", st);
    if (pass == 2)
        conv_full_many_kernel<float><<<grid_dim, 256, 0, st>>>(in, boxes, pass, radius, w_dev, reinterpret_cast<float*>(out));
    else
        conv_full_many_kernel<double><<<grid_dim, 256, 0, st>>>(in, boxes, pass, radius, w_dev, reinterpret_cast<double*>(out));
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" int mad_map_normalise_many(float* maps, const MadDensityBox* boxes_host, int G, const MadDensityBox* boxes,
                                      int radius, float isovalue, void* scratch, void* stream) {
    MAD_CHECK_ARG(maps && boxes && scratch);
    long long totals[5];
    const int rc = check_layout(boxes_host, G, radius, 4, totals);
    if (rc != MAD_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned int* ord = reinterpret_cast<unsigned int*>(scratch);
    MAD_CUDA(cudaMemsetAsync(ord, 0, 4 * (size_t)G, st));
    const long long max_n = max_stage_size(boxes_host, G, radius, 3);
    {
        MAD_PROF("map_max_many_kernel", st);
        map_max_many_kernel<<<dim3(per_structure_blocks(max_n, 256 * 8, G, 8), (unsigned)G), 256, 0, st>>>(maps, boxes, radius, ord);
        MAD_LAUNCH_OK();
    }
    MAD_PROF("map_normalise_many_kernel", st);
    map_normalise_many_kernel<<<dim3(per_structure_blocks(max_n, 256 * 4, G, 16), (unsigned)G), 256, 0, st>>>(
        maps, boxes, radius, ord, isovalue, isovalue != 0.f);
    MAD_LAUNCH_OK();
    return MAD_OK;
}
