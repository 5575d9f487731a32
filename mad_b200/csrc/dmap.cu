// a0: device-side operations of the Dmap container (mad/Dmap.py:49-97): isovalue cut, max
// normalisation, bounding box of the non-zero voxels, crop + zero padding.  The grid stays in HBM;
// these are single streaming passes over it (4-8 B per voxel).
#include <string.h>

#include "common.cuh"

namespace {

__global__ void __launch_bounds__(256)
grid_max_kernel(const float* __restrict__ g, long long n, unsigned int* __restrict__ out_ord) {
    unsigned int m = 0u;                                         // below every finite float's image
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        m = max(m, mad_f2ord(__ldg(g + i)));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
    if ((threadIdx.x & 31) == 0 && m) atomicMax(out_ord, m);
}

__global__ void __launch_bounds__(256)
threshold_normalise_kernel(float* __restrict__ g, long long n, float isovalue, float vmax, int divide) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        g[i] = mad_threshold_normalise_one(g[i], isovalue, vmax, divide);
}

// bbox[0..2] = min index of a non-zero voxel per axis, bbox[3..5] = max (mad/Dmap.py:77-80).
__global__ void __launch_bounds__(256)
grid_bbox_kernel(const float* __restrict__ g, int nx, int ny, int nz, int* __restrict__ bbox) {
    const unsigned plane = (unsigned)ny * (unsigned)nz;
    const unsigned p = blockIdx.x * 256u + threadIdx.x;
    int lo[3] = {1 << 30, 1 << 30, 1 << 30}, hi[3] = {-1, -1, -1};
    if (p < plane) {
        const int y = (int)(p / (unsigned)nz), z = (int)(p - (unsigned)y * (unsigned)nz);
        for (int x = blockIdx.y; x < nx; x += gridDim.y) {
            if (__ldg(g + (long long)x * plane + p) != 0.f) {
                lo[0] = min(lo[0], x); hi[0] = max(hi[0], x);
                lo[1] = min(lo[1], y); hi[1] = max(hi[1], y);
                lo[2] = min(lo[2], z); hi[2] = max(hi[2], z);
            }
        }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[a] = min(lo[a], __shfl_xor_sync(0xFFFFFFFFu, lo[a], o));
            hi[a] = max(hi[a], __shfl_xor_sync(0xFFFFFFFFu, hi[a], o));
        }
        if ((threadIdx.x & 31) == 0 && hi[a] >= 0) {
            atomicMin(bbox + a, lo[a]);
            atomicMax(bbox + 3 + a, hi[a]);
        }
    }
}

__global__ void bbox_init_kernel(int* bbox) {
    if (threadIdx.x < 3) bbox[threadIdx.x] = 1 << 30;
    else if (threadIdx.x < 6) bbox[threadIdx.x] = -1;
}

// out[(cx + 2 pad)(cy + 2 pad)(cz + 2 pad)] = zero-padded copy of the box [x0, x0+cx) x ... of `in`
// (grid3d[minx:maxx+1, ...] followed by np.pad, mad/Dmap.py:86-97).
__global__ void __launch_bounds__(256)
crop_pad_kernel(const float* __restrict__ in, int ny, int nz, int x0, int y0, int z0, int cx, int cy, int cz, int pad,
                float* __restrict__ out) {
    const int oy = cy + 2 * pad, oz = cz + 2 * pad;
    const unsigned plane = (unsigned)oy * (unsigned)oz;
    const unsigned p = blockIdx.x * 256u + threadIdx.x;
    if (p >= plane) return;
    const int y = (int)(p / (unsigned)oz) - pad, z = (int)(p - (p / (unsigned)oz) * (unsigned)oz) - pad;
    const int x = (int)blockIdx.y - pad;
    float v = 0.f;
    if (x >= 0 && x < cx && y >= 0 && y < cy && z >= 0 && z < cz)
        v = __ldg(in + ((long long)(x0 + x) * ny + (y0 + y)) * nz + (z0 + z));
    out[(long long)blockIdx.y * plane + p] = v;
}

}  // namespace

extern "C" int mad_grid_max(const float* grid, long long n, float* out_max, void* stream) {
    MAD_CHECK_ARG(grid && out_max && n > 0);
    cudaStream_t st = (cudaStream_t)stream;
    unsigned int* ord = reinterpret_cast<unsigned int*>(out_max);
    MAD_CUDA(cudaMemsetAsync(ord, 0, sizeof(unsigned int), st));
    const int blocks = (int)std::min<long long>(mad_ceil_div(n, 256 * 8), (long long)mad_sm_count() * 8);
    MAD_PROF("grid_max_kernel", st);
    grid_max_kernel<<<std::max(blocks, 1), 256, 0, st>>>(grid, n, ord);
    MAD_LAUNCH_OK();
    return MAD_OK;   // *out_max holds the ORDERED image; mad_grid_max_decode turns it into the float
}

extern "C" float mad_grid_max_decode(unsigned int ord) {
    const unsigned int u = mad_ord2bits(ord);
    float f;
    memcpy(&f, &u, sizeof(f));
    return f;
}

extern "C" int mad_threshold_normalise(float* grid, long long n, float isovalue, float vmax, int divide, void* stream) {
    MAD_CHECK_ARG(grid && n > 0);
    const int blocks = (int)std::min<long long>(mad_ceil_div(n, 256 * 4), (long long)mad_sm_count() * 16);
    MAD_PROF("threshold_normalise_kernel", stream);
    threshold_normalise_kernel<<<std::max(blocks, 1), 256, 0, (cudaStream_t)stream>>>(grid, n, isovalue, vmax, divide);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" int mad_grid_bbox(const float* grid, int nx, int ny, int nz, int* bbox6, void* stream) {
    MAD_CHECK_ARG(grid && bbox6 && nx > 0 && ny > 0 && nz > 0 && (long long)ny * nz < (1LL << 31));
    cudaStream_t st = (cudaStream_t)stream;
    bbox_init_kernel<<<1, 32, 0, st>>>(bbox6);
    dim3 grid_dim((unsigned)mad_ceil_div((long long)ny * nz, 256), (unsigned)std::min(nx, 64));
    MAD_PROF("grid_bbox_kernel", st);
    grid_bbox_kernel<<<grid_dim, 256, 0, st>>>(grid, nx, ny, nz, bbox6);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" int mad_crop_pad3d(const float* in, int nx, int ny, int nz, int x0, int y0, int z0, int cx, int cy, int cz,
                              int pad, float* out, void* stream) {
    MAD_CHECK_ARG(in && out && pad >= 0 && cx > 0 && cy > 0 && cz > 0);
    MAD_CHECK_ARG(x0 >= 0 && y0 >= 0 && z0 >= 0 && x0 + cx <= nx && y0 + cy <= ny && z0 + cz <= nz);
    MAD_CHECK_ARG(cx + 2 * pad <= 65535);
    dim3 grid_dim((unsigned)mad_ceil_div((long long)(cy + 2 * pad) * (cz + 2 * pad), 256), (unsigned)(cx + 2 * pad));
    MAD_PROF("crop_pad_kernel", stream);
    crop_pad_kernel<<<grid_dim, 256, 0, (cudaStream_t)stream>>>(in, ny, nz, x0, y0, z0, cx, cy, cz, pad, out);
    MAD_LAUNCH_OK();
    return MAD_OK;
}
