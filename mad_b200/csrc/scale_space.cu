// Scale-space stage of the MaD hot path for B200 (sm_100a):
//   a1  zero padding                         (np.pad,                    mad/MapSpace.py:117-118)
//   a2  2x cubic-spline upsampling + presmooth (interp1d cubic x3 + gaussian_filter, :137-146)
//   a3  LoG response + a4 Gaussian grid        (gaussian_laplace / gaussian_filter, :170-173,182)
//   a4  gradient field                         (np.gradient,              :187)
// All kernels are HBM-bound stencils: marching kernels with register windows for the strided
// axes (coalesced across the contiguous z index), shared-memory row staging for the z axis.
#include <stdlib.h>
#include <type_traits>

#include "common.cuh"

// ------------------------------------------------------------------------------------------
// a1: zero padding
// ------------------------------------------------------------------------------------------
// One warp per output row (x, y): no per-element division, lanes sweep z (coalesced stores; the source row, when the row
// is not padding, is read with the same lanes shifted by `pad`).
__global__ void __launch_bounds__(256)
pad3d_kernel(const float* __restrict__ in, int nx, int ny, int nz, int pad, float* __restrict__ out, int ox, int oy, int oz) {
    const int lane = threadIdx.x & 31;
    const long long rows = (long long)ox * oy;
    for (long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); row < rows; row += (long long)gridDim.x * 8) {
        const int x = (int)(row / oy), y = (int)(row - (long long)x * oy);
        const int sx = x - pad, sy = y - pad;
        float* o = out + row * oz;
        if (sx < 0 || sx >= nx || sy < 0 || sy >= ny) {
            for (int z = lane; z < oz; z += 32) o[z] = 0.f;
        } else {
            const float* src = in + ((long long)sx * ny + sy) * nz - pad;
            for (int z = lane; z < oz; z += 32) o[z] = (z >= pad && z < nz + pad) ? __ldg(src + z) : 0.f;
        }
    }
}

extern "C" int mad_pad3d(const float* in, int nx, int ny, int nz, int pad, float* out, void* stream) {
    MAD_CHECK_ARG(in && out && nx > 0 && ny > 0 && nz > 0 && pad >= 0);
    const int ox = nx + 2 * pad, oy = ny + 2 * pad, oz = nz + 2 * pad;
    const long long rows = (long long)ox * oy;
    int blocks = (int)std::min<long long>(mad_ceil_div(rows, 8), (long long)mad_sm_count() * 32);
    MAD_PROF("pad3d_kernel", stream);
    pad3d_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(in, nx, ny, nz, pad, out, ox, oy, oz);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

// ------------------------------------------------------------------------------------------
// a2: not-a-knot cubic spline at half steps (+ Gaussian presmoothing along the same axis)
//
// Along one line y[0..n-1] with second derivatives M (unit spacing):
//   M[i-1] + 4 M[i] + M[i+1] = 6 d_i,  d_i = y[i-1] - 2 y[i] + y[i+1]      (1 <= i <= n-2)
//   not-a-knot: M[0]-2M[1]+M[2] = 0, M[n-3]-2M[n-2]+M[n-1] = 0  =>  M[1] = d_1, M[n-2] = d_{n-2}
//   u[2i] = y[i],  u[2i+1] = (y[i]+y[i+1])/2 - (M[i]+M[i+1])/16
// The remaining [1 4 1] system for M[2..n-3] is solved by the Thomas recurrence STREAMING:
// the forward sweep is exact from the line start; the backward sweep for a chunk of 32 samples
// starts 32 samples ahead, where the neglected term has decayed by (2-sqrt3)^32 = 5e-19, i.e.
// below float64 rounding (and it starts from the true last row near the line end).  So no
// O(n) scratch per line is needed: a 64-entry ring per thread in shared memory.
// The presmoothing Gaussian (reflect boundary) of the same axis is applied on the fly to the
// upsampled samples through a register window.  Separable operators on different axes commute,
// so the per-axis fusion equals SciPy's "3 interpolations then 3 filters" up to f64 rounding.
// ------------------------------------------------------------------------------------------
struct SplineParams {
    double cprime[40];  // Thomas pivots c'_i = 1/(4 - c'_{i-1}), c'_2 = 1/4 (constant beyond ~i=25)
    double gw[9];       // presmoothing weights gw[|j|], j = 0..GR
    int long_min;       // lines of at least this many samples take spline_line_long (>= 64; env MAD_SPLINE_GENERIC: never)
};

template <int GR>
struct GaussStream {
    double w[2 * GR + 1];
    int cnt;   // values pushed so far
    int kout;  // next output index
    __device__ __forceinline__ void init() {
        cnt = 0;
        kout = 0;
#pragma unroll
        for (int i = 0; i < 2 * GR + 1; ++i) w[i] = 0.0;
    }
    template <class IO>
    __device__ __forceinline__ void emit(IO& io, const double* gw) {
        double acc = w[GR] * gw[0];
#pragma unroll
        for (int jj = GR; jj >= 1; --jj) acc = fma(w[GR - jj] + w[GR + jj], gw[jj], acc);
        io.put(kout++, acc);
    }
    template <class IO>
    __device__ __forceinline__ void push(double v, IO& io, const double* gw) {
        if (GR == 0) {
            io.put(kout++, v);
            return;
        }
#pragma unroll
        for (int i = 0; i < 2 * GR; ++i) w[i] = w[i + 1];
        w[2 * GR] = v;
        ++cnt;
        if (cnt == GR + 1) {  // u[0..GR] sit in w[GR..2GR]: mirror them (reflect: u[-1-t] = u[t])
#pragma unroll
            for (int t = 0; t < GR; ++t) w[GR - 1 - t] = w[GR + t];
            emit(io, gw);
        } else if (cnt > GR + 1) {
            emit(io, gw);
        }
    }
    // p-th push of the line with p known at compile time (unrolled head chunk): the fill / mirror / emit cases fold away
    template <class IO>
    __device__ __forceinline__ void push_at(int p, double v, IO& io, const double* gw) {
#pragma unroll
        for (int i = 0; i < 2 * GR; ++i) w[i] = w[i + 1];
        w[2 * GR] = v;
        ++cnt;
        if (p == GR) {
#pragma unroll
            for (int t = 0; t < GR; ++t) w[GR - 1 - t] = w[GR + t];
        }
        if (p >= GR) emit(io, gw);
    }
    // interior of the line: the window is full, every push emits
    template <class IO>
    __device__ __forceinline__ void push_steady(double v, IO& io, const double* gw) {
#pragma unroll
        for (int i = 0; i < 2 * GR; ++i) w[i] = w[i + 1];
        w[2 * GR] = v;
        ++cnt;
        emit(io, gw);
    }
    template <class IO>
    __device__ __forceinline__ void finish(IO& io, const double* gw) {
        if (GR == 0) return;
        // virtual sample N+t equals u[N-1-t], which sits in slot 2GR-2t at that moment
#pragma unroll
        for (int t = 0; t < GR; ++t) push(w[2 * GR - 2 * t], io, gw);
    }
};

// ring slot of sample i: i mod 48 (48 = chunk + look-ahead; exact for i < 130 000)
__device__ __forceinline__ int ring_slot(int i) { return i - 48 * ((i * 43691) >> 21); }

// Lines of n >= 64 samples (every real map: the padded grids are >= 100 long).  Same arithmetic, in the same order, as
// spline_line below; what differs is the control flow, which is straight-line everywhere but in the last <= 18 samples:
//   head     forward rows 2..31 in two batches of 15 loads, then chunk 0 with the varying pivots as immediates and the
//            Gaussian window's fill / mirror cases folded at compile time;
//   interior chunks of 16 samples while the 32-row look-ahead stays below the last row (s + 50 < n);
//   final    ONE sweep whose look-ahead reaches the last row: the back substitution starts at the true last row, so it
//            yields M for every remaining row (35..50 of them); they are parked in the ring and the remaining samples
//            are emitted without further sweeps: two unrolled blocks of 16, then a compact loop for the last 3..18.
template <int GR, int RS, class IO>
__device__ __forceinline__ void spline_line_long(IO& io, const int n, const SplineParams& prm, double* ring) {
    constexpr int rs = RS;
    const double cinf = prm.cprime[39];
    const int last = n - 3;
    const double M1 = (io.y(0) - 2.0 * io.y(1)) + io.y(2);
    const double Mn2 = (io.y(n - 3) - 2.0 * io.y(n - 2)) + io.y(n - 1);
    double xprev = 0.0;
    double ya = io.y(1), yb = io.y(2);
    GaussStream<GR> gs;
    gs.init();

    // forward rows f0 .. f0+15 into seg[0..15] with the limit pivot
    auto forward16 = [&](int f0, double* seg) {
        double yy[16];
        io.load_run(f0 + 1, yy);
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const double x = fma(6.0, (ya - 2.0 * yb) + yy[q], -xprev) * cinf;    // forward row: ONE rounding of 6 d - x', on every path
            seg[q * rs] = x;
            xprev = x;
            ya = yb;
            yb = yy[q];
        }
    };
    // samples s0 .. s0+15 and the half steps after them; seg holds M[s0 .. s0+15], Mnext = M[s0+16]
    auto emit16 = [&](int s0, const double* seg, double M0, double Mnext, auto head_c) {
        constexpr bool HEAD = decltype(head_c)::value;
        double yn[17];                                                    // y[s0 .. s0+16]
        io.load_run(s0, yn);
        double yi = yn[0];
        double Mi = M0;
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            double Mn = (q < 15) ? seg[(q < 15 ? q + 1 : 0) * rs] : Mnext;
            if (HEAD && q == 0) Mn = M1;                                  // M[1]
            const double h = 0.5 * (yi + yn[q + 1]) - (Mi + Mn) * 0.0625;
            if (HEAD) {
                gs.push_at(2 * q, yi, io, prm.gw);
                gs.push_at(2 * q + 1, h, io, prm.gw);
            } else {
                gs.push_steady(yi, io, prm.gw);
                gs.push_steady(h, io, prm.gw);
            }
            Mi = Mn;
            yi = yn[q + 1];
        }
        io.chunk_done();
    };

    // ---- head: rows 2..31 forward (pivots still converging: immediates), then chunk 0 ----
    {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            double yy[15];
            io.load_run(3 + 15 * h, yy);
#pragma unroll
            for (int q = 0; q < 15; ++q) {
                const int f = 2 + 15 * h + q;
                const double a = (f == 2) ? M1 : xprev;                  // row 2: x' = 0, the not-a-knot term takes its place
                const double x = fma(6.0, (ya - 2.0 * yb) + yy[q], -a) * prm.cprime[f];
                ring[f * rs] = x;
                xprev = x;
                ya = yb;
                yb = yy[q];
            }
        }
        double* r0 = ring;
        double* r1 = ring + 16 * rs;
        double* r2 = ring + 32 * rs;
        forward16(32, r2);
        double M = r2[15 * rs];
#pragma unroll
        for (int d = 14; d >= 0; --d) M = fma(-cinf, M, r2[d * rs]);
#pragma unroll
        for (int d = 15; d >= 1; --d) M = fma(-cinf, M, r1[d * rs]);
        const double Me = fma(-cinf, M, r1[0]);
        M = Me;
#pragma unroll
        for (int d = 15; d >= 2; --d) {
            M = fma(-prm.cprime[d], M, r0[d * rs]);
            r0[d * rs] = M;
        }
        r0[rs] = M1;                                                      // M[1]; M now holds M[2]
        emit16(0, r0, 2.0 * M1 - M, Me, std::true_type{});
    }

    // ---- interior chunks ----
    int s = 16, b0 = 16;
    for (; s + 50 < n; s += 16, b0 = (b0 == 32) ? 0 : b0 + 16) {
        double* r0 = ring + b0 * rs;                                  // samples s    .. s+15
        double* r1 = ring + ((b0 >= 32) ? b0 - 32 : b0 + 16) * rs;    // samples s+16 .. s+31
        double* r2 = ring + ((b0 >= 16) ? b0 - 16 : b0 + 32) * rs;    // samples s+32 .. s+47
        forward16(s + 32, r2);
        double M = r2[15 * rs];
#pragma unroll
        for (int d = 14; d >= 0; --d) M = fma(-cinf, M, r2[d * rs]);
#pragma unroll
        for (int d = 15; d >= 1; --d) M = fma(-cinf, M, r1[d * rs]);
        const double Me = fma(-cinf, M, r1[0]);                       // M[s+16]
        M = Me;
#pragma unroll
        for (int d = 15; d >= 0; --d) {
            M = fma(-cinf, M, r0[d * rs]);
            r0[d * rs] = M;
        }
        emit16(s, r0, r0[0], Me, std::false_type{});
    }

    // ---- final sweep at s (n - 50 <= s <= n - 35): rows s+32 .. last forward, then M for all rows last .. s ----
    {
        double* r0 = ring + b0 * rs;
        double* r1 = ring + ((b0 >= 32) ? b0 - 32 : b0 + 16) * rs;
        double* r2 = ring + ((b0 >= 16) ? b0 - 16 : b0 + 32) * rs;
        const int nf = last - (s + 32) + 1;                           // 1 .. 16 forward rows are left
        {
            double yy[16];
#pragma unroll
            for (int q = 0; q < 16; ++q) yy[q] = (q < nf) ? io.y(s + 33 + q) : 0.0;
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                if (q < nf) {
                    const double a = (q == nf - 1) ? xprev + Mn2 : xprev;   // the last row's not-a-knot term
                    const double x = fma(6.0, (ya - 2.0 * yb) + yy[q], -a) * cinf;
                    r2[q * rs] = x;
                    xprev = x;
                    ya = yb;
                    yb = yy[q];
                }
            }
        }
        // rows above `last` do not exist: from M = 0 the first existing row gives M = x[last] exactly
        double M = 0.0;
#pragma unroll
        for (int d = 15; d >= 0; --d) {
            if (d < nf) {
                M = fma(-cinf, M, r2[d * rs]);
                r2[d * rs] = M;
            }
        }
#pragma unroll
        for (int d = 15; d >= 0; --d) {
            M = fma(-cinf, M, r1[d * rs]);
            r1[d * rs] = M;
        }
#pragma unroll
        for (int d = 15; d >= 0; --d) {
            M = fma(-cinf, M, r0[d * rs]);
            r0[d * rs] = M;
        }
        const double Mlast = r2[(nf - 1) * rs];                       // M[n-3]
        emit16(s, r0, r0[0], r1[0], std::false_type{});
        emit16(s + 16, r1, r1[0], r2[0], std::false_type{});
        // ---- the last 3 .. 18 samples: rows s+32 .. n-1 (M of rows <= last in r2, the two end rows from the not-a-knot rule) ----
        int i = s + 32;
        double yi = io.y(i);
        double Mi = r2[0];
#pragma unroll 1
        for (; i < n; ++i) {
            gs.push_steady(yi, io, prm.gw);
            if (i + 1 < n) {
                const int i1 = i + 1;
                const int d1 = min(i1 - (s + 32), 15);                // in-range ring row also where the value is not used
                const double Mr = r2[d1 * rs];
                const double Mn = (i1 == n - 2) ? Mn2 : (i1 == n - 1) ? 2.0 * Mn2 - Mlast : Mr;
                const double yn = io.y(i1);
                gs.push_steady(0.5 * (yi + yn) - (Mi + Mn) * 0.0625, io, prm.gw);
                Mi = Mn;
                yi = yn;
            }
        }
    }
    gs.finish(io, prm.gw);
    io.chunk_done();
}

template <int GR, int RS, class IO>
__device__ __forceinline__ void spline_line(IO& io, const int n, const SplineParams& prm, double* ring) {
    if (GR > 0 && n >= prm.long_min) {
        spline_line_long<GR, RS>(io, n, prm, ring);
        return;
    }
    // short lines (and the radius-0 filter): one generic chunk loop with every boundary case in it
    constexpr int C = 16, L = 32;
    constexpr int rs = RS;                         // ring stride in doubles
    const double cinf = prm.cprime[39];            // the pivots have converged to 2 - sqrt(3) long before i = 39
    int b0 = 0;                                    // ring slot of sample s (s is a multiple of 16: 0, 16, 32, 0, ...)
    const int last = n - 3;
    const double M1 = (io.y(0) - 2.0 * io.y(1)) + io.y(2);
    const double Mn2 = (io.y(n - 3) - 2.0 * io.y(n - 2)) + io.y(n - 1);
    double M2v = 0.0, Mn3v = 0.0;
    int fwd = 2;
    double xprev = 0.0;
    double ya = io.y(1), yb = io.y(2);
    GaussStream<GR> gs;
    gs.init();
    for (int s = 0; s < n; s += C, b0 = (b0 == 32) ? 0 : b0 + 16) {
        const int e = min(s + C, n);
        const int top = min(e + L - 1, last);
        while (fwd <= top) {  // forward Thomas sweep, loads batched 8 deep to keep HBM requests in flight
            const int nb = min(8, top - fwd + 1);
            double yy[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) yy[q] = (q < nb) ? io.y(fwd + 1 + q) : 0.0;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                if (q < nb) {
                    const double yc = yy[q];
                    double a = (fwd == 2) ? M1 : xprev;                  // the same roundings as spline_line_long, row by row:
                    if (fwd == last) a += Mn2;                           // boundary terms join x', then ONE fma per row
                    const double x = fma(6.0, (ya - 2.0 * yb) + yc, -a) * prm.cprime[fwd < 39 ? fwd : 39];
                    ring[ring_slot(fwd) * rs] = x;
                    xprev = x;
                    ya = yb;
                    yb = yc;
                    ++fwd;
                }
            }
        }
        const int lo = max(s, 2);
        double Me = 0.0;
        if (lo <= last) {
            int j = top;
            double M = ring[ring_slot(j) * rs];
            for (;;) {
                if (j == last) Mn3v = M;
                if (j == 2) M2v = M;
                if (j < e) ring[ring_slot(j) * rs] = M;
                else if (j == e) Me = M;
                if (j == lo) break;
                --j;
                M = fma(-prm.cprime[j < 39 ? j : 39], M, ring[ring_slot(j) * rs]);
            }
        }
        auto Mval = [&](int i) -> double {
            if (i == 0) return 2.0 * M1 - M2v;
            if (i == 1) return M1;
            if (i == n - 2) return Mn2;
            if (i == n - 1) return 2.0 * Mn2 - Mn3v;
            if (i == e) return Me;
            return ring[ring_slot(i) * rs];
        };
        double Mi = Mval(s);
        double yi = io.y(s);
        for (int i0 = s; i0 < e; i0 += 8) {
            double yy[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) yy[q] = (i0 + q < e && i0 + q + 1 < n) ? io.y(i0 + q + 1) : 0.0;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int i = i0 + q;
                if (i < e) {
                    gs.push(yi, io, prm.gw);
                    if (i + 1 < n) {
                        const double Mn = Mval(i + 1);
                        const double yn = yy[q];
                        gs.push(0.5 * (yi + yn) - (Mi + Mn) * 0.0625, io, prm.gw);
                        Mi = Mn;
                        yi = yn;
                    }
                }
            }
        }
        io.chunk_done();
    }
    gs.finish(io, prm.gw);
    io.chunk_done();
}

// Lines along a strided axis: thread (o, j) owns line  in[o*n*inner + j + i*inner].
template <typename TIn, typename TOut>
struct StridedIO {
    const TIn* yin;
    TOut* uout;          // next output (the outputs of a line are written strictly in order)
    int stride;          // elements between consecutive samples of the line (< 2^31: one IMAD.WIDE per address)
    __device__ __forceinline__ double y(int i) const { return (double)__ldg(yin + (long long)i * stride); }
    // samples i0 .. i0+CNT-1: one 64-bit multiply for the run, then a running pointer
    template <int CNT>
    __device__ __forceinline__ void load_run(int i0, double (&v)[CNT]) const {
        const TIn* p = yin + (long long)i0 * stride;
#pragma unroll
        for (int q = 0; q < CNT; ++q) {
            v[q] = (double)__ldg(p);
            p += stride;
        }
    }
    __device__ __forceinline__ void put(int, double v) {
        *uout = (TOut)v;
        uout += stride;
    }
    __device__ __forceinline__ void chunk_done() {}
};

template <typename TIn, typename TOut, int GR>
__global__ void __launch_bounds__(128)
spline_up_strided_kernel(const TIn* __restrict__ in, TOut* __restrict__ out, int n, long long inner,
                         long long total_lines, SplineParams prm) {
    extern __shared__ double ring_s[];  // [48][blockDim.x]
    const long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (g >= total_lines) return;
    const long long o = g / inner, j = g % inner;
    StridedIO<TIn, TOut> io;
    io.yin = in + o * (long long)n * inner + j;
    io.uout = out + o * (long long)(2 * n - 1) * inner + j;
    io.stride = (int)inner;
    spline_line<GR, 128>(io, n, prm, ring_s + threadIdx.x);
}

// Lines along the contiguous axis: one warp owns 32 consecutive lines; the input lines are staged
// in shared memory with coalesced loads, outputs are staged per chunk and flushed row by row.
constexpr int kZStage = 49;  // >= 2*16 outputs per chunk (+ 2*GR at the end); odd row stride (in doubles) avoids bank conflicts
struct ZLineIO {
    const float* yline;   // this lane's line in global memory (read through L1: a sector serves 8 steps)
    double* ostage;       // [32][kZStage]
    double* out;          // global, first line of this warp
    long long N;          // output line length (2n-1)
    int lines_valid;      // lines of this warp that exist
    int lane;
    int kbase, cnt;
    __device__ __forceinline__ double y(int i) const { return (double)__ldg(yline + i); }
    template <int CNT>
    __device__ __forceinline__ void load_run(int i0, double (&v)[CNT]) const {
#pragma unroll
        for (int q = 0; q < CNT; ++q) v[q] = (double)__ldg(yline + i0 + q);
    }
    __device__ __forceinline__ void put(int k, double v) {
        ostage[lane * kZStage + (k - kbase)] = v;
        ++cnt;
    }
    __device__ __forceinline__ void chunk_done() {
        __syncwarp();
        for (int r = 0; r < lines_valid; ++r)
            for (int t = lane; t < cnt; t += 32) out[r * N + kbase + t] = ostage[r * kZStage + t];
        kbase += cnt;
        cnt = 0;
        __syncwarp();
    }
};

// Lines along the contiguous axis: a warp owns 32 consecutive lines (lane = line).  Inputs are read
// straight from global memory (each lane walks its own line; the 32-byte sectors are reused from
// L1 for 8 steps), outputs are staged per chunk in shared memory and flushed row by row (coalesced).
// 4 warps per CTA, each with its own ring and output stage: no block-level barrier.
template <int GR>
__global__ void __launch_bounds__(128)
spline_up_z_kernel(const float* __restrict__ in, double* __restrict__ out, int n, long long total_lines,
                   int npad, SplineParams prm) {
    extern __shared__ double zs[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double* ring = zs + (size_t)warp * (48 * 32 + 32 * kZStage);   // [48][32]
    double* ostage = ring + 48 * 32;                                // [32][kZStage]
    const long long l0 = ((long long)blockIdx.x * 4 + warp) * 32;
    if (l0 >= total_lines) return;
    const int valid = (int)min((long long)32, total_lines - l0);
    ZLineIO io;
    io.yline = in + (l0 + min(lane, valid - 1)) * n;               // tail lanes recompute the last line
    io.ostage = ostage;
    io.out = out + l0 * (long long)(2 * n - 1);
    io.N = 2 * n - 1;
    io.lines_valid = valid;
    io.lane = lane;
    io.kbase = 0;
    io.cnt = 0;
    (void)npad;
    spline_line<GR, 32>(io, n, prm, ring + lane);
}

static bool fill_spline_params(SplineParams& p, const double* gw, int radius) {
    p.cprime[0] = p.cprime[1] = 0.0;
    p.cprime[2] = 0.25;
    for (int i = 3; i < 40; ++i) p.cprime[i] = 1.0 / (4.0 - p.cprime[i - 1]);
    for (int j = 0; j < 9; ++j) p.gw[j] = 0.0;
    for (int j = 0; j <= radius; ++j) p.gw[j] = gw ? gw[radius + j] : (j == 0 ? 1.0 : 0.0);
    p.long_min = getenv("MAD_SPLINE_GENERIC") ? 0x7fffffff : 64;
    return p.cprime[15] == p.cprime[39];   // the unrolled chunks use the limit pivot for every row >= 15
}

extern "C" size_t mad_upsample_workspace_bytes(int bx, int by, int bz) {
    size_t a = (size_t)bx * by * (2 * (size_t)bz - 1) * sizeof(double);
    size_t b = (2 * (size_t)bx - 1) * by * (2 * (size_t)bz - 1) * sizeof(double);
    return mad_align_up(a, 256) + mad_align_up(b, 256);
}

template <int GR>
static int upsample_launch(const float* base, int bx, int by, int bz, const SplineParams& prm, float* up,
                           double* wsA, double* wsB, cudaStream_t st) {
    // pass Z (contiguous axis, smallest array): f32 [bx][by][bz] -> f64 [bx][by][2bz-1]
    {
        const long long lines = (long long)bx * by;
        const int npad = bz | 1;
        const size_t smem = (size_t)4 * (48 * 32 + 32 * kZStage) * sizeof(double);
        MAD_CUDA(cudaFuncSetAttribute(spline_up_z_kernel<GR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        MAD_PROF("spline_up_z_kernel", st);
        spline_up_z_kernel<GR><<<(unsigned)mad_ceil_div(lines, 128), 128, smem, st>>>(base, wsA, bz, lines, npad, prm);
        MAD_LAUNCH_OK();
    }
    const size_t ring_smem = 48 * 128 * sizeof(double);
    // pass X: f64 [bx][by][Z] -> f64 [2bx-1][by][Z],  Z = 2bz-1
    {
        const long long inner = (long long)by * (2 * bz - 1);
        MAD_CUDA(cudaFuncSetAttribute(spline_up_strided_kernel<double, double, GR>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ring_smem));
        MAD_PROF("spline_up_x_kernel", st);
        spline_up_strided_kernel<double, double, GR>
            <<<(unsigned)mad_ceil_div(inner, 128), 128, ring_smem, st>>>(wsA, wsB, bx, inner, inner, prm);
        MAD_LAUNCH_OK();
    }
    // pass Y: f64 [X][by][Z] -> f32 [X][2by-1][Z],  X = 2bx-1
    {
        const long long inner = 2 * bz - 1;
        const long long lines = (long long)(2 * bx - 1) * inner;
        MAD_CUDA(cudaFuncSetAttribute(spline_up_strided_kernel<double, float, GR>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ring_smem));
        MAD_PROF("spline_up_y_kernel", st);
        spline_up_strided_kernel<double, float, GR>
            <<<(unsigned)mad_ceil_div(lines, 128), 128, ring_smem, st>>>(wsB, up, by, inner, lines, prm);
        MAD_LAUNCH_OK();
    }
    return MAD_OK;
}

extern "C" int mad_upsample_presmooth(const float* base, int bx, int by, int bz, const double* gauss_w_host,
                                      int radius, float* up, void* workspace, size_t workspace_bytes,
                                      void* stream) {
    MAD_CHECK_ARG(base && up && workspace);
    MAD_CHECK_ARG(bx >= 5 && by >= 5 && bz >= 5);
    MAD_CHECK_ARG(radius >= 0 && radius <= 8 && (radius == 0 || gauss_w_host));
    MAD_CHECK_ARG(2 * bx - 1 > radius && 2 * by - 1 > radius && 2 * bz - 1 > radius);
    MAD_CHECK_ARG(workspace_bytes >= mad_upsample_workspace_bytes(bx, by, bz));
    MAD_CHECK_ARG((long long)by * (2 * (long long)bz - 1) < 0x7fffffffLL);      // line strides are 32-bit element counts
    SplineParams prm;
    if (!fill_spline_params(prm, gauss_w_host, radius)) {
        mad_set_error("mad_upsample_presmooth: Thomas pivots have not converged by row 15 on this host");
        return MAD_ERR_ARG;
    }
    double* wsA = reinterpret_cast<double*>(workspace);
    double* wsB = reinterpret_cast<double*>(reinterpret_cast<char*>(workspace) +
                                            mad_align_up((size_t)bx * by * (2 * (size_t)bz - 1) * sizeof(double), 256));
    cudaStream_t st = (cudaStream_t)stream;
    switch (radius) {
        case 0: return upsample_launch<0>(base, bx, by, bz, prm, up, wsA, wsB, st);
        case 1: return upsample_launch<1>(base, bx, by, bz, prm, up, wsA, wsB, st);
        case 2: return upsample_launch<2>(base, bx, by, bz, prm, up, wsA, wsB, st);
        case 3: return upsample_launch<3>(base, bx, by, bz, prm, up, wsA, wsB, st);
        case 4: return upsample_launch<4>(base, bx, by, bz, prm, up, wsA, wsB, st);
        case 6: return upsample_launch<6>(base, bx, by, bz, prm, up, wsA, wsB, st);
        case 8: return upsample_launch<8>(base, bx, by, bz, prm, up, wsA, wsB, st);
        default:
            mad_set_error("mad_upsample_presmooth: presmoothing radius %d not instantiated (0-4, 6, 8)", radius);
            return MAD_ERR_ARG;
    }
}

// ------------------------------------------------------------------------------------------
// a3/a4: LoG + Gaussian with SciPy's pass structure.
//   pass X:  f         -> P0 = g*f,  Q0 = g''*f
//   pass Y:  P0, Q0    -> P01 = g*P0, R = g''*P0, S = g*Q0
//   pass Z:  P01, R, S -> gauss = g*P01;  LoG = (g*S + g*R) + g''*P01;  out = max(0, -scale*LoG)
// Every 1-D result is rounded to float32 (as SciPy stores it) before the next pass consumes it.
// ------------------------------------------------------------------------------------------
struct ConvW {
    double w0[17];  // order-0 weights, index |j|
    double w2[17];  // order-2 weights, index |j|
};

template <typename ACC> struct Wt;
template <> struct Wt<double> { static __device__ __forceinline__ double get(double w) { return w; } };
template <> struct Wt<float> { static __device__ __forceinline__ float get(double w) { return (float)w; } };

// The sliding windows hold the samples ALREADY CONVERTED to the accumulation type: one
// F2F.F64.F32 per loaded sample instead of one per tap (the conversion runs at 1/8 of the FP64
// FMA rate and was the bound of the first version of these kernels).
template <int R, typename ACC>
__device__ __forceinline__ void conv_both(const ACC* win, int t, const ConvW& w, float& o0, float& o2) {
    const ACC c = win[t + R];
    ACC a0 = c * Wt<ACC>::get(w.w0[0]);
    ACC a2 = c * Wt<ACC>::get(w.w2[0]);
#pragma unroll
    for (int jj = R; jj >= 1; --jj) {
        const ACC s = win[t + R - jj] + win[t + R + jj];
        a0 = fma(s, Wt<ACC>::get(w.w0[jj]), a0);
        a2 = fma(s, Wt<ACC>::get(w.w2[jj]), a2);
    }
    o0 = (float)a0;
    o2 = (float)a2;
}

template <int R, typename ACC>
__device__ __forceinline__ float conv_g(const ACC* win, int t, const ConvW& w) {
    ACC a0 = win[t + R] * Wt<ACC>::get(w.w0[0]);
#pragma unroll
    for (int jj = R; jj >= 1; --jj) {
        const ACC s = win[t + R - jj] + win[t + R + jj];
        a0 = fma(s, Wt<ACC>::get(w.w0[jj]), a0);
    }
    return (float)a0;
}

// Tap-outer forms of the two routines above for T outputs at once: the loop over the taps is outermost, so the T
// (or 2 T) accumulator chains advance in lock step and every FP64 instruction has T independent neighbours
// (the per-output summation order is unchanged, hence the same bits).
template <int R, int T, typename ACC>
__device__ __forceinline__ void conv_both_rows(const ACC* win, const ConvW& w, float* o0, float* o2) {
    ACC a0[T], a2[T];
#pragma unroll
    for (int t = 0; t < T; ++t) {
        a0[t] = win[t + R] * Wt<ACC>::get(w.w0[0]);
        a2[t] = win[t + R] * Wt<ACC>::get(w.w2[0]);
    }
#pragma unroll
    for (int jj = R; jj >= 1; --jj) {
#pragma unroll
        for (int t = 0; t < T; ++t) {
            const ACC s = win[t + R - jj] + win[t + R + jj];
            a0[t] = fma(s, Wt<ACC>::get(w.w0[jj]), a0[t]);
            a2[t] = fma(s, Wt<ACC>::get(w.w2[jj]), a2[t]);
        }
    }
#pragma unroll
    for (int t = 0; t < T; ++t) { o0[t] = (float)a0[t]; o2[t] = (float)a2[t]; }
}

template <int R, int T, typename ACC>
__device__ __forceinline__ void conv_g_rows(const ACC* win, const ConvW& w, float* o0) {
    ACC a0[T];
#pragma unroll
    for (int t = 0; t < T; ++t) a0[t] = win[t + R] * Wt<ACC>::get(w.w0[0]);
#pragma unroll
    for (int jj = R; jj >= 1; --jj) {
#pragma unroll
        for (int t = 0; t < T; ++t) {
            const ACC s = win[t + R - jj] + win[t + R + jj];
            a0[t] = fma(s, Wt<ACC>::get(w.w0[jj]), a0[t]);
        }
    }
#pragma unroll
    for (int t = 0; t < T; ++t) o0[t] = (float)a0[t];
}

__device__ __forceinline__ void cp_async4(float* smem_dst, const float* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// MODE 0: pass X (in0=f; o0=P0, o1=Q0).  MODE 1: pass Y (in0=P0, in1=Q0; o0=P01, o1=R, o2=S).
// One thread per line, marching along the (strided) axis; consecutive threads own consecutive z,
// so every load and store of a warp is one coalesced 128-byte line.  Samples travel
// global -> shared through cp.async (LDGSTS) into a private per-thread ring of D rows, PF groups
// of T rows ahead of the arithmetic: the HBM latency is covered by ~24 rows in flight per thread
// without spending registers on them, and no block-level barrier is needed (a thread only ever
// reads what it copied itself).  The reflect boundary is applied when the copy is issued.
template <int R, typename ACC, int MODE>
__global__ void __launch_bounds__(128)
log_pass_strided_kernel(const float* __restrict__ in0, const float* __restrict__ in1, float* __restrict__ o0,
                        float* __restrict__ o1, float* __restrict__ o2, int n, long long inner,
                        long long total_lines, int seg_len, ConvW w) {
    constexpr int T = ((2 * R) % 8 == 0) ? 8 : 4, W = T + 2 * R;
    constexpr int NA = MODE == 1 ? 2 : 1;
    constexpr int D = 32, PF = D / T - 1;          // ring depth (rows) and groups in flight ahead
    constexpr int G0 = 2 * R / T;                  // groups that make up the initial window
    static_assert((2 * R) % T == 0, "window prologue must be whole groups");
    extern __shared__ float ring[];                // [D][NA][128]
    const long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (g >= total_lines) return;
    const long long o = g / inner, j = g % inner;
    const long long base = o * (long long)n * inner + j;
    const int a0 = blockIdx.y * seg_len;
    const int a1 = min(n, a0 + seg_len);
    const int q_end = a1 - a0 + 2 * R;             // samples this thread needs: q = pos - (a0 - R) in [0, q_end)
    float* my = ring + threadIdx.x;
    auto issue = [&](int grp) {
        const int q0 = grp * T;
        float* dst0 = my + ((q0 & (D - 1)) * NA) * 128;          // T divides D: the group's slots are consecutive
        const int p0 = a0 - R + q0;                              // position of the group's first sample on the axis
        if (p0 >= 0 && p0 + T <= n && q0 + T <= q_end) {         // interior: no reflection, one address per group
            const long long off = base + (long long)p0 * inner;
#pragma unroll
            for (int i = 0; i < T; ++i) {
                cp_async4(dst0 + i * NA * 128, in0 + off + (long long)i * inner);
                if (MODE == 1) cp_async4(dst0 + i * NA * 128 + 128, in1 + off + (long long)i * inner);
            }
        } else {
#pragma unroll
            for (int i = 0; i < T; ++i) {
                const int q = q0 + i;
                if (q < q_end) {
                    const long long off = base + (long long)mad_reflect(a0 - R + q, n) * inner;
                    cp_async4(dst0 + i * NA * 128, in0 + off);
                    if (MODE == 1) cp_async4(dst0 + i * NA * 128 + 128, in1 + off);
                }
            }
        }
        cp_async_commit();
    };
    static_assert(G0 <= PF + 1, "the initial window must fit the ring");
#pragma unroll
    for (int grp = 0; grp <= PF; ++grp) issue(grp);         // fill the ring: groups 0 .. PF
    cp_async_wait<PF + 1 - G0>();                           // groups 0 .. G0-1 (the initial window) have landed
    ACC wa[W];
    ACC wb[MODE == 1 ? W : 1];
#pragma unroll
    for (int i = 0; i < 2 * R; ++i) {
        wa[i] = (ACC)my[(i * NA) * 128];
        if (MODE == 1) wb[i] = (ACC)my[(i * NA + 1) * 128];
    }
#pragma unroll
    for (int grp = PF + 1; grp <= PF + G0; ++grp) issue(grp);   // their slots are free again
    int grp = G0;
    for (int a = a0; a < a1; a += T, ++grp) {
        cp_async_wait<PF>();                                 // group `grp` (the T new samples of this step) has landed
#pragma unroll
        for (int i = 0; i < T; ++i) {
            const int slot = (grp * T + i) & (D - 1);
            wa[2 * R + i] = (ACC)my[(slot * NA) * 128];
            if (MODE == 1) wb[2 * R + i] = (ACC)my[(slot * NA + 1) * 128];
        }
        issue(grp + PF + 1);                                 // refill the slots just read
#pragma unroll
        for (int t = 0; t < T; ++t) {
            if (a + t < a1) {
                const long long off = base + (long long)(a + t) * inner;
                float r0, r2;
                conv_both<R, ACC>(wa, t, w, r0, r2);
                o0[off] = r0;
                o1[off] = r2;
                if (MODE == 1) o2[off] = conv_g<R, ACC>(wb, t, w);
            }
        }
#pragma unroll
        for (int i = 0; i < 2 * R; ++i) {
            wa[i] = wa[i + T];
            if (MODE == 1) wb[i] = wb[i + T];
        }
    }
    cp_async_wait<0>();
}

// Pass Z (contiguous axis).  Persistent CTAs walk over batches of rows; the three input rows of the
// NEXT batch travel global -> shared with cp.async (4-byte copies: rows of an odd-length grid are
// only 4-byte aligned; the reflect halo is applied by the copy's source index) while the current
// batch is being convolved, so the HBM latency is hidden behind the FP64 work.  A thread produces
// T consecutive outputs of one row from a register window converted once to the accumulation
// type, one input array after the other; results are staged in shared memory and written as
// whole rows (coalesced).
template <int R, typename ACC>
__global__ void __launch_bounds__(384)
log_pass_z_kernel(const float* __restrict__ P01, const float* __restrict__ Rr, const float* __restrict__ S,
                  float* __restrict__ log_out, float* __restrict__ gauss_out, int nz, long long n_rows,
                  int rows_per_cta, int rs_in, int rs_out, long long n_batches, float scale, ConvW w) {
    constexpr int T = 8, W = T + 2 * R;
    extern __shared__ __align__(16) float zsm[];
    const size_t in_buf = (size_t)3 * rows_per_cta * rs_in;          // floats per input buffer
    float* sout0 = zsm + 2 * in_buf;
    float* sout1 = sout0 + (size_t)rows_per_cta * rs_out;
    const int tid = threadIdx.x;
    const int halo_len = nz + 2 * R;
    auto issue = [&](long long batch, int buf) {
        if (batch < n_batches) {
            const long long row0 = batch * rows_per_cta;
            const int rows = (int)min((long long)rows_per_cta, n_rows - row0);
            float* d0 = zsm + buf * in_buf;
            for (int r = 0; r < rows; ++r) {
                const long long gb = (row0 + r) * nz;
                for (int t = tid; t < halo_len; t += blockDim.x) {
                    const long long src = gb + mad_reflect(t - R, nz);
                    float* d = d0 + r * rs_in + t;
                    cp_async4(d, P01 + src);
                    cp_async4(d + (size_t)rows_per_cta * rs_in, Rr + src);
                    cp_async4(d + (size_t)2 * rows_per_cta * rs_in, S + src);
                }
            }
        }
        cp_async_commit();
    };
    const int n_chunks = (nz + T - 1) / T;
    int buf = 0;
    issue(blockIdx.x, 0);
    for (long long batch = blockIdx.x; batch < n_batches; batch += gridDim.x, buf ^= 1) {
        issue(batch + gridDim.x, buf ^ 1);
        cp_async_wait<1>();                                           // this batch's rows have landed
        __syncthreads();
        const long long row0 = batch * rows_per_cta;
        const int rows = (int)min((long long)rows_per_cta, n_rows - row0);
        const float* sin0 = zsm + buf * in_buf;
        const float* sin1 = sin0 + (size_t)rows_per_cta * rs_in;
        const float* sin2 = sin1 + (size_t)rows_per_cta * rs_in;
        for (int it = tid; it < rows * n_chunks; it += blockDim.x) {
            const int r = it / n_chunks, c = it % n_chunks;
            const int z0 = c * T;
            ACC win[W];
            auto load_window = [&](const float* src) {
                const float4* p = reinterpret_cast<const float4*>(src + r * rs_in + z0);
#pragma unroll
                for (int q = 0; q < W / 4; ++q) {
                    const float4 v = p[q];
                    win[4 * q] = (ACC)v.x; win[4 * q + 1] = (ACC)v.y; win[4 * q + 2] = (ACC)v.z; win[4 * q + 3] = (ACC)v.w;
                }
            };
            float gs[T], t3[T], t2[T], t1[T];
            load_window(sin0);
#pragma unroll
            for (int t = 0; t < T; ++t) conv_both<R, ACC>(win, t, w, gs[t], t3[t]);
            load_window(sin1);
#pragma unroll
            for (int t = 0; t < T; ++t) t2[t] = conv_g<R, ACC>(win, t, w);
            load_window(sin2);
#pragma unroll
            for (int t = 0; t < T; ++t) t1[t] = conv_g<R, ACC>(win, t, w);
#pragma unroll
            for (int t = 0; t < T; ++t) {
                const float lap = __fadd_rn(__fadd_rn(t1[t], t2[t]), t3[t]);
                float m = __fmul_rn(-lap, scale);
                if (m < 0.f) m = 0.f;
                if (z0 + t < nz) {
                    sout0[r * rs_out + z0 + t] = m;
                    sout1[r * rs_out + z0 + t] = gs[t];
                }
            }
        }
        __syncthreads();
        for (int r = 0; r < rows; ++r) {
            const long long gb = (row0 + r) * nz;
            for (int t = tid; t < nz; t += blockDim.x) {
                log_out[gb + t] = sout0[r * rs_out + t];
                gauss_out[gb + t] = sout1[r * rs_out + t];
            }
        }
        // the next iteration's barrier (after its wait) orders these reads of sout before its writes
    }
    cp_async_wait<0>();
}

// Passes Y and Z fused (one launch per octave instead of two, and no P01 / R / S round trip through HBM:
// 17 B per voxel instead of 40).  A CTA owns one x plane and a tile of TZ = 128 - 2R z columns plus the R-column
// halo on either side (reflected at the grid ends): 128 threads, thread t <-> column z0 - R + t.
//   phase A  every thread marches along y exactly like pass Y above (private cp.async ring, float64 register
//            windows) and produces T = 8 rows of P01, R, S for its column, rounded to float32 as SciPy stores them
//            and parked as float64 in a shared-memory stage [3][T][128];
//   phase B  128 work items (row, chunk of CW = 7 z) -- every thread has one: window of CW + 2R staged values per array
//            -> Gaussian and the three Laplacian terms, summed and clamped in float32, written to an output stage;
//   phase C  the T x TZ output tile goes to HBM as whole row segments (coalesced).
// Two barriers per T rows; the HBM latency is covered by the cp.async ring as before.
template <int R, int DEPTH = 32>
struct YzCfg {
    static constexpr int T = 8, W = T + 2 * R, D = DEPTH, PF = D / T - 1, G0 = 2 * R / T;
    static constexpr int TZ = 128 - 2 * R;                      // output columns per CTA
    static constexpr int CH = 128 / T;                          // phase-B chunks per row: T rows x CH chunks = 128 items
    static constexpr int CW = TZ / CH;                          // columns per chunk (7 for R = 8: odd, see below)
    static constexpr int RS = 128;                              // stage row stride in doubles
    static constexpr int OS = TZ;                               // output-stage row stride in floats
    static constexpr size_t ring_bytes = (size_t)D * 2 * 128 * sizeof(float);
    static constexpr size_t stage_bytes = (size_t)3 * T * RS * sizeof(double);
    static constexpr size_t out_bytes = (size_t)2 * T * OS * sizeof(float);
    static constexpr size_t smem = ring_bytes + stage_bytes + out_bytes;
    // R = 8 (the LoG of sigma = 2): 112 columns = 16 chunks of 7.  An odd chunk width makes the chunk-strided window loads
    // of a half-warp (16 items of one row) and the output-stage stores of a warp hit distinct banks with a plain layout.
    static constexpr bool ok = TZ % CH == 0 && (CW % 2) == 1 && (2 * R) % T == 0 && G0 <= PF + 1;
};

template <int R, typename ACC, int MINB, int DEPTH>
__global__ void __launch_bounds__(128, MINB)
log_pass_yz_kernel(const float* __restrict__ P0, const float* __restrict__ Q0, float* __restrict__ log_out,
                   float* __restrict__ gauss_out, int ny, int nz, int n_ztiles, float scale, ConvW w) {
    using C = YzCfg<R, DEPTH>;
    static_assert(C::ok, "the fused pass needs a kernel radius that is a multiple of 4");
    constexpr int T = C::T, W = C::W, D = C::D, PF = C::PF, G0 = C::G0, TZ = C::TZ, CH = C::CH, CW = C::CW, RS = C::RS, OS = C::OS;
    constexpr int WB = CW + 2 * R;                               // phase-B window
    extern __shared__ __align__(16) unsigned char yz_smem[];
    float* ring = reinterpret_cast<float*>(yz_smem);                                    // [D][2][128]
    double* stage = reinterpret_cast<double*>(yz_smem + C::ring_bytes);                 // [3][T][RS]
    float* sout = reinterpret_cast<float*>(yz_smem + C::ring_bytes + C::stage_bytes);   // [2][T][TZ]
    const int tid = threadIdx.x;
    const int x = blockIdx.x / n_ztiles, zt = blockIdx.x - x * n_ztiles;
    const int z0 = zt * TZ;
    int zc = z0 - R + tid;                                       // this thread's column (reflected; clamped when unused)
    if (zc >= nz + R) zc = nz + R - 1;
    zc = mad_reflect(zc, nz);
    const long long plane = (long long)x * ny * nz;
    const long long base = plane + zc;
    const int q_end = ny + 2 * R;                                // samples q = y + R in [0, q_end)
    float* my = ring + tid;
    auto issue = [&](int grp) {
        const int q0 = grp * T;
        float* dst0 = my + ((q0 & (D - 1)) * 2) * 128;           // T divides D: the group's slots are consecutive
        if (q0 >= R && q0 + T <= ny + R) {                       // interior rows: no reflection, one address per group
            const float* p0 = P0 + base + (long long)(q0 - R) * nz;
            const float* p1 = Q0 + base + (long long)(q0 - R) * nz;
#pragma unroll
            for (int i = 0; i < T; ++i) {
                cp_async4(dst0 + i * 256, p0 + (long long)i * nz);
                cp_async4(dst0 + i * 256 + 128, p1 + (long long)i * nz);
            }
        } else {
#pragma unroll
            for (int i = 0; i < T; ++i) {
                const int q = q0 + i;
                if (q < q_end) {
                    const long long off = base + (long long)mad_reflect(q - R, ny) * nz;
                    cp_async4(dst0 + i * 256, P0 + off);
                    cp_async4(dst0 + i * 256 + 128, Q0 + off);
                }
            }
        }
        cp_async_commit();
    };
#pragma unroll
    for (int grp = 0; grp <= PF; ++grp) issue(grp);
    cp_async_wait<PF + 1 - G0>();
    ACC wa[W], wb[W];
#pragma unroll
    for (int i = 0; i < 2 * R; ++i) {
        wa[i] = (ACC)my[(i * 2) * 128];
        wb[i] = (ACC)my[(i * 2 + 1) * 128];
    }
#pragma unroll
    for (int grp = PF + 1; grp <= PF + G0; ++grp) issue(grp);
    const int br = tid / CH, bc = tid - br * CH;                 // phase-B work item: row br, chunk bc
    const bool b_active = (z0 + bc * CW) < nz;
    int grp = G0;
    for (int a = 0; a < ny; a += T, ++grp) {
        // ---- phase A: T rows of P01 / R / S for this column
        cp_async_wait<PF>();
#pragma unroll
        for (int i = 0; i < T; ++i) {
            const int slot = (grp * T + i) & (D - 1);
            wa[2 * R + i] = (ACC)my[(slot * 2) * 128];
            wb[2 * R + i] = (ACC)my[(slot * 2 + 1) * 128];
        }
        issue(grp + PF + 1);
        {
            float r0[T], r2[T], r1[T];
            conv_both_rows<R, T, ACC>(wa, w, r0, r2);
            conv_g_rows<R, T, ACC>(wb, w, r1);
#pragma unroll
            for (int t = 0; t < T; ++t) {
                const int slot = t * RS + tid;
                stage[0 * T * RS + slot] = (double)r0[t];        // P01 (float32-rounded as SciPy stores it)
                stage[1 * T * RS + slot] = (double)r2[t];        // R
                stage[2 * T * RS + slot] = (double)r1[t];        // S
            }
        }
#pragma unroll
        for (int i = 0; i < 2 * R; ++i) {
            wa[i] = wa[i + T];
            wb[i] = wb[i + T];
        }
        __syncthreads();
        // ---- phase B: (row, chunk) items from the staged rows
        const int rows = min(T, ny - a);
        if (b_active && br < rows) {
            ACC win[WB];
            auto load_window = [&](int arr) {
                const double* src = stage + (arr * T + br) * RS + bc * CW;
#pragma unroll
                for (int q = 0; q < WB; ++q) win[q] = (ACC)src[q];
            };
            float gs[CW], t3[CW], t2[CW], t1[CW];
            load_window(0);
            conv_both_rows<R, CW, ACC>(win, w, gs, t3);
            load_window(1);
            conv_g_rows<R, CW, ACC>(win, w, t2);
            load_window(2);
            conv_g_rows<R, CW, ACC>(win, w, t1);
#pragma unroll
            for (int t = 0; t < CW; ++t) {
                const float lap = __fadd_rn(__fadd_rn(t1[t], t2[t]), t3[t]);
                float m = __fmul_rn(-lap, scale);
                if (m < 0.f) m = 0.f;
                sout[(0 * T + br) * OS + bc * CW + t] = m;
                sout[(1 * T + br) * OS + bc * CW + t] = gs[t];
            }
        }
        __syncthreads();
        // ---- phase C: coalesced row segments
        if (tid < TZ && z0 + tid < nz) {                          // thread = column: every row is one coalesced segment
            const float* so = sout + tid;
            float* lo_p = log_out + plane + (long long)a * nz + z0 + tid;
            float* ga_p = gauss_out + plane + (long long)a * nz + z0 + tid;
#pragma unroll
            for (int r = 0; r < T; ++r) {
                if (r < rows) {
                    lo_p[(long long)r * nz] = so[(0 * T + r) * OS];
                    ga_p[(long long)r * nz] = so[(1 * T + r) * OS];
                }
            }
        }
        // the next iteration's first barrier orders these reads of sout before its phase-B writes, and this
        // iteration's second barrier ordered the phase-B reads of the stage before the next phase-A writes
    }
    cp_async_wait<0>();
}

extern "C" size_t mad_log_gauss_workspace_bytes(int nx, int ny, int nz) {
    const size_t v = mad_align_up((size_t)nx * ny * nz * sizeof(float), 256);
    return 5 * v;  // P0, Q0, P01, R, S
}

template <int R, typename ACC>
static int log_gauss_launch(const float* grid, int nx, int ny, int nz, const ConvW& w, float scale, float* log_out,
                            float* gauss_out, float* ws, cudaStream_t st) {
    const size_t v = mad_align_up((size_t)nx * ny * nz * sizeof(float), 256) / sizeof(float);
    float *P0 = ws, *Q0 = ws + v, *P01 = ws + 2 * v, *Rr = ws + 3 * v, *S = ws + 4 * v;
    const int sms = mad_sm_count();
    auto segs_for = [&](long long lines, int n) {
        // enough CTAs to fill the machine (~8 CTAs of 128 threads per SM), segments multiple of 16
        long long ctas = mad_ceil_div(lines, 128);
        int segs = (int)std::max<long long>(1, std::min<long long>(mad_ceil_div((long long)sms * 8, ctas), mad_ceil_div(n, 64)));
        int seg_len = (int)mad_ceil_div(mad_ceil_div(n, segs), 16) * 16;
        return seg_len;
    };
    {
        const long long inner = (long long)ny * nz;
        const int seg_len = segs_for(inner, nx);
        dim3 grid_dim((unsigned)mad_ceil_div(inner, 128), (unsigned)mad_ceil_div(nx, seg_len));
        MAD_PROF("log_pass_x_kernel", st);
        log_pass_strided_kernel<R, ACC, 0><<<grid_dim, 128, 32 * 1 * 128 * sizeof(float), st>>>(grid, nullptr, P0, Q0, nullptr, nx, inner, inner, seg_len, w);
        MAD_LAUNCH_OK();
    }
    // Passes Y and Z are independent per x plane and planes are contiguous, so they CAN run slab by slab through
    // one small set of intermediates that stays in the 126 MB L2 (MAD_LOG_SLAB = planes per slab).  Measured at
    // C2 on B200 it loses: 8 planes 13.1 ms/step, 16: 11.4, 48: 10.5 against 10.0 unslabbed -- the passes are bound
    // by FP64 issue and load latency, not by HBM bytes, and small launches under-fill the machine.  Default: off.
    // Default: passes Y and Z fused in one launch (MAD_LOG_FUSED=0 selects the two-launch path below).
    static const bool fused = !(getenv("MAD_LOG_FUSED") && atoi(getenv("MAD_LOG_FUSED")) == 0);
    if constexpr (YzCfg<R>::ok) if (fused) {
        using C = YzCfg<R, 32>;
        const int n_ztiles = (int)mad_ceil_div(nz, C::TZ);
        const unsigned n_cta = (unsigned)((long long)nx * n_ztiles);
        // 3 CTAs per SM (168 registers); 2 CTAs with 220 registers and 4 CTAs with 128 registers and a 16-row ring
        // measured the same 2.3 ms at C2: the kernel is bound by instruction issue, not by latency (DESIGN.md section 4)
        MAD_CUDA(cudaFuncSetAttribute(log_pass_yz_kernel<R, ACC, 3, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::smem));
        MAD_PROF("log_pass_yz_kernel", st);
        log_pass_yz_kernel<R, ACC, 3, 32><<<n_cta, 128, C::smem, st>>>(P0, Q0, log_out, gauss_out, ny, nz, n_ztiles, scale, w);
        MAD_LAUNCH_OK();
        return MAD_OK;
    }
    const long long plane = (long long)ny * nz;
    static const long long slab_env = getenv("MAD_LOG_SLAB") ? atoll(getenv("MAD_LOG_SLAB")) : 0;
    long long slab = slab_env;
    if (slab <= 0 || slab > nx) slab = nx;
    const int n_chunks = (nz + 7) / 8;
    const int rs_in = (n_chunks * 8 + 2 * R + 3) / 4 * 4;
    const int rs_out = (nz + 3) / 4 * 4;
    const size_t row_bytes = (size_t)(2 * 3 * rs_in + 2 * rs_out) * sizeof(float);   // double-buffered inputs + outputs
    // rows per batch: the value (within ~72 KB of shared memory, 3-4 CTAs per SM) that leaves the fewest
    // idle threads over the rows x chunks work items of a batch (wider CTAs measured slower)
    const int max_rows = (int)std::max<size_t>(1, std::min<size_t>(32, (72 * 1024) / row_bytes));
    int rows = 1;
    double best_eff = -1.0;
    for (int r = 1; r <= max_rows; ++r) {
        const long long work = (long long)r * n_chunks;
        const double eff = (double)work / (double)(mad_ceil_div(work, 128) * 128);
        if (eff > best_eff + 1e-9) { best_eff = eff; rows = r; }
    }
    const size_t smem = rows * row_bytes;
    if (smem > 200 * 1024) {
        mad_set_error("mad_log_gauss: z extent %d too long for the shared-memory row stage", nz);
        return MAD_ERR_ARG;
    }
    MAD_CUDA(cudaFuncSetAttribute(log_pass_z_kernel<R, ACC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 48 * 1024)));
    const int ctas_per_sm = (int)std::max<size_t>(1, std::min<size_t>(4, (size_t)(216 * 1024) / std::max<size_t>(smem, 1)));
    for (long long x0 = 0; x0 < nx; x0 += slab) {
        const int sx = (int)std::min<long long>(slab, nx - x0);
        const long long off = x0 * plane;
        {
            const long long inner = nz;
            const long long lines = (long long)sx * nz;
            const int seg_len = segs_for(lines, ny);
            dim3 grid_dim((unsigned)mad_ceil_div(lines, 128), (unsigned)mad_ceil_div(ny, seg_len));
            MAD_PROF("log_pass_y_kernel", st);
            log_pass_strided_kernel<R, ACC, 1><<<grid_dim, 128, 32 * 2 * 128 * sizeof(float), st>>>(P0 + off, Q0 + off, P01, Rr, S, ny, inner, lines, seg_len, w);
            MAD_LAUNCH_OK();
        }
        {
            const long long n_rows = (long long)sx * ny;
            const long long n_batches = mad_ceil_div(n_rows, rows);
            const unsigned grid_z = (unsigned)std::min<long long>(n_batches, (long long)sms * ctas_per_sm);
            MAD_PROF("log_pass_z_kernel", st);
            log_pass_z_kernel<R, ACC><<<grid_z, 128, smem, st>>>(P01, Rr, S, log_out + off, gauss_out + off, nz, n_rows, rows, rs_in, rs_out, n_batches, scale, w);
            MAD_LAUNCH_OK();
        }
    }
    return MAD_OK;
}

extern "C" int mad_log_gauss(const float* grid, int nx, int ny, int nz, const double* w0_host, const double* w2_host,
                             int radius, float scale, float* log_out, float* gauss_out, void* workspace,
                             size_t workspace_bytes, int exact_f64, void* stream) {
    MAD_CHECK_ARG(grid && log_out && gauss_out && workspace && w0_host && w2_host);
    MAD_CHECK_ARG(radius >= 1 && radius <= 16);
    MAD_CHECK_ARG(nx >= 2 * radius + 1 && ny >= 2 * radius + 1 && nz >= 2 * radius + 1);
    MAD_CHECK_ARG(workspace_bytes >= mad_log_gauss_workspace_bytes(nx, ny, nz));
    ConvW w;
    for (int j = 0; j < 17; ++j) w.w0[j] = w.w2[j] = 0.0;
    for (int j = 0; j <= radius; ++j) {
        w.w0[j] = w0_host[radius + j];
        w.w2[j] = w2_host[radius + j];
    }
    float* ws = reinterpret_cast<float*>(workspace);
    cudaStream_t st = (cudaStream_t)stream;
#define MAD_LOG_CASE(RR)                                                                                   \
    case RR:                                                                                               \
        return exact_f64 ? log_gauss_launch<RR, double>(grid, nx, ny, nz, w, scale, log_out, gauss_out, ws, st) \
                         : log_gauss_launch<RR, float>(grid, nx, ny, nz, w, scale, log_out, gauss_out, ws, st);
    switch (radius) {
        MAD_LOG_CASE(4)
        MAD_LOG_CASE(6)
        MAD_LOG_CASE(8)
        MAD_LOG_CASE(10)
        MAD_LOG_CASE(12)
        default:
            mad_set_error("mad_log_gauss: kernel radius %d not instantiated (4, 6, 8, 10, 12)", radius);
            return MAD_ERR_ARG;
    }
#undef MAD_LOG_CASE
}

// ------------------------------------------------------------------------------------------
// a4: gradient field, float4 (gx, gy, gz, 0) per voxel
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float grad_axis(const float* __restrict__ f, long long c, int i, int n, long long stride) {
    if (i == 0) return __fsub_rn(__ldg(f + c + stride), __ldg(f + c));
    if (i == n - 1) return __fsub_rn(__ldg(f + c), __ldg(f + c - stride));
    return __fmul_rn(__fsub_rn(__ldg(f + c + stride), __ldg(f + c - stride)), 0.5f);
}

// A thread owns one (y, z) column and marches over XS consecutive x planes (blockIdx.y = slab):
// the x neighbours travel through registers (prev / cur / next), so every voxel of the Gaussian
// grid is loaded once for the x and centre terms; the y neighbours are coalesced rows, the z
// neighbours come from L1.  One 32-bit divide per thread; the store is one 16-byte
// (gx, gy, gz, 0) per voxel, 512 contiguous bytes per warp.
constexpr int kGradSlab = 8;
__global__ void __launch_bounds__(256)
gradient_kernel(const float* __restrict__ f, int nx, int ny, int nz, float4* __restrict__ grad) {
    const unsigned plane = (unsigned)ny * (unsigned)nz;
    const unsigned p = blockIdx.x * 256u + threadIdx.x;
    if (p >= plane) return;
    const int y = (int)(p / (unsigned)nz);
    const int z = (int)(p - (unsigned)y * (unsigned)nz);
    const int x0 = blockIdx.y * kGradSlab;
    const int x1 = min(nx, x0 + kGradSlab);
    const long long sx = plane;
    long long c = (long long)x0 * sx + p;
    float prev = (x0 > 0) ? __ldg(f + c - sx) : 0.f;
    float cur = __ldg(f + c);
#pragma unroll 4
    for (int x = x0; x < x1; ++x, c += sx) {
        const float next = (x + 1 < nx) ? __ldg(f + c + sx) : 0.f;
        float4 v;
        if (x == 0) v.x = __fsub_rn(next, cur);
        else if (x == nx - 1) v.x = __fsub_rn(cur, prev);
        else v.x = __fmul_rn(__fsub_rn(next, prev), 0.5f);
        v.y = grad_axis(f, c, y, ny, nz);
        v.z = grad_axis(f, c, z, nz, 1);
        v.w = 0.f;
        grad[c] = v;
        prev = cur;
        cur = next;
    }
}

// Masked form: the orientation / description stages only ever read the gradient inside a box around each keypoint
// (+-2r voxels for the orientation patch, +-(2r-1) sqrt(3) for the rotated lattice; half of that in the base octave), so
// the field is computed on the 8 x 8 x 8 tiles those boxes touch and nowhere else.  flags[tile]: 0 = not needed,
// 1 = requested (computed by the next launch), 2 = computed.  The values written are the same as gradient_kernel's.
constexpr int kTile = 8;
static_assert(kTile == kGradSlab, "a gradient slab is one tile thick");

__global__ void __launch_bounds__(256)
gradient_masked_kernel(const float* __restrict__ f, int nx, int ny, int nz, float4* __restrict__ grad,
                       const uint8_t* __restrict__ flags, int ty, int tz) {
    const unsigned plane = (unsigned)ny * (unsigned)nz;
    const unsigned p = blockIdx.x * 256u + threadIdx.x;
    if (p >= plane) return;
    const int y = (int)(p / (unsigned)nz);
    const int z = (int)(p - (unsigned)y * (unsigned)nz);
    if (flags[((size_t)blockIdx.y * ty + (y >> 3)) * tz + (z >> 3)] != 1) return;
    const int x0 = blockIdx.y * kGradSlab;
    const int x1 = min(nx, x0 + kGradSlab);
    const long long sx = plane;
    long long c = (long long)x0 * sx + p;
    float prev = (x0 > 0) ? __ldg(f + c - sx) : 0.f;
    float cur = __ldg(f + c);
#pragma unroll 4
    for (int x = x0; x < x1; ++x, c += sx) {
        const float next = (x + 1 < nx) ? __ldg(f + c + sx) : 0.f;
        float4 v;
        if (x == 0) v.x = __fsub_rn(next, cur);
        else if (x == nx - 1) v.x = __fsub_rn(cur, prev);
        else v.x = __fmul_rn(__fsub_rn(next, prev), 0.5f);
        v.y = grad_axis(f, c, y, ny, nz);
        v.z = grad_axis(f, c, z, nz, 1);
        v.w = 0.f;
        grad[c] = v;
        prev = cur;
        cur = next;
    }
}

__global__ void gradient_flags_done_kernel(uint8_t* __restrict__ flags, size_t n) {
    const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (i < n && flags[i] == 1) flags[i] = 2;
}

// Requests every tile the box [vox - reach, vox + reach] of keypoint K touches (clipped to the grid); the CTA's threads
// share the tiles.
__device__ __forceinline__ void mark_box(const MadKeypoint& K, int nx, int ny, int nz, int reach, uint8_t* __restrict__ flags) {
    const int ty = (ny + kTile - 1) / kTile, tz = (nz + kTile - 1) / kTile;
    const int ax = max(K.vox[0] - reach, 0) / kTile, bx = min(K.vox[0] + reach, nx - 1) / kTile;
    const int ay = max(K.vox[1] - reach, 0) / kTile, by = min(K.vox[1] + reach, ny - 1) / kTile;
    const int az = max(K.vox[2] - reach, 0) / kTile, bz = min(K.vox[2] + reach, nz - 1) / kTile;
    const int wy = by - ay + 1, wz = bz - az + 1;
    const int total = (bx - ax + 1) * wy * wz;
    for (int t = threadIdx.x; t < total; t += blockDim.x) {
        const int k = t % wz, j = (t / wz) % wy, i = t / (wz * wy);
        uint8_t* fl = flags + ((size_t)(ax + i) * ty + (ay + j)) * tz + (az + k);
        if (*fl == 0) *fl = 1;                                    // benign race: every writer stores 1
    }
}

// One CTA per keypoint: requests every tile its box [vox - reach, vox + reach] touches (clipped to the grid).
__global__ void gradient_mark_kernel(const MadKeypoint* __restrict__ kp, int n_kp, int nx0, int ny0, int nz0, int nx1,
                                     int ny1, int nz1, int reach0, int reach1, uint8_t* __restrict__ flags0,
                                     uint8_t* __restrict__ flags1) {
    const MadKeypoint K = kp[blockIdx.x];
    const int o = K.oct ? 1 : 0;
    const int nx = o ? nx1 : nx0, ny = o ? ny1 : ny0, nz = o ? nz1 : nz0;
    const int reach = o ? reach1 : reach0;
    uint8_t* __restrict__ flags = o ? flags1 : flags0;
    mark_box(K, nx, ny, nz, reach, flags);
    (void)n_kp;
}

// mad_gradient_mark_many: gradient_mark_kernel's work for keypoint b of a batch (CTA b; none at or beyond kp_off[G]), in
// the tiles of its map g (dims [g][6], flags [g][2] device addresses).
__global__ void gradient_mark_many_kernel(const MadKeypoint* __restrict__ kp, const int* __restrict__ kp_off, int G,
                                          const int* __restrict__ dims, const uint64_t* __restrict__ flags_tab, int reach0,
                                          int reach1) {
    const int ki = blockIdx.x;
    if (ki >= kp_off[G]) return;
    const int g = mad_segment_of([&](int k) { return kp_off[k]; }, G, ki);
    const MadKeypoint K = kp[ki];
    const int o = K.oct ? 1 : 0;
    const int* d = dims + 6 * g + 3 * o;
    const int nx = d[0], ny = d[1], nz = d[2];
    const int reach = o ? reach1 : reach0;
    uint8_t* __restrict__ flags = reinterpret_cast<uint8_t*>(flags_tab[2 * g + o]);
    mark_box(K, nx, ny, nz, reach, flags);
}

extern "C" int mad_gradient_mark_many(const MadKeypoint* kp, const int* kp_off, int n_rows, int G, const int* dims,
                                      const uint64_t* flags, int reach_oct0, int reach_oct1, void* stream) {
    MAD_CHECK_ARG(kp_off && dims && flags && G >= 1 && n_rows >= 0 && reach_oct0 >= 0 && reach_oct1 >= 0);
    if (n_rows == 0) return MAD_OK;
    MAD_CHECK_ARG(kp);
    MAD_PROF("gradient_mark_many_kernel", stream);
    gradient_mark_many_kernel<<<n_rows, 128, 0, (cudaStream_t)stream>>>(kp, kp_off, G, dims, flags, reach_oct0, reach_oct1);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" int mad_gradient(const float* gauss, int nx, int ny, int nz, float* grad4, void* stream) {
    MAD_CHECK_ARG(gauss && grad4 && nx >= 2 && ny >= 2 && nz >= 2);
    MAD_CHECK_ARG((reinterpret_cast<uintptr_t>(grad4) & 15) == 0);
    MAD_CHECK_ARG(nx <= 65535 && (long long)ny * nz < (1LL << 31));
    dim3 grid_dim((unsigned)mad_ceil_div((long long)ny * nz, 256), (unsigned)mad_ceil_div(nx, kGradSlab));
    MAD_PROF("gradient_kernel", stream);
    gradient_kernel<<<grid_dim, 256, 0, (cudaStream_t)stream>>>(gauss, nx, ny, nz, reinterpret_cast<float4*>(grad4));
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" size_t mad_gradient_tiles(int nx, int ny, int nz) {
    return (size_t)mad_ceil_div(nx, kTile) * (size_t)mad_ceil_div(ny, kTile) * (size_t)mad_ceil_div(nz, kTile);
}

extern "C" int mad_gradient_mark(const MadKeypoint* kp, int n_kp, const int* dims_oct_host, int reach_oct0, int reach_oct1,
                                 uint8_t* flags_oct0, uint8_t* flags_oct1, void* stream) {
    MAD_CHECK_ARG(dims_oct_host && n_kp >= 0 && reach_oct0 >= 0 && reach_oct1 >= 0);
    if (n_kp == 0) return MAD_OK;
    MAD_CHECK_ARG(kp && flags_oct0 && flags_oct1);
    const int* d = dims_oct_host;
    MAD_PROF("gradient_mark_kernel", stream);
    gradient_mark_kernel<<<n_kp, 128, 0, (cudaStream_t)stream>>>(kp, n_kp, d[0], d[1], d[2], d[3], d[4], d[5], reach_oct0,
                                                               reach_oct1, flags_oct0, flags_oct1);
    MAD_LAUNCH_OK();
    return MAD_OK;
}

extern "C" int mad_gradient_masked(const float* gauss, int nx, int ny, int nz, float* grad4, uint8_t* flags, void* stream) {
    MAD_CHECK_ARG(gauss && grad4 && flags && nx >= 2 && ny >= 2 && nz >= 2);
    MAD_CHECK_ARG((reinterpret_cast<uintptr_t>(grad4) & 15) == 0);
    MAD_CHECK_ARG(nx <= 65535 * kTile && (long long)ny * nz < (1LL << 31));
    const int ty = (int)mad_ceil_div(ny, kTile), tz = (int)mad_ceil_div(nz, kTile);
    dim3 grid_dim((unsigned)mad_ceil_div((long long)ny * nz, 256), (unsigned)mad_ceil_div(nx, kGradSlab));
    {
        MAD_PROF("gradient_masked_kernel", stream);
        gradient_masked_kernel<<<grid_dim, 256, 0, (cudaStream_t)stream>>>(gauss, nx, ny, nz, reinterpret_cast<float4*>(grad4),
                                                                         flags, ty, tz);
        MAD_LAUNCH_OK();
    }
    const size_t n = mad_gradient_tiles(nx, ny, nz);
    MAD_PROF("gradient_flags_done_kernel", stream);
    gradient_flags_done_kernel<<<(unsigned)mad_ceil_div((long long)n, 256), 256, 0, (cudaStream_t)stream>>>(flags, n);
    MAD_LAUNCH_OK();
    return MAD_OK;
}
