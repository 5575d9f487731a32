/*
 * mad_b200.h -- C ABI of libmad_b200.so: the B200 (sm_100a) implementation of MaD's
 * local-feature hot path (scale-space -> detect -> orient -> describe -> match).
 *
 * This is the drop-in boundary (DESIGN.md section 2).  The reference (LBM-EPFL/MaD) is pure Python
 * with no FFI of its own; every entry point below replaces one NumPy/SciPy/scikit-image call
 * site of the reference (cited per function, paths relative to the reference tree), and is
 * what a ctypes stub in the reference's classes would bind (INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _host;
 *   - grids are C-contiguous float32 [x][y][z] (z fastest), as in the reference;
 *   - gradient fields are float4 per voxel (gx, gy, gz, 0), 16-byte aligned;
 *   - `stream` is a cudaStream_t passed as void* (0 = default stream); calls are asynchronous
 *     on that stream unless stated; no hidden allocation: work space is supplied by the caller
 *     (sizes from the *_workspace_bytes helpers);
 *   - return value: 0 = MAD_OK, negative = error (mad_last_error_string() for text).
 */
#ifndef MAD_B200_H
#define MAD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MAD_OK 0
#define MAD_ERR_ARG (-1)      /* bad argument (null pointer, size out of range)              */
#define MAD_ERR_CUDA (-2)     /* a CUDA runtime call or kernel launch failed                  */
#define MAD_ERR_CAPACITY (-3) /* an output list did not fit the caller's buffer               */
#define MAD_ERR_NODEVICE (-4) /* no sm_100 device / wrong architecture for a tcgen05 kernel   */

#define MAD_MAX_ORI 36        /* <= 6 main x 6 secondary orientations per keypoint            */
#define MAD_DSC_LEN 1024      /* 64 sub-blocks x 16 zones                                      */
#define MAD_DSC_REFUSED (1 << 30) /* max_entry of a set that is not a descriptor set (see mad_dsc_prepare) */

/* One detected keypoint (mad/Detector.py:30-45, mad/DensityFeature.py:35-41). */
typedef struct MadKeypoint {
    int32_t vox[3];   /* integer voxel after Newton moves  (DensityFeature.coords)           */
    int32_t oct;      /* 0 = 2x-upsampled octave, 1 = base octave                            */
    float off[3];     /* sub-voxel offset (float32 arithmetic, as NumPy 2 does it)           */
    float val;        /* LoG value at the ORIGINAL peak voxel (mad/Detector.py:35)            */
    int32_t peak[3];  /* original 3x3x3-maximum voxel                                         */
    int32_t accepted; /* 1 = passed check_localize                                            */
} MadKeypoint;

/* One oriented feature = (row in the keypoint table, main zone, secondary zone).
 * Rfinal depends only on (main, sec): see mad_orient_tables. */
typedef struct MadOriented {
    int32_t kp;
    int16_t main_bin;
    int16_t sec_bin;
} MadOriented;

/* EQSP zone table on the device: bounds[zone] = (theta_min, phi_min, theta_max, phi_max) as
 * float64 exactly as parsed from the reference's 4-decimal tables (mad/eqsp/sphere_*.txt). */
typedef struct MadZoneTable {
    int32_t n_zones;          /* 112 or 16                                                    */
    int32_t n_belts;
    const double* bounds;     /* [n_zones][4]                                                 */
    const int32_t* belt_first;/* [n_belts+1] first zone index of each belt                    */
    const double* belt_phi;   /* [n_belts+1] phi bounds of the belts                          */
    const void* fast;         /* device image built once by mad_zone_fast_build (MAD_ZONE_FAST_BYTES), or
                               * NULL: every CTA then derives it from the table itself                */
} MadZoneTable;

/* Builds the float32 fast-classification image of a zone table (guard-banded bounds, see csrc/eqsp_zones.cuh)
 * into fast_out (device, MAD_ZONE_FAST_BYTES); store the pointer in MadZoneTable.fast. */
#define MAD_ZONE_FAST_BYTES 2048
int mad_zone_fast_build(const MadZoneTable* zones_host, void* fast_out, void* stream);

const char* mad_last_error_string(void);
int mad_version(void);
/* Fills (sm_count, cc_major, cc_minor) of the current device. */
int mad_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* Copies `bytes` (a multiple of 4, <= 4096) from device memory to PINNED host memory by a kernel writing over PCIe,
 * not by a copy engine: a small count does not queue behind a large transfer in flight.  dst_host_mapped: the
 * device-visible address of the pinned buffer (equal to the host address under unified addressing).  The host reads
 * the buffer after synchronising the stream or an event recorded behind this call. */
int mad_publish_small(const void* src_dev, void* dst_host_mapped, int bytes, void* stream);

/* Copies `bytes` from device memory to PINNED, device-mapped host memory with n_ctas CTAs storing over PCIe (no copy
 * engine involved, so nothing else queues behind a large download).  Both addresses 16-byte aligned.  The host reads the
 * buffer after synchronising the stream or an event recorded behind this call. */
int mad_copy_to_host(const void* src_dev, void* dst_host_mapped, long long bytes, int n_ctas, void* stream);

/* ---- launch accounting and per-kernel timing (no reference counterpart; measurement only) ---- */
/* Number of kernels this library has launched in this process (CUB-internal kernels count as one
 * per CUB call). */
long long mad_launch_count(void);
/* While enabled, every kernel launch is bracketed by two CUDA events on its stream.  Records
 * accumulate until mad_profile_reset(); mad_profile_get(i) synchronises on record i and returns
 * the kernel's name (static string) and its duration in milliseconds. */
int mad_profile_enable(int on);
int mad_profile_count(void);
int mad_profile_get(int i, const char** name, float* ms);
int mad_profile_reset(void);

/* ---- a0: Dmap container operations on the device-resident grid (mad/Dmap.py:49-97) ------------ */
/* Maximum of the grid.  *out_max_ord (device, 4 bytes) receives an order-preserving integer image
 * of the float maximum; mad_grid_max_decode (host) turns the value read back into the float. */
int mad_grid_max(const float* grid, long long n, float* out_max_ord, void* stream);
float mad_grid_max_decode(unsigned int ord);
/* In place: v < isovalue -> 0 (mad/Dmap.py:50-54), then, if divide, v / vmax as a correctly rounded
 * float32 division (mad/Dmap.py:66-67). */
int mad_threshold_normalise(float* grid, long long n, float isovalue, float vmax, int divide, void* stream);
/* bbox6 (device int[6]) = min x, y, z and max x, y, z of the non-zero voxels (mad/Dmap.py:77-80);
 * max < 0 when the grid is all zero. */
int mad_grid_bbox(const float* grid, int nx, int ny, int nz, int* bbox6, void* stream);
/* out = np.pad(in[x0:x0+cx, y0:y0+cy, z0:z0+cz], pad)  (mad/Dmap.py:86-97). */
int mad_crop_pad3d(const float* in, int nx, int ny, int nz, int x0, int y0, int z0, int cx, int cy, int cz,
                   int pad, float* out, void* stream);

/* ---- a1: zero padding (np.pad, mad/MapSpace.py:117-118) ---------------------------------- */
int mad_pad3d(const float* in, int nx, int ny, int nz, int pad, float* out, void* stream);

/* ---- a2: 2x not-a-knot cubic spline upsampling + Gaussian presmoothing ------------------- */
/* (scipy.interpolate.interp1d(kind='cubic') x3 axes, mad/MapSpace.py:137-146,191-214, then
 *  scipy.ndimage.gaussian_filter(sigma=sig_presmooth), float64 throughout, float32 result).
 *  base: [bx][by][bz] f32;  up: [2bx-1][2by-1][2bz-1] f32.  gauss_w_host: the (2*radius+1)
 *  float64 weights of the presmoothing kernel, centre at [radius]; radius 0 = no smoothing.
 *  Needs every b* >= 5. */
size_t mad_upsample_workspace_bytes(int bx, int by, int bz);
int mad_upsample_presmooth(const float* base, int bx, int by, int bz,
                           const double* gauss_w_host, int radius,
                           float* up, void* workspace, size_t workspace_bytes, void* stream);

/* ---- a3/a4: LoG response, Gaussian-smoothed grid -------------------------------------------- */
/* map_space = max(0, -sigma^2 * gaussian_laplace(grid, sigma)), gauss = gaussian_filter(grid,
 * sigma)  (mad/MapSpace.py:170-173,182), with SciPy's pass structure: 1-D correlations along
 * x, y, z with `reflect` boundaries, accumulated per output in float64 (exact_f64 = 1) or in
 * float32 (exact_f64 = 0) and stored as float32 between passes, the three second-derivative
 * terms summed in float32 as ((x-term + y-term) + z-term).  w0 / w2: the (2*radius+1) float64
 * weights of the order-0 / order-2 kernels (host pointers), radius <= 16. */
size_t mad_log_gauss_workspace_bytes(int nx, int ny, int nz);
int mad_log_gauss(const float* grid, int nx, int ny, int nz,
                  const double* w0_host, const double* w2_host, int radius, float scale,
                  float* log_out, float* gauss_out, void* workspace, size_t workspace_bytes,
                  int exact_f64, void* stream);

/* ---- a4: gradient field (np.gradient, mad/MapSpace.py:187) ---------------------------------- */
/* grad4[x][y][z] = (d/dx, d/dy, d/dz, 0): central differences, one-sided at the two ends. */
int mad_gradient(const float* gauss, int nx, int ny, int nz, float* grad4, void* stream);
/* Masked form of the same field.  Orientator / Descriptor read grad_list only inside a box around each keypoint
 * (mad/Orientator.py:129-155: +-2r up-octave voxels, +-r base; mad/Descriptor.py:123-149: the rotated lattice,
 * +-(2r - 1) sqrt(3) and +-(r - 0.5) sqrt(3)), so the field is computed on the 8x8x8 tiles those boxes touch.
 * flags[mad_gradient_tiles(nx, ny, nz)] (device, zero-initialised by the caller): 0 = not needed, 1 = requested,
 * 2 = computed.  mad_gradient_mark requests the tiles within reach_oct{0,1} voxels of every keypoint's (moved) voxel in
 * its octave; mad_gradient_masked computes the requested tiles (values identical to mad_gradient) and marks them 2.
 * Tiles never requested keep whatever grad4 held.  mad_gradient_mark(all tiles) == mad_gradient. */
size_t mad_gradient_tiles(int nx, int ny, int nz);
int mad_gradient_mark(const MadKeypoint* kp, int n_kp, const int* dims_oct_host, int reach_oct0, int reach_oct1,
                      uint8_t* flags_oct0, uint8_t* flags_oct1, void* stream);
int mad_gradient_masked(const float* gauss, int nx, int ny, int nz, float* grad4, uint8_t* flags, void* stream);

/* ---- a5/a6: keypoint detection + sub-voxel refinement --------------------------------------- */
/* peak_local_max(grid, exclude_border=border, threshold_abs=threshold) + check_localize
 * (mad/Detector.py:26-45,53-123).  Appends one MadKeypoint per 3x3x3 maximum (accepted or
 * not) to cand[0..cap) at *count (device counter, not reset by this call).  Unordered. */
int mad_detect(const float* log_grid, int nx, int ny, int nz, int oct, int border,
               float threshold, MadKeypoint* cand, int cap, int* count, void* stream);

/* Orders candidates canonically (octave asc, value desc, raster index of the peak asc) and
 * keeps the accepted ones: out[0..*out_count).  n = number of candidates (host value).
 * dims_oct = {nx0,ny0,nz0,nx1,ny1,nz1} (host pointer) for the raster index. */
size_t mad_sort_keypoints_workspace_bytes(int n);
int mad_sort_keypoints(const MadKeypoint* cand, int n, const int* dims_oct_host,
                       MadKeypoint* out, int* out_count,
                       void* workspace, size_t workspace_bytes, void* stream);

/* ---- a7-a10: dominant orientations ----------------------------------------------------------- */
/* Orientator.assign_orientations (mad/Orientator.py:68-110 and helpers).  For keypoint i writes
 * n_ori[i] (0..36) and slots[i*36 + j] = main | (sec << 16) in emission order (main asc, sec asc).
 * grad4_oct0 / grad4_oct1 with dims as in mad_sort_keypoints; r = ori_radius//2 (8 for patch 16).
 * r1_table: float64 [n_zones][9], row-major rotation taking zone centre -> +z (identity for 0). */
int mad_orient(const float* grad4_oct0, const float* grad4_oct1, const int* dims_oct_host,
               const MadKeypoint* kp, int n_kp, int r, const MadZoneTable* zones112_host,
               const double* r1_table, int lim_main, int lim_sec,
               int32_t* n_ori, int32_t* slots, void* stream);

/* Exclusive scan of n_ori + scatter: oriented[0..*out_count) in emission order. */
size_t mad_compact_oriented_workspace_bytes(int n_kp);
int mad_compact_oriented(const int32_t* n_ori, const int32_t* slots, int n_kp,
                         MadOriented* oriented, int cap, int* out_count,
                         void* workspace, size_t workspace_bytes, void* stream);

/* ---- a11/a12: descriptors ---------------------------------------------------------------------- */
/* Descriptor.step06_distribute_subeqsp (mad/Descriptor.py:123-202).  dsc[i][1024] int16.
 * rf_table / rf_inv_table: float64 [rf_zones*rf_zones][9] indexed by main*rf_zones+sec: Rfinal and
 * inv(Rfinal) (rf_zones = 112).  r = dsc_radius//2 (8 for patch 16); lattice has 2r points per axis. */
int mad_describe(const float* grad4_oct0, const float* grad4_oct1, const int* dims_oct_host,
                 const MadKeypoint* kp, const MadOriented* oriented, int n_oriented, int r,
                 const MadZoneTable* zones16_host, const double* rf_table, const double* rf_inv_table,
                 int rf_zones, int16_t* dsc, void* stream);

/* ---- a15: descriptor matching (mad/MaD.py:416-424) ---------------------------------------------- */
/* A descriptor set prepared for matching (device pointers; the struct itself lives on the host).
 * norm2: exact integer squared L2 norms.  u8: uint8 copy [rows_padded][1024] (zero rows beyond
 * `rows`, rows_padded a multiple of 128; a multiple of 256 enables the CTA-pair kernel) -- the operand of the
 * tcgen05 kind::i8 kernel, exact while
 * max_entry <= 255 (true for every patch size <= 24: an entry counts the votes of one sub-block).
 * rnorm: float 1/sqrt(norm2) per padded row (0 for zero rows), the fp32 pre-filter's scale.
 * half: optional fp16 copy for the general tensor-core kernel (impl = 2).  That kernel accumulates in fp32, which is
 * exact while every partial sum of a dot product stays <= 2^24: it accepts a pair of sets only if every entry lies in
 * [0, 2048] (exact in fp16) and max_norm2(hi) * max_norm2(lo) <= 2^48 (by Cauchy-Schwarz every dot product, and so
 * every partial sum of non-negative terms, is then <= 2^24).  The SIMT kernel (impl = 1) is exact in int32 for any
 * set whose squared norms fit int32.
 * dsc is only read by the SIMT check kernel (impl = 1).
 * A set with a negative entry or a squared norm >= 2^31 is not a descriptor set: mad_dsc_prepare reports it with
 * max_entry = MAD_DSC_REFUSED, and every matching entry point refuses it (MAD_ERR_ARG). */
typedef struct MadDscSet {
    const int16_t* dsc;   /* [rows][1024] */
    const void* half;     /* [rows_padded][1024] fp16, or NULL */
    const int32_t* norm2; /* [rows] */
    const uint8_t* u8;    /* [rows_padded][1024], or NULL */
    const float* rnorm;   /* [rows_padded], or NULL */
    int32_t rows;
    int32_t rows_padded;
    int32_t max_entry;    /* largest descriptor entry (host copy of what mad_dsc_prepare found; -1 = not known) */
    int32_t max_norm2;    /* largest squared norm (host copy of what mad_dsc_prepare found; -1 = not known) */
} MadDscSet;

/* Fills norm2[rows], rnorm[rows_padded], u8[rows_padded][1024] (may be NULL) and atomically
 * raises *max_entry (device int32, caller zeroes it) to the largest entry seen -- MAD_DSC_REFUSED if an entry is
 * negative or a squared norm is >= 2^31 -- and *max_norm2 (device int32, caller zeroes it; may be NULL) to the
 * largest squared norm. */
int mad_dsc_prepare(const int16_t* dsc, int rows, int rows_padded, int32_t* norm2, float* rnorm,
                    uint8_t* u8, int32_t* max_entry, int32_t* max_norm2, void* stream);
int mad_dsc_norms(const int16_t* dsc, int rows, int32_t* norm2, void* stream);
int mad_dsc_to_half(const int16_t* dsc, int rows, int rows_padded, void* half_out, void* stream);

/* Threshold mode (the parity contract): all (i, j) with  dot(hi_i, lo_j) / sqrt(n_i n_j) > cc in
 * float64 (integer dot and norms exact); zero rows score 0.
 * The lo axis is cut into n_seg = mad_match_segments(M, N, impl) contiguous segments (so that a
 * few hi tiles still fill 148 SMs).  Two passes: COUNT fills seg_count[M][n_seg]; after an
 * exclusive scan over that array in memory order (mad_exclusive_scan_i32_to_i64, n = M*n_seg)
 * FILL writes pair_hi / pair_lo / pair_score starting at seg_offset[i][s], lo ascending -- i.e. the
 * row-major order of np.where(preds > cc) (mad/MaD.py:423-424).
 * impl: 1 = SIMT integer kernel (device-side check), 2 = fp16 tcgen05 kernel (only where it is exact: see MadDscSet).
 * The product path for threshold matching is the ONE-pass mad_match_pairs below; impl 0 (that kernel) has no
 * count / fill form and is REJECTED here with MAD_ERR_ARG and a message (never silently remapped).
 * mad_match_segments(M, N, 0) only sizes the top-k workspace of the uint8 kernel. */
int mad_match_segments(int M, int N, int impl);
int mad_match_count(const MadDscSet* hi, const MadDscSet* lo, double cc, int n_seg, int32_t* seg_count, int impl,
                    void* stream);
int mad_match_fill(const MadDscSet* hi, const MadDscSet* lo, double cc, int n_seg, const int64_t* seg_offset,
                   int32_t* pair_hi, int32_t* pair_lo, double* pair_score, int impl, void* stream);
size_t mad_exclusive_scan_workspace_bytes(int n);
int mad_exclusive_scan_i32_to_i64(const int32_t* in, int n, int64_t* out, int64_t* total,
                                  void* workspace, size_t workspace_bytes, void* stream);

/* One-pass threshold matching on the uint8 tcgen05 kernel (the product path): every pair with
 * cosine > cc is appended, unordered, to cand_key[] (an opaque sort key) and cand_dot[] = exact integer
 * dot product; *count (device, reset by the call) receives the number of pairs FOUND, which may
 * exceed cap -- then only cap were stored and the caller repeats with a larger buffer; a value >= 2^62 reports an
 * internal time-out of the kernel (the list is incomplete and must be discarded).
 * (cand_key holds hi * lo_rows + lo, the row-major rank of the pair.)
 * mad_match_pairs_finish sorts the n stored candidates by (hi, lo) -- the row-major order of
 * np.where(preds > cc), mad/MaD.py:423-424 -- and evaluates the float64 scores. */
int mad_match_pairs(const MadDscSet* hi, const MadDscSet* lo, double cc, uint64_t* cand_key, int32_t* cand_dot,
                    uint64_t cap, uint64_t* count, void* stream);
size_t mad_match_pairs_finish_workspace_bytes(long long n);
int mad_match_pairs_finish(const uint64_t* cand_key, const int32_t* cand_dot, long long n, int hi_rows, int lo_rows,
                           const int32_t* hi_n2, const int32_t* lo_n2, int32_t* pair_hi, int32_t* pair_lo,
                           double* pair_score, void* workspace, size_t workspace_bytes, void* stream);
/* Compact form for the trip to the host: pair_dot = the exact integer dot product instead of the float64 score (12 bytes
 * per pair instead of 16); score = dot / sqrt(|hi|^2 |lo|^2) is recomputed from the norms with the same correctly rounded
 * float64 operations (mad_b200.pipeline.scores_from_dots), i.e. bit-identical to mad_match_pairs_finish's. */
int mad_match_pairs_finish_dot(const uint64_t* cand_key, const int32_t* cand_dot, long long n, int hi_rows, int lo_rows,
                               int32_t* pair_hi, int32_t* pair_lo, int32_t* pair_dot, void* workspace, size_t workspace_bytes,
                               void* stream);

/* Top-k mode (extension, SURVEY.md 8c): per hi row the k best lo rows by (score desc, index asc), where the score is
 * the float64 cosine of the threshold mode (bit for bit) and equal scores go to the lower index; lo_index_base is added
 * to the stored indices (sharded reference axis).  k <= 32.
 * topk_idx[M][k] (-1 padded), topk_score[M][k] float64 (-inf padded); a row whose indices are all -2
 * (MAD_TOPK_INCOMPLETE: an internal hand-off of the kernel timed out) means the list is incomplete -- discard the call's
 * result.  Workspace: per-segment partial lists (mad_match_topk_workspace_bytes).  impl: 0 = uint8 tcgen05 kernel
 * (product; needs max_entry <= 255), 1 = SIMT check kernel, 2 = fp16 tcgen05 kernel (see MadDscSet). */
size_t mad_match_topk_workspace_bytes(int M, int N, int k, int impl);
int mad_match_topk(const MadDscSet* hi, const MadDscSet* lo, int k, int lo_index_base,
                   int32_t* topk_idx, double* topk_score, void* workspace, size_t workspace_bytes,
                   int impl, void* stream);
/* Merges G per-shard top-k lists [G][M][k] into one [M][k] with the same ordering rule (-1 entries are padding); a row
 * with a -2 entry in any input list comes out as all -2 (list incomplete, discard the call's result). */
#define MAD_TOPK_INCOMPLETE (-2)
int mad_topk_merge(const int32_t* idx_in, const double* score_in, int G, int M, int k,
                   int32_t* idx_out, double* score_out, void* stream);

/* ---- next component (SURVEY.md 8f rank 1): per-pair repeatability, mad/MaD.py:426-453 ------------------ */
/* used[idx[i]] = 1 for every i (which features occur in the pair list). */
int mad_mark_used(const int32_t* idx, long long n, uint8_t* used, void* stream);
/* For pair p = (hi, lo): R = inv(Rfinal_lo) . Rfinal_hi; the hi cloud (unique sub-voxel coordinates of the
 * matched hi anchors, [n_hi_cloud][3]) is moved by q = (c - subv_hi) . R^T + subv_lo and
 * repeatability = 100 * #{q with a lo-cloud point closer than dist} / n_hi_cloud.
 * results[p][23] = score, repeatability, lo (index, oct, main), hi (index, oct, main), subv_hi[3], subv_lo[3], R[9]
 * -- the row layout of the reference (mad/MaD.py:451).  *_meta: int32 [D][4] = index, oct_scale, main_bin, sec_bin.
 * The lo cloud comes cell-sorted for a uniform grid of cell size dist: lo_sorted [L][3], cell_start [ncell + 1],
 * near_bits = bitmap of cells whose 27-cell neighbourhood is non-empty; grid_org_host / grid_dims_host (host). */
int mad_repeatability(const int32_t* pair_hi, const int32_t* pair_lo, const double* pair_score, long long n_pairs,
                      const double* hi_subv, const double* lo_subv, const int32_t* hi_meta, const int32_t* lo_meta,
                      const double* rf_table, const double* rf_inv_table, int rf_zones,
                      const double* hi_cloud, int n_hi_cloud, const double* lo_sorted, const int32_t* cell_start,
                      const uint32_t* near_bits, const double* grid_org_host, const int* grid_dims_host,
                      double dist, double* results, void* stream);
/* mad_repeatability in two parts, so that the pairs can be shared out (mad_b200.parallel.match_dsc_sharded):
 * mad_repeat_counts writes counts[p - p0] = #{q with a lo-cloud point closer than dist} for the pairs p in [p0, p1)
 * (mad/MaD.py:430-448, the cKDTree query per pair); mad_repeat_rows writes results[p][23] for all n_pairs pairs from
 * those counts with mad_repeatability's formulas (mad/MaD.py:449-451: repeatability = 100 * count / n_hi_cloud).
 * The arguments mean what they mean for mad_repeatability; counts + rows == mad_repeatability, bit for bit. */
int mad_repeat_counts(const int32_t* pair_hi, const int32_t* pair_lo, long long p0, long long p1,
                      const double* hi_subv, const double* lo_subv, const int32_t* hi_meta, const int32_t* lo_meta,
                      const double* rf_table, const double* rf_inv_table, int rf_zones,
                      const double* hi_cloud, int n_hi_cloud, const double* lo_sorted, const int32_t* cell_start,
                      const uint32_t* near_bits, const double* grid_org_host, const int* grid_dims_host,
                      double dist, int32_t* counts, void* stream);
int mad_repeat_rows(const int32_t* pair_hi, const int32_t* pair_lo, const double* pair_score, long long n_pairs,
                    const double* hi_subv, const double* lo_subv, const int32_t* hi_meta, const int32_t* lo_meta,
                    const double* rf_table, const double* rf_inv_table, int rf_zones, const int32_t* counts,
                    int n_hi_cloud, double* results, void* stream);

/* The anchor clouds and the lo grid of the repeatability loop, on the device (mad/MaD.py:427-428 and the grid above).
 * mad_anchor_cloud: cloud[0..n) = np.unique(subv[used], axis=0) -- the distinct rows of subv [n_rows][3] whose used flag
 * is set, in lexicographic (x, y, z) order, bit for bit (-0.0 is taken as +0.0, as NumPy compares them equal);
 * cloud has room for n_rows rows.  info (device int64[8], written by the call): [0] n, [1] number of used rows with a
 * non-finite coordinate (the caller must refuse the set: the cloud is then meaningless), [2..4] grid dims =
 * floor((max - org) / cell) + 2 (clamped to 2^40), [5..7] the bits of grid_org (device double[3]) = min - cell, all in
 * float64 as NumPy evaluates them.  Read info back once and pass dims / org to the calls below.
 * mad_cloud_grid: for the cloud of n rows (n >= 1), sorted [n][3] = the cloud stably sorted by cell id
 * (np.argsort(kind="stable")), cell_start [ncell + 1] = points in lower cells, near_bits [ceil(ncell / 32)] = cells whose
 * 27-cell neighbourhood (clipped to the grid) holds a point.  ncell = dims0 dims1 dims2 must be < 2^31 (MAD_ERR_ARG
 * otherwise: the repeatability kernel indexes cells in int32). */
size_t mad_anchor_cloud_workspace_bytes(int n_rows);
int mad_anchor_cloud(const double* subv, const uint8_t* used, int n_rows, double cell, double* cloud, double* grid_org,
                     long long* info, void* workspace, size_t workspace_bytes, void* stream);
size_t mad_cloud_grid_workspace_bytes(int n);
int mad_cloud_grid(const double* cloud, int n, const double* grid_org, const long long* grid_dims_host, double cell,
                   double* sorted, int32_t* cell_start, uint32_t* near_bits, void* workspace, size_t workspace_bytes,
                   void* stream);

/* ---- next component (SURVEY.md 8f rank 2): atoms -> density, mad/PDB.py:131-163,215-292 -------------------- */
/* Mass-weighted trilinear splat of n_atoms points (xyz [n][3], mass [n], float64) into grid [px][py][pz] float64
 * (zeroed by the call); min_host = lattice-registered minimum corner, margin = 2 + pad (mad/PDB.py:246-285). */
int mad_density_splat(const double* xyz, const double* mass, int n_atoms, const double* min_host, double voxelsp,
                      int margin, int px, int py, int pz, double* grid, void* stream);
/* grid /= max(grid) in float64 (mad/PDB.py:287); the grid must be non-negative; scratch8 = 8 device bytes. */
int mad_normalise_f64(double* grid, long long n, void* scratch8, void* stream);
/* "full" 1-D convolution with zero extension along the middle axis of in [outer][n][inner] float64 ->
 * out [outer][n + 2 radius][inner] (float64, or float32 if out_is_f32); w_dev: 2 radius + 1 device weights. */
int mad_conv_full_f64(const double* in, long long outer, int n, long long inner, const double* w_dev, int radius,
                      void* out, int out_is_f32, void* stream);

/* ---- next component (SURVEY.md 8f rank 4): scoring reductions and rigid refinement on HBM-resident grids -------- */
/* One pass over the common box of two float32 grids [x][y][z]: box_host[9] = (x1, y1, z1, x2, y2, z2, ex, ey, ez), the box
 * start in each grid and its extent (the bounds of mad/Dmap.py:172-246).  out8 (device float64): [0] sum a b, [1] sum a a,
 * [2] sum b b, [3] sum a a where b > 0, [4] sum b b where a > 0, [5] #(a > isovalue and b > isovalue), [6] #(a > 0 and
 * b > 0), [7] 0 -- everything Dmap.get_CCC_with_grid (mad/Dmap.py:248-258), Dmap.get_CCC_with_dmap (:351-372) and
 * structure_utils.get_overlap (mad/structure_utils.py:254-259) evaluate.  An empty box gives zeros. */
size_t mad_box_scores_workspace_bytes(int ex, int ey, int ez);
int mad_box_scores(const float* g1, int nx1, int ny1, int nz1, const float* g2, int nx2, int ny2, int nz2,
                   const int* box_host, float isovalue, double* out8, void* workspace, size_t workspace_bytes,
                   void* stream);
/* *out (device, reset by the call) = #{grid > thr}: np.count_nonzero(grid > isovalue), mad/Dmap.py:354. */
int mad_grid_count_gt(const float* grid, long long n, float thr, unsigned long long* out, void* stream);
/* Dmap.mask_with (mad/Dmap.py:99-151): g1 is zeroed outside [lo, hi) on any axis and wherever
 * g2[x - shift] < 1e-8; shift / lo / hi are the host integers of :115-136. */
int mad_mask_with(float* g1, int nx1, int ny1, int nz1, const float* g2, int nx2, int ny2, int nz2,
                  const int* shift_host, const int* lo_host, const int* hi_host, void* stream);
/* structure_utils.refine_pdb (mad/structure_utils.py:58-161) for n_problems poses of n_atoms atoms each, one CTA per
 * pose: init [P][n][3] float64 start coordinates, center [P][3] = their mean, max_dist [P] = largest distance from it;
 * grad4 = mad_gradient of the map (np.gradient, float4 per voxel), px / py / pz = device float64 axis coordinates
 * (np.arange(o, voxsp n + o, voxsp)[:n]).  Even steps translate along the summed gradient at the atoms (trilinear, as
 * scipy's RegularGridInterpolator evaluates it), odd steps rotate about the summed torque so that the farthest atom moves
 * step_size; every 4 steps the step is halved when no atom moved further than it; stops when it drops below min_step.
 * coords_out [P][n][3] = final coordinates, meta_out [P][4] = (converged, last step index, NaN flag, final step size). */
int mad_refine_rigid(const float* grad4, int nx, int ny, int nz, const double* px, const double* py, const double* pz,
                     double voxsp, const double* init, const double* center, const double* max_dist, int n_problems,
                     int n_atoms, int n_steps, double max_step, double min_step, double* coords_out, double* meta_out,
                     void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MAD_B200_H */
