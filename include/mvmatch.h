/*
 * mvmatch.h -- C ABI of libmvmatch.so: the B200 (sm_100a) dense-correspondence matching path.
 *
 * This is the drop-in boundary for the matching step of midvision-probe
 * (reference: evals/utils/correspondence.py, evaluate_spair_correspondence.py:59-103).
 * The reference has no FFI of its own on this path -- it calls torch CPU ops and
 * faiss-gpu (correspondence.py:14-23) -- so the entry points below are what a ctypes
 * binding of that path binds: plain pointers, sizes and a CUDA stream handle.
 * No torch types cross this boundary.  INTEGRATION.md shows the reference-side stub.
 *
 * Conventions
 *   - every function returns 0 on success; <0 = argument error (MV_E_*), >0 = cudaError_t.
 *     mv_last_error() returns a thread-local description of the last non-zero return.
 *   - all pointers are DEVICE pointers unless the parameter is documented "host".
 *   - all launches go to `stream`; nothing synchronises the host.
 *   - feature rows are row-major (n, C); feature maps are channel-last (h*w, C).
 *   - "n_dev" parameters are optional device-resident int32 counts (produced by
 *     mv_compact_valid) so a whole pair can be queued without a host round trip;
 *     when NULL the host-side maximum is the live count.
 */
#ifndef MVMATCH_H_
#define MVMATCH_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* mv_stream_t; /* cudaStream_t */

/* ---- error codes -------------------------------------------------------------------- */
#define MV_OK 0
#define MV_E_ARG (-1)       /* bad argument (null pointer, non-positive size, bad enum)   */
#define MV_E_ALIGN (-2)     /* pointer / leading dimension alignment requirement violated  */
#define MV_E_RANGE (-3)     /* size outside the supported range                           */
#define MV_E_WORKSPACE (-4) /* workspace too small                                        */
#define MV_E_ARCH (-5)      /* device is not sm_100                                       */
#define MV_E_DRIVER (-6)    /* driver entry point (cuTensorMapEncodeTiled) unavailable     */

/* ---- enums -------------------------------------------------------------------------- */
/* sampling modes of kernel 1 */
#define MV_SAMPLE_BILINEAR_ZEROS 0 /* F.grid_sample(mode=bilinear, padding_mode=zeros): correspondence.py:173, spair:76-78 */
#define MV_SAMPLE_BICUBIC_CLAMP 1  /* F.interpolate(mode=bicubic, align_corners=False):  correspondence.py:240-241        */
#define MV_SAMPLE_ROWS 2           /* no resampling, rows are taken as they are:          correspondence.py:47-48           */

/* operand types of kernel 2 */
#define MV_DTYPE_BF16 0 /* tcgen05.mma kind::f16, bf16 inputs, fp32 accumulate  */
#define MV_DTYPE_TF32 1 /* tcgen05.mma kind::tf32, fp32 inputs, fp32 accumulate */
#define MV_DTYPE_F16 2  /* tcgen05.mma kind::f16, fp16 inputs (11-bit mantissa at the bf16 rate), fp32 accumulate */

/* role of a row set in a match: queries are the rows of S, targets its columns (f16c rows, see mv_k1_sample_f16c) */
#define MV_ROLE_QUERY 0
#define MV_ROLE_TARGET 1

/* `cluster` argument of kernel 2: 0 / 1 = every SM on its own; 2 / 4 = clusters of that many CTAs with the B tile
 * TMA-multicast; MV_CLUSTER_PAIR = CTA pairs (tcgen05 cta_group::2): one 256 x 256 MMA tile per two SMs */
#define MV_CLUSTER_PAIR 20
#define MV_CLUSTER_AUTO (-1) /* pick between 2-CTA multicast and the CTA pair from the operand type and C */

/* value written in masked / empty slots of similarity outputs */
#define MV_SIM_MASKED (-3.0e38f)

#define MV_MAX_THRESHOLDS 16

/* ---- library ------------------------------------------------------------------------ */
int mv_version(void);
const char* mv_last_error(void);
/* sm count, compute capability and L2 size of `device` (host out-params, any may be NULL) */
int mv_device_info(int device, int* sm_count, int* cc_major, int* cc_minor, int* l2_bytes);

/* ---- host -> device upload of pageable memory -------------------------------------------- */
/* The reference's callers hold plain CPU tensors (.detach().cpu(), evaluate_navi_correspondence.py:149-150): pageable
 * memory, which a plain cudaMemcpyAsync stages on the calling thread at a fifth of the PCIe rate.  mv_h2d_staged copies
 * `bytes` from src_host to dst_device through a pinned ring filled by a small pool of worker threads (MVMATCH_STAGE_THREADS,
 * default: half of the cores, at most 8), one plain cudaMemcpyAsync per 1 MiB chunk on `stream`.  Returns when every chunk has been issued: src_host
 * may be modified afterwards, the transfers complete in stream order.  One upload at a time per process. */
int mv_h2d_staged(void* dst_device, const void* src_host, size_t bytes, mv_stream_t stream);
int mv_h2d_staged_threads(void);

/* ---- layout helpers ------------------------------------------------------------------ */
/* (C, hw) channel-major fp32 map -> (hw, C) channel-last.  prenorm != 0 additionally divides
 * every pixel's C-vector by max(||.||_2, 1e-12)  (SPair: F.normalize(feats, p=2, dim=1),
 * evaluate_spair_correspondence.py:59).  norm_scratch: hw floats, required when prenorm. */
int mv_chw_to_hwc(const float* src_chw, float* dst_hwc, int C, int hw, int prenorm, float* norm_scratch,
                  mv_stream_t stream);

/* Backbone outputs in reduced precision (bf16 / fp16 under autocast) or already channel-last: any of
 * {fp32, bf16, fp16} x {(C, hw) channel-major, (hw, C) channel-last} -> the fp32 channel-last map kernel 1 reads.
 * The widening is exact: results equal the reference run on feats.float().  (SURVEY §8f.1: the hand-off of the
 * backbone output without the fp32 CPU round trip of evaluate_navi_correspondence.py:149-150.) */
#define MV_FEAT_F32 0
#define MV_FEAT_BF16 1
#define MV_FEAT_F16 2
int mv_feat_to_hwc_f32(const void* src, int dtype, int channel_last, int C, int hw, float* dst_hwc, mv_stream_t stream);

/* Row-major stable compaction of the indices i in [0, n) with z[i * z_stride] > 0
 * (correspondence.py:221-222 `xyz[:, 2] > 0`, :247-252 `xyz_grid[2] > 0`).
 * valid_idx: n int32 (first *n_valid are live, ascending); n_valid: 1 int32.  n <= 2^20. */
int mv_compact_valid(const float* z, int z_stride, int n, int32_t* valid_idx, int32_t* n_valid, mv_stream_t stream);

/* ---- geometry: per-point source coordinates for kernel 1 ------------------------------- */
/* ScanNet path: grid_to_pointcloud (correspondence.py:147-161) + the projection and NDC
 * normalisation of sample_pointcloud_features (:164-170) + grid_sample's align_corners=False
 * un-normalisation.  For every pixel of the (H, W) depth map:
 *   xyz_all (H*W, 3) = Kinv @ (depth * pixel-centre grid)            [always written]
 * and for the live points listed in valid_idx (after mv_compact_valid on xyz_all[:,2]):
 *   xyz (n, 3) compacted, coords (n, 2) = (ix, iy) in feature-map pixels.
 * Two entry points because the compaction sits between them.  K, Kinv: row-major 3x3, either HOST pointers (the
 * matrix is passed to the kernel by value) or DEVICE pointers (the kernel reads them: the intrinsics can then
 * change between replays of a captured CUDA graph -- ScanNet's differ per scene). */
int mv_geom_backproject(const float* depth, int H, int W, const float* Kinv_host, float* xyz_all, mv_stream_t stream);
int mv_geom_project_coords(const float* xyz_all, const int32_t* valid_idx, const int32_t* n_dev, int n_max,
                           const float* K_host, int H, int W, int h, int w, float* xyz, float* coords,
                           mv_stream_t stream);

/* NAVI path (correspondence.py:240-252): compacted xyz (n,3), uv (n,2) = pixel centres (x+.5, y+.5)
 * of the live pixels of the (3,H,W) xyz grid, and coords (n,2) = bicubic source index
 * (h/H)*(dst+0.5)-0.5 in the (h, w) feature map. */
int mv_geom_grid_coords(const float* xyz_grid, const int32_t* valid_idx, const int32_t* n_dev, int n_max, int H,
                        int W, int h, int w, float* xyz, float* uv, float* coords, mv_stream_t stream);

/* SPair path (evaluate_spair_correspondence.py:71-78): keypoints (n, kp_stride) in image pixels ->
 * kp/image_size*2-1 -> grid_sample align_corners=True un-normalisation ((g+1)/2*(size-1)). */
int mv_geom_keypoint_coords(const float* kps, int kp_stride, int n, float image_size, int h, int w, float* coords,
                            mv_stream_t stream);

/* ---- kernel 1: sample + L2-normalise + cast (HBM-bound) -------------------------------- */
/* For point p < n: row = sample(src, coords[p]) (4-tap bilinear with zero padding, 16-tap Keys
 * cubic A=-0.75 with border clamp, or row p of src itself); if normalize: row /= max(||row||,1e-12)
 * (F.normalize, correspondence.py:47-48).  Writes bf16 and/or fp32 rows.  C % 8 == 0, C <= 8192.
 * out_bf16_lo (optional, needs out_bf16): the SPLIT form of the fp32 row -- bf16(row - float(out_bf16)), so that
 * out_bf16 + out_bf16_lo reproduces the fp32 row to 2^-17 relative in 4 bytes per element instead of the 6 of
 * bf16 + fp32 (kernel 1 is bound by its row writes); consumed by mv_k3_ratio_mutual_split.
 * taps (optional, (n,2) int32): the (x0, y0) = floor(ix), floor(iy) tap origin, for parity tests. */
int mv_k1_sample_normalize(int mode, const float* src, int C, int h, int w, const float* coords,
                           const int32_t* n_dev, int n_max, int normalize, uint16_t* out_bf16, uint16_t* out_bf16_lo,
                           float* out_f32, int32_t* taps, mv_stream_t stream);

/* "f16c" rows: kernel 2's fp16 operand with the precision of a tf32 product at the bf16 rate, for feature sets whose
 * rows are nearly collinear (CNN features: all-positive, mean cosine ~0.9 -- there a bf16 product ranks the
 * wrong neighbour on most rows).  For a target row b and any fixed centre mu (we use the mean direction of the target's
 * source map), a . b = a . (b - mu) + a . mu, so
 *     target row  = [ fp16(b - mu) (C) | 1, 1, 2^-11, 0, 0, 0, 0, 0 ]
 *     query  row  = [ fp16(a)      (C) | p0, p1, p2, 0, 0, 0, 0, 0 ]     p0 + p1 + p2 * 2^-11 = r = a . mu  (fp32)
 * have the inner product a . b with the rounding error of the target scaled by |b - mu| instead of |b|; the ranking
 * along a row AND along a column is that of a . b for every mu.  Row pitch `pitch` >= C + 8 halfs (a multiple of 64 keeps
 * kernel 2's 128-byte TMA rows aligned: an unaligned pitch costs ~20 % of kernel 2); kernel 2 is called through
 * mv_k2_sim_top2_ld with C + 8 columns, that pitch and MV_DTYPE_F16 (columns beyond C + 8 are never read).  out_f16_lo (optional, (n, C) halfs): fp16((y - float(out_f16)) * 2^11) with
 * y = row - center, so that y = hi + lo * 2^-11 to 2^-22 relative (consumed by mv_k3_ratio_mutual_f16c).
 * role: MV_ROLE_QUERY uses dotvec (= the target's centre; NULL -> r = 0), MV_ROLE_TARGET uses center.  Both may be
 * given.  pixdot (optional; h*w floats, n for MV_SAMPLE_ROWS): src[p] . dotvec of every source row (mv_rows_dot); when
 * given, r is the row's own 4- / 16-tap blend of these scalars (times 1/norm) instead of a C-long dot product per row --
 * the same number up to the order of the fp32 sums -- and dotvec is not read.  row_dot (optional, n floats): r.  Other
 * arguments as mv_k1_sample_normalize. */
int mv_k1_sample_f16c(int mode, const float* src, int C, int h, int w, const float* coords, const int32_t* n_dev, int n_max,
                      int normalize, int role, const float* center, const float* dotvec, const float* pixdot, uint16_t* out_f16,
                      int pitch, uint16_t* out_f16_lo, float* out_f32, float* row_dot, int32_t* taps, mv_stream_t stream);

/* The same centring for the tf32 operand type ("tf32c" rows): out_op (n, pitch) fp32 = [tf32_round(row - center) (C) | 8
 * augmentation columns: three tf32-exact pieces of r (query) or (1, 1, 1) (target)], rounded to nearest tf32 here so
 * that the tensor core's truncation of fp32 operands is exact; pitch >= C + 8 (a multiple of 32 keeps the TMA rows
 * 128-byte aligned); kernel 2 takes C + 8 columns with MV_DTYPE_TF32.  out_f32 (n, C): the exact fp32 rows kernel 3 reads. */
int mv_k1_sample_tf32c(int mode, const float* src, int C, int h, int w, const float* coords, const int32_t* n_dev, int n_max,
                       int normalize, int role, const float* center, const float* dotvec, const float* pixdot, float* out_op, int pitch,
                       float* out_f32, int32_t* taps, mv_stream_t stream);

/* out[p] = rows[p] . vec for the n rows of rows (n, C) fp32 (C % 4 == 0): the per-source-pixel dots of the pixdot form. */
int mv_rows_dot(const float* rows, int C, int n, const float* vec, float* out, mv_stream_t stream);

/* The NAVI-style side as ONE tiled kernel (csrc/k1_grid.cu): bicubic upsampling (A = -0.75, align_corners=False, border
 * clamp) of the (h*w, C) map by the integer factors W / w (4 or 8) and H / h (1..8) onto the live pixels of the (H, W)
 * grid, L2-normalise, f16c rows -- the same values as mv_geom_grid_coords + mv_k1_sample_f16c(MV_SAMPLE_BICUBIC_CLAMP)
 * (identical arithmetic per element; the sum of squares is accumulated in another order: <= 1 ulp of the norm).
 * 2-D tiles (the fy output rows of a source-row step share 5 source rows, the pixels of a quad 5 columns) with the
 * channels split over a thread-block cluster whose CTAs exchange their partial sums of squares through distributed
 * shared memory: 3x less L2 traffic than the point-run kernel at C = 3072.
 * rank (H*W int32): row index of every live pixel, -1 elsewhere (mv_rank_of_valid).  Row r = rank[y*W + x] of
 * out_f16 / out_f16_lo is written for every live pixel.  mv_k1_grid_supported says whether a shape is covered. */
int mv_k1_grid_supported(int C, int h, int w, int H, int W);
int mv_rank_of_valid(const int32_t* valid_idx, const int32_t* n_dev, int n_max, int32_t* rank, int n_pixels, mv_stream_t stream);
int mv_k1_grid_f16c(const float* src, int C, int h, int w, int H, int W, const int32_t* rank, int role, const float* center,
                    const float* dotvec, uint16_t* out_f16, int pitch, uint16_t* out_f16_lo, mv_stream_t stream);

/* mu (C floats) = mean over every `step`-th row p < n of rows[p] / max(||rows[p]||, 1e-12); rows (n, C) fp32 (a channel-last
 * feature map or a set of feature rows).  inv_scratch: ceil(n_max / step) floats.  Deterministic. */
int mv_rows_center(const float* rows, int C, int n_max, const int32_t* n_dev, int step, float* inv_scratch, float* mu,
                   mv_stream_t stream);

/* ---- kernel 2's operands in the basis of the source pixels ("low-rank proposal", csrc/lr_gram.cu) ----
 * The dense helpers interpolate every row linearly from an (h*w, C) source map (correspondence.py:164-176 bilinear
 * grid_sample; :240-241 bicubic interpolate), so the cosine similarity of two interpolated, normalised rows
 * (correspondence.py:47-48 + :14-23) is a product over the h*w SOURCE PIXELS of the target image instead of the C
 * channels:  cos(x_i, y_j) = sum_t A[i,t] B[j,t],  A[i,t] = (x_i/|x_i|) . (src1[t]/|src1[t]|),  B[j,t] = W1[j,t] |src1[t]| / |y_j|.
 * The N x M product still runs on kernel 2 (mv_k2_sim_top2_ld, MV_DTYPE_F16, hwp + 8 columns); these entry points build
 * its operands.  hwp = h*w rounded up to a multiple of 8 (<= MV_LR_MAX_SOURCE_PIXELS).
 *   mv_lr_unit_rows    U (hw, C) fp16 = src / |src| per source pixel, snorm (hw) = |src|; src (hw, C) fp32 channel-last.
 *                      The caller stacks both images' U (image k at row offset off_k, pad rows zero) and obtains the
 *                      stacked cosine Gram matrix G (fp32, pitch ld_g) from mv_k2_affinity(U, U).
 *   mv_lr_gram_exact   the other source of G: the Gram matrix of the RAW source rows of both images stacked (image 1 at row /
 *                      column offset off1, a multiple of 32 >= hw), (2 off1, ld_g) fp32, computed on the CUDA cores with blocked
 *                      fp32 accumulation (16 slices of C / 16 channels per entry, fixed-order tree: ~1 ulp, deterministic;
 *                      C % 64 == 0), plus snorm / rsnorm (2 off1): |src[p]| and its reciprocal from the diagonal.  Written: the
 *                      whole cross block (image 0 x image 1, both orientations) and, of the two same-image blocks, the entries
 *                      whose indices are at most `reach` apart (at least those: whole 32 x 32 tiles of the band) -- pass the largest
 *                      index distance between two taps of one point ((T - 1) (w + 1) for T x T taps); the rest of G is left
 *                      untouched.  Exact enough for kernel 3 (mv_k3_ratio_mutual_lr); the tensor-core Gram is not (tcgen05
 *                      accumulates with truncation).
 *   mv_lr_build_query  A_f16 (n, pitch): [fp16(A[i,:] - c_i) (hw) | 0 (to hwp) | c_i, c_i, 0 x 6], c_i = fp16(max_t A[i,t])
 *                      (centring a row on its own maximum keeps the fp16 rounding error of the columns that compete for
 *                      the row's top-2 at ~1e-6, also on nearly collinear CNN features).
 *   mv_lr_build_target B_f16 (m, pitch): [fp16(B[j,:]) scattered into zeros | two fp16 pieces of beta_j = sum_t B[j,t], 0 x 6]
 * so that the product of an A row and a B row over hwp + 8 columns is cos(x_i, y_j) up to the fp16 rounding of A - c and B.
 * coords (n, 2): the continuous source coordinates kernel 1 samples at (mv_geom_project_coords / mv_geom_grid_coords);
 * mode: MV_SAMPLE_BILINEAR_ZEROS or MV_SAMPLE_BICUBIC_CLAMP (the taps of kernel 1); off_own / off_tgt: this image's and the
 * target image's offset in G.  Scales, by the kind of G:   cosine Gram of unit rows: tapscale = this image's snorm, query
 * colscale = NULL;   raw Gram: tapscale = NULL, query colscale = the target's rsnorm.  The target's snorm argument is the
 * target image's |src| in both cases.  inv_norm_out (optional, n floats): 1 / max(|x_i|, 1e-12) of every point.
 *   mv_k3_ratio_mutual_lr  kernel 3's ratio / mutual step on the raw Gram: the fp32 cosine distances of every query's two
 *                      candidates (row_idx from kernel 2) as 1 - (sum_{a,b} W0[i,a] W1[j,b] G[off_q + s_a, off_t + t_b]) inv_q[i] inv_t[j]
 *                      -- 16 (bilinear) / 256 (bicubic) Gram entries per candidate instead of three C-long rows -- then exactly
 *                      mv_k3_ratio_mutual's outputs (correspondence.py:53-58, :72-77, :105-121).  With it the interpolated
 *                      rows are never materialised: kernel 1 does not run. */
#define MV_LR_MAX_SOURCE_PIXELS 1024
int mv_lr_unit_rows(const float* src_hwc, int C, int hw, void* U_f16, float* snorm, mv_stream_t stream);
int mv_lr_gram_exact(const float* src0_hwc, const float* src1_hwc, int C, int hw, int off1, int reach, float* G, int ld_g,
                     float* snorm, float* rsnorm, mv_stream_t stream);
int mv_lr_build_query(int mode, const float* coords, const int32_t* n_dev, int n_max, int h, int w, const float* tapscale,
                      const float* colscale, const float* G, int ld_g, int off_own, int off_tgt, void* A_f16, int pitch, int hwp,
                      float* inv_norm_out, mv_stream_t stream);
int mv_lr_build_target(int mode, const float* coords, const int32_t* n_dev, int n_max, int h, int w, const float* tapscale,
                       const float* snorm, const float* G, int ld_g, int off_own, void* B_f16, int pitch, int hwp,
                       float* inv_norm_out, mv_stream_t stream);
int mv_k3_ratio_mutual_lr(int mode, const float* coords_q, const float* coords_t, const float* inv_q, const float* inv_t,
                          const float* G, int ld_g, int off_q, int off_t, int h, int w, const int32_t* n_dev, int n_max,
                          int32_t* row_idx, const unsigned long long* col_best, int ratio_test, float* dists, float* weight,
                          uint8_t* mutual, mv_stream_t stream);

/* ---- kernel 2: similarity GEMM with fused row top-2 / column arg-max (tensor-core bound) -- */
/* S = A @ B^T (n x m, never written).  Replaces faiss GpuIndexFlatL2.search(k<=2)
 * (correspondence.py:14-23) for L2-normalised rows, where the L2 order equals the cosine order
 * (correspondence.py:27-43).
 *   row_val/row_idx (n_max, 2): the two largest S[i, :] and their columns, best first, ties to the
 *                               lower column; missing entries = MV_SIM_MASKED / -1.
 *   col_best (m_max) optional : packed arg-max over rows of S[:, j]; decode with mv_k2_unpack_col.
 * A, B: bf16 (MV_DTYPE_BF16), fp16 (MV_DTYPE_F16) or fp32 (MV_DTYPE_TF32), 16-byte aligned, C % 8 == 0 (16-bit) / C % 4 == 0.
 * cluster: 0 or 1 = one CTA per SM on its own; 2 or 4 = thread-block clusters of that many CTAs working on
 * consecutive row blocks with the B tile loaded once and TMA-multicast to all of them; MV_CLUSTER_PAIR = the two
 * CTAs of a cluster issue ONE 256-row MMA (cta_group::2), each holding half of the B tile.
 * workspace from mv_k2_workspace_bytes. */
size_t mv_k2_workspace_bytes(int n_max, int m_max);
int mv_k2_sim_top2(const void* A, const void* B, int n_max, int m_max, int C, const int32_t* n_dev,
                   const int32_t* m_dev, int dtype, int cluster, float* row_val, int32_t* row_idx,
                   unsigned long long* col_best, void* workspace, size_t workspace_bytes, mv_stream_t stream);
/* the same with explicit row pitches lda / ldb (elements, >= C, a multiple of 16 bytes): only the first C columns of a row
 * are read (f16c rows: C = channels + 8, pitch rounded up to 128 bytes) */
int mv_k2_sim_top2_ld(const void* A, int lda, const void* B, int ldb, int n_max, int m_max, int C, const int32_t* n_dev,
                      const int32_t* m_dev, int dtype, int cluster, float* row_val, int32_t* row_idx,
                      unsigned long long* col_best, void* workspace, size_t workspace_bytes, mv_stream_t stream);
/* The same GEMM with the similarity matrix WRITTEN OUT as well: S_out (n_max, ld_s) fp32, S[i][j] = A[i] . B[j] (rows / columns
 * beyond the live counts are left untouched).  For consumers that need the matrix itself -- MaskCut's normalised affinity
 * feats^T @ feats (evals/models/maskcut_processor.py:77-78) -- instead of its row top-2 / column arg-max, which are still
 * produced (the epilogue is the same kernel; S_out == NULL is exactly mv_k2_sim_top2_ld). */
int mv_k2_affinity(const void* A, int lda, const void* B, int ldb, int n_max, int m_max, int C, const int32_t* n_dev,
                   const int32_t* m_dev, int dtype, int cluster, float* S_out, int ld_s, float* row_val, int32_t* row_idx,
                   unsigned long long* col_best, void* workspace, size_t workspace_bytes, mv_stream_t stream);
/* Timing of the GEMM kernel ALONE (for a roofline figure that is not diluted by the col_best memset and the row merge of
 * the same call): after mv_k2_profile_begin(capacity) the next `capacity` calls of mv_k2_sim_top2* / mv_k2_affinity on this
 * host thread record a CUDA event pair right around the launch of the tcgen05 kernel; mv_k2_profile_read waits for them
 * and returns how many durations (milliseconds, call order) it wrote to ms_out (host).  begin(0) switches it off.  Not
 * capturable into a CUDA graph. */
/* Schedule switch of kernel 2: 1 lets the persistent schedule cut tiles along K when a cluster would otherwise get a
 * small non-integer number of tiles ("stream-K": equal k-block counts per SM, head fragments handed over through the
 * workspace).  Default 0 (MVMATCH_K2_STREAMK=1 in the environment starts with 1): measured slower on B200, see
 * csrc/k2_sim.cu.  Returns the previous setting; on < 0 only queries.  Takes effect for launches issued afterwards (a
 * captured CUDA graph keeps the setting it was captured with). */
int mv_k2_set_streamk(int on);
int mv_k2_profile_begin(int capacity);
int mv_k2_profile_read(float* ms_out, int max_n);
/* (n_max, m_max, C) of the recorded launches, three ints each, call order: tells the launches of one call site from another's
 * (the Gram launch of the low-rank proposal and the main product go through the same kernel). */
int mv_k2_profile_dims(int* nmc_out, int max_n);
int mv_k2_unpack_col(const unsigned long long* col_best, int m, float* col_val, int32_t* col_idx, mv_stream_t stream);

/* ---- k > 2 nearest neighbours: kernel 2 with a row top-KP epilogue + an fp32 re-rank ------------ */
/* The same GEMM as mv_k2_sim_top2_ld with an epilogue that keeps the kp (8 or 16) largest S[i, :] of every row instead of
 * the top-2 and the column arg-max:
 *   row_val/row_idx (n_max, kp): values descending, ties to the lower column; missing entries (m < kp, columns past *m_dev,
 *                                rows past *n_dev) = MV_SIM_MASKED / -1.
 * Positions 0 and 1 equal mv_k2_sim_top2_ld's row outputs bit for bit on the same operands and cluster form (stream-K off).
 * The schedule is always tile-granular (mv_k2_set_streamk does not apply) and the launch is not recorded by
 * mv_k2_profile_*.  Other arguments as mv_k2_sim_top2_ld; workspace from mv_k2_topk_workspace_bytes (0 for a bad kp). */
size_t mv_k2_topk_workspace_bytes(int n_max, int m_max, int kp);
int mv_k2_sim_topk_ld(const void* A, int lda, const void* B, int ldb, int n_max, int m_max, int C, const int32_t* n_dev,
                      const int32_t* m_dev, int dtype, int cluster, int kp, float* row_val, int32_t* row_idx, void* workspace,
                      size_t workspace_bytes, mv_stream_t stream);
/* fp32 re-rank of kp candidates per query (cand (n_max, kp) int32, e.g. row_idx above; -1 = no candidate): the distance of
 * query row Q[i] (n_max, ldq) to every candidate row T[j] (ldt) over C columns --
 *   MV_METRIC_L2SQ     sum (q - t)^2                                  (faiss' squared L2)
 *   MV_METRIC_COSINE   1 - q.t / (max(|q|, 1e-8) * max(|t|, 1e-8))    (kernel 3's cosine distance)
 * -- sorted ascending, ties to the lower index; out_dist / out_idx (n_max, k) receive the first k, 1 <= k <= kp
 * (missing: +inf / -1, also for rows past *n_dev).  128-bit loads when C and both pitches are multiples of 4 floats. */
#define MV_METRIC_L2SQ 0
#define MV_METRIC_COSINE 1
int mv_knn_rerank(const float* Q, int ldq, const float* T, int ldt, int C, const int32_t* n_dev, int n_max, const int32_t* cand,
                  int kp, int k, int metric, float* out_dist, int32_t* out_idx, mv_stream_t stream);

/* ---- kernel 3: fp32 distance recompute, ratio test, mutual check, selection, scoring ---- */
/* Per query row i with candidates j0, j1 = row_idx[i]:  d_k = 1 - cos(A32[i], B32[j_k]) in fp32
 * (knn_points, correspondence.py:53-58); candidates are re-ranked so d_0 <= d_1 (row_idx is updated
 * in place); weight = 1 - max(d0,1e-9)/max(d1,1e-9) if ratio_test else d0  (correspondence.py:72-77,
 * :105-121); mutual[i] = (argmax_i' S[i', j0] == i) from col_best (may be NULL -> all 0). */
int mv_k3_ratio_mutual(const float* A32, const float* B32, int C, const int32_t* n_dev, int n_max,
                       int32_t* row_idx, const unsigned long long* col_best, int ratio_test, float* dists,
                       float* weight, uint8_t* mutual, mv_stream_t stream);
/* The same on SPLIT rows (mv_k1_sample_normalize's out_bf16 / out_bf16_lo planes): every element is rebuilt
 * as float(hi) + float(lo) (exact in fp32) before the identical fp32 arithmetic.  C % 8 == 0. */
int mv_k3_ratio_mutual_split(const uint16_t* A_hi, const uint16_t* A_lo, const uint16_t* B_hi, const uint16_t* B_lo, int C,
                             const int32_t* n_dev, int n_max, int32_t* row_idx, const unsigned long long* col_best,
                             int ratio_test, float* dists, float* weight, uint8_t* mutual, mv_stream_t stream);

/* The same on f16c rows (mv_k1_sample_f16c): A_hi (n, pitch) / A_lo (n, C) query rows, B_hi / B_lo target rows,
 * center_B (C floats or NULL) the centre the target rows are relative to; every element is rebuilt as
 * float(hi) + float(lo) * 2^-11 (+ center_B) before the identical fp32 arithmetic. */
int mv_k3_ratio_mutual_f16c(const uint16_t* A_hi, const uint16_t* A_lo, const uint16_t* B_hi, const uint16_t* B_lo, int C, int pitch,
                            const float* center_B, const int32_t* n_dev, int n_max, int32_t* row_idx,
                            const unsigned long long* col_best, int ratio_test, float* dists, float* weight, uint8_t* mutual,
                            mv_stream_t stream);

/* MaskCut's thresholded affinity (evals/models/maskcut_processor.py:103-106): A[i][j] = S[i][j] > tau ? 1 : eps, written as
 * fp32, and count[i] = #{j : S[i][j] > tau} (so that d_i = count + (m - count) * eps is exact in any precision).  S (n, ld_s). */
int mv_affinity_threshold(const float* S, int n, int m, int ld_s, float tau, float eps, float* A_out, int32_t* count, mv_stream_t stream);

/* 2AFC perceptual evaluation (evaluate_model_percepture.py:46-48, :118-122): per sample i the cosine similarities
 * sim_l = cos(ref_i, left_i), sim_r = cos(ref_i, right_i) with torch.nn.functional.cosine_similarity's arithmetic
 * (x . y / (max(|x|, 1e-8) * max(|y|, 1e-8))) and pred_i = sim_l > sim_r ? 0 : 1.  Rows (n, C) fp32, C % 4 == 0. */
int mv_cosine_2afc(const float* ref, const float* left, const float* right, int n, int C, float* sim_left, float* sim_right,
                   int32_t* pred, mv_stream_t stream);

/* get_topk_matches (correspondence.py:125-129): the k = min(num_corr, n) largest weights, sorted
 * descending (ties: lower row first).  sel_* have num_corr entries; k_dev receives k.
 * num_corr <= 16384, n_max <= 2^20. */
int mv_k3_topk_matches(const float* weight, const int32_t* row_idx, const int32_t* n_dev, int n_max,
                       int num_corr, int32_t* sel_src, int32_t* sel_dst, float* sel_weight, int32_t* k_dev,
                       mv_stream_t stream);

/* Scoring of the selected matches (callers: evaluate_navi_correspondence.py:183-212,
 * render_scannet_correspondence.py:211-217, :253-264, :131-147):
 *   p0 = xyz0[sel_src], p1 = xyz1[sel_dst]; p0in1 = p0 @ R^T + t (transformations.py:27-36);
 *   err3d = ||p0in1 - p1||; err2d = ||proj(p0in1) - proj(p1)||, proj = project_3dto2d (:193-196).
 * Integer hit counts are ACCUMULATED (atomicAdd) into hits[]:
 *   hits[0]                      += k                      (matches scored)
 *   hits[1]                      += #mutual among them
 *   hits[2 + t]                  += #(err3d < thr3d[t])            t < n3
 *   hits[2 + n3 + t]             += #(err2d < thr2d[t])            t < n2
 *   hits[2 + n3 + n2 + t]        += #(mutual & err3d < thr3d[t])
 *   hits[2 + 2*n3 + n2 + t]      += #(mutual & err2d < thr2d[t])
 * Rt (3x4), Kproj (3x3), thr3d, thr2d are host arrays.  c_* / err* outputs are optional (NULL). */
int mv_k3_score(const int32_t* sel_src, const int32_t* sel_dst, const int32_t* k_dev, int k_max,
                const float* xyz0, const float* xyz1, const uint8_t* mutual, const float* Rt_host,
                const float* Kproj_host, const float* thr3d_host, int n3, const float* thr2d_host, int n2,
                float* c_xyz0, float* c_xyz1, float* err3d, float* err2d, unsigned long long* hits,
                mv_stream_t stream);

/* Plain gather of rows: dst[i, :] = src[idx[i], :] for i < *k_dev (k_max if NULL); width floats. */
int mv_gather_rows(const float* src, int width, const int32_t* idx, const int32_t* k_dev, int k_max, float* dst,
                   mv_stream_t stream);

/* The return tuple of estimate_correspondence_xyz / _depth (correspondence.py:229-232, :258-263) gathered into ONE
 * buffer of column blocks, each k_max rows: [xyz0 (k_max,3) | xyz1 (k_max,3) | weight (k_max) | uv0 (k_max,2) |
 * uv1 (k_max,2) | n0, n1, k, 0] -- xyz0 = xyz0_all[sel_src], xyz1 = xyz1_all[sel_dst] etc.; the uv blocks exist
 * only when uv0/uv1 are given; the 4-float tail carries the live counts (*n0_dev, *n1_dev, k) so that a host
 * caller needs a single device -> host copy and a single sync.  out: (7 or 11) * k_max + 4 floats. */
int mv_pack_matches(const int32_t* sel_src, const int32_t* sel_dst, const float* sel_weight, const int32_t* k_dev, int k_max,
                    const float* xyz0, const float* xyz1, const float* uv0, const float* uv1, const int32_t* n0_dev,
                    const int32_t* n1_dev, float* out, mv_stream_t stream);

/* argmax_2d (correspondence.py:179-190): flat arg-max (or arg-min) of every row of x (rows, cols),
 * first occurrence on ties; out_flat (rows) int32.  The caller turns flat into (col, row). */
int mv_argmax_rows(const float* x, int rows, int cols, int max_value, int32_t* out_flat, mv_stream_t stream);

/* SPair scoring (evaluate_spair_correspondence.py:83-98, :121): pred (K) = arg-max column of the
 * heat map in the (h, w) feature map -> (col,row)/w; errors (K,K) = ||pred_k - kps_j[l,:2]/image_size||
 * / thresh_scale, 1e3 where kps_i[k,2]*kps_j[l,2] != 1.  Outputs error matrix (K,K, optional),
 * error_same (K; -1 where the keypoint is not in both), error_nn / index_nn (K; -1 likewise) and
 * ACCUMULATES hits[0] += #in_both, hits[1] += #(error_same < pck_thresh) and, when `confusion` is given
 * ((conf_dim, conf_dim) counters, conf_dim >= K), confusion[k][index_nn[k]] += 1 for every keypoint in both
 * images (the matrix evaluate_dataset builds at evaluate_spair_correspondence.py:115-118). K <= 64. */
int mv_k3_spair_errors(const int32_t* pred_flat, int K, int w, const float* kps_i, const float* kps_j,
                       int kp_stride, float image_size, float thresh_scale, float pck_thresh, float* errors,
                       float* error_same, float* error_nn, int32_t* index_nn, unsigned long long* hits,
                       unsigned long long* confusion, int conf_dim, mv_stream_t stream);

/* SPair matching for a BATCH of pairs in one launch (evaluate_spair_correspondence.py:59-103 for every pair of
 * the loop at :108): feats (B, 2, C, h, w) = the backbone output for (image_i, image_j) of each pair, fp32,
 * contiguous; kps_i / kps_j (B, K, kp_stride) = (x, y, valid, ...) in image pixels; thresh_scale (B) on the
 * device.  Per pair: per-pixel L2 normalisation (:59), bilinear key-point gather with align_corners=True
 * (:71-79), K x (h*w) heat map and its arg-max (:82-83) -- all fp32, the heat map never leaves registers --
 * then the scoring of mv_k3_spair_errors.  Outputs (each optional): pred_flat (B, K) int32 flat arg-max pixel,
 * error_same / error_nn (B, K; -1 where the key point is not in both images), index_nn (B, K); hits[0..1] and
 * confusion accumulate as in mv_k3_spair_errors.  K <= 64. */
int mv_spair_match_batch(const float* feats, int B, int C, int h, int w, const float* kps_i, const float* kps_j, int K,
                         int kp_stride, const float* thresh_scale, float image_size, float pck_thresh,
                         int32_t* pred_flat, float* error_same, float* error_nn, int32_t* index_nn,
                         unsigned long long* hits, unsigned long long* confusion, int conf_dim, mv_stream_t stream);

/* mv_spair_match_batch on a map of any MV_FEAT_* element type: feats (B, 2, C, h, w) contiguous fp32, bf16 or fp16 (the
 * output of an autocast backbone), read as it is -- a 16-bit map streams half the bytes and is widened on the chip.
 * Widening is exact and the kernel keeps the fp32 form's channel chunks and summation order, so the outputs are BIT-
 * IDENTICAL to mv_spair_match_batch on the map widened to fp32, in either heat-map precision.  feat_dtype = MV_FEAT_F32
 * is mv_spair_match_batch.  Errors, checked before any CUDA call: an unknown feat_dtype (MV_E_ARG), feats not aligned to
 * its element size (MV_E_ALIGN), and those of mv_spair_match_batch. */
int mv_spair_match_batch_typed(const void* feats, int feat_dtype, int B, int C, int h, int w, const float* kps_i,
                               const float* kps_j, int K, int kp_stride, const float* thresh_scale, float image_size,
                               float pck_thresh, int32_t* pred_flat, float* error_same, float* error_nn, int32_t* index_nn,
                               unsigned long long* hits, unsigned long long* confusion, int conf_dim, mv_stream_t stream);

/* Precision of the batched kernel's heat map (the einsum of evaluate_spair_correspondence.py:82) on the tensor cores:
 * 3 (default) = every product as three tf32 MMAs (hi*hi + hi*lo + lo*hi, ~21 mantissa bits: the arg-max equals the fp32
 * reference's wherever the top-2 heat-map gap exceeds 1e-5); 1 = one tf32 MMA, operands rounded to 10 mantissa bits with
 * fp32 accumulation (arg-max equal wherever the gap exceeds 1e-3, the tolerance of the matching path's tf32 operand type).
 * Returns the previous setting; any other value only queries.  Takes effect for launches issued afterwards. */
int mv_spair_set_heatmap_terms(int terms);

#ifdef __cplusplus
}
#endif
#endif /* MVMATCH_H_ */
