// k1_sample.cu -- kernel 1 of the matching path and its small producers.
//
//   mv_chw_to_hwc            (C,h,w) backbone map -> channel-last (h*w, C), optional per-pixel L2 norm
//   mv_compact_valid         stable compaction of the live (z > 0) pixels
//   mv_geom_*                per-point source coordinates for the three reference call sites
//   mv_k1_sample_normalize   gather/upsample + L2-normalise + bf16/fp32 row writer   (HBM-bound)
//
// Reference behaviour being reproduced (file:line in /root/reference):
//   evals/utils/correspondence.py:132-176  get_grid / grid_to_pointcloud / sample_pointcloud_features
//   evals/utils/correspondence.py:240-252  bicubic upsample + valid-pixel gather
//   evals/utils/correspondence.py:47-48    F.normalize of the sampled rows
//   evaluate_spair_correspondence.py:59-79 per-pixel normalise + keypoint grid_sample(align_corners=True)
//
// Data layout: the source map is channel-last so that every tap is one contiguous C-vector read with
// 128-bit loads; consecutive live points are handled by the same CTA, which stages the source columns they
// share in shared memory once (an 8x upsample re-uses each tap ~8 times along x), so the kernel's traffic is
// the row writes: C*h*w*4 bytes read + n*C*(2 [+4]) bytes written.

#include <cuda_fp16.h>

#include <cstdlib>

#include "common.cuh"
#include "sm100_ptx.cuh"

namespace {

constexpr float K1_NORM_EPS = 1e-12f;  // F.normalize default eps

// ------------------------------------------------------------------------------------------
// (C, hw) -> (hw, C) transpose, optional scale by 1/max(norm, eps)
// ------------------------------------------------------------------------------------------
__global__ void pixel_norm_kernel(const float* __restrict__ src, float* __restrict__ norm, int C, int hw) {
  // block = (32 pixels, 8 channel slices)
  __shared__ float part[8][33];
  const int px = blockIdx.x * 32 + threadIdx.x;
  float ss = 0.f;
  if (px < hw) {
    for (int c = threadIdx.y; c < C; c += 8) {
      float v = __ldg(src + (size_t)c * hw + px);
      ss = fmaf(v, v, ss);
    }
  }
  part[threadIdx.y][threadIdx.x] = ss;
  __syncthreads();
  if (threadIdx.y == 0 && px < hw) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += part[k][threadIdx.x];
    norm[px] = sqrtf(t);
  }
}

__global__ void chw_to_hwc_kernel(const float* __restrict__ src, float* __restrict__ dst, int C, int hw,
                                  const float* __restrict__ norm) {
  __shared__ float tile[32][33];
  const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  // read: x = pixel (contiguous in src), y = channel
  for (int dy = threadIdx.y; dy < 32; dy += 8) {
    int c = c0 + dy, p = p0 + threadIdx.x;
    float v = 0.f;
    if (c < C && p < hw) v = __ldg(src + (size_t)c * hw + p);
    tile[dy][threadIdx.x] = v;
  }
  __syncthreads();
  // write: x = channel (contiguous in dst), y = pixel
  for (int dy = threadIdx.y; dy < 32; dy += 8) {
    int p = p0 + dy, c = c0 + threadIdx.x;
    if (c < C && p < hw) {
      float v = tile[threadIdx.x][dy];
      if (norm) v = __fdiv_rn(v, fmaxf(__ldg(norm + p), K1_NORM_EPS));
      dst[(size_t)p * C + c] = v;
    }
  }
}

// The same transpose with 128-bit accesses on both sides (hw % 4 == 0, C % 4 == 0): a CTA moves a tile of
// 64 channels x 64 pixels; 16 lanes read one channel's 256 contiguous bytes, 16 lanes write one pixel's.
__global__ void __launch_bounds__(256) chw_to_hwc_vec_kernel(const float* __restrict__ src, float* __restrict__ dst,
                                                             int C, int hw, const float* __restrict__ norm) {
  __shared__ float tile[64][65];  // [channel][pixel]
  const int p0 = blockIdx.x * 64, c0 = blockIdx.y * 64;
  const int q = threadIdx.x & 15, r = threadIdx.x >> 4;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int c = c0 + r + 16 * k, p = p0 + 4 * q;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c < C && p < hw) v = __ldg(reinterpret_cast<const float4*>(src + (size_t)c * hw + p));
    float* t = &tile[r + 16 * k][4 * q];
    t[0] = v.x;
    t[1] = v.y;
    t[2] = v.z;
    t[3] = v.w;
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int p = p0 + r + 16 * k, c = c0 + 4 * q;
    if (p < hw && c < C) {
      float4 v = make_float4(tile[4 * q][r + 16 * k], tile[4 * q + 1][r + 16 * k], tile[4 * q + 2][r + 16 * k],
                             tile[4 * q + 3][r + 16 * k]);
      if (norm) {
        const float d = fmaxf(__ldg(norm + p), K1_NORM_EPS);
        v.x = __fdiv_rn(v.x, d);
        v.y = __fdiv_rn(v.y, d);
        v.z = __fdiv_rn(v.z, d);
        v.w = __fdiv_rn(v.w, d);
      }
      *reinterpret_cast<float4*>(dst + (size_t)p * C + c) = v;
    }
  }
}

// Reduced-precision backbone outputs (bf16 / fp16 under autocast): widen to the fp32 channel-last map kernel 1
// reads.  The widening is exact, so the result equals the reference run on feat.float().
template <typename T> __device__ __forceinline__ float feat_to_float(T v);
template <> __device__ __forceinline__ float feat_to_float<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <> __device__ __forceinline__ float feat_to_float<__half>(__half v) { return __half2float(v); }

template <typename T>
__global__ void chw_to_hwc_widen_kernel(const T* __restrict__ src, float* __restrict__ dst, int C, int hw) {
  __shared__ float tile[32][33];
  const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int dy = threadIdx.y; dy < 32; dy += 8) {
    const int c = c0 + dy, p = p0 + threadIdx.x;
    tile[dy][threadIdx.x] = (c < C && p < hw) ? feat_to_float<T>(src[(size_t)c * hw + p]) : 0.f;
  }
  __syncthreads();
  for (int dy = threadIdx.y; dy < 32; dy += 8) {
    const int p = p0 + dy, c = c0 + threadIdx.x;
    if (c < C && p < hw) dst[(size_t)p * C + c] = tile[threadIdx.x][dy];
  }
}

template <typename T>
__global__ void widen_kernel(const T* __restrict__ src, float* __restrict__ dst, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = feat_to_float<T>(src[i]);
}

// ------------------------------------------------------------------------------------------
// stable compaction (n <= 2^20): one CTA per 1024 elements.  A CTA first counts the live elements BEFORE its chunk
// itself (coalesced sweep over the preceding flags: at most n / 1024 loads per thread, all in flight), then places its
// own chunk with a ballot scan -- no inter-CTA communication, no second launch, and the order is the row-major order
// of the reference's boolean mask (correspondence.py:221-222, :247-252).  (Round 1: a single CTA with 19 strided
// elements per thread, 19 us for 19200 depth pixels; now ~3 us.)
// ------------------------------------------------------------------------------------------
constexpr int COMPACT_CHUNK = 1024;
__global__ void __launch_bounds__(COMPACT_CHUNK) compact_valid_kernel(const float* __restrict__ z, int z_stride, int n,
                                                                     int32_t* __restrict__ valid_idx,
                                                                     int32_t* __restrict__ n_valid) {
  __shared__ int warp_tot[32];
  __shared__ int s_before;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int base = blockIdx.x * COMPACT_CHUNK;
  // ---- live elements in [0, base)
  int cnt = 0;
#pragma unroll 4
  for (int i = tid; i < base; i += COMPACT_CHUNK) cnt += (__ldg(z + (size_t)i * z_stride) > 0.f) ? 1 : 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if (lane == 0) warp_tot[wid] = cnt;
  __syncthreads();
  if (wid == 0) {
    int t = warp_tot[lane];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (lane == 0) s_before = t;
  }
  __syncthreads();
  const int before = s_before;
  // ---- this chunk: one element per thread
  const int i = base + tid;
  const bool live = i < n && __ldg(z + (size_t)i * z_stride) > 0.f;
  const uint32_t bal = __ballot_sync(0xffffffffu, live);
  if (lane == 0) warp_tot[wid] = __popc(bal);
  __syncthreads();
  int off = 0, total = 0;
#pragma unroll 8
  for (int w = 0; w < 32; ++w) {
    const int c = warp_tot[w];
    off += (w < wid) ? c : 0;
    total += c;
  }
  if (live) valid_idx[before + off + __popc(bal & ((1u << lane) - 1u))] = i;
  if (blockIdx.x == gridDim.x - 1 && tid == 0) *n_valid = before + total;
}

// ------------------------------------------------------------------------------------------
// geometry
// ------------------------------------------------------------------------------------------
struct Mat3 {
  float m[9];
};

// correspondence.py:132-161: points = depth * (x+.5, y+.5, 1); xyz = Kinv @ points
// A 3x3 matrix argument is either passed by value (host pointer at the ABI) or read from device memory (device
// pointer at the ABI: the matrix can then change between replays of a captured CUDA graph).
__device__ __forceinline__ Mat3 pick_mat3(const Mat3& by_value, const float* __restrict__ dev) {
  if (!dev) return by_value;
  Mat3 m;
#pragma unroll
  for (int i = 0; i < 9; ++i) m.m[i] = __ldg(dev + i);
  return m;
}

__global__ void backproject_kernel(const float* __restrict__ depth, int H, int W, Mat3 Ki_val,
                                   const float* __restrict__ Ki_dev, float* __restrict__ xyz_all) {
  int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= H * W) return;
  const Mat3 Ki = pick_mat3(Ki_val, Ki_dev);
  int y = p / W, x = p - y * W;
  float d = __ldg(depth + p);
  float px = __fmul_rn(d, (float)x + 0.5f), py = __fmul_rn(d, (float)y + 0.5f), pz = d;  // depth * grid
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    float a = __fmul_rn(Ki.m[3 * r + 0], px);
    a = fmaf(Ki.m[3 * r + 1], py, a);
    a = fmaf(Ki.m[3 * r + 2], pz, a);
    xyz_all[(size_t)p * 3 + r] = a;
  }
}

// correspondence.py:164-170 + ATen CPU grid_sampler (align_corners=False): ix = (g+1)*(size/2) - 0.5
__global__ void project_coords_kernel(const float* __restrict__ xyz_all, const int32_t* __restrict__ valid_idx,
                                      const int32_t* __restrict__ n_dev, int n_max, Mat3 K_val,
                                      const float* __restrict__ K_dev, int H, int W, int h, int w,
                                      float* __restrict__ xyz, float* __restrict__ coords) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  int n = n_dev ? min(*n_dev, n_max) : n_max;
  if (i >= n) return;
  const Mat3 K = pick_mat3(K_val, K_dev);
  int p = valid_idx ? valid_idx[i] : i;
  float X = xyz_all[(size_t)p * 3 + 0], Y = xyz_all[(size_t)p * 3 + 1], Z = xyz_all[(size_t)p * 3 + 2];
  xyz[(size_t)i * 3 + 0] = X;
  xyz[(size_t)i * 3 + 1] = Y;
  xyz[(size_t)i * 3 + 2] = Z;
  float uvd[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) {  // uvd = pc @ K^T
    float a = __fmul_rn(X, K.m[3 * r + 0]);
    a = fmaf(Y, K.m[3 * r + 1], a);
    a = fmaf(Z, K.m[3 * r + 2], a);
    uvd[r] = a;
  }
  float den = fmaxf(uvd[2], 1e-9f);
  float u = __fdiv_rn(uvd[0], den), v = __fdiv_rn(uvd[1], den);
  float gx = __fsub_rn(__fdiv_rn(__fmul_rn(2.f, u), (float)W), 1.f);
  float gy = __fsub_rn(__fdiv_rn(__fmul_rn(2.f, v), (float)H), 1.f);
  coords[(size_t)i * 2 + 0] = __fsub_rn(__fmul_rn(__fadd_rn(gx, 1.f), (float)w * 0.5f), 0.5f);
  coords[(size_t)i * 2 + 1] = __fsub_rn(__fmul_rn(__fadd_rn(gy, 1.f), (float)h * 0.5f), 0.5f);
}

// correspondence.py:240-252: bicubic source index scale*(dst+0.5)-0.5, uv = pixel centre, xyz gather
__global__ void grid_coords_kernel(const float* __restrict__ xyz_grid, const int32_t* __restrict__ valid_idx,
                                   const int32_t* __restrict__ n_dev, int n_max, int H, int W, int h, int w,
                                   float* __restrict__ xyz, float* __restrict__ uv, float* __restrict__ coords) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  int n = n_dev ? min(*n_dev, n_max) : n_max;
  if (i >= n) return;
  int p = valid_idx ? valid_idx[i] : i;
  int y = p / W, x = p - y * W;
  const size_t HW = (size_t)H * W;
  if (xyz) {
    xyz[(size_t)i * 3 + 0] = __ldg(xyz_grid + p);
    xyz[(size_t)i * 3 + 1] = __ldg(xyz_grid + HW + p);
    xyz[(size_t)i * 3 + 2] = __ldg(xyz_grid + 2 * HW + p);
  }
  if (uv) {
    uv[(size_t)i * 2 + 0] = (float)x + 0.5f;
    uv[(size_t)i * 2 + 1] = (float)y + 0.5f;
  }
  float sx = (float)w / (float)W, sy = (float)h / (float)H;
  coords[(size_t)i * 2 + 0] = __fsub_rn(__fmul_rn(sx, (float)x + 0.5f), 0.5f);
  coords[(size_t)i * 2 + 1] = __fsub_rn(__fmul_rn(sy, (float)y + 0.5f), 0.5f);
}

// evaluate_spair_correspondence.py:71-78 + ATen CUDA grid_sampler (align_corners=True):
//   g = kp/size*2-1 ; ix = ((g+1)/2)*(w-1)
__global__ void keypoint_coords_kernel(const float* __restrict__ kps, int stride, int n, float image_size, int h,
                                       int w, float* __restrict__ coords) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float kx = __fdiv_rn(kps[(size_t)i * stride + 0], image_size);
  float ky = __fdiv_rn(kps[(size_t)i * stride + 1], image_size);
  float gx = __fsub_rn(__fmul_rn(kx, 2.f), 1.f), gy = __fsub_rn(__fmul_rn(ky, 2.f), 1.f);
  coords[(size_t)i * 2 + 0] = __fmul_rn(__fdiv_rn(__fadd_rn(gx, 1.f), 2.f), (float)(w - 1));
  coords[(size_t)i * 2 + 1] = __fmul_rn(__fdiv_rn(__fadd_rn(gy, 1.f), 2.f), (float)(h - 1));
}

// ------------------------------------------------------------------------------------------
// kernel 1
// ------------------------------------------------------------------------------------------
struct K1Params {
  const float* src;
  const float* coords;
  const int32_t* n_dev;
  int n_max, C, h, w, normalize;
  __nv_bfloat16* out_bf16;  // 16-bit rows: bf16 (fmt16 == 0, pitch C) or fp16 (fmt16 == 1, pitch C + 8: "f16c" rows)
  __nv_bfloat16* out_lo;  // 16-bit residual of the 16-bit rounding: with out_bf16 a copy of the fp32 row in 4 bytes
  float* out_f32;
  int32_t* taps;
  // ---- f16c rows (fmt16 == 1): kernel 2's fp16 operand = [fp16(row - center) | 8 augmentation columns]
  int fmt16;            // 0 = bf16, 1 = fp16 + augmentation columns
  int pitch16;          // row pitch of the fp16 rows in elements (>= C + 8; a multiple of 64 keeps kernel 2's TMA rows 128-byte aligned)
  int role;             // MV_ROLE_QUERY: aug = 3 fp16 pieces of r = row . dotvec;  MV_ROLE_TARGET: aug = (1, 1, 2^-11)
  const float* center;  // (C) or NULL: subtracted from the normalised row before the 16-bit split
  const float* dotvec;  // (C) or NULL
  const float* pixdot;  // (h*w; n for MV_SAMPLE_ROWS) or NULL: src[p] . dotvec per source row, precomputed (mv_rows_dot).  The
                        // row's dot product is then the same blend of 4 / 16 of these scalars instead of C multiply-adds
  float* row_dot;       // (n) or NULL: r in fp32
  // ---- tf32c rows: kernel 2's fp32 (tf32) operand = [tf32_round(row - center) | 8 augmentation columns], pitch pitch_op32
  float* out_op32;
  int pitch_op32;
};

constexpr float K1_LO_SCALE = 2048.f;  // the fp16 residual is stored * 2^11 so that it stays a normal number

__device__ __forceinline__ float4 ld4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void fma4(float4& a, float w, const float4& v) {
  a.x = fmaf(w, v.x, a.x);
  a.y = fmaf(w, v.y, a.y);
  a.z = fmaf(w, v.z, a.z);
  a.w = fmaf(w, v.w, a.w);
}

// Keys cubic convolution, A = -0.75 (ATen UpSample.h cubic_convolution1/2)
__device__ __forceinline__ void cubic_coeffs(float t, float c[4]) {
  const float A = -0.75f;
  float x0 = t + 1.f, x1 = t, x2 = 1.f - t, x3 = 2.f - t;
  c[0] = ((A * x0 - 5.f * A) * x0 + 8.f * A) * x0 - 4.f * A;
  c[1] = ((A + 2.f) * x1 - (A + 3.f)) * x1 * x1 + 1.f;
  c[2] = ((A + 2.f) * x2 - (A + 3.f)) * x2 * x2 + 1.f;
  c[3] = ((A * x3 - 5.f * A) * x3 + 8.f * A) * x3 - 4.f * A;
}

// ------------------------------------------------------------------------------------------
// kernel 1: teams of warps over a shared-memory window of source columns
// ------------------------------------------------------------------------------------------
// A CTA owns a range of consecutive live points and cuts it into SUB-RUNS: maximal prefixes of points that
// lie on one output row and whose taps fall into a window of source columns that fits shared memory.
//   phase S (warp 0): per point scalars (tap origin, 4 blend weights), the window, and GROUPS: up to G
//            consecutive points with the same tap origin, i.e. the same four window columns
//   phase A (all threads): fill the window in shared memory from the L2-resident channel-last map --
//            bicubic: the 4 source rows blended along y ONCE per column (every point of the sub-run has the
//            bit-identical y coordinate), bilinear: the two raw source rows (zeros outside the map)
//   phase B (a TEAM of W warps per group, warp = C / W channels): each warp loads its slice of the four
//            columns once (4 x LDS.128 per 4 channels) and blends it for all G points of the group, so the
//            shared-memory traffic per point is 1/G of a point-at-a-time loop; the rows stay in registers
//            (G x C / W values per warp); the sum of squares is 5 shuffles per point and warp plus one
//            named barrier per group among the W warps; then scale + row stores, contiguous per warp.
// History (profiles/): one CTA per point with taps in registers and a block-wide reduction issued ~37
// instructions per element (2.6 TB/s); one warp per point over the window issues ~10 (W = G = 1, still the
// configuration for C = 3072); the group form cuts the LDS count by G, worth 4 % at C = 2048 (see launch_k1).
constexpr int K1W_PMAX = 32;  // points per sub-run: one warp inspects them with a ballot
// which row outputs exist: bf16 + fp32, fp32 only, bf16 + bf16 residual, or ANY (checked at run time)
constexpr int K1W_OUT_BOTH = 0, K1W_OUT_F32 = 1, K1W_OUT_ANY = 2, K1W_OUT_SPLIT = 3;

template <int W>
struct K1WShared {
  float wt[K1W_PMAX][4];
  int off[K1W_PMAX][4];  // float offsets of the point's four columns / taps in the window
  int g_start[K1W_PMAX], g_cnt[K1W_PMAX];
  float part[2][4][4][4];  // [parity][team][point of the group][warp of the team]: partial sums of squares
  float partd[2][4][4][4]; // the same for row . dotvec
  float rd[K1W_PMAX];      // per point: (unnormalised row) . dotvec from the pixel dots (pixdot form)
  float cy[4];
  int npts, ncols, xbase, y0, ngroups;
  int cur0;  // first point of the sub-run
};

// round to nearest tf32 (10 explicit mantissa bits), ties away from zero: the value the tensor core then reads exactly
__device__ __forceinline__ float tf32_rn(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u); }
__device__ __forceinline__ float4 lds4(const float* q) { return *reinterpret_cast<const float4*>(q); }
__device__ __forceinline__ float dot4(const float4& v, float ss) {
  ss = fmaf(v.x, v.x, ss);
  ss = fmaf(v.y, v.y, ss);
  ss = fmaf(v.z, v.z, ss);
  return fmaf(v.w, v.w, ss);
}

// NITW > 0: C == 128 * NITW * W exactly; a warp holds G rows of C / W channels (G * NITW float4 per lane).
// NITW == 0: any C (multiple of 4), W = G = 1: two passes over the window (sum of squares, then values).
// PW > 0: WARP-SPECIALISED form -- the first PW warps are PRODUCERS (phases S and A of sub-run i + 1 into the second
// window) while the THREADS / 32 CONSUMER warps run phase B of sub-run i; two windows, full / empty mbarriers.  The window
// fill is bound by L2 -> SM bandwidth (128 MB of reads for a NAVI-shaped side) and the row writes by HBM: with one phase
// after the other (PW == 0) a side costs the sum, here the larger of the two.
// BULK > 0: f16c split rows leave through bulk stores: each warp stages its point's hi row (C + 8 fp16, augmentation
// columns included) and lo row (C fp16), BULK pieces of C / BULK channels at a time, in a slot of its own behind the
// window, and its lane 0 copies them to global memory with cp.async.bulk.  The warp goes on as soon as a piece is handed
// over, so the window fill of the next sub-run runs while the last rows of this one drain.
template <int MODE, int NITW, int W, int G, int OUTS, int THREADS, int MINB, int PW = 0, int BULK = 0>
__global__ void __launch_bounds__(THREADS + 32 * PW, MINB) k1_rows_kernel(K1Params p, int nslots, uint32_t c4_magic) {
  static_assert(W == 1 || W == 2 || W == 4, "team size");
  static_assert(G >= 1 && G <= 4 && (THREADS / 32) % W == 0 && (W == 1 || THREADS / 32 / W <= 4), "team layout");
  static_assert(PW == 0 || MODE != MV_SAMPLE_ROWS, "the row-copy mode has no window to produce");
  static_assert(!BULK || (W == 1 && G == 1 && NITW > 0 && OUTS == K1W_OUT_SPLIT && PW == 0 && MODE != MV_SAMPLE_ROWS),
                "bulk row stores: one warp per point, whole rows in registers, f16c split rows only");
  extern __shared__ float4 k1w_dyn[];
  constexpr int NBUF = PW > 0 ? 2 : 1;
  __shared__ K1WShared<W> shb[NBUF];
  __shared__ unsigned long long ws_full[2], ws_empty[2];
  K1WShared<W>& sh0 = shb[0];  // the consumers' partial-sum exchange lives in buffer 0's struct
  const int n = p.n_dev ? min(*p.n_dev, p.n_max) : p.n_max;
  const int C = (NITW > 0) ? NITW * W * 128 : p.C, C4 = C >> 2;
  float* winb[2] = {reinterpret_cast<float*>(k1w_dyn), reinterpret_cast<float*>(k1w_dyn) + (size_t)(PW > 0 ? nslots : 0) * C};
  const int tid = threadIdx.x, lane = tid & 31, wid_all = tid >> 5;
  const int wid = wid_all - PW;  // consumer warp index (negative for a producer warp)
  constexpr int NWARP = THREADS / 32, NTEAM = NWARP / W;
  const int team = wid / W, wsub = wid % W;
  const int cbase = wsub * (C / W);  // this warp's channel slice
  const int ppc = (n + (int)gridDim.x - 1) / (int)gridDim.x;  // from the LIVE count: no idle SMs for a small n
  const int pt_beg = min(blockIdx.x * ppc, n);
  const int pt_end = min(pt_beg + ppc, n);
  const bool has32 = (OUTS == K1W_OUT_BOTH || OUTS == K1W_OUT_F32) || (OUTS == K1W_OUT_ANY && p.out_f32 != nullptr);
  const bool has16 = (OUTS == K1W_OUT_BOTH || OUTS == K1W_OUT_SPLIT) || (OUTS == K1W_OUT_ANY && p.out_bf16 != nullptr);
  const bool haslo = (OUTS == K1W_OUT_SPLIT) || (OUTS == K1W_OUT_ANY && p.out_lo != nullptr);
  const bool normalize = p.normalize != 0;
  int parity = 0;  // of this team's group counter: double-buffers sh.part

  const bool f16c = p.fmt16 != 0;
  const size_t pitch16 = f16c ? (size_t)p.pitch16 : (size_t)C;
  const bool haspd = p.pixdot != nullptr;                    // the dot product comes from per-pixel dots: nothing in the hot loop
  const bool hasdot = p.dotvec != nullptr && !haspd;
  auto scaled = [](float4 o, float inv) {
    o.x *= inv;  // inv == 1 when not normalising: exact
    o.y *= inv;
    o.z *= inv;
    o.w *= inv;
    return o;
  };
  // fp16(o) of 4 channels and the residual * 2^11 (exact scaling): value = hi + lo * 2^-11 carries 22 mantissa bits
  auto f16c_split = [](const float4& o, uint2& hi, uint2& lo) {
    const __half2 h0 = __floats2half2_rn(o.x, o.y), h1 = __floats2half2_rn(o.z, o.w);
    hi.x = *reinterpret_cast<const uint32_t*>(&h0);
    hi.y = *reinterpret_cast<const uint32_t*>(&h1);
    const float2 l = __half22float2(h0), h = __half22float2(h1);
    const __half2 rl = __floats2half2_rn((o.x - l.x) * K1_LO_SCALE, (o.y - l.y) * K1_LO_SCALE);
    const __half2 rh = __floats2half2_rn((o.z - h.x) * K1_LO_SCALE, (o.w - h.y) * K1_LO_SCALE);
    lo.x = *reinterpret_cast<const uint32_t*>(&rl);
    lo.y = *reinterpret_cast<const uint32_t*>(&rh);
  };
  auto centred = [&](int c, float4 o) {
    if (p.center) {  // rows relative to the centre: the 16-bit rounding error scales with |row - center|
      const float4 m = ld4(p.center + c);
      o.x -= m.x;
      o.y -= m.y;
      o.z -= m.z;
      o.w -= m.w;
    }
    return o;
  };
  auto put = [&](int pt, int c, float4 o, float inv) {
    o = scaled(o, inv);
    if (has32) __stcs(reinterpret_cast<float4*>(p.out_f32 + (size_t)pt * C + c), o);
    if (p.out_op32) {  // tf32 operand rows: centred, rounded to nearest tf32 here (the tensor core would truncate)
      float4 y = o;
      if (p.center) {
        const float4 m = ld4(p.center + c);
        y.x -= m.x;
        y.y -= m.y;
        y.z -= m.z;
        y.w -= m.w;
      }
      y.x = tf32_rn(y.x);
      y.y = tf32_rn(y.y);
      y.z = tf32_rn(y.z);
      y.w = tf32_rn(y.w);
      *reinterpret_cast<float4*>(p.out_op32 + (size_t)pt * p.pitch_op32 + c) = y;
    }
    if (has16) {
      o = centred(c, o);
      uint2 pk;
      if (f16c) {
        uint2 pl;
        f16c_split(o, pk, pl);
        *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(p.out_bf16) + (size_t)pt * pitch16 + c) = pk;
        if (haslo) *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(p.out_lo) + (size_t)pt * C + c) = pl;
        return;
      }
      __nv_bfloat162 lo = __floats2bfloat162_rn(o.x, o.y), hi = __floats2bfloat162_rn(o.z, o.w);
      pk.x = *reinterpret_cast<uint32_t*>(&lo);
      pk.y = *reinterpret_cast<uint32_t*>(&hi);
      *reinterpret_cast<uint2*>(p.out_bf16 + (size_t)pt * C + c) = pk;
      if (haslo) {  // residual of the bf16 rounding, itself rounded to bf16: hi + lo carries 16 mantissa bits
        const float2 l = __bfloat1622float2(lo), h = __bfloat1622float2(hi);
        __nv_bfloat162 rl = __floats2bfloat162_rn(o.x - l.x, o.y - l.y), rh = __floats2bfloat162_rn(o.z - h.x, o.w - h.y);
        pk.x = *reinterpret_cast<uint32_t*>(&rl);
        pk.y = *reinterpret_cast<uint32_t*>(&rh);
        *reinterpret_cast<uint2*>(p.out_lo + (size_t)pt * C + c) = pk;
      }
    }
  };
  // the 8 augmentation columns of an f16c row
  auto f16c_aug = [&](float r) {
    __half a[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) a[k] = __float2half_rn(0.f);
    if (p.role == MV_ROLE_TARGET) {
      a[0] = __float2half_rn(1.f);
      a[1] = __float2half_rn(1.f);
      a[2] = __float2half_rn(1.f / K1_LO_SCALE);
    } else {
      a[0] = __float2half_rn(r);
      const float r1 = r - __half2float(a[0]);
      a[1] = __float2half_rn(r1);
      a[2] = __float2half_rn((r1 - __half2float(a[1])) * K1_LO_SCALE);
    }
    return *reinterpret_cast<const uint4*>(a);
  };
  // the augmentation columns (and the fp32 r), written by one lane per row
  auto put_aug = [&](int pt, float r) {
    if (p.row_dot) p.row_dot[pt] = r;
    if (p.out_op32) {  // three tf32-exact pieces of r against (1, 1, 1) of the target rows
      float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0;
      if (p.role == MV_ROLE_TARGET) {
        a0.x = a0.y = a0.z = 1.f;
      } else {
        a0.x = tf32_rn(r);
        a0.y = tf32_rn(r - a0.x);
        a0.z = tf32_rn(r - a0.x - a0.y);
      }
      float* q = p.out_op32 + (size_t)pt * p.pitch_op32 + C;
      *reinterpret_cast<float4*>(q) = a0;
      *reinterpret_cast<float4*>(q + 4) = a1;
    }
    if (!f16c || !has16) return;
    *reinterpret_cast<uint4*>(reinterpret_cast<__half*>(p.out_bf16) + (size_t)pt * pitch16 + C) = f16c_aug(r);
  };
  // x * (1 / max(||x||, eps)) from the per-warp partial sums of squares of the cnt rows of a group; dd (raw row .
  // dotvec) is reduced the same way and comes back as r = (normalised row) . dotvec
  auto inverse_norms = [&](float (&ss)[G], float (&inv)[G], float (&dd)[G]) {
#pragma unroll
    for (int j = 0; j < G; ++j) inv[j] = 1.f;
    if (!normalize && !hasdot) return;
#pragma unroll
    for (int j = 0; j < G; ++j) ss[j] = warp_sum(ss[j]);
    if (hasdot) {
#pragma unroll
      for (int j = 0; j < G; ++j) dd[j] = warp_sum(dd[j]);
    }
    if (W > 1) {
      if (lane == 0) {
#pragma unroll
        for (int j = 0; j < G; ++j) {
          sh0.part[parity][team][j][wsub] = ss[j];
          sh0.partd[parity][team][j][wsub] = dd[j];
        }
      }
      sm100::named_bar_sync(1 + team, W * 32);
#pragma unroll
      for (int j = 0; j < G; ++j) {
        float t = 0.f, u = 0.f;
#pragma unroll
        for (int q = 0; q < W; ++q) {  // fixed order: every warp gets the same bits
          t += sh0.part[parity][team][j][q];
          u += sh0.partd[parity][team][j][q];
        }
        ss[j] = t;
        dd[j] = u;
      }
      parity ^= 1;  // the next group's partials go to the other buffer; its barrier orders the re-use of this one
    }
    if (normalize) {
#pragma unroll
      for (int j = 0; j < G; ++j) inv[j] = __frcp_rn(fmaxf(sqrtf(ss[j]), K1_NORM_EPS));
    }
#pragma unroll
    for (int j = 0; j < G; ++j) dd[j] *= inv[j];
  };
  auto dotacc = [&](const float4& v, const float4& d, float acc) {
    acc = fmaf(v.x, d.x, acc);
    acc = fmaf(v.y, d.y, acc);
    acc = fmaf(v.z, d.z, acc);
    return fmaf(v.w, d.w, acc);
  };
  const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);

  // BULK: stage the warp's row (scaled, centred, split exactly as put / put_aug do) in BULK pieces of C / BULK channels and
  // hand each piece to the bulk-copy engine; the last piece carries the augmentation columns.  Lane 0 issues, commits
  // and waits on the slot's bulk groups.
  constexpr int CP = (NITW > 0 ? NITW * 128 : 4) / (BULK > 0 ? BULK : 1);  // channels per piece
  __half* const stage_hi = reinterpret_cast<__half*>(winb[0] + (size_t)nslots * C) + (size_t)wid_all * (2 * CP + 8);
  __half* const stage_lo = stage_hi + CP + 8;
  auto stage_row = [&](int pt, const float4* acc, float inv, float r) {
#pragma unroll
    for (int k = 0; k < (BULK > 0 ? BULK : 1); ++k) {
      if (lane == 0) sm100::bulk_wait_group_read0();  // the slot's previous piece has been read out
      __syncwarp();
#pragma unroll
      for (int i = 0; i < CP / 128; ++i) {
        const int c = (i * 32 + lane) * 4;
        uint2 hi, lo;
        f16c_split(centred(k * CP + c, scaled(acc[k * (CP / 128) + i], inv)), hi, lo);
        *reinterpret_cast<uint2*>(stage_hi + c) = hi;
        *reinterpret_cast<uint2*>(stage_lo + c) = lo;
      }
      const bool last = k == BULK - 1;
      if (lane == 0 && last) {
        if (p.row_dot) p.row_dot[pt] = r;
        *reinterpret_cast<uint4*>(stage_hi + CP) = f16c_aug(r);
      }
      sm100::fence_proxy_async_smem();  // this lane's generic-proxy writes become visible to the bulk copy
      __syncwarp();
      if (lane == 0) {
        sm100::bulk_store_1d(reinterpret_cast<__half*>(p.out_bf16) + (size_t)pt * pitch16 + k * CP, sm100::smem_u32(stage_hi),
                             (CP + (last ? 8 : 0)) * 2);
        sm100::bulk_store_1d(reinterpret_cast<__half*>(p.out_lo) + (size_t)pt * C + k * CP, sm100::smem_u32(stage_lo), CP * 2);
        sm100::bulk_commit_group();
      }
    }
  };

  if (MODE == MV_SAMPLE_ROWS) {  // rows as they are, no window: a team per row
    for (int pt = pt_beg + team; pt < pt_end; pt += NTEAM) {
      const float* row = p.src + (size_t)pt * C;
      float ss[G], inv[G], dd[G];
#pragma unroll
      for (int j = 0; j < G; ++j) ss[j] = dd[j] = 0.f;
      if (NITW > 0) {
        float4 acc[NITW > 0 ? NITW : 1];
#pragma unroll
        for (int it = 0; it < NITW; ++it) {
          acc[it] = ld4(row + cbase + (it * 32 + lane) * 4);
          ss[0] = dot4(acc[it], ss[0]);
          if (hasdot) dd[0] = dotacc(acc[it], ld4(p.dotvec + cbase + (it * 32 + lane) * 4), dd[0]);
        }
        inverse_norms(ss, inv, dd);
#pragma unroll
        for (int it = 0; it < NITW; ++it) put(pt, cbase + (it * 32 + lane) * 4, acc[it], inv[0]);
      } else {
        if (normalize || hasdot)
          for (int c = lane * 4; c < C; c += 128) {
            const float4 v = ld4(row + c);
            ss[0] = dot4(v, ss[0]);
            if (hasdot) dd[0] = dotacc(v, ld4(p.dotvec + c), dd[0]);
          }
        inverse_norms(ss, inv, dd);
        for (int c = lane * 4; c < C; c += 128) put(pt, c, ld4(row + c), inv[0]);
      }
      if (lane == 0 && wsub == 0) put_aug(pt, haspd ? __ldg(p.pixdot + pt) * inv[0] : dd[0]);
    }
    return;
  }

  constexpr bool CUBIC = (MODE == MV_SAMPLE_BICUBIC_CLAMP);
  const int max_cols = CUBIC ? nslots : (nslots >> 1);
  const int max_dx = max_cols - (CUBIC ? 4 : 2);  // tap origins x0 .. x0 + max_dx share one window

  // ---- phase S (one warp): the sub-run that starts at point `cur`
  auto phase_S = [&](K1WShared<W>& sh, int cur) {
    {
      const int pt = cur + lane;
      const bool live = pt < pt_end;
      float2 xy = make_float2(0.f, 0.f);
      if (live) xy = __ldg(reinterpret_cast<const float2*>(p.coords) + pt);
      const float fx = floorf(xy.x), fy = floorf(xy.y);
      const int x0 = (int)fx, y0 = (int)fy;
      const int x0f = __shfl_sync(0xffffffffu, x0, 0), y0f = __shfl_sync(0xffffffffu, y0, 0);
      const uint32_t iyf = __shfl_sync(0xffffffffu, __float_as_uint(xy.y), 0);
      const int dx = x0 - x0f;
      bool ok = live && y0 == y0f && dx >= 0 && dx <= max_dx;
      if (CUBIC) ok = ok && (__float_as_uint(xy.y) == iyf);  // one y blend serves the whole sub-run
      const uint32_t bal = __ballot_sync(0xffffffffu, ok);
      const int npts = (bal == 0xffffffffu) ? 32 : (__ffs(~bal) - 1);  // leading run of ok lanes (lane 0 always is)
      const int dxmax = __reduce_max_sync(0xffffffffu, lane < npts ? dx : 0);
      const int ncols = dxmax + (CUBIC ? 4 : 2);
      // groups: consecutive points with the same tap origin (=> the same window columns), at most G of them
      const int x0p = __shfl_up_sync(0xffffffffu, x0, 1);
      const uint32_t segm = __ballot_sync(0xffffffffu, lane < npts && (lane == 0 || x0 != x0p));
      const int seg_start = 31 - __clz(segm & (0xffffffffu >> (31 - lane)));  // last segment head at or before this lane
      const bool head = lane < npts && ((lane - seg_start) % G == 0);
      const uint32_t headm = __ballot_sync(0xffffffffu, head);
      if (head) {
        const int gid = __popc(headm & ((1u << lane) - 1u));
        const uint32_t later = (lane == 31) ? 0u : (headm >> (lane + 1));
        const int end = later ? lane + __ffs(later) : npts;
        sh.g_start[gid] = lane;
        sh.g_cnt[gid] = end - lane;
      }
      if (lane < npts) {
        if (p.taps) {
          p.taps[2 * (size_t)pt] = x0;
          p.taps[2 * (size_t)pt + 1] = y0;
        }
        if (CUBIC) {
          float cx[4];
          cubic_coeffs(xy.x - fx, cx);
#pragma unroll
          for (int j = 0; j < 4; ++j) {  // window slot s holds source column clamp(x0f - 1 + s)
            sh.wt[lane][j] = cx[j];
            sh.off[lane][j] = (dx + j) * C;
          }
        } else {
          // ATen GridSamplerKernel.cpp (bilinear, zeros): w = ix - floor(ix), e = 1 - w, n = iy - floor(iy), s = 1 - n
          const float ww = xy.x - fx, we = 1.f - ww, wn = xy.y - fy, ws = 1.f - wn;
          sh.wt[lane][0] = ws * we;  // nw
          sh.wt[lane][1] = ws * ww;  // ne
          sh.wt[lane][2] = wn * we;  // sw
          sh.wt[lane][3] = wn * ww;  // se
          sh.off[lane][0] = dx * C;
          sh.off[lane][1] = (dx + 1) * C;
          sh.off[lane][2] = (ncols + dx) * C;
          sh.off[lane][3] = (ncols + dx + 1) * C;
        }
      }
      if (haspd && lane < npts) {
        // (unnormalised row) . dotvec = the row's own blend applied to the per-pixel dots
        float r = 0.f;
        if (CUBIC) {
          float cx[4], cyl[4];
          cubic_coeffs(xy.x - fx, cx);
          cubic_coeffs(xy.y - fy, cyl);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int xx = min(max(x0 - 1 + i, 0), p.w - 1);
            float yb = 0.f;
#pragma unroll
            for (int j = 0; j < 4; ++j) yb = fmaf(cyl[j], __ldg(p.pixdot + min(max(y0 - 1 + j, 0), p.h - 1) * p.w + xx), yb);
            r = fmaf(cx[i], yb, r);
          }
        } else {
          const float ww = xy.x - fx, we = 1.f - ww, wn = xy.y - fy, ws = 1.f - wn;
          const float wt4[4] = {ws * we, ws * ww, wn * we, wn * ww};
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int xx = x0 + (k & 1), yy = y0 + (k >> 1);
            if (xx >= 0 && xx < p.w && yy >= 0 && yy < p.h) r = fmaf(wt4[k], __ldg(p.pixdot + yy * p.w + xx), r);
          }
        }
        sh.rd[lane] = r;
      }
      if (lane == 0) {
        sh.cur0 = cur;
        sh.npts = npts;
        sh.ncols = ncols;
        sh.xbase = CUBIC ? x0 - 1 : x0;
        sh.y0 = y0;
        sh.ngroups = __popc(headm);
        if (CUBIC) cubic_coeffs(xy.y - fy, sh.cy);
      }
    }
  };

  // ---- phase A (threads t of nt): one flat loop over (window slot, 4 channels), several items = many loads in flight per thread
  auto phase_A = [&](const K1WShared<W>& sh, float* win, int t, int nt) {
    const int ncols = sh.ncols, xbase = sh.xbase, y0 = sh.y0;
    if (CUBIC) {
      const float cy0 = sh.cy[0], cy1 = sh.cy[1], cy2 = sh.cy[2], cy3 = sh.cy[3];
      const size_t rs = (size_t)p.w * C;
      const float* r0 = p.src + (size_t)min(max(y0 - 1, 0), p.h - 1) * rs;
      const float* r1 = p.src + (size_t)min(max(y0, 0), p.h - 1) * rs;
      const float* r2 = p.src + (size_t)min(max(y0 + 1, 0), p.h - 1) * rs;
      const float* r3 = p.src + (size_t)min(max(y0 + 2, 0), p.h - 1) * rs;
      const int items = ncols * C4;
#pragma unroll 4  // 16 loads in flight per thread; 32 measured slower (28.7 vs 27.5 us NAVI side, same box)
      for (int idx = t; idx < items; idx += nt) {
        const int s = (int)__umulhi((uint32_t)idx, c4_magic);  // idx / C4
        const int c = (idx - s * C4) * 4;
        const int xo = min(max(xbase + s, 0), p.w - 1) * C + c;
        const float4 a = ld4(r0 + xo), b = ld4(r1 + xo), cc = ld4(r2 + xo), d = ld4(r3 + xo);
        float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
        fma4(o, cy0, a);
        fma4(o, cy1, b);
        fma4(o, cy2, cc);
        fma4(o, cy3, d);
        *reinterpret_cast<float4*>(win + idx * 4) = o;  // slot s, channel c  ==  float offset s * C + c
      }
    } else {
      const int items = 2 * ncols * C4;
#pragma unroll 8
      for (int idx = t; idx < items; idx += nt) {
        const int slot = (int)__umulhi((uint32_t)idx, c4_magic);  // r * ncols + s
        const int c = (idx - slot * C4) * 4;
        const int r = slot >= ncols ? 1 : 0;
        const int yy = y0 + r, xx = xbase + slot - r * ncols;
        const bool in = yy >= 0 && yy < p.h && xx >= 0 && xx < p.w;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (in) v = ld4(p.src + ((size_t)yy * p.w + xx) * C + c);
        *reinterpret_cast<float4*>(win + idx * 4) = v;
      }
    }
  };

  // ---- phase B (the consumer warps, in teams)
  auto phase_B = [&](K1WShared<W>& sh, const float* win) {
    const int cur = sh.cur0, ngroups = sh.ngroups;
    for (int g = team; g < ngroups; g += NTEAM) {
      const int t0 = sh.g_start[g], cnt = sh.g_cnt[g];
      const float* q0 = win + sh.off[t0][0] + cbase;
      const float* q1 = win + sh.off[t0][1] + cbase;
      const float* q2 = win + sh.off[t0][2] + cbase;
      const float* q3 = win + sh.off[t0][3] + cbase;
      float wt[G][4];
#pragma unroll
      for (int j = 0; j < G; ++j) {
        const int t = t0 + min(j, cnt - 1);  // rows beyond cnt repeat the last point and are not stored
#pragma unroll
        for (int k = 0; k < 4; ++k) wt[j][k] = sh.wt[t][k];
      }
      auto blend = [&](int j, const float4& a, const float4& b, const float4& c, const float4& d) {
        float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
        fma4(o, wt[j][0], a);
        fma4(o, wt[j][1], b);
        fma4(o, wt[j][2], c);
        fma4(o, wt[j][3], d);
        return o;
      };
      float ss[G], inv[G], dd[G];
#pragma unroll
      for (int j = 0; j < G; ++j) ss[j] = dd[j] = 0.f;
      if (NITW > 0) {
        float4 acc[G][NITW > 0 ? NITW : 1];
#pragma unroll
        for (int it = 0; it < NITW; ++it) {
          const int c = (it * 32 + lane) * 4;
          const float4 a = lds4(q0 + c), b = lds4(q1 + c), cc = lds4(q2 + c), d = lds4(q3 + c);
          const float4 dv = hasdot ? ld4(p.dotvec + cbase + c) : zero4;
#pragma unroll
          for (int j = 0; j < G; ++j) {
            acc[j][it] = blend(j, a, b, cc, d);
            ss[j] = dot4(acc[j][it], ss[j]);
            if (hasdot) dd[j] = dotacc(acc[j][it], dv, dd[j]);
          }
        }
        inverse_norms(ss, inv, dd);
        if (BULK) {
          stage_row(cur + t0, acc[0], inv[0], haspd ? sh.rd[t0] * inv[0] : dd[0]);
          continue;
        }
#pragma unroll
        for (int j = 0; j < G; ++j) {
          if (j < cnt) {
#pragma unroll
            for (int it = 0; it < NITW; ++it) put(cur + t0 + j, cbase + (it * 32 + lane) * 4, acc[j][it], inv[j]);
            if (lane == 0 && wsub == 0) put_aug(cur + t0 + j, haspd ? sh.rd[t0 + j] * inv[j] : dd[j]);
          }
        }
      } else {  // W == G == 1
        if (normalize || hasdot)
          for (int c = lane * 4; c < C; c += 128) {
            const float4 v = blend(0, lds4(q0 + c), lds4(q1 + c), lds4(q2 + c), lds4(q3 + c));
            ss[0] = dot4(v, ss[0]);
            if (hasdot) dd[0] = dotacc(v, ld4(p.dotvec + c), dd[0]);
          }
        inverse_norms(ss, inv, dd);
        for (int c = lane * 4; c < C; c += 128)
          put(cur + t0, c, blend(0, lds4(q0 + c), lds4(q1 + c), lds4(q2 + c), lds4(q3 + c)), inv[0]);
        if (lane == 0) put_aug(cur + t0, haspd ? sh.rd[t0] * inv[0] : dd[0]);
      }
    }
  };

  if (PW == 0) {  // one phase after the other, the whole CTA in each
    int cur = pt_beg;
    while (cur < pt_end) {  // uniform across the CTA
      if (wid == 0) phase_S(shb[0], cur);
      __syncthreads();
      phase_A(shb[0], winb[0], tid, THREADS);
      __syncthreads();
      phase_B(shb[0], winb[0]);
      __syncthreads();  // the window and the per-point scalars are rewritten by the next sub-run
      cur += shb[0].npts;
    }
    if (BULK && lane == 0) sm100::bulk_wait_group0();  // the staging slots stay allocated until the rows are written
    return;
  }

  // ---- warp-specialised driver
  using namespace sm100;
  if (tid == 0) {
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_u32(&ws_full[b]), PW);      // one arrival per producer warp
      mbar_init(smem_u32(&ws_empty[b]), NWARP);  // one per consumer warp
    }
    mbar_fence_init();
  }
  __syncthreads();
  if (wid_all < PW) {
    int cur = pt_beg;
    for (uint32_t it = 0;; ++it) {
      const int b = (int)(it & 1u);
      if (it >= 2) mbar_wait(smem_u32(&ws_empty[b]), ((it >> 1) - 1u) & 1u);  // the consumers released this buffer
      if (wid_all == 0) {
        if (cur < pt_end) phase_S(shb[b], cur);
        else if (lane == 0) shb[b].npts = 0;  // end marker
      }
      named_bar_sync(15, PW * 32);  // producers only
      const int npts = shb[b].npts;
      if (npts > 0) phase_A(shb[b], winb[b], tid, PW * 32);
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&ws_full[b]));
      if (npts == 0) break;
      cur += npts;
    }
  } else {
    for (uint32_t it = 0;; ++it) {
      const int b = (int)(it & 1u);
      mbar_wait(smem_u32(&ws_full[b]), (it >> 1) & 1u);
      if (shb[b].npts == 0) break;
      phase_B(shb[b], winb[b]);
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&ws_empty[b]));
    }
  }
}


// ------------------------------------------------------------------------------------------
// centre of a set of rows: mu = mean_p rows[p] / max(||rows[p]||, eps) over every `step`-th row.  Any vector near the
// mean DIRECTION of the normalised rows works as the centre of f16c rows (the ranking is exact for every choice; the
// fp16 rounding error of kernel 2's operands scales with |row - mu|).
// ------------------------------------------------------------------------------------------
// one CTA of 4 warps per row: the row's channels are split over the warps (short dependent-load chains; these small kernels sit
// on the critical path of a synchronous helper call), partial sums added in a fixed order
__device__ __forceinline__ float block4_sum(float v, float* sm4) {
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) sm4[threadIdx.x >> 5] = v;
  __syncthreads();
  return (sm4[0] + sm4[1]) + (sm4[2] + sm4[3]);
}

__global__ void __launch_bounds__(128) center_invnorm_kernel(const float* __restrict__ rows, int C, int n_max,
                                                             const int32_t* __restrict__ n_dev, int step, float* __restrict__ inv) {
  __shared__ float sm4[4];
  const int n = n_dev ? min(*n_dev, n_max) : n_max;
  const int cnt = (n + step - 1) / step;
  const int q = blockIdx.x;
  if (q >= cnt) return;
  const float* r = rows + (size_t)q * step * C;
  float ss = 0.f;
  for (int c = threadIdx.x * 4; c < C; c += 512) ss = dot4(ld4(r + c), ss);
  ss = block4_sum(ss, sm4);
  if (threadIdx.x == 0) inv[q] = 1.f / fmaxf(sqrtf(ss), K1_NORM_EPS);
}

// out[p] = rows[p] . vec (one CTA of 4 warps per row): the per-pixel dots of the pixdot form
__global__ void __launch_bounds__(128) rows_dot_kernel(const float* __restrict__ rows, int C, int n, const float* __restrict__ vec,
                                                       float* __restrict__ out) {
  __shared__ float sm4[4];
  const int q = blockIdx.x;
  if (q >= n) return;
  const float* r = rows + (size_t)q * C;
  float acc = 0.f;
  for (int c = threadIdx.x * 4; c < C; c += 512) {
    const float4 v = ld4(r + c), d = ld4(vec + c);
    acc = fmaf(v.x, d.x, acc);
    acc = fmaf(v.y, d.y, acc);
    acc = fmaf(v.z, d.z, acc);
    acc = fmaf(v.w, d.w, acc);
  }
  acc = block4_sum(acc, sm4);
  if (threadIdx.x == 0) out[q] = acc;
}

// block = 32 channel quads x 16 row groups: group g sums rows q = g, g + 16, ... (independent loads, 4 in flight), the 16
// partial sums are added in a fixed order -> deterministic
__global__ void __launch_bounds__(512) center_mean_kernel(const float* __restrict__ rows, int C, int n_max,
                                                          const int32_t* __restrict__ n_dev, int step,
                                                          const float* __restrict__ inv, float* __restrict__ mu) {
  __shared__ float4 part[16][32];
  const int n = n_dev ? min(*n_dev, n_max) : n_max;
  const int cnt = (n + step - 1) / step;
  const int cq = threadIdx.x & 31, g = threadIdx.x >> 5;
  const int c = (blockIdx.x * 32 + cq) * 4;
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  if (c < C) {
#pragma unroll 4
    for (int q = g; q < cnt; q += 16) fma4(a, __ldg(inv + q), ld4(rows + (size_t)q * step * C + c));
  }
  part[g][cq] = a;
  __syncthreads();
  if (g == 0 && c < C) {
    float4 t = part[0][cq];
#pragma unroll
    for (int k = 1; k < 16; ++k) {
      t.x += part[k][cq].x;
      t.y += part[k][cq].y;
      t.z += part[k][cq].z;
      t.w += part[k][cq].w;
    }
    const float s = cnt > 0 ? 1.f / (float)cnt : 0.f;
    *reinterpret_cast<float4*>(mu + c) = make_float4(t.x * s, t.y * s, t.z * s, t.w * s);
  }
}

template <int MODE, int NITW, int W, int G, int OUTS, int THREADS, int MINB, int PW = 0, int BULK = 0>
int launch_k1_inst(const K1Params& p, cudaStream_t st) {
  const int C = p.C;
  // the bulk-store form's staging slots, one per warp: a piece of the hi row (C / BULK + 8 fp16) + of the lo row (C / BULK fp16)
  const size_t stage = BULK ? (size_t)(THREADS / 32) * (2 * C / (BULK > 0 ? BULK : 1) + 8) * 2 : 0;
  // window bytes per CTA: MINB CTAs per SM share 227 KB (minus ~3 KB static and 1 KB reserved each); the warp-specialised
  // form holds two windows of 108 KB; the bulk-store form gives the window what its staging slots leave of 110 KB
  const int budget = BULK ? (int)((110 << 10) - stage) : (PW > 0 ? 108 : (MINB >= 3 ? 72 : (MINB == 2 ? 108 : 216))) << 10;
  int nslots = budget / (C * 4);
  if (nslots < 4) nslots = 4;    // C <= 8192: 4 slots = 128 KB, one CTA per SM
  if (nslots > 40) nslots = 40;  // more than any 32-point sub-run can use
  const size_t smem = (MODE == MV_SAMPLE_ROWS) ? 0 : (size_t)(PW > 0 ? 2 : 1) * nslots * C * 4 + stage;
  int grid = mv_sm_count() * MINB;
  if (grid > p.n_max) grid = p.n_max;
  if (grid < 1) grid = 1;
  auto kern = k1_rows_kernel<MODE, NITW, W, G, OUTS, THREADS, MINB, PW, BULK>;
  static size_t opted[MV_MAX_DEVICES];  // per instantiation and device: the attribute belongs to the device function
  size_t& opted_in = opted[mv_device_slot()];
  if (opted_in < (44u << 10)) opted_in = 44 << 10;
  if (smem > opted_in) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
      mv_set_error("mv_k1_sample_normalize: cannot opt in to %zu bytes of shared memory: %s", smem,
                   cudaGetErrorString(e));
      return (int)e;
    }
    opted_in = smem;
  }
  const uint32_t C4 = (uint32_t)p.C / 4;
  const uint32_t magic = (uint32_t)((0x100000000ull + C4 - 1) / C4);  // idx / C4 == umulhi(idx, magic) for idx * C4 < 2^32
  kern<<<grid, THREADS + 32 * PW, smem, st>>>(p, nslots, magic);
  MV_LAUNCH_CHECK();
  return MV_OK;
}

template <int MODE>
int launch_k1(const K1Params& p, cudaStream_t st) {
  const int C = p.C;
  int outs = K1W_OUT_ANY;
  if (p.out_f32 && p.out_bf16 && !p.out_lo) outs = K1W_OUT_BOTH;
  else if (p.out_f32 && !p.out_bf16 && !p.out_lo) outs = K1W_OUT_F32;
  else if (!p.out_f32 && p.out_bf16 && p.out_lo) outs = K1W_OUT_SPLIT;
#define K1W_CASE(CC, NITW, W, GG, THREADS, MINB)                                                                      \
  if (C == CC) {                                                                                                      \
    constexpr int G = (MODE == MV_SAMPLE_ROWS) ? 1 : GG;                                                              \
    if (outs == K1W_OUT_BOTH) return launch_k1_inst<MODE, NITW, W, G, K1W_OUT_BOTH, THREADS, MINB>(p, st);            \
    if (outs == K1W_OUT_F32) return launch_k1_inst<MODE, NITW, W, G, K1W_OUT_F32, THREADS, MINB>(p, st);              \
    if (outs == K1W_OUT_SPLIT) return launch_k1_inst<MODE, NITW, W, G, K1W_OUT_SPLIT, THREADS, MINB>(p, st);          \
  }
  // a warp holds G rows of C / W channels.  Measured on B200 (tools/k1_probe.py, split rows): C = 2048 (8x bilinear)
  // 39.6 us with teams of 4 warps x 4 points vs 41.4 us point-at-a-time; C = 3072 (4x bicubic, ~12-17 points per
  // CTA) 31.5 us with teams -- the 72 KB window of a 3-CTA/SM layout splits the short runs -- vs 27.4 us with one
  // warp per point and the whole row (96 registers) in a 108 KB window, so that shape keeps the latter.
  // C = 3072, one CTA per SM with a 216 KB window (MVMATCH_K1_WIDE=1): 30 % less L2 traffic, measured SLOWER (33.7 vs 31.6 us)
  static const bool wide = getenv("MVMATCH_K1_WIDE") && atoi(getenv("MVMATCH_K1_WIDE")) != 0;
  if (wide) {
    K1W_CASE(3072, 24, 1, 1, 384, 1)
  }
  // warp-specialised form (MVMATCH_K1_WS=1, sampling modes only): 4 producer warps + 8 consumer warps, one CTA per SM.
  // Measured on B200 (bench.py --k1-only, same box): NAVI-shaped side 40.7 us vs 35.1 us, ScanNet-shaped side 80.0 vs 53.8 us:
  // at 159-168 registers per thread one CTA per SM leaves 8 consumer warps where the two classic CTAs have 12-16, and 128
  // producer threads keep a third of the window-fill loads in flight -- the overlap does not pay for either.  OFF by default.
  static const bool ws = getenv("MVMATCH_K1_WS") && atoi(getenv("MVMATCH_K1_WS")) != 0;
  if (ws && MODE != MV_SAMPLE_ROWS && outs == K1W_OUT_SPLIT) {
#define K1WS_CASE(CC, NITW, W, GG)                                                                                   \
  if (C == CC) return launch_k1_inst<(MODE == MV_SAMPLE_ROWS ? MV_SAMPLE_BILINEAR_ZEROS : MODE), NITW, W, GG, K1W_OUT_SPLIT, 256, 1, 4>(p, st);
    K1WS_CASE(3072, 24, 1, 1)
    K1WS_CASE(2048, 4, 4, 4)
    K1WS_CASE(768, 6, 1, 4)
#undef K1WS_CASE
  }
  // C = 3072 bicubic f16c split rows (the NAVI-shaped side): rows leave through bulk stores.  With STG rows (the form
  // below) the two CTAs of an SM start together, fill their windows (L2 -> SM reads), THEN write their rows (HBM), one
  // ~17-point sub-run each, and a warp stalls on its own row stores.  Here each warp stages its row in two halves (6160 B
  // slot: 1536 + 8 hi fp16, 1536 lo fp16) and goes on once a half has been read out of the slot; after its last row it
  // goes straight to the next sub-run's window fill while the copies drain.  Shared memory per CTA, 2 CTAs per SM (168
  // registers, 12 warps as before): 6 slots x 6160 B + a 6-column window (72 KB: 12 points per sub-run, ~2 sub-runs per
  // CTA) = 108 KB + 2.4 KB static.  Measured on B200 at 1000 W (bench.py --k1-only, NAVI-shaped side, same box,
  // alternating): 33.5-34.0 us vs 35.0-35.2 us with STG rows.  Rejected on the same box: whole-row slots (12 x 12304 B) with one CTA of
  // 12 warps per SM and a 6-column window, 37.5-38.0 us (the sub-runs of one CTA run strictly one after another); thirds
  // or quarters of a row with a 7-column window, 35.3-35.4 us.
  if constexpr (MODE == MV_SAMPLE_BICUBIC_CLAMP) {
    if (C == 3072 && outs == K1W_OUT_SPLIT && p.fmt16 && !p.out_op32 &&
        ((reinterpret_cast<uintptr_t>(p.out_bf16) | reinterpret_cast<uintptr_t>(p.out_lo)) & 15) == 0)
      return launch_k1_inst<MODE, 24, 1, 1, K1W_OUT_SPLIT, 192, 2, 0, 2>(p, st);
  }
  K1W_CASE(768, 6, 1, 4, 128, 3)    // ViT-B
  K1W_CASE(1024, 4, 2, 4, 256, 2)   // ViT-L
  K1W_CASE(2048, 4, 4, 4, 256, 2)   // ResNet-50 layer4
  K1W_CASE(1536, 6, 2, 2, 256, 2)   // ViT-S 4-block concat
  K1W_CASE(3072, 24, 1, 1, 192, 2)  // ViT-B 4-block concat
  K1W_CASE(4096, 8, 4, 2, 256, 2)   // ViT-L 4-block concat
#undef K1W_CASE
  return launch_k1_inst<MODE, 0, 1, 1, K1W_OUT_ANY, 256, 2>(p, st);
}

Mat3 load_mat3(const float* host) {
  Mat3 m;
  for (int i = 0; i < 9; ++i) m.m[i] = host[i];
  return m;
}

// host pointer -> by value; device pointer -> the kernel reads it (returns the device pointer, else nullptr)
const float* split_mat3_arg(const float* p, Mat3* by_value) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) == cudaSuccess && (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged)) {
    *by_value = Mat3{};
    return p;
  }
  (void)cudaGetLastError();  // unregistered host memory reports an error on old drivers
  *by_value = load_mat3(p);
  return nullptr;
}

}  // namespace

extern "C" {

int mv_chw_to_hwc(const float* src_chw, float* dst_hwc, int C, int hw, int prenorm, float* norm_scratch,
                  mv_stream_t stream) {
  MV_REQUIRE(src_chw && dst_hwc, MV_E_ARG, "mv_chw_to_hwc: null pointer");
  MV_REQUIRE(C > 0 && hw > 0, MV_E_ARG, "mv_chw_to_hwc: C and hw must be positive");
  MV_REQUIRE(!prenorm || norm_scratch, MV_E_ARG, "mv_chw_to_hwc: prenorm needs norm_scratch (hw floats)");
  cudaStream_t st = mv_cuda_stream(stream);
  if (prenorm) {
    pixel_norm_kernel<<<(hw + 31) / 32, dim3(32, 8), 0, st>>>(src_chw, norm_scratch, C, hw);
    MV_LAUNCH_CHECK();
  }
  const float* norm = prenorm ? norm_scratch : nullptr;
  const bool vec = (hw % 4 == 0) && (C % 4 == 0) && ((reinterpret_cast<uintptr_t>(src_chw) & 15) == 0) &&
                   ((reinterpret_cast<uintptr_t>(dst_hwc) & 15) == 0);
  if (vec) {
    dim3 grid((hw + 63) / 64, (C + 63) / 64);
    chw_to_hwc_vec_kernel<<<grid, 256, 0, st>>>(src_chw, dst_hwc, C, hw, norm);
  } else {
    dim3 grid((hw + 31) / 32, (C + 31) / 32);
    chw_to_hwc_kernel<<<grid, dim3(32, 8), 0, st>>>(src_chw, dst_hwc, C, hw, norm);
  }
  MV_LAUNCH_CHECK();
  return MV_OK;
}

int mv_feat_to_hwc_f32(const void* src, int dtype, int channel_last, int C, int hw, float* dst_hwc, mv_stream_t stream) {
  MV_REQUIRE(src && dst_hwc, MV_E_ARG, "mv_feat_to_hwc_f32: null pointer");
  MV_REQUIRE(C > 0 && hw > 0, MV_E_ARG, "mv_feat_to_hwc_f32: C and hw must be positive");
  MV_REQUIRE(dtype == MV_FEAT_F32 || dtype == MV_FEAT_BF16 || dtype == MV_FEAT_F16, MV_E_ARG,
             "mv_feat_to_hwc_f32: unknown feature dtype %d", dtype);
  cudaStream_t st = mv_cuda_stream(stream);
  if (dtype == MV_FEAT_F32) {
    if (channel_last) {
      MV_CUDA(cudaMemcpyAsync(dst_hwc, src, (size_t)C * hw * sizeof(float), cudaMemcpyDeviceToDevice, st));
      return MV_OK;
    }
    return mv_chw_to_hwc(static_cast<const float*>(src), dst_hwc, C, hw, 0, nullptr, stream);
  }
  const size_t total = (size_t)C * hw;
  if (channel_last) {
    const unsigned blocks = (unsigned)((total + 255) / 256);
    if (dtype == MV_FEAT_BF16) widen_kernel<<<blocks, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(src), dst_hwc, total);
    else widen_kernel<<<blocks, 256, 0, st>>>(static_cast<const __half*>(src), dst_hwc, total);
  } else {
    dim3 grid((hw + 31) / 32, (C + 31) / 32);
    if (dtype == MV_FEAT_BF16)
      chw_to_hwc_widen_kernel<<<grid, dim3(32, 8), 0, st>>>(static_cast<const __nv_bfloat16*>(src), dst_hwc, C, hw);
    else chw_to_hwc_widen_kernel<<<grid, dim3(32, 8), 0, st>>>(static_cast<const __half*>(src), dst_hwc, C, hw);
  }
  MV_LAUNCH_CHECK();
  return MV_OK;
}

int mv_compact_valid(const float* z, int z_stride, int n, int32_t* valid_idx, int32_t* n_valid,
                     mv_stream_t stream) {
  MV_REQUIRE(z && valid_idx && n_valid, MV_E_ARG, "mv_compact_valid: null pointer");
  MV_REQUIRE(n >= 0 && n <= (1 << 20) && z_stride >= 1, MV_E_RANGE, "mv_compact_valid: n must be in [0, 2^20]");
  compact_valid_kernel<<<n > 0 ? (n + COMPACT_CHUNK - 1) / COMPACT_CHUNK : 1, COMPACT_CHUNK, 0, mv_cuda_stream(stream)>>>(z, z_stride, n, valid_idx, n_valid);
  MV_LAUNCH_CHECK();
  return MV_OK;
}

int mv_geom_backproject(const float* depth, int H, int W, const float* Kinv_host, float* xyz_all,
                        mv_stream_t stream) {
  MV_REQUIRE(depth && Kinv_host && xyz_all, MV_E_ARG, "mv_geom_backproject: null pointer");
  MV_REQUIRE(H > 0 && W > 0, MV_E_ARG, "mv_geom_backproject: H and W must be positive");
  int n = H * W;
  Mat3 Ki;
  const float* Ki_dev = split_mat3_arg(Kinv_host, &Ki);
  backproject_kernel<<<(n + 255) / 256, 256, 0, mv_cuda_stream(stream)>>>(depth, H, W, Ki, Ki_dev, xyz_all);
  MV_LAUNCH_CHECK();
  return MV_OK;
}

int mv_geom_project_coords(const float* xyz_all, const int32_t* valid_idx, const int32_t* n_dev, int n_max,
                           const float* K_host, int H, int W, int h, int w, float* xyz, float* coords,
                           mv_stream_t stream) {
  MV_REQUIRE(xyz_all && K_host && xyz && coords, MV_E_ARG, "mv_geom_project_coords: null pointer");
  MV_REQUIRE(n_max >= 0 && H > 0 && W > 0 && h > 0 && w > 0, MV_E_ARG, "mv_geom_project_coords: bad sizes");
  if (n_max == 0) return MV_OK;
  Mat3 Km;
  const float* K_dev = split_mat3_arg(K_host, &Km);
  project_coords_kernel<<<(n_max + 255) / 256, 256, 0, mv_cuda_stream(stream)>>>(
      xyz_all, valid_idx, n_dev, n_max, Km, K_dev, H, W, h, w, xyz, coords);
  MV_LAUNCH_CHECK();
  return MV_OK;
}

int mv_geom_grid_coords(const float* xyz_grid, const int32_t* valid_idx, const int32_t* n_dev, int n_max, int H,
                        int W, int h, int w, float* xyz, float* uv, float* coords, mv_stream_t stream) {
  MV_REQUIRE(coords && (xyz_grid || !xyz), MV_E_ARG, "mv_geom_grid_coords: null pointer");
  MV_REQUIRE(n_max >= 0 && H > 0 && W > 0 && h > 0 && w > 0, MV_E_ARG, "mv_geom_grid_coords: bad sizes");
  if (n_max == 0) return MV_OK;
  grid_coords_kernel<<<(n_max + 255) / 256, 256, 0, mv_cuda_stream(stream)>>>(xyz_grid, valid_idx, n_dev, n_max, H,
                                                                             W, h, w, xyz, uv, coords);
  MV_LAUNCH_CHECK();
  return MV_OK;
}

int mv_geom_keypoint_coords(const float* kps, int kp_stride, int n, float image_size, int h, int w,
                            float* coords, mv_stream_t stream) {
  MV_REQUIRE(kps && coords, MV_E_ARG, "mv_geom_keypoint_coords: null pointer");
  MV_REQUIRE(n >= 0 && kp_stride >= 2 && h > 0 && w > 0 && image_size > 0.f, MV_E_ARG,
             "mv_geom_keypoint_coords: bad sizes");
  if (n == 0) return MV_OK;
  keypoint_coords_kernel<<<(n + 127) / 128, 128, 0, mv_cuda_stream(stream)>>>(kps, kp_stride, n, image_size, h, w,
                                                                            coords);
  MV_LAUNCH_CHECK();
  return MV_OK;
}

int mv_rows_center(const float* rows, int C, int n_max, const int32_t* n_dev, int step, float* inv_scratch, float* mu,
                   mv_stream_t stream) {
  MV_REQUIRE(rows && inv_scratch && mu, MV_E_ARG, "mv_rows_center: null pointer");
  MV_REQUIRE(C > 0 && C % 4 == 0 && n_max > 0 && step > 0, MV_E_ARG, "mv_rows_center: C %% 4 == 0, n_max > 0 and step > 0 required");
  MV_REQUIRE(((reinterpret_cast<uintptr_t>(rows) | reinterpret_cast<uintptr_t>(mu)) & 15) == 0, MV_E_ALIGN,
             "mv_rows_center: rows and mu must be 16-byte aligned");
  cudaStream_t st = mv_cuda_stream(stream);
  const int cnt = (n_max + step - 1) / step;
  center_invnorm_kernel<<<cnt, 128, 0, st>>>(rows, C, n_max, n_dev, step, inv_scratch);
  MV_LAUNCH_CHECK();
  center_mean_kernel<<<(C / 4 + 31) / 32, 512, 0, st>>>(rows, C, n_max, n_dev, step, inv_scratch, mu);
  MV_LAUNCH_CHECK();
  return MV_OK;
}

int mv_rows_dot(const float* rows, int C, int n, const float* vec, float* out, mv_stream_t stream) {
  MV_REQUIRE(rows && vec && out, MV_E_ARG, "mv_rows_dot: null pointer");
  MV_REQUIRE(C > 0 && C % 4 == 0 && n >= 0, MV_E_ARG, "mv_rows_dot: C %% 4 == 0 and n >= 0 required");
  MV_REQUIRE(((reinterpret_cast<uintptr_t>(rows) | reinterpret_cast<uintptr_t>(vec)) & 15) == 0, MV_E_ALIGN,
             "mv_rows_dot: rows and vec must be 16-byte aligned");
  if (n == 0) return MV_OK;
  rows_dot_kernel<<<n, 128, 0, mv_cuda_stream(stream)>>>(rows, C, n, vec, out);
  MV_LAUNCH_CHECK();
  return MV_OK;
}

static int k1_entry(const char* who, int mode, const float* src, int C, int h, int w, const float* coords, const int32_t* n_dev,
                    int n_max, int normalize, int fmt16, int pitch16, int role, const float* center, const float* dotvec,
                    const float* pixdot, uint16_t* out16,
                    uint16_t* out16_lo, float* out_f32, float* row_dot, int32_t* taps, mv_stream_t stream, float* out_op32 = nullptr,
                    int pitch_op32 = 0) {
  MV_REQUIRE(src && (out16 || out_f32), MV_E_ARG, "%s: null src or no output", who);
  MV_REQUIRE(!out_op32 || (pitch_op32 >= C + 8 && pitch_op32 % 4 == 0 && (reinterpret_cast<uintptr_t>(out_op32) & 15) == 0), MV_E_ALIGN,
             "%s: the tf32 operand rows need a 16-byte aligned base and a pitch >= C + 8 that is a multiple of 4", who);
  MV_REQUIRE(mode == MV_SAMPLE_BILINEAR_ZEROS || mode == MV_SAMPLE_BICUBIC_CLAMP || mode == MV_SAMPLE_ROWS,
             MV_E_ARG, "%s: unknown mode %d", who, mode);
  MV_REQUIRE(mode == MV_SAMPLE_ROWS || (coords && h > 0 && w > 0), MV_E_ARG,
             "%s: sampling modes need coords and a map size", who);
  MV_REQUIRE(C > 0 && C % 8 == 0 && C <= 8192, MV_E_RANGE, "%s: C=%d must be a multiple of 8, <= 8192", who, C);
  MV_REQUIRE(n_max >= 0, MV_E_ARG, "%s: negative n_max", who);
  MV_REQUIRE(role == MV_ROLE_QUERY || role == MV_ROLE_TARGET, MV_E_ARG, "%s: unknown role %d", who, role);
  MV_REQUIRE(!fmt16 || (pitch16 >= C + 8 && pitch16 % 8 == 0), MV_E_ALIGN, "%s: pitch %d must be >= C + 8 and a multiple of 8", who, pitch16);
  MV_REQUIRE((reinterpret_cast<uintptr_t>(src) & 15) == 0, MV_E_ALIGN, "%s: src must be 16-byte aligned", who);
  MV_REQUIRE(!out_f32 || (reinterpret_cast<uintptr_t>(out_f32) & 15) == 0, MV_E_ALIGN, "%s: out_f32 must be 16-byte aligned", who);
  MV_REQUIRE(!out16 || (reinterpret_cast<uintptr_t>(out16) & (fmt16 ? 15 : 7)) == 0, MV_E_ALIGN,
             "%s: the 16-bit rows must be %d-byte aligned", who, fmt16 ? 16 : 8);
  MV_REQUIRE(!out16_lo || (out16 && (reinterpret_cast<uintptr_t>(out16_lo) & 7) == 0), MV_E_ARG,
             "%s: the residual plane needs the 16-bit rows and 8-byte alignment", who);
  MV_REQUIRE((!center || (reinterpret_cast<uintptr_t>(center) & 15) == 0) && (!dotvec || (reinterpret_cast<uintptr_t>(dotvec) & 15) == 0),
             MV_E_ALIGN, "%s: center / dotvec must be 16-byte aligned", who);
  if (n_max == 0) return MV_OK;

  K1Params p;
  p.src = src;
  p.coords = coords;
  p.n_dev = n_dev;
  p.n_max = n_max;
  p.C = C;
  p.h = h;
  p.w = w;
  p.normalize = normalize;
  p.out_bf16 = reinterpret_cast<__nv_bfloat16*>(out16);
  p.out_lo = reinterpret_cast<__nv_bfloat16*>(out16_lo);
  p.out_f32 = out_f32;
  p.taps = taps;
  p.fmt16 = fmt16;
  p.pitch16 = pitch16;
  p.role = role;
  p.center = center;
  p.dotvec = dotvec;
  p.pixdot = pixdot;
  p.row_dot = row_dot;
  p.out_op32 = out_op32;
  p.pitch_op32 = pitch_op32;

  cudaStream_t st = mv_cuda_stream(stream);
  if (mode == MV_SAMPLE_BILINEAR_ZEROS) return launch_k1<MV_SAMPLE_BILINEAR_ZEROS>(p, st);
  if (mode == MV_SAMPLE_BICUBIC_CLAMP) return launch_k1<MV_SAMPLE_BICUBIC_CLAMP>(p, st);
  return launch_k1<MV_SAMPLE_ROWS>(p, st);
}

int mv_k1_sample_normalize(int mode, const float* src, int C, int h, int w, const float* coords,
                           const int32_t* n_dev, int n_max, int normalize, uint16_t* out_bf16, uint16_t* out_bf16_lo, float* out_f32,
                           int32_t* taps, mv_stream_t stream) {
  return k1_entry("mv_k1_sample_normalize", mode, src, C, h, w, coords, n_dev, n_max, normalize, 0, C, MV_ROLE_QUERY, nullptr, nullptr, nullptr,
                  out_bf16, out_bf16_lo, out_f32, nullptr, taps, stream);
}

int mv_k1_sample_f16c(int mode, const float* src, int C, int h, int w, const float* coords, const int32_t* n_dev, int n_max,
                      int normalize, int role, const float* center, const float* dotvec, const float* pixdot, uint16_t* out_f16, int pitch,
                      uint16_t* out_f16_lo, float* out_f32, float* row_dot, int32_t* taps, mv_stream_t stream) {
  MV_REQUIRE(out_f16, MV_E_ARG, "mv_k1_sample_f16c: out_f16 is required");
  return k1_entry("mv_k1_sample_f16c", mode, src, C, h, w, coords, n_dev, n_max, normalize, 1, pitch, role, center, dotvec, pixdot, out_f16,
                  out_f16_lo, out_f32, row_dot, taps, stream);
}

int mv_k1_sample_tf32c(int mode, const float* src, int C, int h, int w, const float* coords, const int32_t* n_dev, int n_max,
                       int normalize, int role, const float* center, const float* dotvec, const float* pixdot, float* out_op, int pitch,
                       float* out_f32, int32_t* taps, mv_stream_t stream) {
  MV_REQUIRE(out_op && out_f32, MV_E_ARG, "mv_k1_sample_tf32c: out_op and out_f32 are required");
  return k1_entry("mv_k1_sample_tf32c", mode, src, C, h, w, coords, n_dev, n_max, normalize, 0, C, role, center, dotvec, pixdot, nullptr,
                  nullptr, out_f32, nullptr, taps, stream, out_op, pitch);
}

}  // extern "C"
