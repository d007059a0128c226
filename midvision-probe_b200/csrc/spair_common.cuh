// spair_common.cuh -- pieces shared by the two SPair batch implementations: spair_batch.cu (one CTA per pair: the first
// form, and the streaming form for h*w <= 256) and spair_tiled.cu (pixel tiles of a pair spread over many CTAs, for larger
// maps).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

#include "common.cuh"

constexpr float SPB_NORM_EPS = 1e-12f;  // F.normalize default eps

// element type T of the maps: float, or the __nv_bfloat16 / __half output of an autocast backbone.  Every 16-bit value is
// an fp32 value (widening is exact), and every one is also exactly a tf32 value (8 / 11 significant bits, fp32's exponent
// range): the kernels widen on load from global or shared memory and then run the fp32 arithmetic unchanged.
__device__ __forceinline__ float sp_f32(float v) { return v; }
__device__ __forceinline__ float sp_f32(__nv_bfloat16 v) { return __bfloat162float(v); }
__device__ __forceinline__ float sp_f32(__half v) { return __half2float(v); }
// two neighbouring values, one 8-byte (float) or 4-byte (16-bit) aligned load
__device__ __forceinline__ float2 sp_f32x2(const float* v) { return *reinterpret_cast<const float2*>(v); }
__device__ __forceinline__ float2 sp_f32x2(const __nv_bfloat16* v) {
  return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(v));
}
__device__ __forceinline__ float2 sp_f32x2(const __half* v) { return __half22float2(*reinterpret_cast<const __half2*>(v)); }

struct SpairBatchParams {
  const void* feats;  // (B, 2, C, h, w) of the launch's element type
  const float* kps_i;  // (B, K, stride)
  const float* kps_j;
  const float* thresh_scale;  // (B)
  int B, C, h, w, K, stride;
  float image_size, pck;
  int32_t* pred;  // (B, K)
  float* error_same;
  float* error_nn;
  int32_t* index_nn;
  unsigned long long* hits;
  unsigned long long* confusion;
  int conf_dim;
  int stages, cc, rs;  // streaming form: ring depth, channels per half slot, row stride in floats (set by the launcher)
};

// key point k of kps ((x, y) in image pixels at kps[k * stride]) -> its four bilinear taps: kp / size * 2 - 1 -> ((g + 1) / 2) * (size - 1)
// (align_corners=True).  put(t, weight, pixel) for t = nw, ne, sw, se: weight 0 for a tap outside the map (zero padding),
// pixel index clamped into the map.  The arithmetic of the taps in spair_batch.cu's kernels, which keep their inline copy
// (their compiled code stays as it is); the same operations give the same taps, so every form keeps the same key points.
template <class Put>
__device__ __forceinline__ void spair_taps(const float* kps, int k, int stride, float image_size, int h, int w, Put&& put) {
  const float kx = __fdiv_rn(kps[(size_t)k * stride + 0], image_size);
  const float ky = __fdiv_rn(kps[(size_t)k * stride + 1], image_size);
  const float gx = __fsub_rn(__fmul_rn(kx, 2.f), 1.f), gy = __fsub_rn(__fmul_rn(ky, 2.f), 1.f);
  const float ix = __fmul_rn(__fdiv_rn(__fadd_rn(gx, 1.f), 2.f), (float)(w - 1));
  const float iy = __fmul_rn(__fdiv_rn(__fadd_rn(gy, 1.f), 2.f), (float)(h - 1));
  const float fx = floorf(ix), fy = floorf(iy);
  const int x0 = (int)fx, y0 = (int)fy;
  const float ww = ix - fx, we = 1.f - ww, wn = iy - fy, ws = 1.f - wn;
  const float wt[4] = {ws * we, ws * ww, wn * we, wn * ww};
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    const int xx = x0 + (t & 1), yy = y0 + (t >> 1);
    const bool in = xx >= 0 && xx < w && yy >= 0 && yy < h;
    put(t, in ? wt[t] : 0.f, min(max(yy, 0), h - 1) * w + min(max(xx, 0), w - 1));
  }
}

// m16n8k8 tf32 tensor-core step (legacy warp-level MMA: the heat map of a pair is 196 x 20 x 768, far below a tcgen05 tile)
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// x = hi + lo with hi exactly representable in tf32 (the tensor core drops the low 13 mantissa bits of its operands);
// hi*hi + hi*lo + lo*hi carries ~21 mantissa bits ("3xTF32")
// (the AND sits in an asm block: seen by the compiler, it is dropped for the MMA operand -- the tensor core ignores those bits --
// and kept for the subtraction, and the raw values are then MOVed into the operand's register quad: three instructions per
// value instead of two)
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  asm("and.b32 %0, %1, 0xffffe000;" : "=r"(hi) : "r"(__float_as_uint(x)));
  lo = __float_as_uint(x - __uint_as_float(hi));
}

// where q[c][k] of a chunk sits in its buffer.  Tensor-core pass: per K step (8 channels) and N tile j (8 key points) the
// B fragment of lane (g, t) -- channels t and t + 4 of key point 8 j + g, each already split into its tf32 halves -- is one
// float4 {hi(t), hi(t + 4), lo(t), lo(t + 4)} (the register pairs the MMA takes, no moves), lanes in order: a conflict-free
// LDS.128, and the split is done once per value by step Q instead of once per warp by step H.
template <int KT, bool MMA>
__device__ __forceinline__ int sps_q_off(int c, int k) {
  if (!MMA) return c * KT + k;
  constexpr int NT8 = (KT + 7) / 8;
  const int c8 = c & 7;
  return (((c >> 3) * NT8 + (k >> 3)) * 32 + ((k & 7) << 2) + (c8 & 3)) * 4 + (c8 >> 2);
}
template <int KT, bool MMA>
constexpr int sps_q_floats(int cc) {  // one q buffer
  return MMA ? (cc / 8) * ((KT + 7) / 8) * 128 : cc * KT;
}

// host side
int spair_heatmap_terms();  // 3 or 1: mv_spair_set_heatmap_terms
// the tiled form (spair_tiled.cu): workspace bytes for B pairs of C channels and K key points, and the launches
size_t spair_tiled_workspace_bytes(int B, int C, int K);
template <typename T>
int spair_tiled_launch(const SpairBatchParams& p, void* workspace, cudaStream_t st);
