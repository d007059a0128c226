// spair_batch.cu -- SPair-71k keypoint transfer for a BATCH of image pairs in one launch.
//
//   mv_spair_match_batch   per pair: bilinear key-point features of the normalised map, K x (h*w) heat map with
//                          the per-pixel normalisation folded in, arg-max, key-point error matrix, PCK counts
//                          -- one CTA per pair, fp32 arithmetic throughout
//   mv_spair_match_batch_typed   the same on an fp32, bf16 or fp16 map: 16-bit maps are read as they are and widened
//                          on the chip, with the fp32 results of the widened map bit for bit
//
// Reference behaviour being reproduced (file:line in /root/reference):
//   evaluate_spair_correspondence.py:59     feats = F.normalize(feats, p=2, dim=1)
//   evaluate_spair_correspondence.py:71-79  key points / image size -> NDC -> grid_sample(bilinear, align_corners=True)
//   evaluate_spair_correspondence.py:82-83  heatmaps = einsum("k f, f h w -> k h w"); argmax_2d(...) / w
//   evaluate_spair_correspondence.py:86-98  error matrix, validity, error_same / error_nn        (spair_score.cuh)
//   evaluate_spair_correspondence.py:108, :115-121  loop over pairs, confusion matrix, recall
//
// Why a separate kernel: one pair is 2 * K * h*w * C = 6 MFLOP (K = 20, 14 x 14, C = 768) -- a 128-row
// tensor-core tile would be 84 % padding and the ten launches of the per-pair path (kernels 1-3) are pure
// launch latency.  Here the maps are read straight from the backbone's (B, 2, C, h, w) output -- 1.2 MB per
// pair, the HBM floor; image i a second time, from L2 where it is still there (1.33-1.49 MB of DRAM reads per
// pair measured) -- the heat map lives in registers and nothing but K integers per pair is written, so the
// path is bounded by HBM, not by launches.
#include <math_constants.h>
#include <stdlib.h>

#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <type_traits>

#include "common.cuh"
#include "sm100_ptx.cuh"
#include "spair_score.cuh"

namespace {

constexpr int SPB_THREADS = 256;
constexpr int SPB_MAX_HW = 1 << 20;  // pixels per feature map (2500 at the reference's 800 x 800 input)
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

// dynamic shared memory: q[C][KT], the key-point features of the current tile
// blockDim.x = min(SPB_THREADS, h*w rounded up to a warp): thread = pixel in the heat-map pass, so a 14 x 14 map
// runs 7 warps with 87 % of the lanes busy instead of 8 warps with 77 %.
template <typename T, int KT>
__global__ void __launch_bounds__(SPB_THREADS) spair_batch_kernel(SpairBatchParams p) {
  extern __shared__ float4 spb_dyn[];
  __shared__ SpairScoreShared score;
  __shared__ int s_pred[64];
  __shared__ float s_wt[64][4];   // bilinear weight / max(||f_i[tap]||, eps); 0 for a tap outside the map (zero padding)
  __shared__ int s_tap[64][4];    // pixel index of the tap (clamped into the map)
  __shared__ float s_ss[64][4];   // sum of squares of f_i at the tap
  __shared__ float s_bv[SPB_THREADS / 32][KT];
  __shared__ int s_bi[SPB_THREADS / 32][KT];
  const int C = p.C, hw = p.h * p.w, K = p.K;
  float* q = reinterpret_cast<float*>(spb_dyn);
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int nthr = blockDim.x, nwarp = nthr >> 5;

  for (int b = blockIdx.x; b < p.B; b += gridDim.x) {
    const T* fi = static_cast<const T*>(p.feats) + (size_t)b * 2 * C * hw;
    const T* fj = fi + (size_t)C * hw;
    const float* ki = p.kps_i + (size_t)b * K * p.stride;
    const float* kj = p.kps_j + (size_t)b * K * p.stride;

    // ---- key-point taps: kp / size * 2 - 1 -> ((g + 1) / 2) * (size - 1)  (align_corners=True) ----
    if (tid < K) {
      const float kx = __fdiv_rn(ki[(size_t)tid * p.stride + 0], p.image_size);
      const float ky = __fdiv_rn(ki[(size_t)tid * p.stride + 1], p.image_size);
      const float gx = __fsub_rn(__fmul_rn(kx, 2.f), 1.f), gy = __fsub_rn(__fmul_rn(ky, 2.f), 1.f);
      const float ix = __fmul_rn(__fdiv_rn(__fadd_rn(gx, 1.f), 2.f), (float)(p.w - 1));
      const float iy = __fmul_rn(__fdiv_rn(__fadd_rn(gy, 1.f), 2.f), (float)(p.h - 1));
      const float fx = floorf(ix), fy = floorf(iy);
      const int x0 = (int)fx, y0 = (int)fy;
      const float ww = ix - fx, we = 1.f - ww, wn = iy - fy, ws = 1.f - wn;
      const float wt[4] = {ws * we, ws * ww, wn * we, wn * ww};  // nw, ne, sw, se
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const int xx = x0 + (t & 1), yy = y0 + (t >> 1);
        const bool in = xx >= 0 && xx < p.w && yy >= 0 && yy < p.h;
        s_wt[tid][t] = in ? wt[t] : 0.f;
        s_tap[tid][t] = min(max(yy, 0), p.h - 1) * p.w + min(max(xx, 0), p.w - 1);
        s_ss[tid][t] = 0.f;
      }
    }
    __syncthreads();
    // ---- ||f_i|| at the 4K tap pixels only: (tap, channel slice) per thread, 16 independent loads in flight ----
    {
      const int ntap = 4 * K;
      const int slices = max(1, nthr / ntap);
      for (int item = tid; item < ntap * slices; item += nthr) {
        const int tp = item % ntap, sl = item / ntap;
        const T* src = fi + s_tap[tp >> 2][tp & 3];
        float ss = 0.f;
#pragma unroll 16
        for (int c = sl; c < C; c += slices) {
          const float v = sp_f32(__ldg(src + (size_t)c * hw));
          ss = fmaf(v, v, ss);
        }
        atomicAdd(&s_ss[tp >> 2][tp & 3], ss);
      }
    }
    __syncthreads();
    if (tid < 4 * K) {  // fold 1 / max(||f_i[tap]||, eps) into the blend weight
      const int k = tid >> 2, t = tid & 3;
      s_wt[k][t] = __fdiv_rn(s_wt[k][t], fmaxf(sqrtf(s_ss[k][t]), SPB_NORM_EPS));
    }
    __syncthreads();

    for (int k0 = 0; k0 < K; k0 += KT) {
      const int kt = min(KT, K - k0);
      // ---- q[c][k] = sum_t wt * f_i[c][tap] / max(||f_i[tap]||, eps): the grid_sample of the normalised map ----
#pragma unroll 4
      for (int idx = tid; idx < C * KT; idx += nthr) {
        const int c = idx / KT, k = idx - c * KT;
        const int kk = k0 + min(k, kt - 1);
        const T* src = fi + (size_t)c * hw;
        float acc = sp_f32(__ldg(src + s_tap[kk][0])) * s_wt[kk][0];
        acc = fmaf(sp_f32(__ldg(src + s_tap[kk][1])), s_wt[kk][1], acc);
        acc = fmaf(sp_f32(__ldg(src + s_tap[kk][2])), s_wt[kk][2], acc);
        acc = fmaf(sp_f32(__ldg(src + s_tap[kk][3])), s_wt[kk][3], acc);
        q[idx] = (k < kt) ? acc : 0.f;
      }
      __syncthreads();

      // ---- heat[k][px] = (sum_c q[c][k] * f_j[c][px]) / max(||f_j[px]||, eps), f_j read ONCE: the norm is
      //      accumulated in the same pass; running arg-max per thread ----
      float bestv[KT];
      int besti[KT];
#pragma unroll
      for (int k = 0; k < KT; ++k) {
        bestv[k] = -CUDART_INF_F;
        besti[k] = 0x7fffffff;
      }
      for (int px = tid; px < hw; px += nthr) {
        float acc[KT];
#pragma unroll
        for (int k = 0; k < KT; ++k) acc[k] = 0.f;
        float ss = 0.f;
        const T* col = fj + px;
        int c0 = 0;
        for (; c0 + 16 <= C; c0 += 16) {
          float v[16];
#pragma unroll
          for (int u = 0; u < 16; ++u) v[u] = sp_f32(__ldg(col + (size_t)(c0 + u) * hw));  // 16 loads in flight
#pragma unroll
          for (int u = 0; u < 16; ++u) {
            ss = fmaf(v[u], v[u], ss);
            const float4* qc = reinterpret_cast<const float4*>(q + (size_t)(c0 + u) * KT);
#pragma unroll
            for (int k4 = 0; k4 < KT / 4; ++k4) {
              const float4 qq = qc[k4];  // same address in every lane: broadcast
              acc[4 * k4 + 0] = fmaf(qq.x, v[u], acc[4 * k4 + 0]);
              acc[4 * k4 + 1] = fmaf(qq.y, v[u], acc[4 * k4 + 1]);
              acc[4 * k4 + 2] = fmaf(qq.z, v[u], acc[4 * k4 + 2]);
              acc[4 * k4 + 3] = fmaf(qq.w, v[u], acc[4 * k4 + 3]);
            }
          }
        }
        for (; c0 < C; ++c0) {
          const float v = sp_f32(__ldg(col + (size_t)c0 * hw));
          ss = fmaf(v, v, ss);
#pragma unroll
          for (int k = 0; k < KT; ++k) acc[k] = fmaf(q[(size_t)c0 * KT + k], v, acc[k]);
        }
        const float nrm = fmaxf(sqrtf(ss), SPB_NORM_EPS);
#pragma unroll
        for (int k = 0; k < KT; ++k) {
          const float hv = __fdiv_rn(acc[k], nrm);
          if (hv > bestv[k]) {  // pixels are visited in ascending order: the first maximum wins
            bestv[k] = hv;
            besti[k] = px;
          }
        }
      }
#pragma unroll
      for (int k = 0; k < KT; ++k) {
        float v = bestv[k];
        int i = besti[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const float ov = __shfl_xor_sync(0xffffffffu, v, o);
          const int oi = __shfl_xor_sync(0xffffffffu, i, o);
          if (ov > v || (ov == v && oi < i)) {
            v = ov;
            i = oi;
          }
        }
        if (lane == 0) {
          s_bv[wid][k] = v;
          s_bi[wid][k] = i;
        }
      }
      __syncthreads();
      if (tid < kt) {
        float v = s_bv[0][tid];
        int i = s_bi[0][tid];
        for (int wq = 1; wq < nwarp; ++wq) {
          const float ov = s_bv[wq][tid];
          const int oi = s_bi[wq][tid];
          if (ov > v || (ov == v && oi < i)) {
            v = ov;
            i = oi;
          }
        }
        i = (i == 0x7fffffff) ? 0 : i;  // an all-NaN heat map: torch.argmax would return a NaN position; we return 0
        s_pred[k0 + tid] = i;
        if (p.pred) p.pred[(size_t)b * K + k0 + tid] = i;
      }
      __syncthreads();  // q, s_bv are rewritten by the next tile
    }

    spair_score_block(score, s_pred, K, p.w, ki, kj, p.stride, p.image_size, __ldg(p.thresh_scale + b), p.pck, nullptr,
                      p.error_same ? p.error_same + (size_t)b * K : nullptr,
                      p.error_nn ? p.error_nn + (size_t)b * K : nullptr,
                      p.index_nn ? p.index_nn + (size_t)b * K : nullptr, p.hits, p.confusion, p.conf_dim);
  }
}


// ------------------------------------------------------------------------------------------
// the streaming form (the default where it applies: h*w <= 256, C % 8 == 0, 16-byte aligned maps)
// ------------------------------------------------------------------------------------------
// A pair's two maps are ONE contiguous 2 * C * h*w * 4 byte block.  A producer warp streams it through a ring of
// shared-memory slots with 1-D bulk copies (cp.async.bulk, completion on an mbarrier) and runs up to `stages` slots -- across
// the passes and across pairs -- ahead of the 8 consumer warps, which only ever read shared memory:
//   pass N    slots of 2*cc channels of image i: ||f_i[px]||^2 of every pixel (the key points' taps need their norms first)
//   pass QH   slots of cc channels of image i AND the same cc channels of image j: the consumers blend the key-point vectors
//             q of these channels from the i half (step Q), then add the channels' share of the heat map from the j half
//             (step H).  q therefore lives for one slot only (two small buffers) instead of C x KT floats (61 KB at C = 768,
//             which used to cap the ring at 25-37 KB per CTA): the ring takes the shared memory, 75 KB per CTA in flight.
// Image i is read twice, 0.6 MB apart per CTA, 178 MB apart over the chip's 296 CTAs -- more than the 126 MB L2, and a cyclic
// walk through a smaller LRU-like cache hits nothing (ncu before: L2 hit rate 0.4 %, 1.8 MB of DRAM reads per pair against
// 1.2 MB algorithmic).  SPS_QREV: pass QH walks the channels from the last chunk to the first, so that its first i reads are
// the most recently cached ones; SPS_HINTS: pass N loads with L2 evict_last, everything that is read for the last time with
// evict_first (ncu after: 1.33 MB per pair).
// Rows (one channel = h*w floats) keep their h*w pitch in the slot (one bulk copy per half slot).  Padding them to a
// conflict-free pitch needs one 784-byte bulk copy per row and measured 2.59 M pairs/s against 3.18 M for the unpadded rows of
// the same build: small copies cost more than the two-way bank conflicts of the A-fragment loads.
//
// Measured history (SPair-shaped, 2048-2368 pairs per launch, one B200; profiles/r2_spair_diag.txt): round 1 per-thread global
// loads 1.81 M pairs/s; ring of 4 x 8 channels + tensor-core heat map 2.60 M; 2 x 16 channels 2.79 M; score matrix out of static
// shared memory, 3 x 16 channels 3.17 M, 2 x 24 channels 3.35-3.42 M; pass QH with pre-split B fragments 3.29 M; A fragments by
// LDS.64 into the operand quads 3.57 M; dead tile skipped, branch-free K steps 3.64-3.68 M (67-68 % of the HBM copy peak; the
// memory side alone -- consumers that only wait and release, -DSPS_NULL=1 -- runs 4.69 M); 16 consumer warps per CTA: slower
// (2.16 M at the 4 x 8 ring).
#ifndef SPS_CONS_N
#define SPS_CONS_N 256
#endif
constexpr int SPS_CONS = SPS_CONS_N;        // consumer threads: thread = pixel in pass N
constexpr int SPS_WARPS = SPS_CONS / 32;    // each owns 32 pixels (two m16 tiles) in the tensor-core pass
#ifndef SPS_QWARPS
#define SPS_QWARPS 0  // n > 0: n warps that do nothing but step Q, one chunk ahead of step H (0: the eight consumer warps do both).
// Measured: 2 Q warps (11 warps per CTA, 80 registers) 3.48 M pairs/s, 1 Q warp (96 registers; it becomes the critical path)
// 3.03 M, against 3.64 M for 0 -- kept behind the switch with its tests (the parity tests pass in all three builds)
#endif
constexpr int SPS_QW = SPS_QWARPS;
constexpr int SPS_THREADS = SPS_CONS + 32 * SPS_QW + 32;  // + one producer warp
constexpr int SPS_QH = SPS_CONS + 32 * SPS_QW;            // the threads that meet on the q buffers' barriers
static_assert(SPS_CONS == 256, "32 pixels per consumer warp, h*w <= 256");
constexpr int SPS_MAX_STAGES = 8;
#ifndef SPS_CC_N
#define SPS_CC_N 24
#endif
constexpr int SPS_CC = SPS_CC_N;  // channels per half slot (a multiple of 8: the tensor-core pass takes 8 per K step)
static_assert(SPS_CC % 8 == 0 && SPS_CC >= 8, "whole K steps");
#ifndef SPS_CTAS
#define SPS_CTAS 2  // CTAs per SM the kernel is built for (registers) and the launcher plans for (shared memory)
#endif
#ifndef SPS_NULL
#define SPS_NULL 0  // diagnostic build: 1 = consumers only wait and release (the memory side alone), 2 = no step H, 3 = no step Q
#endif
#ifndef SPS_QREV
#define SPS_QREV 1
#endif
#ifndef SPS_HINTS
#define SPS_HINTS 1
#endif

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
// LDS.128, and the split is done once per value by step Q instead of once per warp by step H.  Columns beyond KT stay zero
// from the start of the kernel.
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

// MMA: the heat-map step on the tensor cores -- pixels on M (16 per tile, 2 tiles per warp), key points on N (8 per tile),
// 8 channels per K step, 3xTF32 -- instead of 21 FFMA + 6 LDS per channel and pixel.
// TERMS: 3 = 3xTF32 (fp32-grade heat map, the default), 1 = one tf32 MMA per tile (mv_spair_set_heatmap_terms(1): operands
// rounded to 10 mantissa bits, the north star's "tf32 inputs, fp32 accumulation" -- arg-max equal wherever the fp32 top-2 gap
// of the heat map exceeds 1e-3)
// T = __nv_bfloat16 / __half: the slots hold the 16-bit rows as they are in global memory (half the bytes of a slot, twice
// the ring stages), and pass N, step Q and step H widen what they read.  The channel chunks, their order and each thread's
// channel order are those of T = float, so every fp32 sum is the same sum: the outputs are those of the fp32 kernel on the
// widened map, bit for bit.  Step H's A operand (the map value) is exactly a tf32 value, its 3xTF32 low half zero: the
// lo * hi MMA, whose products are all zero, and the A split are skipped.
template <typename T, int KT, bool MMA, int TERMS = 3>
__global__ void __launch_bounds__(SPS_THREADS, SPS_CTAS) spair_stream_kernel(SpairBatchParams p) {
  using namespace sm100;
  extern __shared__ __align__(16) float4 sps_dyn[];
  __shared__ int s_pred[64];
  __shared__ float s_wt[64][4];
  __shared__ int s_tap[64][4];
  __shared__ float s_bv[SPS_WARPS][KT];
  __shared__ int s_bi[SPS_WARPS][KT];
  __shared__ __align__(8) unsigned long long full[SPS_MAX_STAGES], empty[SPS_MAX_STAGES];
  constexpr bool REV = SPS_QREV && MMA;  // the CUDA-core form keeps the channel order (and the bits) of the first form
  constexpr bool F32 = std::is_same<T, float>::value;
  const int C = p.C, hw = p.h * p.w, K = p.K, rs = hw;
  constexpr int cc = SPS_CC;
  const int nstage = p.stages;
  const int slot_elems = 2 * cc * rs;  // a multiple of 8: slots and the q buffers after them stay 16-byte aligned
  T* ring = reinterpret_cast<T*>(sps_dyn);                          // [stages][2 * cc rows][rs]
  float* qbuf = reinterpret_cast<float*>(ring + (size_t)nstage * slot_elems);  // [2][cc][KT]
  float* pix_ss = qbuf + 2 * sps_q_floats<KT, MMA>(cc);             // [hw]
  float* score_mem = pix_ss + ((hw + 3) & ~3);                      // [K][K + 1] errors, 2 counters
  const SpairScoreView score{score_mem, K + 1, reinterpret_cast<unsigned int*>(score_mem + K * (K + 1))};
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int nchunk = (C + cc - 1) / cc;
  const int nkt = (K + KT - 1) / KT;  // key-point tiles: pass QH repeats per tile
  const bool vec2 = (hw & 1) == 0;  // rows 8-byte aligned: step H reads its A fragments with LDS.64

  if (tid == 0) {
    for (int s = 0; s < nstage; ++s) {
      mbar_init(smem_u32(&full[s]), 1);
      mbar_init(smem_u32(&empty[s]), SPS_WARPS + SPS_QW);
    }
    mbar_fence_init();
  }
  __syncthreads();

  if (wid == SPS_WARPS + SPS_QW) {
    // ===================================== producer warp =====================================
    int stage = 0;
    uint32_t phase = 0;
    // L2 eviction priorities (SPS_HINTS): 1 = what is read again keeps (evict_last), what is read for the last time streams
    // (evict_first); 2 = only the streaming half, the rest at the normal priority
    const uint64_t pol_keep = SPS_HINTS == 1 ? L2_EVICT_LAST : L2_EVICT_NORMAL;
    const uint64_t pol_stream = SPS_HINTS ? L2_EVICT_FIRST : L2_EVICT_NORMAL;
    // rows [c0, c0 + rows) of one map into a slot at float offset `at`
    // (rows * hw * sizeof(T) bytes: a multiple of 16 for every chunk, the tail included, as C and cc are multiples of 8)
    auto rows_in = [&](const T* map, int c0, int rows, int at, uint64_t pol) {
      bulk_load_1d_hint(smem_u32(ring + (size_t)stage * slot_elems + at), map + (size_t)c0 * hw,
                        (uint32_t)(rows * hw) * (uint32_t)sizeof(T), smem_u32(&full[stage]), pol);
    };
    if (lane != 0) return;
    for (int b = blockIdx.x; b < p.B; b += gridDim.x) {
      const T* fi = static_cast<const T*>(p.feats) + (size_t)b * 2 * C * hw;
      const T* fj = fi + (size_t)C * hw;
      for (int c0 = 0; c0 < C; c0 += 2 * cc) {  // pass N
        const int rows = min(2 * cc, C - c0);
        mbar_wait(smem_u32(&empty[stage]), phase ^ 1u);
        mbar_arrive_expect_tx(smem_u32(&full[stage]), (uint32_t)(rows * hw) * (uint32_t)sizeof(T));
        rows_in(fi, c0, rows, 0, pol_keep);
        if (++stage == nstage) { stage = 0; phase ^= 1u; }
      }
      for (int kt = 0; kt < nkt; ++kt) {  // pass QH per key-point tile
        const uint64_t pol_i = kt + 1 < nkt ? pol_keep : pol_stream, pol_j = pol_i;
        for (int cq = 0; cq < nchunk; ++cq) {
          const int c0 = (REV ? nchunk - 1 - cq : cq) * cc, rows = min(cc, C - c0);
          mbar_wait(smem_u32(&empty[stage]), phase ^ 1u);
          mbar_arrive_expect_tx(smem_u32(&full[stage]), (uint32_t)(2 * rows * hw) * (uint32_t)sizeof(T));
          rows_in(fi, c0, rows, 0, pol_i);
          rows_in(fj, c0, rows, cc * rs, pol_j);
          if (++stage == nstage) { stage = 0; phase ^= 1u; }
        }
      }
    }
    return;
  }

  // ===================================== consumers =====================================
  int stage = 0;
  uint32_t phase = 0;
  auto cons_sync = [] { asm volatile("bar.sync 1, %0;" ::"n"(SPS_CONS) : "memory"); };
  auto release = [&] {  // this warp is done with the current slot
    __syncwarp();
    if (lane == 0) mbar_arrive(smem_u32(&empty[stage]));
    if (++stage == nstage) { stage = 0; phase ^= 1u; }
  };
  // named barriers between the Q warps and the H warps (SPS_QW > 0): 2 = the pair's blend weights are folded, 3 + b = q buffer b
  // is full, 5 + b = q buffer b is free again; 7 = the Q warps among themselves.  `g` counts the chunks of this CTA (the same
  // sequence in both roles): chunk g uses buffer g & 1.
  auto bar_sync = [](int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); };
  auto bar_arrive = [](int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); };
  constexpr int QF = sps_q_floats<KT, MMA>(cc);
  unsigned g_chunk = 0;
  const unsigned n_chunks_cta = blockIdx.x < (unsigned)p.B ? (unsigned)((p.B - 1 - blockIdx.x) / gridDim.x + 1) * nkt * nchunk : 0u;

  if (SPS_QW > 0 && wid >= SPS_WARPS) {
    // ===================================== Q warps =====================================
    // step Q of chunk g while the H warps are still on chunk g - 1: lane = (key point, channel group), the key point's four
    // taps and folded weights in registers for the whole tile
    constexpr int QT = 32 * (SPS_QW > 0 ? SPS_QW : 1), G = QT / KT;
    const int ql = tid - SPS_CONS, k = ql % KT, cg = ql / KT;
    const bool q_on = ql < G * KT;
    for (int i = ql; i < 2 * QF; i += QT) qbuf[i] = 0.f;
    bar_sync(7, QT);
    for (int b = blockIdx.x; b < p.B; b += gridDim.x) {
      for (int c0 = 0; c0 < C; c0 += 2 * cc) {  // pass N belongs to the H warps
        mbar_wait(smem_u32(&full[stage]), phase);
        release();
      }
      bar_sync(2, SPS_QH);
      for (int k0 = 0; k0 < K; k0 += KT) {
        const int kt = min(KT, K - k0), kk = k0 + min(k, kt - 1);
        int tap[4];
        float wq[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) tap[t] = s_tap[kk][t], wq[t] = s_wt[kk][t];
        for (int cq = 0; cq < nchunk; ++cq) {
          const int c0 = (REV ? nchunk - 1 - cq : cq) * cc, rows = min(cc, C - c0);
          float* qb = qbuf + (g_chunk & 1) * QF;
          mbar_wait(smem_u32(&full[stage]), phase);
          if (g_chunk >= 2) bar_sync(5 + (g_chunk & 1), SPS_QH);
          const T* sti = ring + (size_t)stage * slot_elems;
          if (q_on) {
            for (int c = cg; c < rows; c += G) {
              const T* src = sti + c * rs;
              float a = sp_f32(src[tap[0]]) * wq[0];
              a = fmaf(sp_f32(src[tap[1]]), wq[1], a);
              a = fmaf(sp_f32(src[tap[2]]), wq[2], a);
              a = fmaf(sp_f32(src[tap[3]]), wq[3], a);
              a = (k < kt) ? a : 0.f;
              if constexpr (MMA) {
                uint32_t hi, lo;
                split_tf32(a, hi, lo);
                float* qd = qb + sps_q_off<KT, MMA>(c, k);
                qd[0] = __uint_as_float(hi);
                qd[2] = __uint_as_float(lo);
              } else {
                qb[sps_q_off<KT, MMA>(c, k)] = a;
              }
            }
          }
          bar_arrive(3 + (g_chunk & 1), SPS_QH);
          release();
          ++g_chunk;
        }
      }
    }
    return;
  }

  const int px = tid;
  const bool has_px = px < hw;
  if (SPS_QW == 0) {
    for (int i = tid; i < 2 * QF; i += SPS_CONS) qbuf[i] = 0.f;
    cons_sync();
  }

  for (int b = blockIdx.x; b < p.B; b += gridDim.x) {
    const float* ki = p.kps_i + (size_t)b * K * p.stride;
    const float* kj = p.kps_j + (size_t)b * K * p.stride;
    // ---- key-point taps: kp / size * 2 - 1 -> ((g + 1) / 2) * (size - 1)  (align_corners=True) ----
    if (tid < K) {
      const float kx = __fdiv_rn(ki[(size_t)tid * p.stride + 0], p.image_size);
      const float ky = __fdiv_rn(ki[(size_t)tid * p.stride + 1], p.image_size);
      const float gx = __fsub_rn(__fmul_rn(kx, 2.f), 1.f), gy = __fsub_rn(__fmul_rn(ky, 2.f), 1.f);
      const float ix = __fmul_rn(__fdiv_rn(__fadd_rn(gx, 1.f), 2.f), (float)(p.w - 1));
      const float iy = __fmul_rn(__fdiv_rn(__fadd_rn(gy, 1.f), 2.f), (float)(p.h - 1));
      const float fx = floorf(ix), fy = floorf(iy);
      const int x0 = (int)fx, y0 = (int)fy;
      const float ww = ix - fx, we = 1.f - ww, wn = iy - fy, ws = 1.f - wn;
      const float wt[4] = {ws * we, ws * ww, wn * we, wn * ww};  // nw, ne, sw, se
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const int xx = x0 + (t & 1), yy = y0 + (t >> 1);
        const bool in = xx >= 0 && xx < p.w && yy >= 0 && yy < p.h;
        s_wt[tid][t] = in ? wt[t] : 0.f;
        s_tap[tid][t] = min(max(yy, 0), p.h - 1) * p.w + min(max(xx, 0), p.w - 1);
      }
    }
    // ---- pass N: ||f_i[px]||^2 of every pixel, channels in ascending order ----
    {
      float ss = 0.f;
      for (int c0 = 0; c0 < C; c0 += 2 * cc) {
        const int rows = min(2 * cc, C - c0);
        mbar_wait(smem_u32(&full[stage]), phase);
        const T* st = ring + (size_t)stage * slot_elems + px;
        if (has_px && SPS_NULL != 1) {
          for (int c = 0; c < rows; c += 8) {
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              const float v = sp_f32(st[(c + u) * rs]);
              ss = fmaf(v, v, ss);
            }
          }
        }
        release();
      }
      if (has_px) pix_ss[px] = ss;
    }
    cons_sync();
    if (tid < 4 * K) {  // fold 1 / max(||f_i[tap]||, eps) into the blend weight
      const int k = tid >> 2, t = tid & 3;
      s_wt[k][t] = __fdiv_rn(s_wt[k][t], fmaxf(sqrtf(pix_ss[s_tap[k][t]]), SPB_NORM_EPS));
    }
    cons_sync();
    if (SPS_QW > 0) bar_arrive(2, SPS_QH);

    for (int k0 = 0; k0 < K; k0 += KT) {
      const int kt = min(KT, K - k0);
      // accumulators of step H.  Tensor-core form: d[i][j][2 r + e] = heat of pixel 32 wid + 16 i + 2 g + r (tile i, fragment
      // row g + 8 r) and key point 8 j + 2 t + e; ssr[i][r] = this lane's share (channels t, t + 4) of that pixel's norm
      constexpr int NT8 = (KT + 7) / 8;
      const int g = lane >> 2, t = lane & 3;
      float d[2][MMA ? NT8 : 1][4];
      float ssr[2][2];
      float acc[MMA ? 1 : KT];
      float ssp = 0.f;
      if constexpr (MMA) {
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          ssr[i][0] = ssr[i][1] = 0.f;
#pragma unroll
          for (int j = 0; j < NT8; ++j) d[i][j][0] = d[i][j][1] = d[i][j][2] = d[i][j][3] = 0.f;
        }
      } else {
#pragma unroll
        for (int k = 0; k < KT; ++k) acc[k] = 0.f;
      }
      const bool warp_live = 32 * wid < hw;  // warp-uniform: this warp's 32 pixels hold at least one of the map
      const bool tile1_live = 32 * wid + 16 < hw;

      for (int cq = 0; cq < nchunk; ++cq) {
        const int c0 = (REV ? nchunk - 1 - cq : cq) * cc, rows = min(cc, C - c0);
        float* qb = qbuf + ((SPS_QW > 0 ? g_chunk : (unsigned)cq) & 1) * QF;
        mbar_wait(smem_u32(&full[stage]), phase);
        const T* sti = ring + (size_t)stage * slot_elems;
        const T* stj = sti + cc * rs;
        // ---- step Q: q[c][k] = sum_t wt * f_i[c][tap] / max(||f_i[tap]||, eps): the grid_sample of the normalised map ----
        for (int idx = tid; idx < rows * KT && SPS_NULL != 1 && SPS_NULL != 3 && SPS_QW == 0; idx += SPS_CONS) {
          const int c = idx / KT, k = idx - c * KT;
          const int kk = k0 + min(k, kt - 1);
          const T* src = sti + c * rs;
          float a = sp_f32(src[s_tap[kk][0]]) * s_wt[kk][0];
          a = fmaf(sp_f32(src[s_tap[kk][1]]), s_wt[kk][1], a);
          a = fmaf(sp_f32(src[s_tap[kk][2]]), s_wt[kk][2], a);
          a = fmaf(sp_f32(src[s_tap[kk][3]]), s_wt[kk][3], a);
          a = (k < kt) ? a : 0.f;
          if constexpr (MMA) {
            uint32_t hi, lo;
            split_tf32(a, hi, lo);
            float* qd = qb + sps_q_off<KT, MMA>(c, k);
            qd[0] = __uint_as_float(hi);
            qd[2] = __uint_as_float(lo);
          } else {
            qb[sps_q_off<KT, MMA>(c, k)] = a;
          }
        }
        if (SPS_QW > 0) bar_sync(3 + (g_chunk & 1), SPS_QH);  // q of this chunk complete (the Q warps have arrived)
        else cons_sync();  // q of this chunk complete; the other buffer is free again once every warp has passed this point
        // ---- step H: heat[k][px] += sum_c q[c][k] * f_j[c][px], the pixel's norm accumulated alongside ----
        if constexpr (MMA) {
          if (warp_live && SPS_NULL != 1 && SPS_NULL != 2) {
            const T* aj = stj + 32 * wid + 2 * g;
            const float4* bq = reinterpret_cast<const float4*>(qb) + lane;
            // the two run-time facts of a K step -- 8-byte loads possible, second tile live -- are dispatched once per chunk, so
            // that the K steps themselves are branch-free and the scheduler can lift the next step's loads above this step's MMAs
            auto h_chunk = [&](auto vec2_c, auto tile1_c) {
            constexpr bool VEC2 = decltype(vec2_c)::value;
            constexpr int NTILE = decltype(tile1_c)::value ? 2 : 1;
            auto kstep = [&](int ks) {  // channels ks .. ks + 7 of the chunk
              uint32_t bh[NT8][2], bl[NT8][2];
#pragma unroll
              for (int j = 0; j < NT8; ++j) {
                const float4 b4 = bq[((ks >> 3) * NT8 + j) * 32];
                bh[j][0] = __float_as_uint(b4.x);
                bh[j][1] = __float_as_uint(b4.y);
                bl[j][0] = __float_as_uint(b4.z);
                bl[j][1] = __float_as_uint(b4.w);
              }
              // A fragments: pixels 16 i + 2 g, + 1 (fragment rows g, g + 8 of tile i) of channels t and t + 4, each pair one
              // LDS.64 straight into its half of the operand's register quad (the tensor core ignores the low mantissa bits, so
              // the loaded values ARE the hi operand).  16-bit rows: each pair one 32-bit load, widened in registers; with an
              // odd h*w every other row starts at an odd element, and all four values are single 16-bit loads.  Pixels beyond
              // h*w read whatever follows in the slot (finite or not: their rows are never looked at).
              const T* r0 = aj + (ks + t) * rs;
              const T* r1 = r0 + 4 * rs;
              float av[2][4];
#pragma unroll
              for (int i = 0; i < NTILE; ++i) {  // NTILE == 1: the warp's second 16 pixels lie beyond the map
                if constexpr (VEC2) {
                  const float2 x0 = sp_f32x2(r0 + 16 * i), x1 = sp_f32x2(r1 + 16 * i);
                  av[i][0] = x0.x, av[i][1] = x0.y, av[i][2] = x1.x, av[i][3] = x1.y;
                } else {
                  av[i][0] = sp_f32(r0[16 * i]), av[i][1] = sp_f32(r0[16 * i + 1]);
                  av[i][2] = sp_f32(r1[16 * i]), av[i][3] = sp_f32(r1[16 * i + 1]);
                }
              }
#pragma unroll
              for (int i = 0; i < NTILE; ++i) {
                ssr[i][0] = fmaf(av[i][0], av[i][0], ssr[i][0]);
                ssr[i][0] = fmaf(av[i][2], av[i][2], ssr[i][0]);
                ssr[i][1] = fmaf(av[i][1], av[i][1], ssr[i][1]);
                ssr[i][1] = fmaf(av[i][3], av[i][3], ssr[i][1]);
                uint32_t ah[4], al[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  if constexpr (F32) split_tf32(av[i][e], ah[e], al[e]);
                  else ah[e] = __float_as_uint(av[i][e]);  // a widened 16-bit value is its own hi half; lo = 0
                }
#pragma unroll
                for (int j = 0; j < NT8; ++j) {
                  if (SPS_NULL != 4 && SPS_NULL != 5 && TERMS == 3 && F32) mma_tf32(d[i][j], al, bh[j][0], bh[j][1]);
                  if (SPS_NULL != 4 && SPS_NULL != 5 && TERMS == 3) mma_tf32(d[i][j], ah, bl[j][0], bl[j][1]);
                  if (SPS_NULL != 5) mma_tf32(d[i][j], ah, bh[j][0], bh[j][1]);
                }
              }
            };
            if (rows == cc) {
#pragma unroll
              for (int ks = 0; ks < cc; ks += 8) kstep(ks);
            } else {
              for (int ks = 0; ks < rows; ks += 8) kstep(ks);
            }
            };
            using Y = std::true_type;
            using N = std::false_type;
            if (vec2) {
              if (tile1_live) h_chunk(Y{}, Y{});
              else h_chunk(Y{}, N{});
            } else {
              if (tile1_live) h_chunk(N{}, Y{});
              else h_chunk(N{}, N{});
            }
          }
        } else {
          if (has_px) {
            const T* sj = stj + px;
            for (int c = 0; c < rows; ++c) {
              const float v = sp_f32(sj[c * rs]);
              ssp = fmaf(v, v, ssp);
              const float4* qc = reinterpret_cast<const float4*>(qb + c * KT);
#pragma unroll
              for (int k4 = 0; k4 < KT / 4; ++k4) {
                const float4 qq = qc[k4];  // same address in every lane: broadcast
                acc[4 * k4 + 0] = fmaf(qq.x, v, acc[4 * k4 + 0]);
                acc[4 * k4 + 1] = fmaf(qq.y, v, acc[4 * k4 + 1]);
                acc[4 * k4 + 2] = fmaf(qq.z, v, acc[4 * k4 + 2]);
                acc[4 * k4 + 3] = fmaf(qq.w, v, acc[4 * k4 + 3]);
              }
            }
          }
        }
        if (SPS_QW > 0) {
          if (g_chunk + 2 < n_chunks_cta) bar_arrive(5 + (g_chunk & 1), SPS_QH);  // this warp is done with the q buffer
          ++g_chunk;
        }
        release();
      }

      // ---- heat / max(||f_j[px]||, eps), arg-max per key point (first pixel among equals) ----
      if constexpr (MMA) {
        // per key point this lane owns (columns 2t, 2t + 1 of every N tile): best of its 4 pixels, then across the 8 row groups
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
          for (int r = 0; r < 2; ++r) {
            float ss = ssr[i][r];
            ss += __shfl_xor_sync(0xffffffffu, ss, 1);
            ss += __shfl_xor_sync(0xffffffffu, ss, 2);
            ssr[i][r] = fmaxf(sqrtf(ss), SPB_NORM_EPS);
          }
#pragma unroll
        for (int j = 0; j < NT8; ++j) {
#pragma unroll
          for (int e2 = 0; e2 < 2; ++e2) {
            float v = -CUDART_INF_F;
            int bi = 0x7fffffff;
#pragma unroll
            for (int i = 0; i < 2; ++i) {
#pragma unroll
              for (int r = 0; r < 2; ++r) {
                const int pxl = 32 * wid + 16 * i + 2 * g + r;  // ascending in (i, r): `>` keeps the first among equals
                const float hv = __fdiv_rn(d[i][j][2 * r + e2], ssr[i][r]);
                if (warp_live && pxl < hw && hv > v) {
                  v = hv;
                  bi = pxl;
                }
              }
            }
#pragma unroll
            for (int o = 4; o < 32; o <<= 1) {
              const float ov = __shfl_xor_sync(0xffffffffu, v, o);
              const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
              if (ov > v || (ov == v && oi < bi)) {
                v = ov;
                bi = oi;
              }
            }
            const int kcol = 8 * j + 2 * t + e2;
            if (g == 0 && kcol < KT) {
              s_bv[wid][kcol] = v;
              s_bi[wid][kcol] = bi;
            }
          }
        }
      } else {
        const float nrm = fmaxf(sqrtf(ssp), SPB_NORM_EPS);
#pragma unroll
        for (int k = 0; k < KT; ++k) {
          float v = has_px ? __fdiv_rn(acc[k], nrm) : -CUDART_INF_F;
          int i = has_px ? px : 0x7fffffff;
          if (!(v > -CUDART_INF_F)) {  // NaN / -inf never win (the first form's `hv > bestv` test against -inf)
            v = -CUDART_INF_F;
            i = 0x7fffffff;
          }
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, v, o);
            const int oi = __shfl_xor_sync(0xffffffffu, i, o);
            if (ov > v || (ov == v && oi < i)) {
              v = ov;
              i = oi;
            }
          }
          if (lane == 0) {
            s_bv[wid][k] = v;
            s_bi[wid][k] = i;
          }
        }
      }
      cons_sync();
      if (tid < kt) {
        float v = s_bv[0][tid];
        int i = s_bi[0][tid];
        for (int wq = 1; wq < SPS_WARPS; ++wq) {
          const float ov = s_bv[wq][tid];
          const int oi = s_bi[wq][tid];
          if (ov > v || (ov == v && oi < i)) {
            v = ov;
            i = oi;
          }
        }
        i = (i == 0x7fffffff) ? 0 : i;  // an all-NaN heat map: torch.argmax would return a NaN position; we return 0
        s_pred[k0 + tid] = i;
        if (p.pred) p.pred[(size_t)b * K + k0 + tid] = i;
      }
      cons_sync();  // s_bv is rewritten by the next tile
    }

    spair_score_block<SPS_CONS>(score, s_pred, K, p.w, ki, kj, p.stride, p.image_size, __ldg(p.thresh_scale + b), p.pck, nullptr,
                                p.error_same ? p.error_same + (size_t)b * K : nullptr,
                                p.error_nn ? p.error_nn + (size_t)b * K : nullptr,
                                p.index_nn ? p.index_nn + (size_t)b * K : nullptr, p.hits, p.confusion, p.conf_dim);
  }
}

int g_spair_terms = 3;  // mv_spair_set_heatmap_terms

// shared-memory plan of the streaming form
struct SpsPlan {
  int cc, rs, stages;
  size_t smem;
  bool ok;
};
SpsPlan sps_plan(const SpairBatchParams& p, int KT, size_t elem) {
  SpsPlan pl{};
  const int hw = p.h * p.w;
  static const int off = getenv("MVMATCH_SPAIR_STREAM") && getenv("MVMATCH_SPAIR_STREAM")[0] == '0';
  if (off || hw > 256 || p.C % 8 != 0 || ((uintptr_t)p.feats & 15) != 0) return pl;
  static const int env_stages = getenv("MVMATCH_SPAIR_STAGES") ? atoi(getenv("MVMATCH_SPAIR_STAGES")) : 0;
  static const bool mma = !(getenv("MVMATCH_SPAIR_MMA") && getenv("MVMATCH_SPAIR_MMA")[0] == '0');
  const int cc = SPS_CC, rs = hw;
  const size_t qf = mma ? (size_t)(cc / 8) * ((KT + 7) / 8) * 128 : (size_t)cc * KT;
  const size_t fixed = (2 * qf + (size_t)((hw + 3) & ~3) + (size_t)((p.K * (p.K + 1) + 2 + 3) & ~3)) * sizeof(float);
  const size_t slot = (size_t)2 * cc * rs * elem;  // 16-bit maps: half the bytes, twice the stages (5 against 2 at 14 x 14)
  // SPS_CTAS CTAs per SM: 227 KB less 1 KB reserved and ~4 KB of static shared memory per CTA
  const size_t budget = ((227u << 10) / SPS_CTAS) - (5u << 10);
  int stages = env_stages > 0 ? env_stages : (fixed + 2 * slot <= budget ? (int)((budget - fixed) / slot) : 2);
  if (stages < 2) stages = 2;
  if (stages > SPS_MAX_STAGES) stages = SPS_MAX_STAGES;
  pl.cc = cc;
  pl.rs = rs;
  pl.stages = stages;
  pl.smem = fixed + stages * slot;
  pl.ok = pl.smem <= (200u << 10);
  return pl;
}

template <typename T, int KT>
int launch_spair_stream(const SpairBatchParams& p, const SpsPlan& pl, cudaStream_t st) {
  // MVMATCH_SPAIR_MMA=0: the heat-map step on the CUDA cores (the arithmetic of the first form)
  static const bool mma = !(getenv("MVMATCH_SPAIR_MMA") && getenv("MVMATCH_SPAIR_MMA")[0] == '0');
  const bool one_term = mma && g_spair_terms == 1;
  auto kern = !mma ? spair_stream_kernel<T, KT, false>
                   : one_term ? spair_stream_kernel<T, KT, true, 1> : spair_stream_kernel<T, KT, true, 3>;
  static size_t opted[MV_MAX_DEVICES][3];
  size_t& opted_in = opted[mv_device_slot()][!mma ? 0 : one_term ? 2 : 1];
  if (pl.smem > opted_in) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem);
    if (e != cudaSuccess) {
      mv_set_error("mv_spair_match_batch: cannot opt in to %zu bytes of shared memory: %s", pl.smem, cudaGetErrorString(e));
      return (int)e;
    }
    opted_in = pl.smem;
  }
  int per_sm = (int)((227u << 10) / (pl.smem + (5u << 10)));  // static shared memory of the kernel is ~4 KB
  if (per_sm < 1) per_sm = 1;
  if (per_sm > SPS_CTAS) per_sm = SPS_CTAS;
  int grid = mv_sm_count() * per_sm;
  if (grid > p.B) grid = p.B;
  SpairBatchParams ps = p;
  ps.stages = pl.stages;
  ps.cc = pl.cc;
  ps.rs = pl.rs;
  kern<<<grid, SPS_THREADS, pl.smem, st>>>(ps);
  MV_LAUNCH_CHECK();
  return MV_OK;
}

template <typename T, int KT>
int launch_spair_batch(const SpairBatchParams& p, cudaStream_t st) {
  const SpsPlan pl = sps_plan(p, KT, sizeof(T));
  if (pl.ok) return launch_spair_stream<T, KT>(p, pl, st);
  const size_t smem = (size_t)p.C * KT * sizeof(float);
  auto kern = spair_batch_kernel<T, KT>;
  static size_t opted[MV_MAX_DEVICES];  // per device; static + dynamic shared memory above 48 KB needs the opt-in
  size_t& opted_in = opted[mv_device_slot()];
  if (opted_in < (24u << 10)) opted_in = 24 << 10;
  if (smem > opted_in) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
      mv_set_error("mv_spair_match_batch: cannot opt in to %zu bytes of shared memory: %s", smem, cudaGetErrorString(e));
      return (int)e;
    }
    opted_in = smem;
  }
  int per_sm = (int)((200u << 10) / (smem + (24u << 10)));  // static shared memory of the kernel is ~21 KB
  if (per_sm < 1) per_sm = 1;
  if (per_sm > 4) per_sm = 4;
  int grid = mv_sm_count() * per_sm;
  if (grid > p.B) grid = p.B;
  int threads = ((p.h * p.w + 31) / 32) * 32;
  if (threads > SPB_THREADS) threads = SPB_THREADS;
  if (threads < 4 * p.K) threads = ((4 * p.K + 31) / 32) * 32;  // the tap set-up uses one thread per tap (K <= 64)
  kern<<<grid, threads, smem, st>>>(p);
  MV_LAUNCH_CHECK();
  return MV_OK;
}

// key-point tile = accumulators per thread; the first form's tile features (C * KT floats) must fit shared memory
template <typename T>
int launch_spair_tiles(const SpairBatchParams& p, cudaStream_t st) {
  const size_t budget = 160u << 10;
  const size_t per_k = (size_t)p.C * sizeof(float);
  const int K = p.K;
  if (K > 24 && 32 * per_k <= budget) return launch_spair_batch<T, 32>(p, st);
  if (K > 20 && 24 * per_k <= budget) return launch_spair_batch<T, 24>(p, st);
  if (K > 16 && 20 * per_k <= budget) return launch_spair_batch<T, 20>(p, st);  // SPair-71k: up to 20 key points for most classes
  if (K > 12 && 16 * per_k <= budget) return launch_spair_batch<T, 16>(p, st);
  if (K > 8 && 12 * per_k <= budget) return launch_spair_batch<T, 12>(p, st);
  return launch_spair_batch<T, 8>(p, st);
}

// mv_spair_match_batch (feat_dtype = MV_FEAT_F32) and mv_spair_match_batch_typed; `fn` names the entry point in errors
int spair_match_batch(const char* fn, const void* feats, int feat_dtype, int B, int C, int h, int w, const float* kps_i,
                      const float* kps_j, int K, int kp_stride, const float* thresh_scale, float image_size, float pck_thresh,
                      int32_t* pred_flat, float* error_same, float* error_nn, int32_t* index_nn, unsigned long long* hits,
                      unsigned long long* confusion, int conf_dim, mv_stream_t stream) {
  MV_REQUIRE(feat_dtype == MV_FEAT_F32 || feat_dtype == MV_FEAT_BF16 || feat_dtype == MV_FEAT_F16, MV_E_ARG,
             "%s: unknown feature dtype %d", fn, feat_dtype);
  MV_REQUIRE(B >= 0 && C > 0 && h > 0 && w > 0, MV_E_ARG, "%s: bad sizes", fn);
  MV_REQUIRE((B == 0 || K == 0) || (feats && kps_i && kps_j && thresh_scale), MV_E_ARG, "%s: null pointer", fn);
  const uintptr_t elem = feat_dtype == MV_FEAT_F32 ? 4 : 2;
  MV_REQUIRE(((uintptr_t)feats & (elem - 1)) == 0, MV_E_ALIGN, "%s: feats must be aligned to its %d-byte elements", fn,
             (int)elem);
  MV_REQUIRE(h * w <= SPB_MAX_HW, MV_E_RANGE, "%s: h*w=%d exceeds %d pixels", fn, h * w, SPB_MAX_HW);
  MV_REQUIRE(K >= 0 && K <= 64, MV_E_RANGE, "%s: K=%d must be in [0, 64]", fn, K);
  MV_REQUIRE(kp_stride >= 3 && image_size > 0.f, MV_E_ARG, "%s: bad key-point layout", fn);
  MV_REQUIRE(!confusion || conf_dim >= K, MV_E_ARG, "%s: conf_dim=%d must be >= K=%d", fn, conf_dim, K);
  if (B == 0 || K == 0) return MV_OK;
  MV_REQUIRE(8 * (size_t)C * sizeof(float) <= (160u << 10), MV_E_RANGE, "%s: C=%d too large for the key-point tile", fn, C);
  SpairBatchParams p;
  p.feats = feats;
  p.kps_i = kps_i;
  p.kps_j = kps_j;
  p.thresh_scale = thresh_scale;
  p.B = B;
  p.C = C;
  p.h = h;
  p.w = w;
  p.K = K;
  p.stride = kp_stride;
  p.image_size = image_size;
  p.pck = pck_thresh;
  p.pred = pred_flat;
  p.error_same = error_same;
  p.error_nn = error_nn;
  p.index_nn = index_nn;
  p.hits = hits;
  p.confusion = confusion;
  p.conf_dim = conf_dim;
  p.stages = p.cc = p.rs = 0;
  cudaStream_t st = mv_cuda_stream(stream);
  if (feat_dtype == MV_FEAT_BF16) return launch_spair_tiles<__nv_bfloat16>(p, st);
  if (feat_dtype == MV_FEAT_F16) return launch_spair_tiles<__half>(p, st);
  return launch_spair_tiles<float>(p, st);
}

}  // namespace

extern "C" {

int mv_spair_match_batch(const float* feats, int B, int C, int h, int w, const float* kps_i, const float* kps_j, int K,
                         int kp_stride, const float* thresh_scale, float image_size, float pck_thresh,
                         int32_t* pred_flat, float* error_same, float* error_nn, int32_t* index_nn,
                         unsigned long long* hits, unsigned long long* confusion, int conf_dim, mv_stream_t stream) {
  return spair_match_batch("mv_spair_match_batch", feats, MV_FEAT_F32, B, C, h, w, kps_i, kps_j, K, kp_stride, thresh_scale,
                           image_size, pck_thresh, pred_flat, error_same, error_nn, index_nn, hits, confusion, conf_dim, stream);
}

int mv_spair_match_batch_typed(const void* feats, int feat_dtype, int B, int C, int h, int w, const float* kps_i,
                               const float* kps_j, int K, int kp_stride, const float* thresh_scale, float image_size,
                               float pck_thresh, int32_t* pred_flat, float* error_same, float* error_nn, int32_t* index_nn,
                               unsigned long long* hits, unsigned long long* confusion, int conf_dim, mv_stream_t stream) {
  return spair_match_batch("mv_spair_match_batch_typed", feats, feat_dtype, B, C, h, w, kps_i, kps_j, K, kp_stride,
                           thresh_scale, image_size, pck_thresh, pred_flat, error_same, error_nn, index_nn, hits, confusion,
                           conf_dim, stream);
}

int mv_spair_set_heatmap_terms(int terms) {
  const int prev = g_spair_terms;
  if (terms == 1 || terms == 3) g_spair_terms = terms;
  return prev;
}

}  // extern "C"
