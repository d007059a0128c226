// k3_score.cu -- kernel 3 of the matching path: everything after the nearest-neighbour search.
//
//   mv_k3_ratio_mutual   fp32 recompute of the two cosine distances per query, re-rank, Lowe ratio
//                        weight, mutual-nearest-neighbour flag
//   mv_k3_topk_matches   the num_corr largest weights, sorted (radix select + bitonic sort, one CTA)
//   mv_k3_mutual_select  two-sided mutual test on the forward and reverse re-ranked candidates, min weight, and the
//                        top num_corr of the mutual queries (k on the device)
//   mv_k3_score          Rt transform, K projection, 3-D / 2-D errors, integer threshold hit counts
//   mv_gather_rows       row gather for the helper's return tuples
//   mv_k3_spair_errors   SPair keypoint error matrix, error_same / error_nn, PCK hit counts
//
// Reference behaviour being reproduced (file:line in /root/reference):
//   evals/utils/correspondence.py:53-58    X_f_nn = Y_f[X_nn]; dists = 1 - cosine_similarity(...)
//   evals/utils/correspondence.py:72-77    idx_1[..., 0]; ratio weights or dists[:, 0]
//   evals/utils/correspondence.py:105-121  calculate_ratio_test (both clamps at 1e-9)
//   evals/utils/correspondence.py:125-129  get_topk_matches (torch.topk, sorted descending)
//   evals/utils/correspondence.py:193-196  project_3dto2d
//   evals/utils/transformations.py:27-36   transform_points_Rt
//   evaluate_navi_correspondence.py:186-212, render_scannet_correspondence.py:211-217, :253-264  errors, recall
//   evaluate_spair_correspondence.py:83-98, :121  SPair errors and PCK
#include <cuda_fp16.h>

#include <cstdlib>
#include <math_constants.h>

#include "common.cuh"
#include "spair_score.cuh"

namespace {

constexpr float COS_EPS = 1e-8f;     // torch.nn.functional.cosine_similarity default eps
constexpr float RATIO_CLAMP = 1e-9f; // calculate_ratio_test clamps
constexpr float MISSING_DIST = 2.0f; // distance reported for a candidate that does not exist (m < 2)
constexpr float F16C_ZERO_SS = 1e-10f;  // f16c target rows: squared norms below this are the rebuild residual of a zero row

// ------------------------------------------------------------------------------------------
// ratio / mutual: one warp per query row
// ------------------------------------------------------------------------------------------
// Row storage: fp32 rows, or SPLIT rows = two bf16 planes hi = bf16(x), lo = bf16(x - hi) written by kernel 1;
// hi + lo is exact in fp32 and differs from x by <= 2^-17 |x| per element, which moves 1 - cos by ~1e-7.
struct RowsF32 {
  const float* A;
  const float* B;
};
struct RowsSplit {
  const __nv_bfloat16* A_hi;
  const __nv_bfloat16* A_lo;
  const __nv_bfloat16* B_hi;
  const __nv_bfloat16* B_lo;
};

// f16c rows (mv_k1_sample_f16c): hi (pitch C + 8) + lo * 2^-11 (pitch C), target rows relative to a centre
struct RowsF16c {
  const __half* A_hi;
  const __half* A_lo;
  const __half* B_hi;
  const __half* B_lo;
  const float* center_B;  // may be null
  int pitch;              // row pitch of the hi planes (>= C + 8)
  const float* center_A;  // may be null: the reverse pass of a mutual match, whose query rows are target-role rows
};

__device__ __forceinline__ void f16c8(const __half* hi, const __half* lo, int c8, float (&out)[8]) {
  const uint4 h = __ldg(reinterpret_cast<const uint4*>(hi) + c8), l = __ldg(reinterpret_cast<const uint4*>(lo) + c8);
  const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&hw[k]));
    const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&lw[k]));
    out[2 * k] = fmaf(b.x, 1.f / 2048.f, a.x);  // exact: 11 + 11 mantissa bits
    out[2 * k + 1] = fmaf(b.y, 1.f / 2048.f, a.y);
  }
}

__device__ __forceinline__ void acc5(float v, float a, float b, float& xx, float& aa, float& bb, float& xa, float& xb) {
  xx = fmaf(v, v, xx);
  aa = fmaf(a, a, aa);
  bb = fmaf(b, b, bb);
  xa = fmaf(v, a, xa);
  xb = fmaf(v, b, xb);
}

__device__ __forceinline__ void split8(const __nv_bfloat16* hi, const __nv_bfloat16* lo, int c8, float (&out)[8]) {
  const uint4 h = __ldg(reinterpret_cast<const uint4*>(hi) + c8), l = __ldg(reinterpret_cast<const uint4*>(lo) + c8);
  const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
  for (int k = 0; k < 4; ++k) {  // bf16 -> fp32 is a 16-bit shift
    out[2 * k] = __uint_as_float(hw[k] << 16) + __uint_as_float(lw[k] << 16);
    out[2 * k + 1] = __uint_as_float(hw[k] & 0xffff0000u) + __uint_as_float(lw[k] & 0xffff0000u);
  }
}

// A TEAM of W warps per query (W = 1, 2 or 4 by C): each warp owns a contiguous 1/W of the channels, so the serial chain
// of a row is C / (8 * 32 * W) chunk loads deep instead of C / 256 -- the kernel is bound by the DRAM latency of the row
// reads (ncu round 2: 74 % of the samples on long-scoreboard stalls, 81 MB read in 27.6 us = 2.9 TB/s with one warp per
// row at C = 3072).  The five partial sums meet in shared memory and are added in a fixed order.
constexpr int RATIO_THREADS = 128;
template <typename ROWS, int W>
__global__ void __launch_bounds__(RATIO_THREADS, 6) k3_ratio_mutual_kernel(ROWS rows, int C, const int32_t* __restrict__ n_dev, int n_max,
                                                              int32_t* __restrict__ row_idx,
                                                              const unsigned long long* __restrict__ col_best,
                                                              int ratio_test, float* __restrict__ dists,
                                                              float* __restrict__ weight, uint8_t* __restrict__ mutual) {
  constexpr int TEAMS = RATIO_THREADS / 32 / W;
  __shared__ float part[TEAMS][W][5];
  const int n = n_dev ? min(*n_dev, n_max) : n_max;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int team = wid / W, wsub = wid % W;
  const int i = blockIdx.x * TEAMS + team;
  const bool live = i < n;
  int j0 = -1, j1 = -1;
  float xx = 0.f, aa = 0.f, bb = 0.f, xa = 0.f, xb = 0.f;
  if (live) {
    j0 = row_idx[2 * (size_t)i];
    j1 = row_idx[2 * (size_t)i + 1];
    if constexpr (sizeof(ROWS) == sizeof(RowsF32)) {
      const float4* x = reinterpret_cast<const float4*>(rows.A + (size_t)i * C);
      const float4* y0 = reinterpret_cast<const float4*>(rows.B + (size_t)max(j0, 0) * C);
      const float4* y1 = reinterpret_cast<const float4*>(rows.B + (size_t)max(j1, 0) * C);
      const int q = ((C >> 2) + W - 1) / W, beg = wsub * q, end = min(beg + q, C >> 2);
      for (int c = beg + lane; c < end; c += 32) {
        const float4 v = __ldg(x + c), a = __ldg(y0 + c), b = __ldg(y1 + c);
        xx = fmaf(v.x, v.x, xx); xx = fmaf(v.y, v.y, xx); xx = fmaf(v.z, v.z, xx); xx = fmaf(v.w, v.w, xx);
        aa = fmaf(a.x, a.x, aa); aa = fmaf(a.y, a.y, aa); aa = fmaf(a.z, a.z, aa); aa = fmaf(a.w, a.w, aa);
        bb = fmaf(b.x, b.x, bb); bb = fmaf(b.y, b.y, bb); bb = fmaf(b.z, b.z, bb); bb = fmaf(b.w, b.w, bb);
        xa = fmaf(v.x, a.x, xa); xa = fmaf(v.y, a.y, xa); xa = fmaf(v.z, a.z, xa); xa = fmaf(v.w, a.w, xa);
        xb = fmaf(v.x, b.x, xb); xb = fmaf(v.y, b.y, xb); xb = fmaf(v.z, b.z, xb); xb = fmaf(v.w, b.w, xb);
      }
    } else if constexpr (sizeof(ROWS) == sizeof(RowsF16c)) {
      const size_t P = (size_t)rows.pitch;
      const size_t ox = (size_t)i * C, o0 = (size_t)max(j0, 0) * C, o1 = (size_t)max(j1, 0) * C;
      const __half* xh = rows.A_hi + (size_t)i * P;
      const __half* ah = rows.B_hi + (size_t)max(j0, 0) * P;
      const __half* bh = rows.B_hi + (size_t)max(j1, 0) * P;
      const int q = ((C >> 3) + W - 1) / W, beg = wsub * q, end = min(beg + q, C >> 3);
#pragma unroll 3
      for (int c8 = beg + lane; c8 < end; c8 += 32) {
        float v[8], a[8], b[8];
        f16c8(xh, rows.A_lo + ox, c8, v);
        f16c8(ah, rows.B_lo + o0, c8, a);
        f16c8(bh, rows.B_lo + o1, c8, b);
        if (rows.center_A) {
          const float4 m0 = __ldg(reinterpret_cast<const float4*>(rows.center_A) + 2 * c8);
          const float4 m1 = __ldg(reinterpret_cast<const float4*>(rows.center_A) + 2 * c8 + 1);
          const float mu[8] = {m0.x, m0.y, m0.z, m0.w, m1.x, m1.y, m1.z, m1.w};
#pragma unroll
          for (int k = 0; k < 8; ++k) v[k] += mu[k];
        }
        if (rows.center_B) {
          const float4 m0 = __ldg(reinterpret_cast<const float4*>(rows.center_B) + 2 * c8);
          const float4 m1 = __ldg(reinterpret_cast<const float4*>(rows.center_B) + 2 * c8 + 1);
          const float mu[8] = {m0.x, m0.y, m0.z, m0.w, m1.x, m1.y, m1.z, m1.w};
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            a[k] += mu[k];
            b[k] += mu[k];
          }
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) acc5(v[k], a[k], b[k], xx, aa, bb, xa, xb);
      }
    } else {
      const size_t ox = (size_t)i * C, o0 = (size_t)max(j0, 0) * C, o1 = (size_t)max(j1, 0) * C;
      const int q = ((C >> 3) + W - 1) / W, beg = wsub * q, end = min(beg + q, C >> 3);
#pragma unroll 2
      for (int c8 = beg + lane; c8 < end; c8 += 32) {
        float v[8], a[8], b[8];
        split8(rows.A_hi + ox, rows.A_lo + ox, c8, v);
        split8(rows.B_hi + o0, rows.B_lo + o0, c8, a);
        split8(rows.B_hi + o1, rows.B_lo + o1, c8, b);
#pragma unroll
        for (int k = 0; k < 8; ++k) acc5(v[k], a[k], b[k], xx, aa, bb, xa, xb);
      }
    }
    xx = warp_sum(xx); aa = warp_sum(aa); bb = warp_sum(bb); xa = warp_sum(xa); xb = warp_sum(xb);
  }
  if (W > 1) {
    if (lane == 0) {
      float* q = part[team][wsub];
      q[0] = xx; q[1] = aa; q[2] = bb; q[3] = xa; q[4] = xb;
    }
    __syncthreads();
    if (wsub == 0 && lane == 0) {
      xx = aa = bb = xa = xb = 0.f;
#pragma unroll
      for (int w = 0; w < W; ++w) {  // fixed order
        const float* q = part[team][w];
        xx += q[0]; aa += q[1]; bb += q[2]; xa += q[3]; xb += q[4];
      }
    }
  }
  if (!live || lane != 0 || wsub != 0) return;
  if constexpr (sizeof(ROWS) == sizeof(RowsF16c)) {
    // a zero target row stored relative to the centre rebuilds as hi + lo * 2^-11 + mu: a residual of up to ~2^-21 |mu| per
    // element (norm ~4e-8 for |mu| ~ 1), not 0, whose cosine with the query is rounding noise.  The rows are L2-normalised
    // (norm 1, or 0 for a zero input row), so a rebuilt row below F16C_ZERO_SS is that residual: cosine 0, as for a zero row
    if (rows.center_B) {
      if (aa < F16C_ZERO_SS) xa = 0.f;
      if (bb < F16C_ZERO_SS) xb = 0.f;
    }
    if (rows.center_A && xx < F16C_ZERO_SS) xa = xb = 0.f;
  }
  const float nx = fmaxf(sqrtf(xx), COS_EPS);
  float d0 = j0 >= 0 ? 1.f - xa / (nx * fmaxf(sqrtf(aa), COS_EPS)) : MISSING_DIST;
  float d1 = j1 >= 0 ? 1.f - xb / (nx * fmaxf(sqrtf(bb), COS_EPS)) : MISSING_DIST;
  if (j1 >= 0 && (d1 < d0 || (d1 == d0 && j1 < j0))) {  // fp32 order wins over the tensor-core order
    const float td = d0; d0 = d1; d1 = td;
    const int tj = j0; j0 = j1; j1 = tj;
    row_idx[2 * (size_t)i] = j0;
    row_idx[2 * (size_t)i + 1] = j1;
  }
  if (dists) {
    dists[2 * (size_t)i] = d0;
    dists[2 * (size_t)i + 1] = d1;
  }
  if (weight) {
    float w = d0;
    if (ratio_test) w = 1.f - __fdiv_rn(fmaxf(d0, RATIO_CLAMP), fmaxf(fmaxf(d1, RATIO_CLAMP), RATIO_CLAMP));
    weight[i] = w;
  }
  if (mutual) {
    uint8_t f = 0;
    if (col_best && j0 >= 0) {
      const unsigned long long pk = col_best[j0];
      f = (pk != 0ull && (0xffffffffu - (uint32_t)(pk & 0xffffffffull)) == (uint32_t)i) ? 1 : 0;
    }
    mutual[i] = f;
  }
}

// W warps per query by the row length: deeper rows get more warps (shorter dependent-load chains)
template <typename ROWS>
void launch_ratio(const ROWS& rows, int C, const int32_t* n_dev, int n_max, int32_t* row_idx, const unsigned long long* col_best,
                  int ratio_test, float* dists, float* weight, uint8_t* mutual, cudaStream_t st) {
  static const int forced = getenv("MVMATCH_RATIO_W") ? atoi(getenv("MVMATCH_RATIO_W")) : 0;
  // measured in the 4-lane pipeline (bench.py, same box): NAVI-shaped 4153 pairs/s with teams of 4 vs 4353 with one warp per query,
  // ScanNet-shaped 917 vs 917 -- the other lanes already hide this kernel's load latency -- so one warp per query stays the default
  const int W = forced ? forced : 1;
  const int teams = RATIO_THREADS / 32 / W;
  const unsigned grid = (unsigned)((n_max + teams - 1) / teams);
  if (W == 4) k3_ratio_mutual_kernel<ROWS, 4><<<grid, RATIO_THREADS, 0, st>>>(rows, C, n_dev, n_max, row_idx, col_best, ratio_test, dists, weight, mutual);
  else if (W == 2) k3_ratio_mutual_kernel<ROWS, 2><<<grid, RATIO_THREADS, 0, st>>>(rows, C, n_dev, n_max, row_idx, col_best, ratio_test, dists, weight, mutual);
  else k3_ratio_mutual_kernel<ROWS, 1><<<grid, RATIO_THREADS, 0, st>>>(rows, C, n_dev, n_max, row_idx, col_best, ratio_test, dists, weight, mutual);
}

// ------------------------------------------------------------------------------------------
// adjacent similarity consumers (SURVEY 8f.4)
// ------------------------------------------------------------------------------------------
// MaskCut: A = S > tau ? 1 : eps and the per-row counts (maskcut_processor.py:103-106); one warp per row
__global__ void affinity_threshold_kernel(const float* __restrict__ S, int n, int m, int ld_s, float tau, float eps,
                                          float* __restrict__ A_out, int32_t* __restrict__ count) {
  const int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (i >= n) return;
  int c = 0;
  for (int j = lane; j < m; j += 32) {
    const bool on = S[(size_t)i * ld_s + j] > tau;
    c += on ? 1 : 0;
    if (A_out) A_out[(size_t)i * m + j] = on ? 1.f : eps;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if (lane == 0 && count) count[i] = c;
}

// 2AFC: cos(ref, left), cos(ref, right) per sample (F.cosine_similarity, eps 1e-8) and the prediction; one warp per sample
__global__ void cosine_2afc_kernel(const float* __restrict__ ref, const float* __restrict__ left, const float* __restrict__ right,
                                   int n, int C, float* __restrict__ sim_left, float* __restrict__ sim_right,
                                   int32_t* __restrict__ pred) {
  const int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (i >= n) return;
  const float4* x = reinterpret_cast<const float4*>(ref + (size_t)i * C);
  const float4* a = reinterpret_cast<const float4*>(left + (size_t)i * C);
  const float4* b = reinterpret_cast<const float4*>(right + (size_t)i * C);
  float xx = 0.f, aa = 0.f, bb = 0.f, xa = 0.f, xb = 0.f;
  for (int c = lane; c < (C >> 2); c += 32) {
    const float4 v = __ldg(x + c), p = __ldg(a + c), q = __ldg(b + c);
    acc5(v.x, p.x, q.x, xx, aa, bb, xa, xb);
    acc5(v.y, p.y, q.y, xx, aa, bb, xa, xb);
    acc5(v.z, p.z, q.z, xx, aa, bb, xa, xb);
    acc5(v.w, p.w, q.w, xx, aa, bb, xa, xb);
  }
  xx = warp_sum(xx); aa = warp_sum(aa); bb = warp_sum(bb); xa = warp_sum(xa); xb = warp_sum(xb);
  if (lane != 0) return;
  const float nx = fmaxf(sqrtf(xx), COS_EPS);
  const float sl = xa / (nx * fmaxf(sqrtf(aa), COS_EPS)), sr = xb / (nx * fmaxf(sqrtf(bb), COS_EPS));
  if (sim_left) sim_left[i] = sl;
  if (sim_right) sim_right[i] = sr;
  if (pred) pred[i] = sl > sr ? 0 : 1;
}

// ------------------------------------------------------------------------------------------
// top-k of the weights (single CTA, 1024 threads): radix select the k-th key, stable pick among the
// ties, bitonic sort of the k winners by (weight desc, row asc)
// 20 us for 5 k weights / k = 1000.  Measured and rejected: caching the keys in shared memory (20.2 us, the five
// passes are not load-bound) and __match_any_sync-aggregated histogram atomics (36.8 us: the match instruction
// costs more than the same-address shared atomics it saves).
// ------------------------------------------------------------------------------------------
constexpr int TOPK_THREADS = 1024;

__global__ void __launch_bounds__(TOPK_THREADS) k3_topk_kernel(const float* __restrict__ weight,
                                                               const int32_t* __restrict__ row_idx,
                                                               const int32_t* __restrict__ n_dev, int n_max, int num_corr,
                                                               int kpad, int32_t* __restrict__ sel_src,
                                                               int32_t* __restrict__ sel_dst, float* __restrict__ sel_weight,
                                                               int32_t* __restrict__ k_dev) {
  extern __shared__ unsigned long long sortbuf[];  // kpad entries
  __shared__ int hist[256];
  // one private histogram per warp: weights share their top key bytes (ratio weights live in [0, 1]), so a single
  // histogram serialises on a handful of bins (round 2: 20 -> 12 us at n = 5024, 43 -> 17 us at n = 18231)
  __shared__ int whist[TOPK_THREADS / 64][256];  // two warps per histogram: 16 KB (the sort buffer needs the rest of the 48 KB)
  __shared__ int warp_tot[32];
  __shared__ int s_incl[256];
  __shared__ uint32_t s_prefix;
  __shared__ int s_remaining, s_gt;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int n = n_dev ? min(*n_dev, n_max) : n_max;
  const int k = min(num_corr, n);
  if (tid == 0 && k_dev) *k_dev = k;
  if (k <= 0) return;

  // the keys of this thread stay in registers across the passes when n is small enough (every BASELINE shape)
  constexpr int KPT = 20;
  const bool cached = n <= KPT * TOPK_THREADS;
  uint32_t mykeys[KPT];
  if (cached) {
#pragma unroll
    for (int q = 0; q < KPT; ++q) {
      const int i = q * TOPK_THREADS + tid;
      mykeys[q] = i < n ? f32_orderable(__ldg(weight + i)) : 0u;
    }
  }
  // ---- radix select, most significant byte first
  uint32_t prefix = 0, mask = 0;
  int remaining = k;
  for (int pass = 3; pass >= 0; --pass) {
    for (int b = tid; b < (TOPK_THREADS / 64) * 256; b += TOPK_THREADS) (&whist[0][0])[b] = 0;
    __syncthreads();
    if (cached) {
#pragma unroll
      for (int q = 0; q < KPT; ++q) {
        const uint32_t key = mykeys[q];
        if (q * TOPK_THREADS + tid < n && (key & mask) == prefix) atomicAdd(&whist[wid >> 1][(key >> (8 * pass)) & 255], 1);
      }
    } else {
      for (int i = tid; i < n; i += TOPK_THREADS) {
        const uint32_t key = f32_orderable(weight[i]);
        if ((key & mask) == prefix) atomicAdd(&whist[wid >> 1][(key >> (8 * pass)) & 255], 1);
      }
    }
    __syncthreads();
    if (tid < 256) {
      int t = 0;
#pragma unroll 8
      for (int w = 0; w < TOPK_THREADS / 64; ++w) t += whist[w][tid];
      hist[tid] = t;
    }
    __syncthreads();
    // suffix sums of the 256 bins by the first 8 warps: bin b is the pivot when above(b) < remaining <= above(b) + hist[b]
    if (tid < 256) {
      const int h = hist[tid];
      int incl = h;  // inclusive suffix sum inside the warp (towards higher bins)
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t2 = __shfl_down_sync(0xffffffffu, incl, o);
        if (lane + o < 32) incl += t2;
      }
      if (lane == 0) warp_tot[wid] = incl;  // total of this warp's 32 bins
      __syncwarp();
      s_incl[tid] = incl;
    }
    __syncthreads();
    if (tid < 256) {
      int above = s_incl[tid] - hist[tid];
      for (int w = wid + 1; w < 8; ++w) above += warp_tot[w];
      if (above < remaining && remaining <= above + hist[tid]) {
        s_prefix = prefix | ((uint32_t)tid << (8 * pass));
        s_remaining = remaining - above;
      }
    }
    __syncthreads();
    prefix = s_prefix;
    remaining = s_remaining;
    mask |= 0xffu << (8 * pass);
  }
  const uint32_t T = prefix;          // k-th largest key
  const int n_gt = k - remaining;     // keys strictly above it; `remaining` ties are taken in row order
  if (tid == 0) s_gt = 0;
  for (int q = tid; q < kpad; q += TOPK_THREADS) sortbuf[q] = 0ull;
  __syncthreads();

  int eq_seen = 0;  // ties in earlier chunks (uniform)
  for (int base = 0; base < n; base += TOPK_THREADS) {
    const int i = base + tid;
    uint32_t key = 0;
    bool gt = false, eq = false;
    if (i < n) {
      key = f32_orderable(weight[i]);
      gt = key > T;
      eq = key == T;
    }
    const uint32_t bal = __ballot_sync(0xffffffffu, eq);
    if (lane == 0) warp_tot[wid] = __popc(bal);
    __syncthreads();
    int before = 0, total = 0;
#pragma unroll 8
    for (int w = 0; w < 32; ++w) {
      const int c = warp_tot[w];
      before += (w < wid) ? c : 0;
      total += c;
    }
    const unsigned long long packed = ((unsigned long long)key << 32) | (unsigned long long)(0xffffffffu - (uint32_t)i);
    if (gt) sortbuf[atomicAdd(&s_gt, 1)] = packed;
    if (eq) {
      const int r = eq_seen + before + __popc(bal & ((1u << lane) - 1u));
      if (r < remaining) sortbuf[n_gt + r] = packed;
    }
    eq_seen += total;
    __syncthreads();
  }

  if (kpad <= TOPK_THREADS) {
    // ---- bitonic sort with one element per thread: compare-exchange distances below 32 are warp shuffles,
    // the 15 longer ones go through (ping-pong) shared memory with one barrier each -- 15 barriers, not 55
    unsigned long long v = (tid < kpad) ? sortbuf[tid] : 0ull;
    __syncthreads();
    unsigned long long* pp = sortbuf;  // 2 x 1024 entries (the launch sizes shared memory for that)
    int flip = 0;
    for (int size = 2; size <= TOPK_THREADS; size <<= 1) {
      const bool desc = (tid & size) == 0;
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        unsigned long long o;
        if (stride < 32) {
          o = __shfl_xor_sync(0xffffffffu, v, stride);
        } else {
          unsigned long long* buf = pp + flip * TOPK_THREADS;
          buf[tid] = v;
          __syncthreads();
          o = buf[tid ^ stride];
          flip ^= 1;
        }
        const bool keep_max = (((tid & stride) == 0) == desc);
        v = keep_max ? (v > o ? v : o) : (v < o ? v : o);
      }
    }
    if (tid < k) {
      const int i = (int)(0xffffffffu - (uint32_t)(v & 0xffffffffull));
      sel_src[tid] = i;
      sel_dst[tid] = row_idx[2 * (size_t)i];
      sel_weight[tid] = weight[i];
    }
    return;
  }
  // ---- bitonic sort, descending
  for (int size = 2; size <= kpad; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int q = tid; q < (kpad >> 1); q += TOPK_THREADS) {
        const int lo = 2 * q - (q & (stride - 1));
        const int hi = lo + stride;
        const bool desc = (lo & size) == 0;
        const unsigned long long a = sortbuf[lo], b = sortbuf[hi];
        if ((a < b) == desc) {
          sortbuf[lo] = b;
          sortbuf[hi] = a;
        }
      }
      __syncthreads();
    }
  }
  for (int r = tid; r < k; r += TOPK_THREADS) {
    const int i = (int)(0xffffffffu - (uint32_t)(sortbuf[r] & 0xffffffffull));
    sel_src[r] = i;
    sel_dst[r] = row_idx[2 * (size_t)i];
    sel_weight[r] = weight[i];
  }
}

// ------------------------------------------------------------------------------------------
// mutual matches: query i is mutual iff the re-ranked best row of its re-ranked best column is i again.  The selection
// weight of a mutual query is min(w_f(i), w_r(j(i))) with the ratio test, w_f(i) (= d0) without; every other query gets
// -inf, which sorts below every mutual one, and the count of mutual queries goes to *k_dev (zeroed before)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k3_mutual_combine_kernel(const int32_t* __restrict__ row_idx, const float* __restrict__ weight_f,
                                                                const int32_t* __restrict__ col_idx, const float* __restrict__ weight_r,
                                                                const int32_t* __restrict__ n_dev, int n_max, int ratio_test,
                                                                float* __restrict__ weight, uint8_t* __restrict__ mutual,
                                                                int32_t* __restrict__ count) {
  __shared__ int s_count;
  if (threadIdx.x == 0) s_count = 0;
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = n_dev ? min(*n_dev, n_max) : n_max;
  bool mu = false;
  if (i < n) {
    const int j = row_idx[2 * (size_t)i];
    mu = j >= 0 && col_idx[2 * (size_t)j] == i;
    const float wf = weight_f[i];
    weight[i] = mu ? (ratio_test ? fminf(wf, weight_r[j]) : wf) : -CUDART_INF_F;
    if (mutual) mutual[i] = mu ? 1 : 0;
  }
  const uint32_t b = __ballot_sync(0xffffffffu, mu);
  if ((threadIdx.x & 31) == 0 && b) atomicAdd(&s_count, __popc(b));
  __syncthreads();
  if (threadIdx.x == 0 && s_count) atomicAdd(count, s_count);
}

__global__ void k3_clamp_count_kernel(int32_t* __restrict__ k_dev, int num_corr) {
  if (*k_dev > num_corr) *k_dev = num_corr;
}

// ------------------------------------------------------------------------------------------
// scoring
// ------------------------------------------------------------------------------------------
struct ScoreParams {
  float Rt[12];
  float K[9];
  float thr3d[MV_MAX_THRESHOLDS];
  float thr2d[MV_MAX_THRESHOLDS];
  int n3, n2;
};

__device__ __forceinline__ void project(const float* K, float x, float y, float z, float& u, float& v) {
  // xyz @ K^T, then / clamp(z', 1e-9)   (project_3dto2d)
  const float a = fmaf(z, K[2], fmaf(y, K[1], x * K[0]));
  const float b = fmaf(z, K[5], fmaf(y, K[4], x * K[3]));
  const float c = fmaxf(fmaf(z, K[8], fmaf(y, K[7], x * K[6])), 1e-9f);
  u = __fdiv_rn(a, c);
  v = __fdiv_rn(b, c);
}

__global__ void __launch_bounds__(256) k3_score_kernel(const int32_t* __restrict__ sel_src,
                                                       const int32_t* __restrict__ sel_dst,
                                                       const int32_t* __restrict__ k_dev, int k_max,
                                                       const float* __restrict__ xyz0, const float* __restrict__ xyz1,
                                                       const uint8_t* __restrict__ mutual, ScoreParams sp,
                                                       float* __restrict__ c_xyz0, float* __restrict__ c_xyz1,
                                                       float* __restrict__ err3d, float* __restrict__ err2d,
                                                       unsigned long long* __restrict__ hits) {
  __shared__ unsigned int cnt[2 + 4 * MV_MAX_THRESHOLDS];
  const int ncnt = 2 + 2 * (sp.n3 + sp.n2);
  for (int q = threadIdx.x; q < ncnt; q += blockDim.x) cnt[q] = 0;
  __syncthreads();
  const int k = k_dev ? min(*k_dev, k_max) : k_max;
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = r < k;
  float e3 = CUDART_INF_F, e2 = CUDART_INF_F;
  bool mu = false;
  if (live) {
    const int s = sel_src[r], d = sel_dst[r];
    const float px = xyz0[3 * (size_t)s], py = xyz0[3 * (size_t)s + 1], pz = xyz0[3 * (size_t)s + 2];
    const float qx = xyz1[3 * (size_t)d], qy = xyz1[3 * (size_t)d + 1], qz = xyz1[3 * (size_t)d + 2];
    // points @ R^T + t  (transform_points_Rt)
    const float tx = fmaf(pz, sp.Rt[2], fmaf(py, sp.Rt[1], px * sp.Rt[0])) + sp.Rt[3];
    const float ty = fmaf(pz, sp.Rt[6], fmaf(py, sp.Rt[5], px * sp.Rt[4])) + sp.Rt[7];
    const float tz = fmaf(pz, sp.Rt[10], fmaf(py, sp.Rt[9], px * sp.Rt[8])) + sp.Rt[11];
    const float dx = tx - qx, dy = ty - qy, dz = tz - qz;
    e3 = sqrtf(fmaf(dz, dz, fmaf(dy, dy, dx * dx)));
    float u0, v0, u1, v1;
    project(sp.K, tx, ty, tz, u0, v0);
    project(sp.K, qx, qy, qz, u1, v1);
    const float du = u0 - u1, dv = v0 - v1;
    e2 = sqrtf(fmaf(dv, dv, du * du));
    mu = mutual ? mutual[s] != 0 : false;
    if (c_xyz0) { c_xyz0[3 * (size_t)r] = px; c_xyz0[3 * (size_t)r + 1] = py; c_xyz0[3 * (size_t)r + 2] = pz; }
    if (c_xyz1) { c_xyz1[3 * (size_t)r] = qx; c_xyz1[3 * (size_t)r + 1] = qy; c_xyz1[3 * (size_t)r + 2] = qz; }
    if (err3d) err3d[r] = e3;
    if (err2d) err2d[r] = e2;
  }
  const int lane = threadIdx.x & 31;
  auto tally = [&](int slot, bool flag) {
    const unsigned b = __ballot_sync(0xffffffffu, flag);
    if (lane == 0 && b) atomicAdd(&cnt[slot], (unsigned)__popc(b));
  };
  tally(0, live);
  tally(1, live && mu);
  for (int t = 0; t < sp.n3; ++t) {
    const bool h = live && e3 < sp.thr3d[t];
    tally(2 + t, h);
    tally(2 + sp.n3 + sp.n2 + t, h && mu);
  }
  for (int t = 0; t < sp.n2; ++t) {
    const bool h = live && e2 < sp.thr2d[t];
    tally(2 + sp.n3 + t, h);
    tally(2 + 2 * sp.n3 + sp.n2 + t, h && mu);
  }
  __syncthreads();
  for (int q = threadIdx.x; q < ncnt; q += blockDim.x)
    if (cnt[q]) atomicAdd(&hits[q], (unsigned long long)cnt[q]);
}

__global__ void gather_rows_kernel(const float* __restrict__ src, int width, const int32_t* __restrict__ idx,
                                   const int32_t* __restrict__ k_dev, int k_max, float* __restrict__ dst) {
  const int k = k_dev ? min(*k_dev, k_max) : k_max;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)k * width) return;
  const int r = (int)(t / width), c = (int)(t - (long long)r * width);
  dst[t] = src[(size_t)idx[r] * width + c];
}

// The helper's whole return tuple in one buffer of column blocks, each k_max rows long:
//   [xyz0 (k_max,3) | xyz1 (k_max,3) | weight (k_max) | uv0 (k_max,2) | uv1 (k_max,2) | n0, n1, k, 0]
// (uv blocks only when uv0 != NULL).  Rows beyond the live k are left untouched.
__global__ void pack_matches_kernel(const int32_t* __restrict__ sel_src, const int32_t* __restrict__ sel_dst,
                                    const float* __restrict__ sel_weight, const int32_t* __restrict__ k_dev, int k_max,
                                    const float* __restrict__ xyz0, const float* __restrict__ xyz1,
                                    const float* __restrict__ uv0, const float* __restrict__ uv1,
                                    const int32_t* __restrict__ n0_dev, const int32_t* __restrict__ n1_dev,
                                    float* __restrict__ out) {
  const int k = k_dev ? min(*k_dev, k_max) : k_max;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const size_t K = (size_t)k_max;
  if (t == 0) {  // live counts ride along (exact in fp32 below 2^24)
    float* tail = out + (uv0 ? 11 : 7) * K;
    tail[0] = n0_dev ? (float)*n0_dev : -1.f;
    tail[1] = n1_dev ? (float)*n1_dev : -1.f;
    tail[2] = (float)k;
    tail[3] = 0.f;
  }
  if (t >= k) return;
  const int a = sel_src[t], b = sel_dst[t];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    out[(size_t)t * 3 + c] = xyz0[(size_t)a * 3 + c];
    out[3 * K + (size_t)t * 3 + c] = xyz1[(size_t)b * 3 + c];
  }
  out[6 * K + t] = sel_weight[t];
  if (uv0) {
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      out[7 * K + (size_t)t * 2 + c] = uv0[(size_t)a * 2 + c];
      out[9 * K + (size_t)t * 2 + c] = uv1[(size_t)b * 2 + c];
    }
  }
}

// argmax_2d: one warp per row, first occurrence wins
__global__ void __launch_bounds__(256) argmax_rows_kernel(const float* __restrict__ x, int rows, int cols, int max_value,
                                                          int32_t* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= rows) return;
  const float* row = x + (size_t)r * cols;
  float best = max_value ? -CUDART_INF_F : CUDART_INF_F;
  int bi = 0x7fffffff;
  for (int c = lane; c < cols; c += 32) {
    const float v = __ldg(row + c);
    if (max_value ? (v > best) : (v < best)) { best = v; bi = c; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    const bool take = max_value ? (ov > best || (ov == best && oi < bi)) : (ov < best || (ov == best && oi < bi));
    if (take) { best = ov; bi = oi; }
  }
  if (lane == 0) out[r] = bi == 0x7fffffff ? 0 : bi;
}

// ------------------------------------------------------------------------------------------
// SPair
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k3_spair_kernel(const int32_t* __restrict__ pred_flat, int K, int w,
                                                       const float* __restrict__ kps_i, const float* __restrict__ kps_j,
                                                       int stride, float image_size, float thresh_scale, float pck,
                                                       float* __restrict__ errors, float* __restrict__ error_same,
                                                       float* __restrict__ error_nn, int32_t* __restrict__ index_nn,
                                                       unsigned long long* __restrict__ hits,
                                                       unsigned long long* __restrict__ confusion, int conf_dim) {
  __shared__ SpairScoreShared sh;
  spair_score_block(sh, pred_flat, K, w, kps_i, kps_j, stride, image_size, thresh_scale, pck, errors, error_same,
                    error_nn, index_nn, hits, confusion, conf_dim);
}

}  // namespace

extern "C" {

int mv_k3_ratio_mutual(const float* A32, const float* B32, int C, const int32_t* n_dev, int n_max, int32_t* row_idx,
                       const unsigned long long* col_best, int ratio_test, float* dists, float* weight,
                       uint8_t* mutual, mv_stream_t stream) {
  MV_REQUIRE(A32 && B32 && row_idx, MV_E_ARG, "mv_k3_ratio_mutual: null pointer");
  MV_REQUIRE(C > 0 && C % 4 == 0, MV_E_ALIGN, "mv_k3_ratio_mutual: C=%d must be a positive multiple of 4", C);
  MV_REQUIRE(((uintptr_t)A32 & 15) == 0 && ((uintptr_t)B32 & 15) == 0, MV_E_ALIGN,
             "mv_k3_ratio_mutual: A32 and B32 must be 16-byte aligned");
  MV_REQUIRE(n_max >= 0, MV_E_ARG, "mv_k3_ratio_mutual: negative n_max");
  if (n_max == 0) return MV_OK;
  RowsF32 rows{A32, B32};
  launch_ratio(rows, C, n_dev, n_max, row_idx, col_best, ratio_test, dists, weight, mutual, mv_cuda_stream(stream));
  MV_LAUNCH_CHECK();
  return MV_OK;
}

int mv_k3_ratio_mutual_split(const uint16_t* A_hi, const uint16_t* A_lo, const uint16_t* B_hi, const uint16_t* B_lo, int C,
                             const int32_t* n_dev, int n_max, int32_t* row_idx, const unsigned long long* col_best,
                             int ratio_test, float* dists, float* weight, uint8_t* mutual, mv_stream_t stream) {
  MV_REQUIRE(A_hi && A_lo && B_hi && B_lo && row_idx, MV_E_ARG, "mv_k3_ratio_mutual_split: null pointer");
  MV_REQUIRE(C > 0 && C % 8 == 0, MV_E_ALIGN, "mv_k3_ratio_mutual_split: C=%d must be a positive multiple of 8", C);
  MV_REQUIRE((((uintptr_t)A_hi | (uintptr_t)A_lo | (uintptr_t)B_hi | (uintptr_t)B_lo) & 15) == 0, MV_E_ALIGN,
             "mv_k3_ratio_mutual_split: the row planes must be 16-byte aligned");
  MV_REQUIRE(n_max >= 0, MV_E_ARG, "mv_k3_ratio_mutual_split: negative n_max");
  if (n_max == 0) return MV_OK;
  RowsSplit rows{reinterpret_cast<const __nv_bfloat16*>(A_hi), reinterpret_cast<const __nv_bfloat16*>(A_lo),
                 reinterpret_cast<const __nv_bfloat16*>(B_hi), reinterpret_cast<const __nv_bfloat16*>(B_lo)};
  launch_ratio(rows, C, n_dev, n_max, row_idx, col_best, ratio_test, dists, weight, mutual, mv_cuda_stream(stream));
  MV_LAUNCH_CHECK();
  return MV_OK;
}

int mv_k3_ratio_mutual_f16c(const uint16_t* A_hi, const uint16_t* A_lo, const uint16_t* B_hi, const uint16_t* B_lo, int C, int pitch,
                            const float* center_B, const int32_t* n_dev, int n_max, int32_t* row_idx,
                            const unsigned long long* col_best, int ratio_test, float* dists, float* weight, uint8_t* mutual,
                            mv_stream_t stream) {
  MV_REQUIRE(A_hi && A_lo && B_hi && B_lo && row_idx, MV_E_ARG, "mv_k3_ratio_mutual_f16c: null pointer");
  MV_REQUIRE(C > 0 && C % 8 == 0, MV_E_ALIGN, "mv_k3_ratio_mutual_f16c: C=%d must be a positive multiple of 8", C);
  MV_REQUIRE((((uintptr_t)A_hi | (uintptr_t)A_lo | (uintptr_t)B_hi | (uintptr_t)B_lo | (uintptr_t)center_B) & 15) == 0, MV_E_ALIGN,
             "mv_k3_ratio_mutual_f16c: the row planes and the centre must be 16-byte aligned");
  MV_REQUIRE(n_max >= 0 && pitch >= C + 8 && pitch % 8 == 0, MV_E_ARG, "mv_k3_ratio_mutual_f16c: negative n_max or bad pitch %d", pitch);
  if (n_max == 0) return MV_OK;
  RowsF16c rows{reinterpret_cast<const __half*>(A_hi), reinterpret_cast<const __half*>(A_lo), reinterpret_cast<const __half*>(B_hi),
                reinterpret_cast<const __half*>(B_lo), center_B, pitch};
  launch_ratio(rows, C, n_dev, n_max, row_idx, col_best, ratio_test, dists, weight, mutual, mv_cuda_stream(stream));
  MV_LAUNCH_CHECK();
  return MV_OK;
}

int mv_k3_ratio_mutual_f16c_ab(const uint16_t* A_hi, const uint16_t* A_lo, const uint16_t* B_hi, const uint16_t* B_lo, int C,
                               int pitch, const float* center_A, const float* center_B, const int32_t* n_dev, int n_max,
                               int32_t* row_idx, const unsigned long long* col_best, int ratio_test, float* dists, float* weight,
                               uint8_t* mutual, mv_stream_t stream) {
  MV_REQUIRE(A_hi && A_lo && B_hi && B_lo && row_idx, MV_E_ARG, "mv_k3_ratio_mutual_f16c_ab: null pointer");
  MV_REQUIRE(C > 0 && C % 8 == 0, MV_E_ALIGN, "mv_k3_ratio_mutual_f16c_ab: C=%d must be a positive multiple of 8", C);
  MV_REQUIRE((((uintptr_t)A_hi | (uintptr_t)A_lo | (uintptr_t)B_hi | (uintptr_t)B_lo | (uintptr_t)center_A | (uintptr_t)center_B) & 15) == 0,
             MV_E_ALIGN, "mv_k3_ratio_mutual_f16c_ab: the row planes and the centres must be 16-byte aligned");
  MV_REQUIRE(n_max >= 0 && pitch >= C + 8 && pitch % 8 == 0, MV_E_ARG, "mv_k3_ratio_mutual_f16c_ab: negative n_max or bad pitch %d",
             pitch);
  if (n_max == 0) return MV_OK;
  RowsF16c rows{reinterpret_cast<const __half*>(A_hi), reinterpret_cast<const __half*>(A_lo), reinterpret_cast<const __half*>(B_hi),
                reinterpret_cast<const __half*>(B_lo), center_B, pitch, center_A};
  launch_ratio(rows, C, n_dev, n_max, row_idx, col_best, ratio_test, dists, weight, mutual, mv_cuda_stream(stream));
  MV_LAUNCH_CHECK();
  return MV_OK;
}

int mv_k3_mutual_select(const int32_t* row_idx, const float* weight_f, const int32_t* col_idx, const float* weight_r,
                        const int32_t* n_dev, int n_max, int ratio_test, int num_corr, float* weight, uint8_t* mutual,
                        int32_t* sel_src, int32_t* sel_dst, float* sel_weight, int32_t* k_dev, mv_stream_t stream) {
  MV_REQUIRE(row_idx && weight_f && col_idx && weight_r && weight && sel_src && sel_dst && sel_weight && k_dev, MV_E_ARG,
             "mv_k3_mutual_select: null pointer");
  MV_REQUIRE(n_max >= 0 && n_max <= (1 << 20), MV_E_RANGE, "mv_k3_mutual_select: n_max must be in [0, 2^20]");
  MV_REQUIRE(num_corr >= 0 && num_corr <= 16384, MV_E_RANGE, "mv_k3_mutual_select: num_corr must be in [0, 16384]");
  cudaStream_t st = mv_cuda_stream(stream);
  MV_CUDA(cudaMemsetAsync(k_dev, 0, sizeof(int32_t), st));
  if (n_max == 0 || num_corr == 0) return MV_OK;
  k3_mutual_combine_kernel<<<(n_max + 255) / 256, 256, 0, st>>>(row_idx, weight_f, col_idx, weight_r, n_dev, n_max, ratio_test, weight,
                                                                mutual, k_dev);
  MV_LAUNCH_CHECK();
  // the non-mutual queries carry -inf: the first min(num_corr, #mutual) selected are exactly the mutual ones
  int rc = mv_k3_topk_matches(weight, row_idx, n_dev, n_max, num_corr, sel_src, sel_dst, sel_weight, nullptr, stream);
  if (rc) return rc;
  k3_clamp_count_kernel<<<1, 1, 0, st>>>(k_dev, num_corr);
  MV_LAUNCH_CHECK();
  return MV_OK;
}

int mv_affinity_threshold(const float* S, int n, int m, int ld_s, float tau, float eps, float* A_out, int32_t* count, mv_stream_t stream) {
  MV_REQUIRE(S && (A_out || count), MV_E_ARG, "mv_affinity_threshold: null pointer");
  MV_REQUIRE(n >= 0 && m >= 0 && ld_s >= m, MV_E_ARG, "mv_affinity_threshold: bad sizes");
  if (n == 0) return MV_OK;
  affinity_threshold_kernel<<<(n + 7) / 8, 256, 0, mv_cuda_stream(stream)>>>(S, n, m, ld_s, tau, eps, A_out, count);
  MV_LAUNCH_CHECK();
  return MV_OK;
}

int mv_cosine_2afc(const float* ref, const float* left, const float* right, int n, int C, float* sim_left, float* sim_right,
                   int32_t* pred, mv_stream_t stream) {
  MV_REQUIRE(ref && left && right && (sim_left || sim_right || pred), MV_E_ARG, "mv_cosine_2afc: null pointer");
  MV_REQUIRE(n >= 0 && C > 0 && C % 4 == 0, MV_E_ALIGN, "mv_cosine_2afc: C=%d must be a positive multiple of 4", C);
  MV_REQUIRE((((uintptr_t)ref | (uintptr_t)left | (uintptr_t)right) & 15) == 0, MV_E_ALIGN, "mv_cosine_2afc: rows must be 16-byte aligned");
  if (n == 0) return MV_OK;
  cosine_2afc_kernel<<<(n + 7) / 8, 256, 0, mv_cuda_stream(stream)>>>(ref, left, right, n, C, sim_left, sim_right, pred);
  MV_LAUNCH_CHECK();
  return MV_OK;
}

int mv_k3_topk_matches(const float* weight, const int32_t* row_idx, const int32_t* n_dev, int n_max, int num_corr,
                       int32_t* sel_src, int32_t* sel_dst, float* sel_weight, int32_t* k_dev, mv_stream_t stream) {
  MV_REQUIRE(weight && row_idx && sel_src && sel_dst && sel_weight, MV_E_ARG, "mv_k3_topk_matches: null pointer");
  MV_REQUIRE(n_max >= 0 && n_max <= (1 << 20), MV_E_RANGE, "mv_k3_topk_matches: n_max must be in [0, 2^20]");
  MV_REQUIRE(num_corr >= 0 && num_corr <= 16384, MV_E_RANGE, "mv_k3_topk_matches: num_corr must be in [0, 16384]");
  cudaStream_t st = mv_cuda_stream(stream);
  const int kmax = num_corr < n_max ? num_corr : n_max;
  if (kmax == 0) {
    if (k_dev) MV_CUDA(cudaMemsetAsync(k_dev, 0, sizeof(int32_t), st));
    return MV_OK;
  }
  int kpad = 2;
  while (kpad < kmax) kpad <<= 1;
  const size_t smem = (size_t)(kpad > 2 * TOPK_THREADS ? kpad : 2 * TOPK_THREADS) * sizeof(unsigned long long);
  static size_t smem_set_dev[MV_MAX_DEVICES];  // the attribute is per device
  size_t& smem_set = smem_set_dev[mv_device_slot()];
  if (smem > 28 * 1024 && smem > smem_set) {  // the kernel also has ~19 KB of static shared memory
    MV_CUDA(cudaFuncSetAttribute(k3_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    smem_set = smem;
  }
  k3_topk_kernel<<<1, TOPK_THREADS, smem, st>>>(weight, row_idx, n_dev, n_max, num_corr, kpad, sel_src, sel_dst,
                                                sel_weight, k_dev);
  MV_LAUNCH_CHECK();
  return MV_OK;
}

int mv_k3_score(const int32_t* sel_src, const int32_t* sel_dst, const int32_t* k_dev, int k_max, const float* xyz0,
                const float* xyz1, const uint8_t* mutual, const float* Rt_host, const float* Kproj_host,
                const float* thr3d_host, int n3, const float* thr2d_host, int n2, float* c_xyz0, float* c_xyz1,
                float* err3d, float* err2d, unsigned long long* hits, mv_stream_t stream) {
  MV_REQUIRE(sel_src && sel_dst && xyz0 && xyz1 && Rt_host && Kproj_host && hits, MV_E_ARG, "mv_k3_score: null pointer");
  MV_REQUIRE(n3 >= 0 && n3 <= MV_MAX_THRESHOLDS && n2 >= 0 && n2 <= MV_MAX_THRESHOLDS, MV_E_RANGE,
             "mv_k3_score: at most %d thresholds per list", MV_MAX_THRESHOLDS);
  MV_REQUIRE((n3 == 0 || thr3d_host) && (n2 == 0 || thr2d_host), MV_E_ARG, "mv_k3_score: null threshold list");
  MV_REQUIRE(k_max >= 0, MV_E_ARG, "mv_k3_score: negative k_max");
  if (k_max == 0) return MV_OK;
  ScoreParams sp;
  for (int i = 0; i < 12; ++i) sp.Rt[i] = Rt_host[i];
  for (int i = 0; i < 9; ++i) sp.K[i] = Kproj_host[i];
  for (int i = 0; i < MV_MAX_THRESHOLDS; ++i) {
    sp.thr3d[i] = i < n3 ? thr3d_host[i] : 0.f;
    sp.thr2d[i] = i < n2 ? thr2d_host[i] : 0.f;
  }
  sp.n3 = n3;
  sp.n2 = n2;
  k3_score_kernel<<<(k_max + 255) / 256, 256, 0, mv_cuda_stream(stream)>>>(sel_src, sel_dst, k_dev, k_max, xyz0, xyz1,
                                                                          mutual, sp, c_xyz0, c_xyz1, err3d, err2d, hits);
  MV_LAUNCH_CHECK();
  return MV_OK;
}

int mv_gather_rows(const float* src, int width, const int32_t* idx, const int32_t* k_dev, int k_max, float* dst,
                   mv_stream_t stream) {
  MV_REQUIRE(src && idx && dst, MV_E_ARG, "mv_gather_rows: null pointer");
  MV_REQUIRE(width > 0 && k_max >= 0, MV_E_ARG, "mv_gather_rows: bad sizes");
  if (k_max == 0) return MV_OK;
  const long long total = (long long)k_max * width;
  gather_rows_kernel<<<(unsigned)((total + 255) / 256), 256, 0, mv_cuda_stream(stream)>>>(src, width, idx, k_dev, k_max, dst);
  MV_LAUNCH_CHECK();
  return MV_OK;
}

int mv_pack_matches(const int32_t* sel_src, const int32_t* sel_dst, const float* sel_weight, const int32_t* k_dev, int k_max,
                    const float* xyz0, const float* xyz1, const float* uv0, const float* uv1, const int32_t* n0_dev,
                    const int32_t* n1_dev, float* out, mv_stream_t stream) {
  MV_REQUIRE(sel_src && sel_dst && sel_weight && xyz0 && xyz1 && out, MV_E_ARG, "mv_pack_matches: null pointer");
  MV_REQUIRE((uv0 == nullptr) == (uv1 == nullptr), MV_E_ARG, "mv_pack_matches: uv0 and uv1 go together");
  MV_REQUIRE(k_max >= 0, MV_E_ARG, "mv_pack_matches: negative k_max");
  pack_matches_kernel<<<(k_max + 255) / 256 + (k_max == 0 ? 1 : 0), 256, 0, mv_cuda_stream(stream)>>>(
      sel_src, sel_dst, sel_weight, k_dev, k_max, xyz0, xyz1, uv0, uv1, n0_dev, n1_dev, out);
  MV_LAUNCH_CHECK();
  return MV_OK;
}

int mv_argmax_rows(const float* x, int rows, int cols, int max_value, int32_t* out_flat, mv_stream_t stream) {
  MV_REQUIRE(x && out_flat, MV_E_ARG, "mv_argmax_rows: null pointer");
  MV_REQUIRE(rows >= 0 && cols > 0, MV_E_ARG, "mv_argmax_rows: bad sizes");
  if (rows == 0) return MV_OK;
  argmax_rows_kernel<<<(rows + 7) / 8, 256, 0, mv_cuda_stream(stream)>>>(x, rows, cols, max_value, out_flat);
  MV_LAUNCH_CHECK();
  return MV_OK;
}

int mv_k3_spair_errors(const int32_t* pred_flat, int K, int w, const float* kps_i, const float* kps_j, int kp_stride,
                       float image_size, float thresh_scale, float pck_thresh, float* errors, float* error_same,
                       float* error_nn, int32_t* index_nn, unsigned long long* hits, unsigned long long* confusion,
                       int conf_dim, mv_stream_t stream) {
  MV_REQUIRE(pred_flat && kps_i && kps_j, MV_E_ARG, "mv_k3_spair_errors: null pointer");
  MV_REQUIRE(K >= 0 && K <= 64, MV_E_RANGE, "mv_k3_spair_errors: K=%d must be in [0, 64]", K);
  MV_REQUIRE(w > 0 && kp_stride >= 3 && image_size > 0.f, MV_E_ARG, "mv_k3_spair_errors: bad sizes");
  MV_REQUIRE(!confusion || conf_dim >= K, MV_E_ARG, "mv_k3_spair_errors: conf_dim=%d must be >= K=%d", conf_dim, K);
  if (K == 0) return MV_OK;
  k3_spair_kernel<<<1, 256, 0, mv_cuda_stream(stream)>>>(pred_flat, K, w, kps_i, kps_j, kp_stride, image_size,
                                                         thresh_scale, pck_thresh, errors, error_same, error_nn,
                                                         index_nn, hits, confusion, conf_dim);
  MV_LAUNCH_CHECK();
  return MV_OK;
}

}  // extern "C"
