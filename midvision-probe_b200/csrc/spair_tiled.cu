// spair_tiled.cu -- the tiled form of the SPair batch match (mv_spair_match_batch_tiled), for maps above 256 pixels:
// 50 x 50 at the reference's 800-pixel input with a /16 backbone, 57 x 57 with a /14 one.
//
// spair_batch.cu runs one CTA per pair.  At these shapes its key-point tile (C * KT floats, 98 KB at C = 768, K = 30) leaves
// one CTA per SM, so a batch of 16 pairs keeps 16 SMs busy, and its heat map runs on the CUDA cores.  Here one pair is
// spread over many CTAs in four launches on the caller's stream (no host sync: the sequence can be captured in a graph):
//   1. norm   (pair, 32-channel slice): partial sums of squares of f_i at the 4K tap pixels; resets the pair's arg-max slots
//   2. q      (pair, 24-channel chunk): the slices' partials summed in slice order, the blend weights folded with
//             1 / max(||f_i[tap]||, eps), q[c][k] = sum_t w_t f_i[c][tap_t] in fp32, written split into tf32 hi / lo in
//             the B-fragment order of step H (sps_q_off)
//   3. tile   (pair, key-point tile, 256-pixel tile): a producer warp streams the tile's rows of image j, 24 channels at
//             a time, together with that chunk's q fragments, through an mbarrier ring; eight consumer warps run step H
//             of the streaming form (mma.sync m16n8k8, 3xTF32 or one term) and accumulate ||f_j[p]||^2 from the A
//             fragments.  Each warp merges its per-key-point best into the pair's slot with a 64-bit atomicMax on
//             (order-preserving value bits, inverted pixel index): the largest value wins and, among equal values, the
//             lowest pixel; NaN and -inf never take part, so a heat map without a candidate leaves the slot at 0 (pixel 0),
//             the rule of the other forms.  Max is order-independent: the result does not depend on scheduling.
//   4. score  (pair): the slots become pred, then spair_score_block, once per pair.
// Channel slices, channel chunks and every per-thread summation order are fixed by C and K alone -- not by the element
// type, the batch size or the grid -- so a 16-bit map gives the bits of its fp32 widening, and a pair gives the same bits
// alone or inside any batch.
//
// Row alignment: a tile's row segment starts 16-byte aligned only when h*w * sizeof(T) % 16 == 0 (not for bf16 50 x 50,
// 5000-byte rows, nor for any odd h*w).  Each row is therefore one bulk copy of its enclosing 16-byte aligned window,
// landing at the start of its slot row, and the consumers add the row's element offset e(c) = (row start) mod (16 /
// sizeof(T)), which they compute from the same indices.  The window of the very last row may extend up to 15 bytes past
// the map's last element, inside the 16-byte granule that holds it (never onto another page).
#include <math_constants.h>

#include <type_traits>

#include "common.cuh"
#include "sm100_ptx.cuh"
#include "spair_common.cuh"
#include "spair_score.cuh"

namespace {

constexpr int SPT_WARPS = 8;                    // consumer warps: 32 pixels (two m16 tiles) each
constexpr int SPT_PIX = 32 * SPT_WARPS;         // pixels per tile
constexpr int SPT_THREADS = 32 * SPT_WARPS + 32;  // + one producer warp
constexpr int SPT_CC = 24;                      // channels per ring slot: three K steps
constexpr int SPT_SLICE = 32;                   // channels per tap-norm partial
constexpr int SPT_MAX_STAGES = 8;
constexpr int SPT_CTAS = 2;                     // CTAs per SM the tile kernel is built for (registers) and planned for (shared)
static_assert(SPT_CC % 8 == 0, "whole K steps");

// slot row pitch in elements: room for a 256-pixel window that starts up to 16 bytes early, and a pitch of 8 banks modulo 32
// (fp32: 264 floats; 16-bit: 136 words) so that the four rows t = 0..3 of an A-fragment load fall into distinct banks
template <typename T>
constexpr int spt_rs() { return sizeof(T) == 4 ? 264 : 272; }
template <typename T, int KT>
constexpr int spt_slot_bytes() { return SPT_CC * spt_rs<T>() * (int)sizeof(T) + sps_q_floats<KT, true>(SPT_CC) * 4; }

int spt_kt(int K) { return K <= 8 ? 8 : K <= 16 ? 16 : K <= 24 ? 24 : 32; }

// workspace: [B][K] arg-max slots | [B][S][4K] tap-norm partials | [B][nkt][nchunk][QF] q fragments, each 16-byte aligned
struct SptLayout {
  int KT, nkt, nchunk, S, qf;
  size_t part, q, total;
};
SptLayout spt_layout(int B, int C, int K) {
  SptLayout L;
  L.KT = spt_kt(K);
  L.nkt = (K + L.KT - 1) / L.KT;
  L.nchunk = (C + SPT_CC - 1) / SPT_CC;
  L.S = (C + SPT_SLICE - 1) / SPT_SLICE;
  L.qf = (SPT_CC / 8) * (L.KT / 8) * 128;
  auto r16 = [](size_t x) { return (x + 15) & ~(size_t)15; };
  L.part = r16((size_t)B * K * sizeof(unsigned long long));
  L.q = L.part + r16((size_t)B * L.S * 4 * K * sizeof(float));
  L.total = L.q + (size_t)B * L.nkt * L.nchunk * L.qf * sizeof(float);
  return L;
}

// ---- 1. norm: grid (B, S), thread = tap (4K of them) ----
template <typename T>
__global__ void __launch_bounds__(256) spair_tiled_norm_kernel(SpairBatchParams p, float* part, unsigned long long* best, int S) {
  const int b = blockIdx.x, s = blockIdx.y, tid = threadIdx.x, K = p.K, hw = p.h * p.w;
  if (s == 0 && tid < K) best[(size_t)b * K + tid] = 0ull;  // no candidate yet (graph replays start clean)
  if (tid >= 4 * K) return;
  int tap = 0;
  spair_taps(p.kps_i + (size_t)b * K * p.stride, tid >> 2, p.stride, p.image_size, p.h, p.w, [&](int t, float, int tp) {
    if (t == (tid & 3)) tap = tp;
  });
  const T* src = static_cast<const T*>(p.feats) + (size_t)b * 2 * p.C * hw + tap;
  const int c0 = s * SPT_SLICE, c1 = min(p.C, c0 + SPT_SLICE);
  float ss = 0.f;
#pragma unroll 16
  for (int c = c0; c < c1; ++c) {
    const float v = sp_f32(__ldg(src + (size_t)c * hw));
    ss = fmaf(v, v, ss);
  }
  part[((size_t)b * S + s) * 4 * K + tid] = ss;
}

// ---- 2. q: grid (B, nchunk) ----
template <typename T, int KT>
__global__ void __launch_bounds__(256) spair_tiled_q_kernel(SpairBatchParams p, const float* part, float* q, int S) {
  __shared__ float s_wt[64][4];  // bilinear weight / max(||f_i[tap]||, eps); 0 for a tap outside the map
  __shared__ int s_tap[64][4];
  constexpr int QF = sps_q_floats<KT, true>(SPT_CC);
  const int b = blockIdx.x, cq = blockIdx.y, nchunk = gridDim.y, tid = threadIdx.x;
  const int K = p.K, C = p.C, hw = p.h * p.w, nkt = (K + KT - 1) / KT;
  if (tid < 4 * K) {
    const int k = tid >> 2, t = tid & 3;
    float wt = 0.f;
    int tap = 0;
    spair_taps(p.kps_i + (size_t)b * K * p.stride, k, p.stride, p.image_size, p.h, p.w, [&](int tt, float w_, int tp) {
      if (tt == t) wt = w_, tap = tp;
    });
    const float* pp = part + (size_t)b * S * 4 * K + tid;
    float ss = pp[0];
    for (int s = 1; s < S; ++s) ss += pp[(size_t)s * 4 * K];  // slice order
    s_tap[k][t] = tap;
    s_wt[k][t] = __fdiv_rn(wt, fmaxf(sqrtf(ss), SPB_NORM_EPS));
  }
  __syncthreads();
  const int c0 = cq * SPT_CC, rows = min(SPT_CC, C - c0);
  const T* fi = static_cast<const T*>(p.feats) + (size_t)b * 2 * C * hw + (size_t)c0 * hw;
  for (int kt = 0; kt < nkt; ++kt) {
    float* qc = q + (((size_t)b * nkt + kt) * nchunk + cq) * QF;
    for (int idx = tid; idx < SPT_CC * KT; idx += blockDim.x) {
      const int c = idx / KT, k = idx - c * KT, kk = kt * KT + k;
      float a = 0.f;  // channels past C and key points past K: zero B-fragment entries
      if (c < rows && kk < K) {
        const T* src = fi + (size_t)c * hw;
        a = sp_f32(__ldg(src + s_tap[kk][0])) * s_wt[kk][0];
        a = fmaf(sp_f32(__ldg(src + s_tap[kk][1])), s_wt[kk][1], a);
        a = fmaf(sp_f32(__ldg(src + s_tap[kk][2])), s_wt[kk][2], a);
        a = fmaf(sp_f32(__ldg(src + s_tap[kk][3])), s_wt[kk][3], a);
      }
      uint32_t hi, lo;
      split_tf32(a, hi, lo);
      float* qd = qc + sps_q_off<KT, true>(c, k);
      qd[0] = __uint_as_float(hi);
      qd[2] = __uint_as_float(lo);
    }
  }
}

// ---- 3. tile: persistent CTAs over the work units u = ((b * nkt + kt) * npt + pixel tile) ----
struct SptTileParams {
  const void* feats;
  const float* q;
  unsigned long long* best;
  int C, hw, K, nkt, npt, nchunk, units, stages;
};

template <typename T, int KT, int TERMS>
__global__ void __launch_bounds__(SPT_THREADS, SPT_CTAS) spair_tiled_kernel(SptTileParams p) {
  using namespace sm100;
  extern __shared__ __align__(16) float4 spt_dyn[];
  __shared__ __align__(8) unsigned long long full[SPT_MAX_STAGES], empty[SPT_MAX_STAGES];
  constexpr bool F32 = std::is_same<T, float>::value;
  constexpr int NT8 = KT / 8, QF = sps_q_floats<KT, true>(SPT_CC), RS = spt_rs<T>(), AL = 16 / (int)sizeof(T);
  constexpr int ROWS_BYTES = SPT_CC * RS * (int)sizeof(T), SLOT = spt_slot_bytes<T, KT>();
  const int C = p.C, hw = p.hw, K = p.K, nstage = p.stages;
  char* ring = reinterpret_cast<char*>(spt_dyn);
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;

  if (tid == 0) {
    for (int s = 0; s < nstage; ++s) {
      mbar_init(smem_u32(&full[s]), 1);
      mbar_init(smem_u32(&empty[s]), SPT_WARPS);
    }
    mbar_fence_init();
  }
  __syncthreads();

  if (wid == SPT_WARPS) {
    // ===================================== producer warp =====================================
    // lane r < rows copies row c0 + r of the tile (its aligned window), lane 31 the chunk's q fragments
    int stage = 0;
    uint32_t phase = 0;
    for (int u = blockIdx.x; u < p.units; u += gridDim.x) {
      const int pt = u % p.npt, bk = u / p.npt, kt = bk % p.nkt, b = bk / p.nkt;
      const int p0 = pt * SPT_PIX, npx = min(SPT_PIX, hw - p0);
      const T* fj = static_cast<const T*>(p.feats) + (size_t)(2 * b + 1) * C * hw + p0;
      const float* qs = p.q + ((size_t)b * p.nkt + kt) * p.nchunk * QF;
      for (int cq = 0; cq < p.nchunk; ++cq) {
        const int c0 = cq * SPT_CC, rows = min(SPT_CC, C - c0);
        uintptr_t src = 0;
        uint32_t bytes = 0;
        if (lane < rows) {
          const uintptr_t a = reinterpret_cast<uintptr_t>(fj + (size_t)(c0 + lane) * hw);
          src = a & ~(uintptr_t)15;
          bytes = (uint32_t)(((a + (uintptr_t)npx * sizeof(T) + 15) & ~(uintptr_t)15) - src);
        } else if (lane == 31) {
          src = reinterpret_cast<uintptr_t>(qs + (size_t)cq * QF);
          bytes = QF * 4;
        }
        const uint32_t total = __reduce_add_sync(0xffffffffu, bytes);
        char* slot = ring + (size_t)stage * SLOT;
        mbar_wait(smem_u32(&empty[stage]), phase ^ 1u);
        if (lane == 0) mbar_arrive_expect_tx(smem_u32(&full[stage]), total);
        __syncwarp();
        if (lane < rows)
          bulk_load_1d_hint(smem_u32(slot + lane * RS * (int)sizeof(T)), reinterpret_cast<const void*>(src), bytes,
                            smem_u32(&full[stage]), L2_EVICT_FIRST);  // image j is read once
        else if (lane == 31)
          bulk_load_1d(smem_u32(slot + ROWS_BYTES), reinterpret_cast<const void*>(src), bytes, smem_u32(&full[stage]));
        if (++stage == nstage) { stage = 0; phase ^= 1u; }
      }
    }
    return;
  }

  // ===================================== consumers =====================================
  int stage = 0;
  uint32_t phase = 0;
  const int g = lane >> 2, t = lane & 3;
  const bool vec2 = (hw & 1) == 0;  // every row offset even: A fragments as pixel pairs
  const int hwm = hw & (AL - 1);
  for (int u = blockIdx.x; u < p.units; u += gridDim.x) {
    const int pt = u % p.npt, bk = u / p.npt, kt = bk % p.nkt, b = bk / p.nkt;
    const int p0 = pt * SPT_PIX, px0 = p0 + 32 * wid;
    const bool warp_live = px0 < hw;  // warp-uniform: this warp's 32 pixels hold at least one of the map
    const bool tile1_live = px0 + 16 < hw;
    // element offset of the tile's row c in its slot row: (index of the row's first pixel in feats) mod AL
    const int jb = (int)(((size_t)(2 * b + 1) * C * hw + p0) & (size_t)(AL - 1));
    // d[i][j][2 r + e] = heat of pixel px0 + 16 i + 2 g + r and key point 8 j + 2 t + e; ssr[i][r] = this lane's share
    // (channels t, t + 4 of every K step) of that pixel's norm
    float d[2][NT8][4];
    float ssr[2][2];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      ssr[i][0] = ssr[i][1] = 0.f;
#pragma unroll
      for (int j = 0; j < NT8; ++j) d[i][j][0] = d[i][j][1] = d[i][j][2] = d[i][j][3] = 0.f;
    }

    for (int cq = 0; cq < p.nchunk; ++cq) {
      const int c0 = cq * SPT_CC, rows = min(SPT_CC, C - c0);
      mbar_wait(smem_u32(&full[stage]), phase);
      const char* slot = ring + (size_t)stage * SLOT;
      if (warp_live) {
        const T* aj = reinterpret_cast<const T*>(slot) + 32 * wid + 2 * g;
        const float4* bq = reinterpret_cast<const float4*>(slot + ROWS_BYTES) + lane;
        // step H of the streaming form (spair_batch.cu), with each row read at its element offset
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
            const int ca = c0 + ks + t;
            const T* r0 = aj + (ks + t) * RS + ((jb + ca * hwm) & (AL - 1));
            const T* r1 = aj + (ks + t + 4) * RS + ((jb + (ca + 4) * hwm) & (AL - 1));
            float av[2][4];
#pragma unroll
            for (int i = 0; i < NTILE; ++i) {
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
                if (TERMS == 3 && F32) mma_tf32(d[i][j], al, bh[j][0], bh[j][1]);
                if (TERMS == 3) mma_tf32(d[i][j], ah, bl[j][0], bl[j][1]);
                mma_tf32(d[i][j], ah, bh[j][0], bh[j][1]);
              }
            }
          };
          if (rows == SPT_CC) {
#pragma unroll
            for (int ks = 0; ks < SPT_CC; ks += 8) kstep(ks);
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
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&empty[stage]));
      if (++stage == nstage) { stage = 0; phase ^= 1u; }
    }

    // ---- heat / max(||f_j[px]||, eps); per key point the warp's best, merged into the pair's slot ----
    if (warp_live) {
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
              const int pxl = px0 + 16 * i + 2 * g + r;  // ascending in (i, r): `>` keeps the first among equals
              const float hv = __fdiv_rn(d[i][j][2 * r + e2], ssr[i][r]);
              if (pxl < hw && hv > v) {  // NaN and -inf never win
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
          const int kg = kt * KT + 8 * j + 2 * t + e2;
          if (g == 0 && kg < K && bi != 0x7fffffff) {
            // -0 and +0 are equal values: one key for both, so that the lower pixel wins as it does between the warps' lanes
            const uint32_t vb = f32_orderable(v == 0.f ? 0.f : v);
            atomicMax(p.best + (size_t)b * K + kg, ((unsigned long long)vb << 32) | (uint32_t)~(uint32_t)bi);
          }
        }
      }
    }
  }
}

// ---- 4. score: one CTA per pair ----
__global__ void __launch_bounds__(128) spair_tiled_score_kernel(SpairBatchParams p, const unsigned long long* best) {
  __shared__ SpairScoreShared score;
  __shared__ int s_pred[64];
  const int b = blockIdx.x, K = p.K;
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    const unsigned long long v = best[(size_t)b * K + k];
    const int i = v ? (int)~(uint32_t)v : 0;  // no candidate (an all-NaN heat map): pixel 0, as in the other forms
    s_pred[k] = i;
    if (p.pred) p.pred[(size_t)b * K + k] = i;
  }
  __syncthreads();
  const float* ki = p.kps_i + (size_t)b * K * p.stride;
  const float* kj = p.kps_j + (size_t)b * K * p.stride;
  spair_score_block(score, s_pred, K, p.w, ki, kj, p.stride, p.image_size, __ldg(p.thresh_scale + b), p.pck, nullptr,
                    p.error_same ? p.error_same + (size_t)b * K : nullptr, p.error_nn ? p.error_nn + (size_t)b * K : nullptr,
                    p.index_nn ? p.index_nn + (size_t)b * K : nullptr, p.hits, p.confusion, p.conf_dim);
}

template <typename T, int KT, int TERMS>
int spt_launch_tiles(const SptTileParams& tp, cudaStream_t st) {
  constexpr size_t slot = spt_slot_bytes<T, KT>();
  // SPT_CTAS CTAs per SM: 227 KB less 1 KB reserved per CTA and the kernel's few static bytes
  const size_t budget = ((227u << 10) / SPT_CTAS) - (2u << 10);
  int stages = (int)(budget / slot);
  if (stages > SPT_MAX_STAGES) stages = SPT_MAX_STAGES;
  if (stages < 2) stages = 2;
  const size_t smem = stages * slot;
  auto kern = spair_tiled_kernel<T, KT, TERMS>;
  static size_t opted[MV_MAX_DEVICES];
  size_t& opted_in = opted[mv_device_slot()];
  if (smem > opted_in) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
      mv_set_error("mv_spair_match_batch_tiled: cannot opt in to %zu bytes of shared memory: %s", smem, cudaGetErrorString(e));
      return (int)e;
    }
    opted_in = smem;
  }
  SptTileParams ps = tp;
  ps.stages = stages;
  int grid = mv_sm_count() * SPT_CTAS;
  if (grid > ps.units) grid = ps.units;
  kern<<<grid, SPT_THREADS, smem, st>>>(ps);
  MV_LAUNCH_CHECK();
  return MV_OK;
}

template <typename T, int KT>
int spt_launch(const SpairBatchParams& p, const SptLayout& L, char* ws, cudaStream_t st) {
  unsigned long long* best = reinterpret_cast<unsigned long long*>(ws);
  float* part = reinterpret_cast<float*>(ws + L.part);
  float* q = reinterpret_cast<float*>(ws + L.q);
  const int hw = p.h * p.w;
  spair_tiled_norm_kernel<T><<<dim3(p.B, L.S), (4 * p.K + 31) / 32 * 32, 0, st>>>(p, part, best, L.S);
  MV_LAUNCH_CHECK();
  spair_tiled_q_kernel<T, KT><<<dim3(p.B, L.nchunk), 256, 0, st>>>(p, part, q, L.S);
  MV_LAUNCH_CHECK();
  SptTileParams tp;
  tp.feats = p.feats;
  tp.q = q;
  tp.best = best;
  tp.C = p.C;
  tp.hw = hw;
  tp.K = p.K;
  tp.nkt = L.nkt;
  tp.npt = (hw + SPT_PIX - 1) / SPT_PIX;
  tp.nchunk = L.nchunk;
  tp.units = p.B * L.nkt * tp.npt;
  tp.stages = 0;
  const int rc = spair_heatmap_terms() == 1 ? spt_launch_tiles<T, KT, 1>(tp, st) : spt_launch_tiles<T, KT, 3>(tp, st);
  if (rc != MV_OK) return rc;
  spair_tiled_score_kernel<<<p.B, 128, 0, st>>>(p, best);
  MV_LAUNCH_CHECK();
  return MV_OK;
}

}  // namespace

size_t spair_tiled_workspace_bytes(int B, int C, int K) {
  if (B == 0 || K == 0) return 0;
  return spt_layout(B, C, K).total + 16;  // + room to align the caller's pointer to 16 bytes
}

template <typename T>
int spair_tiled_launch(const SpairBatchParams& p, void* workspace, cudaStream_t st) {
  const SptLayout L = spt_layout(p.B, p.C, p.K);
  const long long units = (long long)p.B * L.nkt * ((p.h * p.w + SPT_PIX - 1) / SPT_PIX);
  MV_REQUIRE(units <= 0x7fffffff, MV_E_RANGE, "mv_spair_match_batch_tiled: B=%d too large", p.B);
  char* ws = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(workspace) + 15) & ~(uintptr_t)15);
  switch (L.KT) {
    case 8: return spt_launch<T, 8>(p, L, ws, st);
    case 16: return spt_launch<T, 16>(p, L, ws, st);
    case 24: return spt_launch<T, 24>(p, L, ws, st);
    default: return spt_launch<T, 32>(p, L, ws, st);
  }
}
template int spair_tiled_launch<float>(const SpairBatchParams&, void*, cudaStream_t);
template int spair_tiled_launch<__nv_bfloat16>(const SpairBatchParams&, void*, cudaStream_t);
template int spair_tiled_launch<__half>(const SpairBatchParams&, void*, cudaStream_t);
