// knn_rerank.cu -- fp32 re-rank of the k-NN candidates that kernel 2's top-KP epilogue proposes (mv_k2_sim_topk_ld).
//
// The tensor cores only propose: for every query the KP candidate columns are re-scored from the fp32 rows, in the
// reference's arithmetic, sorted ascending (ties: lower index) and the first k kept -- the k > 2 form of what kernel 3
// does for two candidates (evals/utils/correspondence.py:53-58).
//   MV_METRIC_L2SQ    sum_c (q_c - t_c)^2                                 (faiss' squared L2, correspondence.py:14-23)
//   MV_METRIC_COSINE  1 - q.t / (max(|q|, 1e-8) max(|t|, 1e-8))            (F.cosine_similarity, correspondence.py:58)
// One warp per query; lane j < KP ends up holding candidate j's distance and the sort is a rank count over the lanes.
#include <math_constants.h>

#include "common.cuh"

namespace {

constexpr float COS_EPS = 1e-8f;  // torch.nn.functional.cosine_similarity default eps
constexpr int WARPS = 8;

// Row loads: VEC = 128-bit (C, both pitches multiples of 4 floats, 16-byte aligned rows), otherwise one float per lane.
template <bool VEC, bool COS>
__global__ void __launch_bounds__(WARPS * 32) knn_rerank_kernel(const float* __restrict__ Q, int ldq, const float* __restrict__ T,
                                                                 int ldt, int C, const int32_t* __restrict__ n_dev, int n_max,
                                                                 const int32_t* __restrict__ cand, int kp, int k,
                                                                 float* __restrict__ out_dist, int32_t* __restrict__ out_idx) {
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * WARPS + (threadIdx.x >> 5);
  if (i >= n_max) return;
  const int n = n_dev ? min(*n_dev, n_max) : n_max;
  float* dst_d = out_dist + (size_t)i * k;
  int32_t* dst_i = out_idx + (size_t)i * k;
  if (i >= n) {
    if (lane < k) {
      dst_d[lane] = CUDART_INF_F;
      dst_i[lane] = -1;
    }
    return;
  }
  const float* q = Q + (size_t)i * ldq;
  float qq = 0.f;
  if (COS) {
    if (VEC) {
      for (int c = 4 * lane; c < C; c += 128) {
        const float4 x = __ldg(reinterpret_cast<const float4*>(q + c));
        qq = fmaf(x.x, x.x, qq); qq = fmaf(x.y, x.y, qq); qq = fmaf(x.z, x.z, qq); qq = fmaf(x.w, x.w, qq);
      }
    } else {
      for (int c = lane; c < C; c += 32) qq = fmaf(q[c], q[c], qq);
    }
    qq = warp_sum(qq);
  }
  float my_d = CUDART_INF_F;
  int my_j = -1;
  for (int j = 0; j < kp; ++j) {
    const int cj = __ldg(cand + (size_t)i * kp + j);
    if (cj < 0) continue;  // warp-uniform
    const float* t = T + (size_t)cj * ldt;
    float s = 0.f, tt = 0.f;
    if (VEC) {
#pragma unroll 2  // the compiler's default unroll of 4 spills 4 bytes in the L2 form
      for (int c = 4 * lane; c < C; c += 128) {
        const float4 x = __ldg(reinterpret_cast<const float4*>(q + c));
        const float4 y = __ldg(reinterpret_cast<const float4*>(t + c));
        if (COS) {
          s = fmaf(x.x, y.x, s); s = fmaf(x.y, y.y, s); s = fmaf(x.z, y.z, s); s = fmaf(x.w, y.w, s);
          tt = fmaf(y.x, y.x, tt); tt = fmaf(y.y, y.y, tt); tt = fmaf(y.z, y.z, tt); tt = fmaf(y.w, y.w, tt);
        } else {
          const float d0 = x.x - y.x, d1 = x.y - y.y, d2 = x.z - y.z, d3 = x.w - y.w;
          s = fmaf(d0, d0, s); s = fmaf(d1, d1, s); s = fmaf(d2, d2, s); s = fmaf(d3, d3, s);
        }
      }
    } else {
      for (int c = lane; c < C; c += 32) {
        const float x = q[c], y = t[c];
        if (COS) {
          s = fmaf(x, y, s);
          tt = fmaf(y, y, tt);
        } else {
          const float d = x - y;
          s = fmaf(d, d, s);
        }
      }
    }
    s = warp_sum(s);
    float dist = s;
    if (COS) {
      tt = warp_sum(tt);
      dist = 1.f - s / (fmaxf(sqrtf(qq), COS_EPS) * fmaxf(sqrtf(tt), COS_EPS));
    }
    if (lane == j) {
      my_d = dist;
      my_j = cj;
    }
  }
  // rank of every live candidate among the live ones: ascending distance, ties to the lower index
  int rank = 0;
  for (int l = 0; l < kp; ++l) {
    const float dl = __shfl_sync(0xffffffffu, my_d, l);
    const int jl = __shfl_sync(0xffffffffu, my_j, l);
    rank += (jl >= 0 && (dl < my_d || (dl == my_d && jl < my_j))) ? 1 : 0;
  }
  const int live = __popc(__ballot_sync(0xffffffffu, my_j >= 0));
  if (my_j >= 0 && rank < k) {
    dst_d[rank] = my_d;
    dst_i[rank] = my_j;
  }
  if (lane >= live && lane < k) {  // fewer live candidates than k: faiss' (inf, -1)
    dst_d[lane] = CUDART_INF_F;
    dst_i[lane] = -1;
  }
}

}  // namespace

extern "C" {

int mv_knn_rerank(const float* Q, int ldq, const float* T, int ldt, int C, const int32_t* n_dev, int n_max, const int32_t* cand,
                  int kp, int k, int metric, float* out_dist, int32_t* out_idx, mv_stream_t stream) {
  MV_REQUIRE(Q && T && cand && out_dist && out_idx, MV_E_ARG, "mv_knn_rerank: null pointer");
  MV_REQUIRE(metric == MV_METRIC_L2SQ || metric == MV_METRIC_COSINE, MV_E_ARG, "mv_knn_rerank: unknown metric %d", metric);
  MV_REQUIRE(kp == 8 || kp == 16, MV_E_RANGE, "mv_knn_rerank: kp=%d must be 8 or 16", kp);
  MV_REQUIRE(k >= 1 && k <= kp, MV_E_RANGE, "mv_knn_rerank: k=%d must be in [1, kp=%d]", k, kp);
  MV_REQUIRE(C > 0 && ldq >= C && ldt >= C, MV_E_ARG, "mv_knn_rerank: C must be positive and the row pitches >= C");
  MV_REQUIRE(n_max >= 0 && n_max <= (1 << 20), MV_E_RANGE, "mv_knn_rerank: n_max must be in [0, 2^20]");
  if (n_max == 0) return MV_OK;
  const bool vec = C % 4 == 0 && ldq % 4 == 0 && ldt % 4 == 0 && ((uintptr_t)Q & 15) == 0 && ((uintptr_t)T & 15) == 0;
  const bool cos = metric == MV_METRIC_COSINE;
  const dim3 grid((n_max + WARPS - 1) / WARPS), block(WARPS * 32);
  cudaStream_t st = mv_cuda_stream(stream);
  if (vec && cos) knn_rerank_kernel<true, true><<<grid, block, 0, st>>>(Q, ldq, T, ldt, C, n_dev, n_max, cand, kp, k, out_dist, out_idx);
  else if (vec) knn_rerank_kernel<true, false><<<grid, block, 0, st>>>(Q, ldq, T, ldt, C, n_dev, n_max, cand, kp, k, out_dist, out_idx);
  else if (cos) knn_rerank_kernel<false, true><<<grid, block, 0, st>>>(Q, ldq, T, ldt, C, n_dev, n_max, cand, kp, k, out_dist, out_idx);
  else knn_rerank_kernel<false, false><<<grid, block, 0, st>>>(Q, ldq, T, ldt, C, n_dev, n_max, cand, kp, k, out_dist, out_idx);
  MV_LAUNCH_CHECK();
  return MV_OK;
}

}  // extern "C"
