// k2_sim.cu -- kernel 2: S = A @ B^T on tcgen05 tensor cores with the row top-2 and the column arg-max
// fused into the epilogue.  The n x m similarity matrix only ever exists as 128 x 256 fp32 tiles in TMEM.
//
// Replaces, for L2-normalised rows (where the L2 order is the cosine order, correspondence.py:27-43):
//   evals/utils/correspondence.py:14-23   faiss.GpuIndexFlatL2(res, C).add(target).search(query, k<=2)
//   evaluate_spair_correspondence.py:82-83 einsum("k f, f h w -> k h w") + argmax_2d   (row arg-max)
//
// Structure (one persistent CTA per SM, 20 warps, warp-specialised):
//   warp 0      TMA producer : A tile 128 x 128B and B tile 256 x 128B per k-block into a 4-stage
//                              128B-swizzled shared-memory ring; with MC > 1 the B tile is loaded in MC
//                              slices, each multicast to the MC CTAs of the cluster (they work on MC
//                              consecutive row blocks and the same column tile)
//   warp 1      MMA issuer   : one thread, tcgen05.mma M=128 N=256 K=16 (bf16) / K=8 (tf32), fp32
//                              accumulators in TMEM, two accumulator buffers (2 x 256 = all 512 columns)
//   warp 2      TMEM allocator
//   warps 4..19 epilogue     : four warps per TMEM lane quarter, each owning a quarter of the tile's columns;
//                              tcgen05.ld 32 rows x 16 columns per warp; thread = one row of S.  (Round 2: 16 warps
//                              instead of 8 -- the epilogue was latency-bound at IPC 1.2 per SM; 19200^2 x 768 went
//                              from 0.411 to 0.384 ms, the 312-column low-rank product from 0.328 to 0.277 ms.)
//                              rows   : running (max1, idx1, max2, idx2) in registers across the column
//                                       tiles of a row block; a chunk is only scanned when its maximum
//                                       beats the current second best
//                              columns: warp-wide max in one CREDUX.MAX.F32 + ballot for the owning row,
//                                       4 warps combined through shared memory, then one packed
//                                       (orderable value << 32 | ~row) atomicMax per column per tile,
//                                       skipped when a plain load already shows a better entry
// Scheduling: the (super row block, column tile) list is cut into gridDim/MC equal contiguous ranges, so
// every SM gets the same number of tiles (+-1); a row block that is split between CTAs leaves partial
// top-2 records in the workspace which k2_merge_rows_kernel folds (ties: lower column).
//
// The same main loop also serves k > 2 nearest neighbours (k2_sim_topk_kernel, mv_k2_sim_topk_ld): its epilogue keeps
// the KP (8 or 16) best columns of every row in registers -- a list sorted descending, updated by an unrolled
// compare-and-shift -- and does no column work.  A chunk is only looked at when its maximum beats the list's last entry;
// then its best column is inserted and knocked out until none beats it.  Partial lists go to the workspace like the
// top-2 records and k2_merge_topk_kernel folds them into (n_max, KP) outputs.  Stream-K is never used there.
#include <cuda.h>

#include <stdlib.h>

#include <vector>
#include <math_constants.h>

#include "common.cuh"
#include "sm100_ptx.cuh"

namespace {

using namespace sm100;

constexpr int BM = 128;           // rows of S per tile (UMMA M)
constexpr int BN = 256;           // columns of S per tile (UMMA N)
constexpr int ROW_BYTES = 128;    // one swizzle-128B row: 64 bf16 or 32 fp32 along K
constexpr int A_STAGE_BYTES = BM * ROW_BYTES;  // 16 KB
// single-CTA tiles keep the whole 256-row B tile per stage (48 KB, 4 stages); a CTA pair (cta_group::2) keeps
// only its half of B (32 KB, 6 stages): the tensor cores of both SMs read both halves
constexpr int MAX_STAGES = 6;
#ifndef MV_K2_PAIR_STAGES
// 6 stages = 192 KB ring.  4 stages (128 KB) run the NAVI shape equally fast (1298 vs 1303 TFLOP/s) and would let a
// 72 KB kernel-1 CTA share the SM; measured in the 3-lane pipeline that co-residency LOSES 4 % pairs/s (the small
// kernel-1 configuration is slower and kernel 2 drops from 1188 to 1160 TFLOP/s), so the deep ring stays.
#define MV_K2_PAIR_STAGES 6
#endif
template <bool PAIR> struct Ring {
  static constexpr int B_ROWS = PAIR ? BN / 2 : BN;
  static constexpr int STAGE_BYTES = A_STAGE_BYTES + B_ROWS * ROW_BYTES;
  static constexpr int STAGES = PAIR ? MV_K2_PAIR_STAGES : 4;
  static constexpr int BYTES = STAGES * STAGE_BYTES;
};
constexpr int K2_THREADS = 640;   // 4 control warps + 16 epilogue warps
constexpr int EPI_PARTS = 4;      // epilogue warps per TMEM lane quarter: each owns 256 / EPI_PARTS columns of the tile
constexpr int EPI_CW = 16;        // columns per TMEM read (chunk)
constexpr int PART_COLS = BN / EPI_PARTS, PART_CHUNKS = PART_COLS / EPI_CW;
constexpr int EPI_WARP0 = 4;
constexpr int COL_SMEM_BYTES = 2 * 4 * BN * 8;  // [2 buffers][4 warps][256 columns] (max bits, ballot)
// Epilogue shape of a kernel variant: KP == 0 is the top-2 + column arg-max epilogue above; KP > 0 the row top-KP one.
template <int KP> struct Epi {
  // a 16-entry list (32 registers) spills at the 96 registers of 20 warps: 12 warps, 168 registers
  static constexpr int PARTS = KP == 16 ? 2 : EPI_PARTS;
  static constexpr int THREADS = 32 * EPI_WARP0 + 128 * PARTS;
  static constexpr int CHUNKS = BN / PARTS / EPI_CW;
};
static_assert(Epi<0>::THREADS == K2_THREADS, "the top-2 kernel keeps its 20 warps");
template <bool PAIR> constexpr int k2_smem_bytes() { return 1024 /*align slack*/ + Ring<PAIR>::BYTES + COL_SMEM_BYTES + 256 /*barriers*/; }

struct K2Sched {
  // tiles are numbered t = sb * n_ct + ct and cut into tk work UNITS each; cluster c owns the units
  // [c*W/G, (c+1)*W/G).  Built on the device from the LIVE row counts, so a problem whose counts only exist in
  // device memory is balanced like any other.
  //   tk == 1       : a unit is a tile (every SM gets the same number of tiles +-1)
  //   tk == kblocks : "stream-K": a unit is one k-block of a tile, so every SM gets the same number of k-blocks
  //                   +-1.  A cluster whose range starts inside a tile computes that tile's LAST k-blocks first
  //                   (its head fragment), stores the raw accumulators to the workspace and raises a flag; the
  //                   cluster that holds the tile's k-block 0 OWNS the tile: it runs the fused epilogue on its
  //                   own accumulators + that fragment.  Chosen when a cluster has few tiles (the NAVI shape:
  //                   5.4 tiles per SM would otherwise cost the time of 6).
  unsigned long long T;  // n_sb * n_ct
  unsigned long long W;  // T * tk
  int G;                 // clusters that own work: min(clusters in the grid, T)
  int n_ct;              // column tiles
  int n_sb;              // super row blocks (MC * 128 rows)
  int tk;                // units per tile
};
constexpr int SK_MIN_KBLOCKS = 8;         // stream-K only when a tile has enough k-blocks to be worth cutting
constexpr int SK_MAX_TILES_PER_CLUSTER = 16;  // ... and few enough tiles per cluster for the tail to matter
constexpr int FRAG_BYTES = BM * BN * 4;   // raw accumulators of one CTA's 128 x 256 tile

struct K2Params {
  const int32_t* n_dev;
  const int32_t* m_dev;
  int n_max, m_max, kblocks;
  int tail_steps;   // MMA K-steps that carry data in the LAST k-block (1..4): K extents need not fill the 128-byte row
  uint32_t ab_fmt;  // tcgen05 instruction-descriptor operand format: 0 = fp16, 1 = bf16 (kind::f16), 2 = tf32
  int clusters;     // clusters in the grid
  int streamk;      // 1 = the schedule may cut tiles along K (see K2Sched)
  float4* frag;     // gridDim.x slots of FRAG_BYTES: head-fragment accumulators, slot = contributing CTA
  uint32_t* flags;  // gridDim.x flags, zeroed before the launch: 1 = the CTA's head fragment is in memory
  float4* partial;  // (clusters + n_sb_max) slots of MC * 128 rows x 2 column halves of {max1, idx1, max2, idx2}; slot = cluster + sb
  unsigned long long* col_best;
  float* S_out;     // optional (n_max, ld_s) fp32: the similarity tile is also written out (affinity consumers, mv_k2_affinity)
  int ld_s;
};

__host__ __device__ inline K2Sched make_sched(int n, int m, int mc, int clusters, int kblocks, int streamk) {
  K2Sched s;
  s.n_sb = (n + 128 * mc - 1) / (128 * mc);
  s.n_ct = (m + 256 - 1) / 256;
  s.T = (unsigned long long)s.n_sb * s.n_ct;
  // every cluster below G owns at least one tile, so the clusters that share a row block are consecutive
  s.G = clusters;
  if ((unsigned long long)s.G > s.T) s.G = (int)s.T;
  if (s.G < 1) s.G = 1;
  // T >= G makes every range at least one tile's worth of units long: a tile is shared by at most two clusters and
  // every cluster holds the k-block 0 of at least one tile
  const bool sk = streamk && kblocks >= SK_MIN_KBLOCKS && s.T % (unsigned long long)s.G != 0 &&
                  s.T < (unsigned long long)SK_MAX_TILES_PER_CLUSTER * (unsigned long long)s.G;
  s.tk = sk ? kblocks : 1;
  s.W = s.T * (unsigned long long)s.tk;
  return s;
}

// first unit of cluster c
__host__ __device__ inline unsigned long long sched_begin(const K2Sched& s, int c) {
  return (unsigned long long)c * s.W / (unsigned long long)s.G;
}
// cluster that owns tile t (the one whose range holds the tile's first unit)
__host__ __device__ inline int sched_owner(const K2Sched& s, unsigned long long t) {
  const unsigned long long u = t * (unsigned long long)s.tk;
  return (int)(((u + 1) * (unsigned long long)s.G + s.W - 1) / s.W) - 1;
}

__device__ __forceinline__ bool better(float x, int j, float y, int k) {
  return x > y || (x == y && (unsigned)j < (unsigned)k);
}

// Insert (x, j) into a list sorted descending, dropping its last entry.  Static indices only: the list stays in registers.
// BY_INDEX = false compares values alone, for candidates that arrive in ascending column order (an equal value then
// already sits in the list with a lower column); true breaks ties by the lower column (better()).
template <int KP, bool BY_INDEX>
__device__ __forceinline__ void list_insert(float (&lv)[KP], int (&li)[KP], float x, int j) {
  bool up[KP];  // x goes above entry r
#pragma unroll
  for (int r = 0; r < KP; ++r) up[r] = BY_INDEX ? better(x, j, lv[r], li[r]) : x > lv[r];
#pragma unroll
  for (int r = KP - 1; r > 0; --r) {
    lv[r] = up[r - 1] ? lv[r - 1] : (up[r] ? x : lv[r]);
    li[r] = up[r - 1] ? li[r - 1] : (up[r] ? j : li[r]);
  }
  lv[0] = up[0] ? x : lv[0];
  li[0] = up[0] ? j : li[0];
}

struct __align__(8) Barriers {
  unsigned long long full[MAX_STAGES];
  unsigned long long empty[MAX_STAGES];
  unsigned long long tmem_full[2];
  unsigned long long tmem_empty[2];
  uint32_t tmem_base;
};

// MC: CTAs per cluster (consecutive row blocks of one super row block).  PAIR (MC == 2): the two CTAs form a
// cta_group::2 pair -- ONE 256 x 256 MMA per k-step issued by the rank-0 CTA, each CTA supplying its 128 rows of
// A and its 128 of the 256 columns of B and receiving its 128 rows of the accumulator in its own TMEM.
// KP selects the epilogue (Epi<KP>); the producer, MMA issuer, TMEM allocation and schedule are shared.
template <bool TF32, int MC, bool PAIR, int KP>
__device__ __forceinline__ void k2_body(const CUtensorMap& tmA, const CUtensorMap& tmB, const K2Params& p) {
  static_assert(!PAIR || MC == 2, "a CTA pair is a cluster of two");
  static_assert(KP == 0 || KP == 8 || KP == 16, "row lists of 8 or 16 entries");
  constexpr int STAGES = Ring<PAIR>::STAGES;
  constexpr int STAGE_BYTES = Ring<PAIR>::STAGE_BYTES;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_al = smem_raw + (smem_base - smem_u32(smem_raw));
  constexpr int RING_BYTES = Ring<PAIR>::BYTES;
  uint2* col_smem = reinterpret_cast<uint2*>(smem_al + RING_BYTES);
  Barriers* bars = reinterpret_cast<Barriers*>(smem_al + RING_BYTES + COL_SMEM_BYTES);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rank = (MC > 1) ? (int)cluster_ctarank() : 0;
  const int cluster_id = blockIdx.x / MC;
  const int n = p.n_dev ? min(*p.n_dev, p.n_max) : p.n_max;
  const int m = p.m_dev ? min(*p.m_dev, p.m_max) : p.m_max;

  // clusters beyond sch.G (fewer tiles than clusters) own nothing
  const K2Sched sch = make_sched(n, m, MC, p.clusters, p.kblocks, KP ? 0 : p.streamk);
  const bool has_work = cluster_id < sch.G && sch.T > 0;
  const unsigned long long u_beg = has_work ? sched_begin(sch, cluster_id) : 0ull;
  const unsigned long long u_end = has_work ? sched_begin(sch, cluster_id + 1) : 0ull;
  const unsigned tk = (unsigned)sch.tk;
  // stream-K pieces of this cluster's range (all zero when tk == 1): the head fragment = k-blocks [head_k0, kblocks) of
  // tile head_tile, computed FIRST and handed to the previous cluster; the owned tiles [t_beg, t_end); the last owned
  // tile only up to k-block tail_k (the next cluster's head fragment supplies the rest), computed LAST
  const int head_k0 = (int)(u_beg % tk);
  const unsigned long long head_tile = u_beg / tk;
  const int tail_k = (int)(u_end % tk);
  const unsigned long long t_beg = (u_beg + tk - 1) / tk;
  const unsigned long long t_end = (u_end + tk - 1) / tk;
  // The range is walked starting at its first row-block boundary and wrapping around, so that every CTA sweeps
  // the column tiles in phase (all at column ~s mod n_ct at step s): the B tiles in flight are then the same
  // few for the whole chip and the L2 working set is the active A blocks + a narrow window of B, instead of
  // all of B (which overflows the 126 MB L2 once (n + m) * C * 2 bytes does).
  const unsigned long long t_len = t_end - t_beg;
  unsigned long long t_rot = (t_beg + (unsigned)sch.n_ct - 1) / (unsigned)sch.n_ct * (unsigned)sch.n_ct;
  if (t_rot >= t_end || tk > 1) t_rot = t_beg;  // stream-K keeps the order: the tail tile has to come last
  const unsigned long long t_head = t_end - t_rot;  // steps [0, t_head) map to [t_rot, t_end), the rest to [t_beg, t_rot)
#define MV_K2_TILE_AT(step) ((step) < t_head ? t_rot + (step) : t_beg + ((step) - t_head))
  // work items of this cluster, in execution order: [head fragment] + owned tiles
  const unsigned long long n_items = t_len + (head_k0 ? 1u : 0u);
  struct Item {
    unsigned long long t;
    int kb0, kb1;
    int kind;  // 0 = whole tile, 1 = head fragment (store the accumulators), 2 = tail tile (add the next cluster's fragment)
  };
  auto item_at = [&](unsigned long long s) -> Item {
    Item it;
    if (head_k0) {
      if (s == 0) {
        it.t = head_tile; it.kb0 = head_k0; it.kb1 = p.kblocks; it.kind = 1;
        return it;
      }
      s -= 1;
    }
    it.t = MV_K2_TILE_AT(s);
    const bool last = tail_k != 0 && s + 1 == t_len;
    it.kb0 = 0;
    it.kb1 = last ? tail_k : p.kblocks;
    it.kind = last ? 2 : 0;
    return it;
  };
  constexpr int KE = TF32 ? 32 : 64;  // K elements per 128-byte row

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(smem_u32(&bars->full[s]), 1);
      mbar_init(smem_u32(&bars->empty[s]), PAIR ? 1 : MC);  // PAIR: one multicast commit of the pair's MMA
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(smem_u32(&bars->tmem_full[a]), 1);
      mbar_init(smem_u32(&bars->tmem_empty[a]), PAIR ? 8 * Epi<KP>::PARTS : 4 * Epi<KP>::PARTS);  // PAIR: the epilogue warps of BOTH CTAs (rank 0's barrier)
    }
    mbar_fence_init();
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 2) {
    if (PAIR) tmem_alloc_512_pair(smem_u32(&bars->tmem_base));
    else tmem_alloc_512(smem_u32(&bars->tmem_base));
  }
  tc_fence_before();
  if (MC > 1) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(&bars->tmem_base);

  if (warp == 0) {
    // ===================================== TMA producer =====================================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (unsigned long long step = 0; step < n_items; ++step) {
        const Item it = item_at(step);
        const unsigned long long t = it.t;
        const int sb = (int)(t / (unsigned)sch.n_ct), ct = (int)(t - (unsigned long long)sb * sch.n_ct);
        const int row0 = (sb * MC + rank) * BM, col0 = ct * BN;
        for (int kb = it.kb0; kb < it.kb1; ++kb) {
          mbar_wait(smem_u32(&bars->empty[stage]), phase ^ 1u);
          const uint32_t full = smem_u32(&bars->full[stage]);
          const uint32_t sa = smem_base + stage * STAGE_BYTES, sbm = sa + A_STAGE_BYTES;
          if (PAIR) {
            // both CTAs' loads complete on rank 0's barrier, which expects the bytes of the whole pair
            const uint32_t full0 = map_to_cta(full, 0);
            if (rank == 0) mbar_arrive_expect_tx(full, 2 * STAGE_BYTES);
            tma_load_2d_pair(sa, &tmA, full0, kb * KE, row0);
            tma_load_2d_pair(sbm, &tmB, full0, kb * KE, col0 + rank * (BN / 2));
            if (++stage == STAGES) { stage = 0; phase ^= 1u; }
            continue;
          }
          mbar_arrive_expect_tx(full, STAGE_BYTES);
          tma_load_2d(sa, &tmA, full, kb * KE, row0);
          if (MC == 1) {
            tma_load_2d(sbm, &tmB, full, kb * KE, col0);
          } else {
            constexpr int SLICE = BN / MC;
            tma_load_2d_mc(sbm + rank * SLICE * ROW_BYTES, &tmB, full, kb * KE, col0 + rank * SLICE,
                           (uint16_t)((1u << MC) - 1));
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================================== MMA issuer =======================================
    // The whole warp walks the (warp-uniform) loop; one elected lane issues.  Everything the issuing thread
    // executes per k-block is a barrier wait, two integer multiply-adds and ONE asm block.
    const uint32_t idesc = umma_idesc((int)p.ab_fmt, PAIR ? 2 * BM : BM, BN);
    const int kb_last = p.kblocks - 1;
    const uint32_t tail_steps = (uint32_t)p.tail_steps;
    const uint64_t desc0 = umma_desc_sw128(smem_base);  // stage 0, A tile; later tiles add (bytes >> 4) to the low word
    const bool leader = elect_one() && (!PAIR || rank == 0);  // PAIR: only the rank-0 CTA issues
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (unsigned long long step = 0; (!PAIR || rank == 0) && step < n_items; ++step) {
      const Item it = item_at(step);
      const int kb_first = it.kb0;
      mbar_wait(smem_u32(&bars->tmem_empty[acc]), acc_phase ^ 1u);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)acc * BN;
      for (int kb = it.kb0; kb < it.kb1; ++kb) {
        mbar_wait(smem_u32(&bars->full[stage]), phase);
        tc_fence_after();
        if (leader) {
          const uint64_t da = desc0 + (uint64_t)((uint32_t)stage * (STAGE_BYTES >> 4));
          const uint64_t db = da + (uint64_t)(A_STAGE_BYTES >> 4);
          if (kb == kb_last && tail_steps < 4u) {  // partial last k-block (e.g. the 8 augmentation columns of f16c rows)
            umma_kblock_tail<TF32, PAIR ? 2 : (MC == 1 ? 0 : 1)>(d_tmem, da, db, idesc, (uint32_t)(kb != kb_first), smem_u32(&bars->empty[stage]),
                                                               (uint16_t)((1u << MC) - 1), tail_steps);
          } else if (PAIR) umma_kblock_pair<TF32>(d_tmem, da, db, idesc, (uint32_t)(kb != kb_first), smem_u32(&bars->empty[stage]));
          else if (MC == 1) umma_kblock<TF32>(d_tmem, da, db, idesc, (uint32_t)(kb != kb_first), smem_u32(&bars->empty[stage]));
          else umma_kblock_mc<TF32>(d_tmem, da, db, idesc, (uint32_t)(kb != kb_first), smem_u32(&bars->empty[stage]),
                                    (uint16_t)((1u << MC) - 1));
        }
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
      if (leader) {
        if (PAIR) umma_commit_pair(smem_u32(&bars->tmem_full[acc]), (uint16_t)3);
        else umma_commit(smem_u32(&bars->tmem_full[acc]));
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1u;
    }
  } else if (KP > 0 && warp >= EPI_WARP0) {
    if constexpr (KP > 0) {
      // ================================ top-KP epilogue (rows only) ================================
      // same warp layout as the top-2 epilogue: Epi<KP>::PARTS warps per TMEM lane quarter, thread = one row of the tile
      // and one column part.  Columns reach a thread in ascending order within a row block, so value comparisons alone
      // keep ties on the lower column.
      constexpr int PARTS = Epi<KP>::PARTS, CHUNKS = Epi<KP>::CHUNKS;
      const int ew = warp & 3;
      const int part = (warp - EPI_WARP0) >> 2;
      const int e = ew * 32 + lane;
      float lv[KP];
      int li[KP];
      int cur_sb = -1;
      int acc = 0;
      uint32_t acc_phase = 0;
      auto flush = [&](int sb) {
        float4* dst = p.partial + (((size_t)(cluster_id + sb) * (BM * MC) + rank * BM + e) * PARTS + part) * (KP / 2);
#pragma unroll
        for (int r = 0; r < KP / 2; ++r)
          dst[r] = make_float4(lv[2 * r], __int_as_float(li[2 * r]), lv[2 * r + 1], __int_as_float(li[2 * r + 1]));
      };
      auto chunk_max = [](const float (&v)[EPI_CW]) {
        float g[EPI_CW / 2];
#pragma unroll
        for (int q = 0; q < EPI_CW / 2; ++q) g[q] = fmaxf(v[2 * q], v[2 * q + 1]);
#pragma unroll
        for (int w = EPI_CW / 4; w > 0; w >>= 1)
#pragma unroll
          for (int q = 0; q < w; ++q) g[q] = fmaxf(g[q], g[q + w]);
        return g[0];
      };
      for (unsigned long long step = 0; step < n_items; ++step) {
        const unsigned long long t = item_at(step).t;
        const int sb = (int)(t / (unsigned)sch.n_ct), ct = (int)(t - (unsigned long long)sb * sch.n_ct);
        if (sb != cur_sb) {
          if (cur_sb >= 0) flush(cur_sb);
#pragma unroll
          for (int r = 0; r < KP; ++r) {
            lv[r] = -CUDART_INF_F;
            li[r] = -1;
          }
          cur_sb = sb;
        }
        const int row0 = (sb * MC + rank) * BM, col0 = ct * BN;
        const bool edge = (row0 + BM > n) || (col0 + BN > m);
        const bool row_ok = row0 + e < n;

        mbar_wait(smem_u32(&bars->tmem_full[acc]), acc_phase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + (uint32_t)acc * BN + ((uint32_t)(ew * 32) << 16);
#pragma unroll 1
        for (int ch = part * CHUNKS; ch < (part + 1) * CHUNKS; ++ch) {
          float v[EPI_CW];
          tmem_ld_32x16(taddr + ch * EPI_CW, v);
          const int cb = col0 + ch * EPI_CW;
          if (edge) {
#pragma unroll
            for (int q = 0; q < EPI_CW; ++q) v[q] = (row_ok && cb + q < m) ? v[q] : -CUDART_INF_F;
          }
          // insert the chunk's best column (the lowest of equal ones) and knock it out, while it beats the last entry
          float best = chunk_max(v);
          while (best > lv[KP - 1]) {
            int qb = 0;
#pragma unroll
            for (int q = EPI_CW - 1; q >= 0; --q) qb = v[q] == best ? q : qb;
            list_insert<KP, false>(lv, li, best, cb + qb);
#pragma unroll
            for (int q = 0; q < EPI_CW; ++q) v[q] = q == qb ? -CUDART_INF_F : v[q];
            best = chunk_max(v);
          }
          __syncwarp();  // the next tcgen05.ld is warp-collective
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (PAIR) mbar_arrive_cluster(map_to_cta(smem_u32(&bars->tmem_empty[acc]), 0));
          else mbar_arrive(smem_u32(&bars->tmem_empty[acc]));
        }
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1u;
      }
      if (cur_sb >= 0) flush(cur_sb);
    }
  } else if (warp >= EPI_WARP0) {
    // ===================================== epilogue =========================================
    // four warps per TMEM lane quarter, each owning a quarter of the tile's columns:
    // with a single epilogue warp per scheduler the dependent-issue latencies of the reduce chain are exposed
    const int ew = warp & 3;           // TMEM lane quarter this warp may read
    const int half = (warp - EPI_WARP0) >> 2;  // "part": columns [PART_COLS * half, PART_COLS * half + PART_COLS) of the tile
    const int e = ew * 32 + lane;      // row inside the tile; also column-combine slot
    float m1 = -CUDART_INF_F, m2 = -CUDART_INF_F;
    int i1 = -1, i2 = -1;
    int cur_sb = -1;
    int acc = 0;
    uint32_t acc_phase = 0;

    auto flush = [&](int sb) {
      p.partial[((size_t)(cluster_id + sb) * (BM * MC) + rank * BM + e) * EPI_PARTS + half] =
          make_float4(m1, __int_as_float(i1), m2, __int_as_float(i2));
    };

    // fragment slots: [chunk of 32 columns][4 columns][row] float4, so that the 128 rows of a column group are contiguous
    float4* const frag_mine = p.frag + (size_t)blockIdx.x * (FRAG_BYTES / 16) + e;
    const float4* const frag_next = p.frag + (size_t)(blockIdx.x + MC) * (FRAG_BYTES / 16) + e;  // same rank, next cluster
    for (unsigned long long step = 0; step < n_items; ++step) {
      const Item it = item_at(step);
      const unsigned long long t = it.t;
      const int sb = (int)(t / (unsigned)sch.n_ct), ct = (int)(t - (unsigned long long)sb * sch.n_ct);
      if (it.kind == 1) {
        // ---- head fragment: raw accumulators to the workspace, then the flag the owning cluster waits for
        mbar_wait(smem_u32(&bars->tmem_full[acc]), acc_phase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + (uint32_t)acc * BN + ((uint32_t)(ew * 32) << 16);
#pragma unroll 1
        for (int ch = half * PART_CHUNKS; ch < (half + 1) * PART_CHUNKS; ++ch) {
          float v[EPI_CW];
          tmem_ld_32x16(taddr + ch * EPI_CW, v);
#pragma unroll
          for (int q = 0; q < EPI_CW / 4; ++q)
            __stcg(frag_mine + (size_t)(ch * (EPI_CW / 4) + q) * BM, make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]));
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (PAIR) mbar_arrive_cluster(map_to_cta(smem_u32(&bars->tmem_empty[acc]), 0));
          else mbar_arrive(smem_u32(&bars->tmem_empty[acc]));
        }
        __threadfence();
        named_bar_sync(5, 128 * EPI_PARTS);  // all epilogue warps have stored and fenced
        if (threadIdx.x == EPI_WARP0 * 32) st_release_gpu(p.flags + blockIdx.x, 1u);
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1u;
        continue;
      }
      if (sb != cur_sb) {
        if (cur_sb >= 0) flush(cur_sb);
        m1 = m2 = -CUDART_INF_F;
        i1 = i2 = -1;
        cur_sb = sb;
      }
      const int row0 = (sb * MC + rank) * BM, col0 = ct * BN;
      const bool edge = (row0 + BM > n) || (col0 + BN > m);
      const bool row_ok = row0 + e < n;
      uint2* colw = col_smem + (size_t)acc * (4 * BN) + ew * BN;

      mbar_wait(smem_u32(&bars->tmem_full[acc]), acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t)acc * BN + ((uint32_t)(ew * 32) << 16);
      const bool add_frag = it.kind == 2;
      if (add_frag) {  // the rest of this tile's K range: the next cluster computed it first thing
        if (lane == 0) flag_wait(p.flags + blockIdx.x + MC);
        __syncwarp();
      }

#pragma unroll 1
      for (int ch = half * PART_CHUNKS; ch < (half + 1) * PART_CHUNKS; ++ch) {
        float v[EPI_CW];
        tmem_ld_32x16(taddr + ch * EPI_CW, v);
        if (add_frag) {
#pragma unroll
          for (int q = 0; q < EPI_CW / 4; ++q) {
            const float4 f = __ldcg(frag_next + (size_t)(ch * (EPI_CW / 4) + q) * BM);
            v[4 * q] += f.x;
            v[4 * q + 1] += f.y;
            v[4 * q + 2] += f.z;
            v[4 * q + 3] += f.w;
          }
        }
        const int cb = col0 + ch * EPI_CW;
        if (edge) {
#pragma unroll
          for (int q = 0; q < EPI_CW; ++q) v[q] = (row_ok && cb + q < m) ? v[q] : -CUDART_INF_F;
        }
        if (p.S_out != nullptr && row_ok) {  // similarity-only consumers (MaskCut's affinity): the tile goes to memory as well
          float* dst = p.S_out + (size_t)(row0 + e) * p.ld_s + cb;
          if (cb + EPI_CW <= m) {
#pragma unroll
            for (int q = 0; q < EPI_CW; q += 4) *reinterpret_cast<float4*>(dst + q) = make_float4(v[q], v[q + 1], v[q + 2], v[q + 3]);
          } else {
#pragma unroll
            for (int q = 0; q < EPI_CW; ++q)
              if (cb + q < m) dst[q] = v[q];
          }
        }
        // ---- rows: this thread's row against its running top-2.  Only groups of 8 columns whose maximum
        // beats the current second best are scanned (rare after the first tiles of a row block).
#ifdef MV_K2_EXP_NO_ROWS
        if (v[ch] > m2) { m2 = v[ch]; i2 = cb; }
#else
        float g[EPI_CW / 8];
#pragma unroll
        for (int u = 0; u < EPI_CW / 8; ++u) {
          const float a = fmaxf(fmaxf(v[8 * u], v[8 * u + 1]), fmaxf(v[8 * u + 2], v[8 * u + 3]));
          const float b = fmaxf(fmaxf(v[8 * u + 4], v[8 * u + 5]), fmaxf(v[8 * u + 6], v[8 * u + 7]));
          g[u] = fmaxf(a, b);
        }
        if (fmaxf(g[0], g[1]) > m2) {
#pragma unroll
          for (int u = 0; u < EPI_CW / 8; ++u) {
            if (g[u] > m2) {
#pragma unroll
              for (int q = 8 * u; q < 8 * u + 8; ++q) {
                const float x = v[q];
                if (x > m2) {
                  if (x > m1) { m2 = m1; i2 = i1; m1 = x; i1 = cb + q; }
                  else { m2 = x; i2 = cb + q; }
                }
              }
            }
          }
        }
#endif
        // ---- columns: max over the warp's 32 rows and which row holds it
        // (measured and rejected, round 2: prefiltering groups of 8 columns against the columns' current records --
        // thresholds fetched one tile ahead into shared memory, the CREDUX / ballot path only for groups some row of the
        // warp can improve, ~20 % of them -- is SLOWER: 0.418 vs 0.340 ms at 18231^2 x 312, 0.477 vs 0.411 ms at
        // 19200^2 x 768.  The unconditional loop below is software-pipelined by the compiler (32 independent CREDUX in
        // flight); behind a branch every taken group pays the CREDUX -> FSETP -> VOTE latency chain, plus one more barrier
        // per tile.  Without any column work the K = 312 launch takes 0.267 ms: the rows + TMEM reads are the larger part.
        // Also measured and rejected: the TMEM read of chunk c + 1 in flight while chunk c is processed (two register
        // buffers, 168 registers): 0.375 vs 0.340 ms at K = 312, 0.432 vs 0.411 ms at 19200^2 x 768.  And: keeping the A
        // tiles of a row block resident in shared memory for its whole column sweep at K <= 384 (the ring then carries B
        // tiles only, a third less L2 -> shared-memory traffic): 0.337 vs 0.339 ms at K = 312 -- no change, and K = 256 takes
        // 0.354 ms: at small K the tile time (~4.7 us per 128 x 256 tile) does not depend on K or on the operand traffic at
        // all, it is the epilogue's own instruction stream (TMEM reads alone: 128 KB per tile at 64 B/clk = 2048 of ~9000 clk).)
#ifndef MV_K2_EXP_NO_COLS
#pragma unroll
        for (int q = 0; q < EPI_CW; q += 2) {
          const float x0 = warp_max_f32(v[q]), x1 = warp_max_f32(v[q + 1]);
          const uint32_t b0 = __ballot_sync(0xffffffffu, v[q] == x0);
          const uint32_t b1 = __ballot_sync(0xffffffffu, v[q + 1] == x1);
          if (lane == 0)
            *reinterpret_cast<uint4*>(colw + ch * EPI_CW + q) = make_uint4(__float_as_uint(x0), b0, __float_as_uint(x1), b1);
        }
#endif
      }
      // accumulator drained: hand the TMEM buffer back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR) mbar_arrive_cluster(map_to_cta(smem_u32(&bars->tmem_empty[acc]), 0));  // the MMA issuer lives in rank 0
        else mbar_arrive(smem_u32(&bars->tmem_empty[acc]));
      }

      // combine the 4 warps' column results of this part; thread e < PART_COLS owns column e + PART_COLS * half
      named_bar_sync(1 + half, 128);
      const uint2* colr = col_smem + (size_t)acc * (4 * BN);
      if (e < PART_COLS) {
        const int c = e + half * PART_COLS;
        float best = -CUDART_INF_F;
        int brow = 0;
#pragma unroll
        for (int w = 0; w < 4; ++w) {
          const uint2 r = colr[w * BN + c];
          const float x = __uint_as_float(r.x);
          if (x > best) { best = x; brow = w * 32 + __ffs((int)r.y) - 1; }
        }
        const int col = col0 + c;
        if (best > -CUDART_INF_F && col < m) {
          const unsigned long long packed =
              ((unsigned long long)f32_orderable(best) << 32) | (unsigned long long)(0xffffffffu - (uint32_t)(row0 + brow));
          unsigned long long* dst = p.col_best + col;
          if (packed > __ldcg(dst)) atomicMax(dst, packed);
        }
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1u;
    }
    if (cur_sb >= 0) flush(cur_sb);
  }

  // ---- teardown
  __syncwarp();
  tc_fence_before();
  if (MC > 1) cluster_sync_all(); else __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    if (PAIR) tmem_dealloc_512_pair(tmem_base);
    else tmem_dealloc_512(tmem_base);
  }
}

template <bool TF32, int MC, bool PAIR>
__global__ void __launch_bounds__(K2_THREADS, 1)
    k2_sim_top2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, K2Params p) {
  k2_body<TF32, MC, PAIR, 0>(tmA, tmB, p);
}

template <bool TF32, int MC, bool PAIR, int KP>
__global__ void __launch_bounds__(Epi<KP>::THREADS, 1)
    k2_sim_topk_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, K2Params p) {
  k2_body<TF32, MC, PAIR, KP>(tmA, tmB, p);
}

// fold the partial top-KP lists of every row (Epi<KP>::PARTS column parts per CTA that worked on the row); write
// (n_max, KP) values descending / indices, ties to the lower column, missing entries MV_MASKED_F / -1
template <int MC, int KP>
__global__ void k2_merge_topk_kernel(int clusters, const float4* __restrict__ partial, const int32_t* __restrict__ n_dev, int n_max,
                                     const int32_t* __restrict__ m_dev, int m_max, float* __restrict__ row_val,
                                     int32_t* __restrict__ row_idx) {
  constexpr int PARTS = Epi<KP>::PARTS;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_max) return;
  const int n = n_dev ? min(*n_dev, n_max) : n_max;
  const int m = m_dev ? min(*m_dev, m_max) : m_max;
  float lv[KP];
  int li[KP];
#pragma unroll
  for (int r = 0; r < KP; ++r) {
    lv[r] = -CUDART_INF_F;
    li[r] = -1;
  }
  if (i < n && m > 0) {
    const K2Sched s = make_sched(n, m, MC, clusters, 1, 0);
    const int sb = i / (BM * MC);
    const int c_first = sched_owner(s, (unsigned long long)sb * s.n_ct);
    const int c_last = sched_owner(s, (unsigned long long)(sb + 1) * s.n_ct - 1);
    for (int c = c_first; c <= c_last; ++c) {
      for (int q = 0; q < PARTS; ++q) {
        const float4* rec = partial + (((size_t)(c + sb) * (BM * MC) + (i - sb * BM * MC)) * PARTS + q) * (KP / 2);
        // each partial list is sorted: stop at its first entry that does not make the list
#pragma unroll 1
        for (int h = 0; h < KP / 2; ++h) {
          const float4 r = rec[h];
          const int ja = __float_as_int(r.y), jb = __float_as_int(r.w);
          if (ja < 0 || !better(r.x, ja, lv[KP - 1], li[KP - 1])) break;
          list_insert<KP, true>(lv, li, r.x, ja);
          if (jb < 0 || !better(r.z, jb, lv[KP - 1], li[KP - 1])) break;
          list_insert<KP, true>(lv, li, r.z, jb);
        }
      }
    }
  }
#pragma unroll
  for (int r = 0; r < KP; ++r) {
    row_val[(size_t)KP * i + r] = li[r] >= 0 ? lv[r] : MV_MASKED_F;
    row_idx[(size_t)KP * i + r] = li[r];
  }
}

// fold the partial top-2 records of every row; write (n_max, 2) value / index pairs
template <int MC>
__global__ void k2_merge_rows_kernel(int clusters, int kblocks, int streamk, const float4* __restrict__ partial, const int32_t* __restrict__ n_dev,
                                     int n_max, const int32_t* __restrict__ m_dev, int m_max, float* __restrict__ row_val,
                                     int32_t* __restrict__ row_idx) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_max) return;
  const int n = n_dev ? min(*n_dev, n_max) : n_max;
  const int m = m_dev ? min(*m_dev, m_max) : m_max;
  float m1 = -CUDART_INF_F, m2 = -CUDART_INF_F;
  int i1 = -1, i2 = -1;
  if (i < n && m > 0) {
    const K2Sched s = make_sched(n, m, MC, clusters, kblocks, streamk);
    const int sb = i / (BM * MC);
    const int c_first = sched_owner(s, (unsigned long long)sb * s.n_ct);
    const int c_last = sched_owner(s, (unsigned long long)(sb + 1) * s.n_ct - 1);
    for (int c = c_first; c <= c_last; ++c) {
      const float4* rec = partial + ((size_t)(c + sb) * (BM * MC) + (i - sb * BM * MC)) * EPI_PARTS;
      float xs[2 * EPI_PARTS];
      int js[2 * EPI_PARTS];
#pragma unroll
      for (int q = 0; q < EPI_PARTS; ++q) {  // the column parts of every tile, in column order
        const float4 r = rec[q];
        xs[2 * q] = r.x;
        xs[2 * q + 1] = r.z;
        js[2 * q] = __float_as_int(r.y);
        js[2 * q + 1] = __float_as_int(r.w);
      }
#pragma unroll
      for (int u = 0; u < 2 * EPI_PARTS; ++u) {
        if (js[u] < 0) continue;
        if (better(xs[u], js[u], m1, i1)) { m2 = m1; i2 = i1; m1 = xs[u]; i1 = js[u]; }
        else if (better(xs[u], js[u], m2, i2)) { m2 = xs[u]; i2 = js[u]; }
      }
    }
  }
  row_val[2 * (size_t)i + 0] = i1 >= 0 ? m1 : MV_MASKED_F;
  row_val[2 * (size_t)i + 1] = i2 >= 0 ? m2 : MV_MASKED_F;
  row_idx[2 * (size_t)i + 0] = i1;
  row_idx[2 * (size_t)i + 1] = i2;
}

__global__ void k2_unpack_col_kernel(const unsigned long long* __restrict__ col_best, int m, float* __restrict__ col_val,
                                     int32_t* __restrict__ col_idx) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  const unsigned long long pk = col_best[j];
  if (pk == 0ull) {
    if (col_val) col_val[j] = MV_MASKED_F;
    if (col_idx) col_idx[j] = -1;
  } else {
    if (col_val) col_val[j] = orderable_f32((uint32_t)(pk >> 32));
    if (col_idx) col_idx[j] = (int32_t)(0xffffffffu - (uint32_t)(pk & 0xffffffffull));
  }
}

// ---- host side -----------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(sym);
  }
  return fn;
}

// (rows, C) row-major operand -> tensor map with a (box_rows x 128 bytes) 128B-swizzled box
int make_operand_map(CUtensorMap* tm, const void* base, int rows, int C, int ld, int dtype, int box_rows) {
  const bool tf32 = dtype == MV_DTYPE_TF32;
  EncodeTiledFn enc = get_encode_tiled();
  MV_REQUIRE(enc, MV_E_DRIVER, "mv_k2_sim_top2: cuTensorMapEncodeTiled is not available from this driver");
  const int esz = tf32 ? 4 : 2;
  cuuint64_t gdim[2] = {(cuuint64_t)C, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)ld * esz};  // row pitch; columns >= C are out of bounds = zero fill
  cuuint32_t box[2] = {(cuuint32_t)(ROW_BYTES / esz), (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapDataType dt = tf32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                      : (dtype == MV_DTYPE_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16);
  CUresult r = enc(tm, dt, 2,
                   const_cast<void*>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  MV_REQUIRE(r == CUDA_SUCCESS, MV_E_DRIVER, "mv_k2_sim_top2: cuTensorMapEncodeTiled failed (CUresult %d)", (int)r);
  return MV_OK;
}

size_t k2_partial_bytes(int n_max, int mc, int clusters) {
  const int n_sb_max = (n_max + BM * mc - 1) / (BM * mc);
  return ((size_t)(clusters + n_sb_max) * (BM * mc) * EPI_PARTS * sizeof(float4) + 255) / 256 * 256;
}
// stream-K area behind the partial records: one flag and one accumulator-fragment slot per CTA of the grid
constexpr size_t SK_FLAG_BYTES = 1024;  // >= 4 * 148, keeps the fragments 256-byte aligned
size_t k2_streamk_bytes(int ctas) { return SK_FLAG_BYTES + (size_t)ctas * FRAG_BYTES; }

// The K-cut schedule is OFF by default: measured on B200 at the NAVI shape (tools/k2_streamk_ab.py, same process,
// kernel timed alone) 117.6 us against 111.6 us of the tile-granular schedule back to back, 125 against 122 us for
// isolated launches.  Equalising the k-blocks per SM buys nothing because the kernel is not limited per SM: it runs at the
// power-capped sustained rate of the chip (sw_power_cap in every run; frac_sustained 1.0 in the bench line), so the SMs that
// finish early lower the power draw and the others clock higher; the K-cut only adds 38 MB of fragment traffic and one
// extra epilogue per SM.  MVMATCH_K2_STREAMK=1 or
// mv_k2_set_streamk(1) switches it on (tests/test_gpu_k2.py runs it).
int g_k2_streamk = -1;
int k2_streamk_enabled() {
  if (g_k2_streamk < 0) {
    const char* e = getenv("MVMATCH_K2_STREAMK");
    g_k2_streamk = (e && e[0] == '1') ? 1 : 0;
  }
  return g_k2_streamk;
}

int pick_mc(int cluster) { return cluster <= 1 ? 1 : (cluster >= 4 ? 4 : 2); }

// persistent grid: one CTA per SM, but never more clusters than can be resident at once (GPC
// boundaries strand SMs for cluster sizes that do not divide a GPC), or the grid runs in two waves
template <bool TF32, int MC, bool PAIR, int KP>
constexpr auto k2_kernel() {
  if constexpr (KP == 0) return k2_sim_top2_kernel<TF32, MC, PAIR>;
  else return k2_sim_topk_kernel<TF32, MC, PAIR, KP>;
}

template <bool TF32, int MC, bool PAIR = false, int KP = 0>
int k2_max_clusters() {
  static int cache[MV_MAX_DEVICES];
  int& cached = cache[mv_device_slot()];
  if (cached) return cached;
  auto kern = k2_kernel<TF32, MC, PAIR, KP>();
  int n = mv_sm_count() / MC;
  constexpr int K2_SMEM_BYTES = k2_smem_bytes<PAIR>();
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, K2_SMEM_BYTES) == cudaSuccess && MC > 1) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(mv_sm_count() / MC * MC);
    cfg.blockDim = dim3(Epi<KP>::THREADS);
    cfg.dynamicSmemBytes = K2_SMEM_BYTES;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = MC;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int act = 0;
    if (cudaOccupancyMaxActiveClusters(&act, kern, &cfg) == cudaSuccess && act > 0 && act < n) n = act;
  }
  (void)cudaGetLastError();
  cached = n > 0 ? n : 1;
  return cached;
}

template <int KP = 0>
int k2_grid(int mc, bool tf32, bool pair = false) {
  int clusters;
  if (mc == 1) clusters = mv_sm_count();
  else if (pair) clusters = tf32 ? k2_max_clusters<true, 2, true, KP>() : k2_max_clusters<false, 2, true, KP>();
  else if (mc == 2) clusters = tf32 ? k2_max_clusters<true, 2, false, KP>() : k2_max_clusters<false, 2, false, KP>();
  else clusters = tf32 ? k2_max_clusters<true, 4, false, KP>() : k2_max_clusters<false, 4, false, KP>();
  return clusters * mc;
}

template <bool TF32, int MC, bool PAIR = false, int KP = 0>
int launch_k2(const CUtensorMap& tmA, const CUtensorMap& tmB, const K2Params& p, int grid, cudaStream_t st) {
  auto kern = k2_kernel<TF32, MC, PAIR, KP>();
  constexpr int K2_SMEM_BYTES = k2_smem_bytes<PAIR>();
  static bool done[MV_MAX_DEVICES];
  bool& attr_done = done[mv_device_slot()];
  if (!attr_done) {
    MV_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, K2_SMEM_BYTES));
    attr_done = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(Epi<KP>::THREADS);
  cfg.dynamicSmemBytes = K2_SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = MC;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  MV_CUDA(cudaLaunchKernelEx(&cfg, kern, tmA, tmB, p));
  return MV_OK;
}

// the instantiation for an operand type and cluster form
template <int KP>
int launch_k2_form(bool tf32, int mc, bool pair, const CUtensorMap& tmA, const CUtensorMap& tmB, const K2Params& p, int grid,
                   cudaStream_t st) {
  if (pair) return tf32 ? launch_k2<true, 2, true, KP>(tmA, tmB, p, grid, st) : launch_k2<false, 2, true, KP>(tmA, tmB, p, grid, st);
  if (tf32) {
    if (mc == 1) return launch_k2<true, 1, false, KP>(tmA, tmB, p, grid, st);
    if (mc == 2) return launch_k2<true, 2, false, KP>(tmA, tmB, p, grid, st);
    return launch_k2<true, 4, false, KP>(tmA, tmB, p, grid, st);
  }
  if (mc == 1) return launch_k2<false, 1, false, KP>(tmA, tmB, p, grid, st);
  if (mc == 2) return launch_k2<false, 2, false, KP>(tmA, tmB, p, grid, st);
  return launch_k2<false, 4, false, KP>(tmA, tmB, p, grid, st);
}

// partial top-KP lists: (clusters + n_sb_max) slots of MC * 128 rows x Epi<KP>::PARTS column parts x KP (value, index) pairs
size_t k2_topk_partial_bytes(int n_max, int mc, int clusters, int kp) {
  const int n_sb_max = (n_max + BM * mc - 1) / (BM * mc);
  const int parts = kp == 8 ? Epi<8>::PARTS : Epi<16>::PARTS;
  return ((size_t)(clusters + n_sb_max) * (BM * mc) * parts * kp * sizeof(float2) + 255) / 256 * 256;
}

// ---- optional timing of the GEMM kernel alone (bench.py's roofline): events recorded right around the launch of
// k2_sim_top2_kernel, so that the figure is the kernel's own duration and not memset + kernel + row merge
struct K2Profile {
  std::vector<cudaEvent_t> ev;  // 2 per recorded launch
  std::vector<int> dims;        // (n_max, m_max, C) per recorded launch
  int capacity = 0, count = 0;
};
thread_local K2Profile g_k2_prof;

// operand checks shared by the kernel-2 entry points; no CUDA call
int k2_check_operands(const char* fn, int lda, int ldb, int n_max, int m_max, int C, int dtype, const void* A, const void* B,
                      const void* workspace) {
  MV_REQUIRE(lda >= C && ldb >= C && (lda * (dtype == MV_DTYPE_TF32 ? 4 : 2)) % 16 == 0 && (ldb * (dtype == MV_DTYPE_TF32 ? 4 : 2)) % 16 == 0,
             MV_E_ALIGN, "%s: row pitches (%d, %d) must be >= C and a multiple of 16 bytes", fn, lda, ldb);
  MV_REQUIRE(dtype == MV_DTYPE_BF16 || dtype == MV_DTYPE_TF32 || dtype == MV_DTYPE_F16, MV_E_ARG, "%s: unknown dtype %d", fn, dtype);
  MV_REQUIRE(n_max > 0 && m_max > 0 && C > 0, MV_E_ARG, "%s: sizes must be positive", fn);
  MV_REQUIRE(n_max <= (1 << 20) && m_max <= (1 << 20), MV_E_RANGE, "%s: at most 2^20 rows per side", fn);
  const bool tf32 = dtype == MV_DTYPE_TF32;
  MV_REQUIRE(C % (tf32 ? 4 : 8) == 0, MV_E_ALIGN, "%s: C=%d must be a multiple of %d", fn, C, tf32 ? 4 : 8);
  MV_REQUIRE(((uintptr_t)A & 15) == 0 && ((uintptr_t)B & 15) == 0 && ((uintptr_t)workspace & 15) == 0, MV_E_ALIGN,
             "%s: A, B and workspace must be 16-byte aligned", fn);
  return MV_OK;
}

// A launch of kernel 2 whose arguments passed k2_check_operands: device check, cluster form, grid and the parameters
// every epilogue shares (the caller fills in the outputs and the workspace pointers)
struct K2Launch {
  K2Params p;
  int grid, mc;
  bool tf32, pair;
};
template <int KP>
int k2_prepare(const char* fn, int n_max, int m_max, int C, const int32_t* n_dev, const int32_t* m_dev, int dtype, int cluster,
               K2Launch& k) {
  int dev = 0, cc = 0;
  MV_CUDA(cudaGetDevice(&dev));
  MV_CUDA(cudaDeviceGetAttribute(&cc, cudaDevAttrComputeCapabilityMajor, dev));
  MV_REQUIRE(cc == 10, MV_E_ARCH, "%s: needs an sm_100 device (found compute capability %d.x)", fn, cc);
  k.tf32 = dtype == MV_DTYPE_TF32;
  if (cluster == MV_CLUSTER_AUTO) {
    // measured on B200 (tools/k2_sweep.sh): once a tile's MMA time clearly exceeds its epilogue time (K >= 1536
    // bf16 / 768 tf32 elements) the CTA pair wins (1612 vs 1520 TFLOP/s at 19200^2 x 2048); below that the
    // epilogue co-limits and the looser coupling of two multicast CTAs is faster (1423 vs 1343 at K = 768)
    cluster = (C >= (k.tf32 ? 768 : 1536)) ? MV_CLUSTER_PAIR : 2;
  }
  k.pair = cluster == MV_CLUSTER_PAIR;  // cta_group::2: two SMs on one 256 x 256 MMA tile
  k.mc = k.pair ? 2 : pick_mc(cluster);
  // (5.4 tiles per SM at the NAVI shape leave 10 % of the last tile-time idle; running two pairs' kernel 2 side by
  // side on half the SMs each -- 10.8 tiles per SM -- was measured: same pairs/s, the pipeline's other kernels
  // already fill that tail)
  k.grid = k2_grid<KP>(k.mc, k.tf32, k.pair);
  K2Params& p = k.p;
  p = K2Params{};
  p.clusters = k.grid / k.mc;
  p.n_dev = n_dev;
  p.m_dev = m_dev;
  p.n_max = n_max;
  p.m_max = m_max;
  const int ke = k.tf32 ? 32 : 64;
  p.kblocks = (C + ke - 1) / ke;
  const int kstep = ke / 4;  // K elements per MMA: 16 (16-bit operands) / 8 (tf32)
  p.tail_steps = (C - (p.kblocks - 1) * ke + kstep - 1) / kstep;
  p.ab_fmt = k.tf32 ? 2u : (dtype == MV_DTYPE_F16 ? 0u : 1u);
  return MV_OK;
}

int k2_operand_maps(CUtensorMap* tmA, CUtensorMap* tmB, const void* A, int lda, const void* B, int ldb, int n_max, int m_max,
                    int C, int dtype, int mc) {
  int rc = make_operand_map(tmA, A, n_max, C, lda, dtype, BM);
  if (rc) return rc;
  return make_operand_map(tmB, B, m_max, C, ldb, dtype, BN / mc);
}

size_t k2_topk_workspace_bytes(int n_max, int kp) {
  size_t worst = 0;
  for (int mc = 1; mc <= 4; mc *= 2) {
    const size_t b = k2_topk_partial_bytes(n_max, mc, mv_sm_count() / mc, kp);
    if (b > worst) worst = b;
  }
  return worst;
}

}  // namespace

extern "C" {

int mv_k2_set_streamk(int on) {
  const int prev = k2_streamk_enabled();
  if (on >= 0) g_k2_streamk = on ? 1 : 0;
  return prev;
}

int mv_k2_profile_begin(int capacity) {
  MV_REQUIRE(capacity >= 0 && capacity <= (1 << 16), MV_E_RANGE, "mv_k2_profile_begin: capacity out of range");
  K2Profile& pr = g_k2_prof;
  for (cudaEvent_t e : pr.ev) cudaEventDestroy(e);
  pr.ev.clear();
  pr.count = 0;
  pr.capacity = capacity;
  pr.ev.resize((size_t)2 * capacity);
  pr.dims.assign((size_t)3 * capacity, 0);
  for (auto& e : pr.ev) MV_CUDA(cudaEventCreate(&e));
  return MV_OK;
}

int mv_k2_profile_dims(int* nmc_out, int max_n) {
  K2Profile& pr = g_k2_prof;
  const int n = pr.count < max_n ? pr.count : max_n;
  for (int i = 0; i < 3 * n; ++i) nmc_out[i] = pr.dims[i];
  return n;
}

int mv_k2_profile_read(float* ms_out, int max_n) {
  K2Profile& pr = g_k2_prof;
  const int n = pr.count < max_n ? pr.count : max_n;
  for (int i = 0; i < n; ++i) {
    MV_CUDA(cudaEventSynchronize(pr.ev[2 * i + 1]));
    MV_CUDA(cudaEventElapsedTime(ms_out + i, pr.ev[2 * i], pr.ev[2 * i + 1]));
  }
  return n;
}

size_t mv_k2_workspace_bytes(int n_max, int m_max) {
  (void)m_max;
  if (n_max <= 0) return 256 + k2_streamk_bytes(mv_sm_count());
  size_t worst = 0;
  for (int mc = 1; mc <= 4; mc *= 2) {
    const size_t b = k2_partial_bytes(n_max, mc, mv_sm_count() / mc);
    if (b > worst) worst = b;
  }
  return worst + 256 + k2_streamk_bytes(mv_sm_count());
}

int mv_k2_sim_top2(const void* A, const void* B, int n_max, int m_max, int C, const int32_t* n_dev,
                   const int32_t* m_dev, int dtype, int cluster, float* row_val, int32_t* row_idx,
                   unsigned long long* col_best, void* workspace, size_t workspace_bytes, mv_stream_t stream) {
  return mv_k2_sim_top2_ld(A, C, B, C, n_max, m_max, C, n_dev, m_dev, dtype, cluster, row_val, row_idx, col_best, workspace,
                           workspace_bytes, stream);
}

int mv_k2_sim_top2_ld(const void* A, int lda, const void* B, int ldb, int n_max, int m_max, int C, const int32_t* n_dev,
                      const int32_t* m_dev, int dtype, int cluster, float* row_val, int32_t* row_idx,
                      unsigned long long* col_best, void* workspace, size_t workspace_bytes, mv_stream_t stream) {
  return mv_k2_affinity(A, lda, B, ldb, n_max, m_max, C, n_dev, m_dev, dtype, cluster, nullptr, 0, row_val, row_idx, col_best, workspace,
                        workspace_bytes, stream);
}

int mv_k2_affinity(const void* A, int lda, const void* B, int ldb, int n_max, int m_max, int C, const int32_t* n_dev,
                   const int32_t* m_dev, int dtype, int cluster, float* S_out, int ld_s, float* row_val, int32_t* row_idx,
                   unsigned long long* col_best, void* workspace, size_t workspace_bytes, mv_stream_t stream) {
  MV_REQUIRE(!S_out || (ld_s >= m_max && ld_s % 4 == 0 && ((uintptr_t)S_out & 15) == 0), MV_E_ALIGN,
             "mv_k2_affinity: S_out must be 16-byte aligned with a row pitch >= m_max that is a multiple of 4 floats");
  MV_REQUIRE(A && B && row_val && row_idx && col_best && workspace, MV_E_ARG, "mv_k2_sim_top2: null pointer");
  int rc = k2_check_operands("mv_k2_sim_top2", lda, ldb, n_max, m_max, C, dtype, A, B, workspace);
  if (rc) return rc;
  K2Launch k;
  rc = k2_prepare<0>("mv_k2_sim_top2", n_max, m_max, C, n_dev, m_dev, dtype, cluster, k);
  if (rc) return rc;
  K2Params& p = k.p;
  const size_t part_bytes = k2_partial_bytes(n_max, k.mc, p.clusters);
  const size_t need = part_bytes + k2_streamk_bytes(k.grid);
  MV_REQUIRE(workspace_bytes >= need, MV_E_WORKSPACE, "mv_k2_sim_top2: workspace has %zu bytes, %zu needed",
             workspace_bytes, need);
  p.partial = reinterpret_cast<float4*>(workspace);
  p.flags = reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(workspace) + part_bytes);
  p.frag = reinterpret_cast<float4*>(reinterpret_cast<uint8_t*>(workspace) + part_bytes + SK_FLAG_BYTES);
  p.streamk = k2_streamk_enabled();
  p.col_best = col_best;
  p.S_out = S_out;
  p.ld_s = ld_s;

  CUtensorMap tmA, tmB;
  rc = k2_operand_maps(&tmA, &tmB, A, lda, B, ldb, n_max, m_max, C, dtype, k.mc);
  if (rc) return rc;

  cudaStream_t st = mv_cuda_stream(stream);
  MV_CUDA(cudaMemsetAsync(col_best, 0, (size_t)m_max * sizeof(unsigned long long), st));
  if (p.streamk) MV_CUDA(cudaMemsetAsync(p.flags, 0, SK_FLAG_BYTES, st));
  K2Profile& pr = g_k2_prof;
  const bool timed = pr.count < pr.capacity;
  if (timed) MV_CUDA(cudaEventRecord(pr.ev[2 * pr.count], st));
  rc = launch_k2_form<0>(k.tf32, k.mc, k.pair, tmA, tmB, p, k.grid, st);
  if (rc) return rc;
  if (timed) {
    MV_CUDA(cudaEventRecord(pr.ev[2 * pr.count + 1], st));
    pr.dims[3 * pr.count] = n_max;
    pr.dims[3 * pr.count + 1] = m_max;
    pr.dims[3 * pr.count + 2] = C;
    ++pr.count;
  }
  const int mt = 256;
  const int mc = k.mc;
  if (mc == 1) k2_merge_rows_kernel<1><<<(n_max + mt - 1) / mt, mt, 0, st>>>(p.clusters, p.kblocks, p.streamk, p.partial, n_dev, n_max, m_dev, m_max, row_val, row_idx);
  else if (mc == 2) k2_merge_rows_kernel<2><<<(n_max + mt - 1) / mt, mt, 0, st>>>(p.clusters, p.kblocks, p.streamk, p.partial, n_dev, n_max, m_dev, m_max, row_val, row_idx);
  else k2_merge_rows_kernel<4><<<(n_max + mt - 1) / mt, mt, 0, st>>>(p.clusters, p.kblocks, p.streamk, p.partial, n_dev, n_max, m_dev, m_max, row_val, row_idx);
  MV_LAUNCH_CHECK();
  return MV_OK;
}

size_t mv_k2_topk_workspace_bytes(int n_max, int m_max, int kp) {
  (void)m_max;
  if (kp != 8 && kp != 16) return 0;
  return k2_topk_workspace_bytes(n_max > 0 ? n_max : 1, kp);
}

int mv_k2_sim_topk_ld(const void* A, int lda, const void* B, int ldb, int n_max, int m_max, int C, const int32_t* n_dev,
                      const int32_t* m_dev, int dtype, int cluster, int kp, float* row_val, int32_t* row_idx, void* workspace,
                      size_t workspace_bytes, mv_stream_t stream) {
  MV_REQUIRE(A && B && row_val && row_idx && workspace, MV_E_ARG, "mv_k2_sim_topk_ld: null pointer");
  MV_REQUIRE(kp == 8 || kp == 16, MV_E_RANGE, "mv_k2_sim_topk_ld: kp=%d must be 8 or 16", kp);
  int rc = k2_check_operands("mv_k2_sim_topk_ld", lda, ldb, n_max, m_max, C, dtype, A, B, workspace);
  if (rc) return rc;
  // the worst case over the cluster forms, so that the check needs no device
  const size_t need = k2_topk_workspace_bytes(n_max, kp);
  MV_REQUIRE(workspace_bytes >= need, MV_E_WORKSPACE, "mv_k2_sim_topk_ld: workspace has %zu bytes, %zu needed",
             workspace_bytes, need);
  K2Launch k;
  rc = kp == 8 ? k2_prepare<8>("mv_k2_sim_topk_ld", n_max, m_max, C, n_dev, m_dev, dtype, cluster, k)
               : k2_prepare<16>("mv_k2_sim_topk_ld", n_max, m_max, C, n_dev, m_dev, dtype, cluster, k);
  if (rc) return rc;
  K2Params& p = k.p;
  p.partial = reinterpret_cast<float4*>(workspace);
  p.streamk = 0;  // tile-granular schedule only: no head fragments, no flags

  CUtensorMap tmA, tmB;
  rc = k2_operand_maps(&tmA, &tmB, A, lda, B, ldb, n_max, m_max, C, dtype, k.mc);
  if (rc) return rc;
  cudaStream_t st = mv_cuda_stream(stream);
  rc = kp == 8 ? launch_k2_form<8>(k.tf32, k.mc, k.pair, tmA, tmB, p, k.grid, st)
               : launch_k2_form<16>(k.tf32, k.mc, k.pair, tmA, tmB, p, k.grid, st);
  if (rc) return rc;
  const int mt = 128, blocks = (n_max + mt - 1) / mt;
  const int mc = k.mc;
  if (kp == 8) {
    if (mc == 1) k2_merge_topk_kernel<1, 8><<<blocks, mt, 0, st>>>(p.clusters, p.partial, n_dev, n_max, m_dev, m_max, row_val, row_idx);
    else if (mc == 2) k2_merge_topk_kernel<2, 8><<<blocks, mt, 0, st>>>(p.clusters, p.partial, n_dev, n_max, m_dev, m_max, row_val, row_idx);
    else k2_merge_topk_kernel<4, 8><<<blocks, mt, 0, st>>>(p.clusters, p.partial, n_dev, n_max, m_dev, m_max, row_val, row_idx);
  } else {
    if (mc == 1) k2_merge_topk_kernel<1, 16><<<blocks, mt, 0, st>>>(p.clusters, p.partial, n_dev, n_max, m_dev, m_max, row_val, row_idx);
    else if (mc == 2) k2_merge_topk_kernel<2, 16><<<blocks, mt, 0, st>>>(p.clusters, p.partial, n_dev, n_max, m_dev, m_max, row_val, row_idx);
    else k2_merge_topk_kernel<4, 16><<<blocks, mt, 0, st>>>(p.clusters, p.partial, n_dev, n_max, m_dev, m_max, row_val, row_idx);
  }
  MV_LAUNCH_CHECK();
  return MV_OK;
}

int mv_k2_unpack_col(const unsigned long long* col_best, int m, float* col_val, int32_t* col_idx, mv_stream_t stream) {
  MV_REQUIRE(col_best && (col_val || col_idx), MV_E_ARG, "mv_k2_unpack_col: null pointer");
  MV_REQUIRE(m >= 0, MV_E_ARG, "mv_k2_unpack_col: negative m");
  if (m == 0) return MV_OK;
  k2_unpack_col_kernel<<<(m + 255) / 256, 256, 0, mv_cuda_stream(stream)>>>(col_best, m, col_val, col_idx);
  MV_LAUNCH_CHECK();
  return MV_OK;
}

}  // extern "C"
