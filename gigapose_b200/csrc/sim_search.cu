// Fused query<->template patch-similarity search for sm_100a (row a4 of SURVEY.md §8; replaces
// LocalSimilarity.test, reference src/models/matching.py:188-316 with helpers :63-113).
//
// One work item = one (query b, template n) pair = one 256(t) x 256(s) x 1024(c) similarity tile, computed by a 2-CTA
// cluster on the two SMs of a TPC as ONE M=256 x N=256 UMMA stream (tcgen05 cta_group::2).  CTA r of the pair owns the
// query rows t in [128r, 128r+128) and stages HALF of the template slab (s rows [128r, 128r+128)); the leader issues the
// instructions, which read both CTAs' shared memory, and every CTA drains its own 128 accumulator rows.  Persistent
// pairs walk the item list:
//   warp 0   : TMA producer  -- streams K-blocks of the query / template descriptor planes into a 6-stage smem ring
//   warp 1   : UMMA issuer   -- leader only: tcgen05.mma (cta_group::2, M=256, N=256, K=16, bf16 -> fp32) into TMEM;
//                               consecutive items alternate between two 256-column accumulators, so the epilogue of one
//                               item overlaps the tensor work of the next
//   warp 2   : TMEM allocator
//   warps 4-11: epilogue     -- tcgen05.ld the fp32 tile, apply masks + threshold (matching.py:234-236), row
//                               max/arg-max (t->s) in registers, column max/arg-max (s->t) with redux.sync +
//                               ballot, cycle-consistency / validity masks (matching.py:80-113,247-271) and the
//                               per-template score (matching.py:274-278).  The [B,N,256,256] similarity tensor
//                               never reaches HBM; per item only a 1.5 KB record + one float are written.
// The column maxima (idx_src2tar: arg-max over ALL 256 query patches) of the two halves are exchanged through
// distributed shared memory (st.shared::cluster + mbarrier release / acquire at cluster scope); the leader sums the
// per-template score in ascending-t warp order.
// Against a 1-CTA form (M = 128, the two t-halves of a tile back to back) the template planes are streamed from L2 / HBM
// once per item instead of once per t-half, and each SM's tensor core reads 4 KB + 4 KB of operands per instruction
// instead of 4 KB + 8 KB; that form was measured slower at both precisions and removed (profiles/r02_stress_c5shard.json).
//
// Precision: descriptors are stored as two bf16 planes (hi = bf16(x), lo = bf16(x - hi)); the tile is accumulated
// as hi*hi + hi*lo + lo*hi in fp32 (3 tensor-core passes, ~2^-17 relative operand error), so the thresholded /
// arg-max'ed results agree with the reference's fp32 einsum up to fp32 accumulation-order noise.  `passes = 1`
// runs hi*hi only (plain bf16 tensor-core similarity, 3x less tensor work, not index-exact).
#include "gigapose_kernels.h"
#include "common.cuh"
#include <cstdio>

namespace gp {

namespace {

constexpr int kP = 256;                         // patches per crop (16 x 16)
constexpr int kC = 1024;                        // descriptor channels
constexpr int kBlockK = 32;                     // bf16 elements per stage row: 64 B = SWIZZLE_64B span
constexpr int kRowBytes = kBlockK * 2;
constexpr int kHalfRows = 128;                  // t-rows per CTA of a pair
constexpr int kQPlaneBytes = kHalfRows * kRowBytes;   // 8 KB : 128 rows x 64 B
constexpr int kNumKBlocks = kC / kBlockK;       // 32
constexpr int kEpiWarps = 8;
constexpr int kEpiThreads = kEpiWarps * 32;     // 256
constexpr int kThreads = 4 * 32 + kEpiThreads;  // 384
constexpr int kTmemCols = 512;                  // two 128 x 256 fp32 accumulators (double buffered)

// Item order: queries (sorted by object) are taken in chunks of kQueryChunk; inside a chunk the template index is the
// outer loop.  CTAs that run together then share template tiles (queries of one object are adjacent) AND touch at
// most kQueryChunk query tiles, so both operands stay L2-resident whatever the batch size (at B = 256 with one query
// per object the plain template-major order re-read every query tile from HBM once per template).
constexpr int kQueryChunk = 32;
__device__ __forceinline__ void decode_item(int item, int B, int T, int& j, int& n) {
  const int per_chunk = kQueryChunk * T;
  const int c = item / per_chunk, r = item - c * per_chunk;
  const int q0 = c * kQueryChunk;
  const int qc = min(kQueryChunk, B - q0);
  n = r / qc;
  j = q0 + (r - n * qc);
}

constexpr int kPairStages = 6;
constexpr int kPairStageBytes = 4 * kQPlaneBytes;            // q_hi, q_lo, t_hi half, t_lo half: 32 KB
constexpr uint32_t kIdescPair = umma_idesc_f16(256, 256, /*bf16*/ 1);

struct __align__(8) SimPairTail {
  float smask[kP];
  float tmask[kP];
  float pmax[4][kP];                            // partial column max per group of 32 of THIS CTA's t-rows
  float half_cmax[2][kP];                       // [slot] column max over the PEER's 128 t-rows (written by the peer)
  float cmax[kP];                               // score_src2tar (both halves combined)
  float rmax_s[kHalfRows];                      // score_tar2src of this CTA's rows
  float rowp_max[2][kHalfRows];                 // [column half][row]
  float red[2][kEpiWarps];                      // leader: [0..3] own warps, [4..7] the peer's (written by the peer)
  uint8_t pidx[4][kP];
  uint8_t half_cidx[2][kP];
  uint8_t cidx[kP];                             // idx_src2tar
  uint8_t ridx_s[kHalfRows];                    // idx_tar2src
  uint8_t rowp_idx[2][kHalfRows];
  uint64_t full_bar[kPairStages];
  uint64_t empty_bar[kPairStages];
  uint64_t tmem_full_bar[2];
  uint64_t tmem_empty_bar[2];
  uint64_t xchg_bar[2];                         // peer's column maxima for item slot (item & 1) have landed
  uint64_t sum_bar[2];                          // leader only: the peer's partial score sums have landed
  uint32_t tmem_base;
};
constexpr int kPairSmemBytes = 1024 + kPairStages * kPairStageBytes + sizeof(SimPairTail);
static_assert(kPairSmemBytes <= 227 * 1024, "shared memory budget");
}  // namespace

template <bool kDebug>
__global__ void __launch_bounds__(kThreads, 1)
sim_search_pair_kernel(const __grid_constant__ CUtensorMap tm_q_hi, const __grid_constant__ CUtensorMap tm_q_lo,
                       const __grid_constant__ CUtensorMap tm_t_hi, const __grid_constant__ CUtensorMap tm_t_lo,
                       SimSearchParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  SimPairTail& tail = *reinterpret_cast<SimPairTail*>(smem + kPairStages * kPairStageBytes);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int passes = p.passes;
  const uint32_t rank = cluster_ctarank();                 // 0 = leader; owns t rows [128 rank, 128 rank + 128)
  // One-item striding: the B_o queries of an object that share a template tile are consecutive items, i.e. they run on
  // B_o different pairs AT THE SAME TIME and their reads of the tile coalesce in L2 (2.46 GB of DRAM traffic at c2 against
  // 1.39 GB algorithmic, ncu).  Handing each pair a block of consecutive items instead was measured worse (3.04 GB): the
  // other 73 pairs stream 146 MB through the 126 MB L2 between two visits of a tile by the same pair.
  const int first_item = (int)(blockIdx.x >> 1), item_step = (int)(gridDim.x >> 1);
#define GP_PAIR_ITEMS(...) for (int item = first_item; item < p.num_items; item += item_step __VA_ARGS__)

  if (threadIdx.x == 0) {
    for (int s = 0; s < kPairStages; ++s) { mbar_init(&tail.full_bar[s], 1); mbar_init(&tail.empty_bar[s], 1); }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tail.tmem_full_bar[a], 1);
      mbar_init(&tail.tmem_empty_bar[a], 2 * kEpiWarps);   // both CTAs' epilogue warps report to the leader
      mbar_init(&tail.xchg_bar[a], kEpiWarps);             // the peer's 8 epilogue warps
      mbar_init(&tail.sum_bar[a], 1);
    }
    fence_barrier_init();
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_q_hi); tma_prefetch_desc(&tm_t_hi);
    if (passes == 3) { tma_prefetch_desc(&tm_q_lo); tma_prefetch_desc(&tm_t_lo); }
  }
  if (warp == 2) tmem_alloc_pair(&tail.tmem_base, kTmemCols);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                                      // the peer's barriers and TMEM exist before anything reaches across
  tc_fence_after();
  const uint32_t tmem_base = tail.tmem_base;

  if (warp == 0) {
    // ======================================= TMA producer (both CTAs) =======================================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      const uint32_t tx_bytes = (passes == 3 ? 2 : 1) * 2 * (2 * kQPlaneBytes);     // both CTAs: 128 q rows + 128 t rows each
      GP_PAIR_ITEMS() {
        int j, n;
        decode_item(item, p.B, p.T, j, n);
        const int b = p.perm[j];
        const int t_img = p.q_obj[b] * p.T + n;
        for (int kb = 0; kb < kNumKBlocks; ++kb) {
          mbar_wait(&tail.empty_bar[stage], phase ^ 1);
          uint8_t* st = smem + stage * kPairStageBytes;
          if (rank == 0) mbar_arrive_expect_tx(&tail.full_bar[stage], tx_bytes);
          const int q_row = (b * kNumKBlocks + kb) * kP + (int)rank * kHalfRows;
          const int t_row = (t_img * kNumKBlocks + kb) * kP + (int)rank * kHalfRows;
          tma_load_2d_pair(st, &tm_q_hi, &tail.full_bar[stage], 0, q_row);
          tma_load_2d_pair(st + 2 * kQPlaneBytes, &tm_t_hi, &tail.full_bar[stage], 0, t_row);
          if (passes == 3) {
            tma_load_2d_pair(st + 3 * kQPlaneBytes, &tm_t_lo, &tail.full_bar[stage], 0, t_row);
            tma_load_2d_pair(st + kQPlaneBytes, &tm_q_lo, &tail.full_bar[stage], 0, q_row);
          }
          if (++stage == kPairStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ======================================= UMMA issuer (leader only) ======================================
    if (lane == 0 && rank == 0) {
      int stage = 0; uint32_t phase = 0, unit = 0;
      GP_PAIR_ITEMS(, ++unit) {
        const uint32_t acc = unit & 1u;
        mbar_wait(&tail.tmem_empty_bar[acc], ((unit >> 1) & 1u) ^ 1u);
        tc_fence_after();
        const uint32_t d = tmem_base + acc * 256;
        for (int kb = 0; kb < kNumKBlocks; ++kb) {
          mbar_wait(&tail.full_bar[stage], phase);
          tc_fence_after();
          const uint32_t st = smem_u32(smem + stage * kPairStageBytes);
          const uint32_t q_hi = st, q_lo = st + kQPlaneBytes, t_hi = st + 2 * kQPlaneBytes, t_lo = st + 3 * kQPlaneBytes;
#pragma unroll
          for (int pass = 0; pass < 3; ++pass) {
            if (pass < passes) {
              const uint32_t a = (pass == 2 ? q_lo : q_hi);
              const uint32_t bsm = (pass == 1 ? t_lo : t_hi);
#pragma unroll
              for (int k16 = 0; k16 < kBlockK / 16; ++k16) {
                const uint32_t accum = (kb | pass | k16) != 0 ? 1u : 0u;
                umma_f16_pair(d, umma_desc_kmajor<kRowBytes>(a + k16 * 32), umma_desc_kmajor<kRowBytes>(bsm + k16 * 32),
                              kIdescPair, accum);
              }
            }
          }
          umma_commit_pair(&tail.empty_bar[stage]);           // frees the stage in BOTH CTAs
          if (++stage == kPairStages) { stage = 0; phase ^= 1; }
        }
        umma_commit_pair(&tail.tmem_full_bar[acc]);            // accumulators of both CTAs complete
      }
    }
  } else if (warp >= 4) {
    // ========================================= epilogue (both CTAs) =========================================
    const int e = warp - 4;
    const int q = e & 3, ch = e >> 2;
    const int tid = e * 32 + lane;           // 0..255: column owned in the combine steps
    const int r = q * 32 + lane;             // row within this CTA's 128 rows
    const int t_row = (int)rank * kHalfRows + r;
    const float thr = p.sim_threshold;
    const uint32_t peer = rank ^ 1u;
    uint32_t unit = 0;
    GP_PAIR_ITEMS(, ++unit) {
      int j, n;
      decode_item(item, p.B, p.T, j, n);
      const int b = p.perm[j];
      const size_t rec = (size_t)b * p.T + n;
      const uint32_t acc = unit & 1u, slot = unit & 1u, xpar = (unit >> 1) & 1u;
      tail.smask[tid] = p.bank_mask[((size_t)p.q_obj[b] * p.T + n) * kP + tid];
      tail.tmask[tid] = p.q_mask[(size_t)b * kP + tid];
      named_barrier_sync(1, kEpiThreads);

      const float tm = tail.tmask[t_row];
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * 256 + ch * 128;
      mbar_wait(&tail.tmem_full_bar[acc], (unit >> 1) & 1u);
      tc_fence_after();
      float rmax = -1.0f;
      int ridx = 0;
#pragma unroll 1
      for (int c0 = 0; c0 < 128; c0 += 32) {
        uint32_t v32[32];
        tmem_ld_32x32(taddr + c0, v32);
        tmem_ld_wait();
        const int s0 = ch * 128 + c0;
        uint32_t keep_m = 0, keep_b = 1;
#pragma unroll
        for (int jj = 0; jj < 32; ++jj) {
          if (kDebug) p.debug_tile[((size_t)item * kP + t_row) * kP + s0 + jj] = __uint_as_float(v32[jj]);
          float v = __uint_as_float(v32[jj]) * tail.smask[s0 + jj];         // matching.py:234
          v = v * tm;                                                        // matching.py:235
          v = (v < thr) ? 0.0f : v;                                          // matching.py:236
          if (v > rmax) { rmax = v; ridx = s0 + jj; }
          const uint32_t bits = __float_as_uint(v);
          const uint32_t m = __reduce_max_sync(0xffffffffu, bits);
          const uint32_t bal = __ballot_sync(0xffffffffu, bits == m);
          if (lane == jj) { keep_m = m; keep_b = bal; }
        }
        tail.pmax[q][s0 + lane] = __uint_as_float(keep_m);
        tail.pidx[q][s0 + lane] = (uint8_t)((int)rank * kHalfRows + q * 32 + __ffs(keep_b) - 1);
      }
      tail.rowp_max[ch][r] = rmax;
      tail.rowp_idx[ch][r] = (uint8_t)ridx;
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(&tail.tmem_empty_bar[acc], 0);      // accumulator back to the leader's UMMA warp
      named_barrier_sync(1, kEpiThreads);
      if (ch == 0) {                          // merge the two column halves of row r (ties: lower s wins)
        float a = tail.rowp_max[0][r];
        uint8_t ai = tail.rowp_idx[0][r];
        const float c = tail.rowp_max[1][r];
        if (c > a) { a = c; ai = tail.rowp_idx[1][r]; }
        tail.rmax_s[r] = a;
        tail.ridx_s[r] = ai;
      }
      // column tid: maximum over this CTA's 128 rows (ascending t, strict > keeps the first), sent to the peer
      float best = tail.pmax[0][tid];
      uint8_t bi = tail.pidx[0][tid];
#pragma unroll
      for (int g = 1; g < 4; ++g) {
        const float v = tail.pmax[g][tid];
        if (v > best) { best = v; bi = tail.pidx[g][tid]; }
      }
      st_cluster_f32(mapa_u32(smem_u32(&tail.half_cmax[slot][tid]), peer), best);
      st_cluster_u8(mapa_u32(smem_u32(&tail.half_cidx[slot][tid]), peer), bi);
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(&tail.xchg_bar[slot], peer);        // release: the stores above are visible
      mbar_wait_cluster(&tail.xchg_bar[slot], xpar);
      {
        const float ov = tail.half_cmax[slot][tid];
        const uint8_t oi = tail.half_cidx[slot][tid];
        // lower t wins ties: the leader's half (t < 128) comes first
        float lo_v = rank == 0 ? best : ov, hi_v = rank == 0 ? ov : best;
        uint8_t lo_i = rank == 0 ? bi : oi, hi_i = rank == 0 ? oi : bi;
        if (hi_v > lo_v) { lo_v = hi_v; lo_i = hi_i; }
        tail.cmax[tid] = lo_v;
        tail.cidx[tid] = lo_i;
      }
      named_barrier_sync(1, kEpiThreads);

      // matching.py:247-271 for this CTA's query patches t = 128 rank + tid (threads 0..127)
      float s_contrib = 0.f, s_mall = 0.f;
      if (tid < kHalfRows) {
        const int t = (int)rank * kHalfRows + tid;
        const float rm = tail.rmax_s[tid];
        const int ri = tail.ridx_s[tid];
        const float tmv = tail.tmask[t];
        const bool mask_sim = rm >= thr;
        const int back = tail.cidx[ri];
        const float dx = (float)(back & 15) - (float)(t & 15);
        const float dy = (float)(back >> 4) - (float)(t >> 4);
        const bool mask_cycle = (sqrtf(dx * dx + dy * dy) <= p.patch_threshold) && (tail.cmax[ri] >= thr);
        float mnz = tmv * tail.smask[ri];
        mnz = mnz * (tail.cidx[t] != 0 ? 1.0f : 0.0f);
        mnz = mnz * (ri != 0 ? 1.0f : 0.0f);
        const float mall = (mask_sim && mask_cycle) ? mnz : 0.0f;
        s_contrib = rm * mall;
        s_mall = mall;
        p.rec_score[rec * kP + t] = rm;
        p.rec_idx[rec * kP + t] = (uint8_t)ri;
        p.rec_valid[rec * kP + t] = (mall != 0.0f) ? 1 : 0;
      }
      if (e < 4) {                             // epilogue warps 0..3 hold the patches: red[] lists the 8 sums in ascending t
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
          s_contrib += __shfl_xor_sync(0xffffffffu, s_contrib, off);
          s_mall += __shfl_xor_sync(0xffffffffu, s_mall, off);
        }
        if (lane == 0) {
          if (rank == 0) {
            tail.red[0][e] = s_contrib;
            tail.red[1][e] = s_mall;
          } else {
            st_cluster_f32(mapa_u32(smem_u32(&tail.red[0][4 + e]), 0), s_contrib);
            st_cluster_f32(mapa_u32(smem_u32(&tail.red[1][4 + e]), 0), s_mall);
          }
        }
      }
      named_barrier_sync(1, kEpiThreads);
      if (tid == 0) {
        if (rank != 0) {
          mbar_arrive_cluster(&tail.sum_bar[slot], 0);                      // release after the barrier above: all 8 stores done
        } else {
          mbar_wait_cluster(&tail.sum_bar[slot], xpar);
          float a = 0.f, m = 0.f;
#pragma unroll
          for (int g = 0; g < kEpiWarps; ++g) { a += tail.red[0][g]; m += tail.red[1][g]; }
          p.sim_avg[rec] = (m > 0.f) ? a / (float)kP : 0.0f;                // matching.py:274-278
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                                      // the leader's UMMAs / commits and the DSMEM stores reach across until here
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, kTmemCols);
  }
}
#undef GP_PAIR_ITEMS

// ------------------------------------------------------------------------------------------------------------
// top-k template selection (matching.py:279) + compact candidate records
// ------------------------------------------------------------------------------------------------------------
// One CTA per query.  k rounds of block-wide arg-max over the per-template scores; ties break towards the lowest
// template index (torch.topk leaves tie order unspecified).  Emits one compact record per winner:
//   cand_score[b,k] f32, cand_id[b,k] i32 (GLOBAL template id = local * id_stride + id_offset),
//   cand_pts_score[b,k,256] f32, cand_idx[b,k,256] u8, cand_valid[b,k,256] u8
__global__ void __launch_bounds__(256)
topk_select_kernel(TopkSelectParams p) {
  extern __shared__ float s_val[];                 // [T]
  __shared__ float s_wv[8];
  __shared__ int s_wi[8];
  __shared__ int s_win;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < p.T; i += 256) s_val[i] = p.sim_avg[(size_t)b * p.T + i];
  __syncthreads();
  for (int kk = 0; kk < p.k; ++kk) {
    float bv = -INFINITY;
    int bi = 0x7fffffff;
    for (int i = tid; i < p.T; i += 256) {
      const float v = s_val[i];
      if (v != -INFINITY && (v > bv || (v == bv && i < bi))) { bv = v; bi = i; }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, off);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
      if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    if (lane == 0) { s_wv[warp] = bv; s_wi[warp] = bi; }
    __syncthreads();
    if (tid == 0) {
      for (int w = 1; w < 8; ++w)
        if (s_wv[w] > bv || (s_wv[w] == bv && s_wi[w] < bi)) { bv = s_wv[w]; bi = s_wi[w]; }
      s_win = bi;
      const size_t o = (size_t)b * p.k + kk;
      if (bi < p.T) {
        p.cand_score[o] = bv;
        p.cand_id[o] = bi * p.id_stride + p.id_offset;
        s_val[bi] = -INFINITY;                     // exclude from later rounds (scores themselves are >= 0)
      } else {                                     // fewer than k local templates: padding candidate
        p.cand_score[o] = -INFINITY;
        p.cand_id[o] = 0x7fffffff;
      }
    }
    __syncthreads();
    const int win = s_win;
    const size_t o = ((size_t)b * p.k + kk) * kP + tid;
    if (win < p.T) {
      const size_t r = ((size_t)b * p.T + win) * kP + tid;
      p.cand_pts_score[o] = p.rec_score[r];
      p.cand_idx[o] = p.rec_idx[r];
      p.cand_valid[o] = p.rec_valid[r];
    } else {
      p.cand_pts_score[o] = 0.f;
      p.cand_idx[o] = 0;
      p.cand_valid[o] = 0;
    }
    __syncthreads();
  }
}

// Merge G per-shard candidate lists (G = 1 on a single GPU) into the global top-k and expand the winners into the
// reference's output format (matching.py:282-316, format_prediction :29-61):
//   id_src[B,k] i64, score_src[B,k] f32, score_pts[B,k,256] f32, tar_pts/src_pts[B,k,256,2] i64 (-1 = invalid).
// Candidates are laid out [G][B][k]; ordering = score descending, then global template id ascending.
template <typename T>
__device__ __forceinline__ const T* rank_ptr(const T* base, int g, size_t rank_stride_bytes, size_t dense_elems) {
  return rank_stride_bytes ? reinterpret_cast<const T*>(reinterpret_cast<const char*>(base) + (size_t)g * rank_stride_bytes)
                           : base + (size_t)g * dense_elems;
}

__global__ void __launch_bounds__(256)
topk_merge_expand_kernel(TopkMergeParams p) {
  __shared__ int s_sel[32];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int ncand = p.G * p.k;
  const size_t bk = (size_t)p.B * p.k;
  if (tid == 0) {
    // tiny selection sort over <= 64 candidates: score descending, then global template id ascending
    unsigned long long used = 0;
    for (int kk = 0; kk < p.k; ++kk) {
      float bv = 0.f; int bid = 0; int bc = -1;
      for (int c = 0; c < ncand; ++c) {
        if (used >> c & 1ull) continue;
        const int g = c / p.k, j = c - g * p.k;
        const size_t o = (size_t)b * p.k + j;
        const float v = rank_ptr(p.cand_score, g, p.rank_stride_bytes, bk)[o];
        const int id = rank_ptr(p.cand_id, g, p.rank_stride_bytes, bk)[o];
        if (bc < 0 || v > bv || (v == bv && id < bid)) { bv = v; bid = id; bc = c; }
      }
      used |= 1ull << bc;
      s_sel[kk] = bc;
    }
  }
  __syncthreads();
  for (int kk = 0; kk < p.k; ++kk) {
    const int c = s_sel[kk];
    const int g = c / p.k, j = c - g * p.k;
    const size_t o = (size_t)b * p.k + j;
    const size_t dst = (size_t)b * p.k + kk;
    if (tid == 0) {
      p.id_src[dst] = (long long)rank_ptr(p.cand_id, g, p.rank_stride_bytes, bk)[o];
      p.score_src[dst] = rank_ptr(p.cand_score, g, p.rank_stride_bytes, bk)[o];
    }
    const int t = tid;
    const bool valid = rank_ptr(p.cand_valid, g, p.rank_stride_bytes, bk * kP)[o * kP + t] != 0;
    const int s = rank_ptr(p.cand_idx, g, p.rank_stride_bytes, bk * kP)[o * kP + t];
    p.score_pts[dst * kP + t] = rank_ptr(p.cand_pts_score, g, p.rank_stride_bytes, bk * kP)[o * kP + t];
    longlong2 tp, sp;
    tp.x = valid ? (long long)(t & 15) : -1ll;
    tp.y = valid ? (long long)(t >> 4) : -1ll;
    sp.x = valid ? (long long)(s & 15) : -1ll;
    sp.y = valid ? (long long)(s >> 4) : -1ll;
    reinterpret_cast<longlong2*>(p.tar_pts)[dst * kP + t] = tp;
    reinterpret_cast<longlong2*>(p.src_pts)[dst * kP + t] = sp;
    if (p.out_rel_scale && p.cand_rel_scale)
      p.out_rel_scale[dst * kP + t] = rank_ptr(p.cand_rel_scale, g, p.rank_stride_bytes, bk * kP)[o * kP + t];
    if (p.out_rel_inplane && p.cand_rel_inplane)
      reinterpret_cast<float2*>(p.out_rel_inplane)[dst * kP + t] =
          reinterpret_cast<const float2*>(rank_ptr(p.cand_rel_inplane, g, p.rank_stride_bytes, bk * kP * 2))[o * kP + t];
  }
}

// ------------------------------------------------------------------------------------------------------------
// host-side launchers
// ------------------------------------------------------------------------------------------------------------
cudaError_t launch_sim_search(const CUtensorMap& q_hi, const CUtensorMap& q_lo, const CUtensorMap& t_hi,
                              const CUtensorMap& t_lo, const SimSearchParams& p, int num_sms, cudaStream_t stream) {
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(sim_search_pair_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPairSmemBytes);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(sim_search_pair_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPairSmemBytes);
    if (e != cudaSuccess) return e;
    configured = true;
  }
  if (p.num_items <= 0) return cudaSuccess;
  const int clusters = p.num_items < num_sms / 2 ? p.num_items : num_sms / 2;   // one 2-CTA cluster per item
  auto kernel = p.debug_tile ? sim_search_pair_kernel<true> : sim_search_pair_kernel<false>;
  return launch_ex(kernel, dim3(2 * clusters), dim3(kThreads), kPairSmemBytes, stream, 2, q_hi, q_lo, t_hi, t_lo, p);
}

cudaError_t launch_topk_select(const TopkSelectParams& p, cudaStream_t stream) {
  if (p.B <= 0) return cudaSuccess;
  topk_select_kernel<<<p.B, 256, p.T * sizeof(float), stream>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_topk_merge_expand(const TopkMergeParams& p, cudaStream_t stream) {
  if (p.B <= 0) return cudaSuccess;
  topk_merge_expand_kernel<<<p.B, 256, 0, stream>>>(p);
  return cudaGetLastError();
}

int sim_search_smem_bytes() { return kPairSmemBytes; }

}  // namespace gp
