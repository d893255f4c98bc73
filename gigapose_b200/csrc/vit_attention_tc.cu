// Multi-head self-attention of the ViT-L/14 forward on TMA + tcgen05 (row a1; 257 tokens, 16 heads x 64).
//
// Persistent CTAs (one per SM) walk the (crop, head) items; the TMA producer runs ahead of the tensor pipe, so the next
// item's Q / K / V tiles land while the current item's softmax and P.V still run (K and Q are free as soon as the last
// S = Q K^T of an item has retired), and barrier setup / TMEM allocation / cold instruction fetch are paid once per SM
// instead of once per item.  Per item: K and V of the head (272 key rows: 257 + padding) are TMA-staged once into shared
// memory as bf16 hi/lo planes (SWIZZLE_128B, 128-byte rows); the 257 query rows go through in three 128-row tiles:
//   S = Q K^T          tcgen05.mma SS, M=128, N=256+16, K=64      (A = Q tile, B = K, both K-major)   -> TMEM [0,272)
//   softmax            256 threads, two per query row (keys [0,128) and [128,257); the two warps of a TMEM lane quarter
//                      exchange row max / row sum through shared memory): tcgen05.ld S, fp32 max / ex2 / sum; P is
//                      written back to TMEM as packed bf16 pairs (hi over the first 16 columns of the 32-column S
//                      chunk it came from -- already consumed by the same thread -- lo next to S)
//   O = P V            tcgen05.mma TS, M=128, N=64, K=272          (A = P from TMEM, B = V as MN-major operand)
//   epilogue           tcgen05.ld O, divide by the row sum, store bf16 hi/lo planes (A operand of the proj GEMM)
// Both products use the fp32-faithful split: S = Qh Kh + Qh Kl + Ql Kh, O = Ph Vh + Ph Vl + Pl Vh.
// The 257th query row (token 256) would cost a third 128-row tile; one extra warp computes it with fp32 FMAs from the
// same shared-memory K / V planes while the tensor pipeline runs.
// Warp roles: warp 0 TMA producer (+ TMEM alloc), warp 1 UMMA issuer, warps 2-9 softmax / epilogue, warp 10 last row.
#include "gigapose_kernels.h"
#include "common.cuh"
#include <cuda_bf16.h>

namespace gp {

namespace {

constexpr int kTok = 257, kDim = 1024, kHeads = 16, kHd = 64;
constexpr int kKeys = 272;                         // 17 x 16
constexpr int kRow = 128;                          // bytes per smem row (64 bf16) = SWIZZLE_128B span
constexpr int kKVPlane = kKeys * kRow;             // 34 KB
constexpr int kQPlane = 128 * kRow;                // 16 KB
constexpr int kQTiles = 2;                         // tokens 0..255 on the tensor path; token 256 on one SIMT warp
constexpr int kSoftmaxWarps = 8;
constexpr int kThreads = (2 + kSoftmaxWarps + 1) * 32;
// TMEM columns: S [0,288) (the MMAs write [0,272); P_hi of keys [32c,32c+32) later overwrites columns [32c,32c+16)),
// P_lo [288,432), O [432,496)
constexpr uint32_t kColS = 0, kColPlo = 288, kColO = 432;
constexpr uint32_t kIdescS256 = umma_idesc_f16(128, 256, 1);
constexpr uint32_t kIdescS16 = umma_idesc_f16(128, 16, 1);
constexpr uint32_t kIdescPV = umma_idesc_f16(128, 64, 1, /*B MN-major*/ 1);

struct __align__(8) AttnTail {
  uint64_t k_full, v_full, k_empty, v_empty, q_full[2], q_empty[2], s_full, p_ready, o_full;
  uint32_t tmem_base;
};
constexpr int kSmem = 1024 + 4 * kKVPlane + 4 * kQPlane + sizeof(AttnTail);

// (a, b) -> packed bf16x2 hi word (a in the low half) and the bf16x2 of the residuals: 6 instructions per pair
__device__ __forceinline__ void split_pair(float a, float b, uint32_t& hi, uint32_t& lo) {
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(b), "f"(a));
  const float ra = a - __uint_as_float(hi << 16), rb = b - __uint_as_float(hi & 0xffff0000u);
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(rb), "f"(ra));
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// exp(x / 8) = 2^(x * log2(e) / 8); the 1/sqrt(64) logit scale is folded into the constant
constexpr float kExpScale = 0.125f * 1.4426950408889634f;
// fp32 value of element `col` of row `row` in a [rows][64] bf16 hi/lo tile stored with the 128-byte TMA swizzle
// (`lo` may be null: plain bf16 mode)
__device__ __forceinline__ float2 ld_pair_sw128(const uint8_t* hi, const uint8_t* lo, int row, int col) {
  const uint32_t off = (uint32_t)row * 128u + ((((uint32_t)col >> 3) ^ ((uint32_t)row & 7u)) << 4) + (((uint32_t)col & 7u) << 1);
  const uint32_t h = *reinterpret_cast<const uint32_t*>(hi + off);
  const uint32_t l = lo ? *reinterpret_cast<const uint32_t*>(lo + off) : 0u;
  return make_float2(__uint_as_float(h << 16) + __uint_as_float(l << 16),
                     __uint_as_float(h & 0xffff0000u) + __uint_as_float(l & 0xffff0000u));
}

}  // namespace

// cycle stamps of CTA 300 (a warm, second-wave CTA; CTA 0 for small grids) (diagnostics: gp_debug_attention_timeline)
__device__ long long g_attn_stamp[32];
#define STAMP(i) do { if (blockIdx.x == (gridDim.x > 300 ? 300u : 0u)) g_attn_stamp[i] = clock64(); } while (0)

template <int kPasses>        // 3 = fp32-faithful split products, 1 = plain bf16 (a template parameter: the other mode's code
__global__ void __launch_bounds__(kThreads, 1)   // and registers stay out of the instruction stream)
attention_tc_kernel(const __grid_constant__ CUtensorMap tm_hi_128, const __grid_constant__ CUtensorMap tm_lo_128,
                    const __grid_constant__ CUtensorMap tm_hi_16, const __grid_constant__ CUtensorMap tm_lo_16,
                    const __nv_bfloat16* __restrict__ qkv_hi, const __nv_bfloat16* __restrict__ qkv_lo,
                    __nv_bfloat16* __restrict__ out_hi, __nv_bfloat16* __restrict__ out_lo, int crop_stride, int num_items) {
  constexpr int passes = kPasses;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sK[2] = {smem, smem + kKVPlane};                                   // hi, lo
  uint8_t* sV[2] = {smem + 2 * kKVPlane, smem + 3 * kKVPlane};
  uint8_t* sQ = smem + 4 * kKVPlane;                                          // [buf][hi|lo]
  AttnTail& tail = *reinterpret_cast<AttnTail*>(smem + 4 * kKVPlane + 4 * kQPlane);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // item -> (crop, head) and the first rows of its operands: head-major planes [q|k|v][crop][head][token][64]
  auto coords = [&](int item, int& head, int& row0, int& rq, int& rk, int& rv) {
    const int img = item / kHeads;
    head = item % kHeads;
    row0 = img * kTok;                               // first token row of this crop in the [M, 1024] output planes
    rq = ((0 * crop_stride + img) * kHeads + head) * kTok;
    rk = ((1 * crop_stride + img) * kHeads + head) * kTok;
    rv = ((2 * crop_stride + img) * kHeads + head) * kTok;
  };

  if (threadIdx.x == 0) {
    mbar_init(&tail.k_full, 1);
    mbar_init(&tail.v_full, 1);
    mbar_init(&tail.k_empty, 2);                       // last S = Q K^T retired (tcgen05.commit) + the token-256 warp is done with K
    mbar_init(&tail.v_empty, 2);                       // last P V retired + the token-256 warp is done with V
    for (int i = 0; i < 2; ++i) { mbar_init(&tail.q_full[i], 1); mbar_init(&tail.q_empty[i], 1); }
    mbar_init(&tail.s_full, 1);
    mbar_init(&tail.p_ready, kSoftmaxWarps);
    mbar_init(&tail.o_full, 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(&tail.tmem_base, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tail.tmem_base;
  if (threadIdx.x == 0) STAMP(0);

  if (warp == 0) {
    // ============================== TMA producer ==============================
    if (lane == 0) {
      const int np = passes == 3 ? 2 : 1;
      tma_prefetch_desc(&tm_hi_128); tma_prefetch_desc(&tm_hi_16);
      if (np == 2) { tma_prefetch_desc(&tm_lo_128); tma_prefetch_desc(&tm_lo_16); }
      // order of issue = order of need: Q tile 0, K (for S), then V (only needed after the first softmax), Q tile 1.
      // Every buffer is filled once per item; fill number `it` waits for release number `it - 1` (parity (it & 1) ^ 1,
      // which a fresh barrier passes at once).
      int it = 0;
      for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
        int head, row0, rq, rk, rv;
        coords(item, head, row0, rq, rk, rv);
        const uint32_t free_par = (uint32_t)(it & 1) ^ 1u;
        mbar_wait(&tail.q_empty[0], free_par);
        mbar_arrive_expect_tx(&tail.q_full[0], (uint32_t)(np * kQPlane));
        tma_load_2d(sQ, &tm_hi_128, &tail.q_full[0], 0, rq);
        if (np == 2) tma_load_2d(sQ + kQPlane, &tm_lo_128, &tail.q_full[0], 0, rq);
        mbar_wait(&tail.k_empty, free_par);
        mbar_arrive_expect_tx(&tail.k_full, (uint32_t)(np * kKVPlane));
        for (int pl = 0; pl < np; ++pl) {
          const CUtensorMap* m128 = pl ? &tm_lo_128 : &tm_hi_128;
          const CUtensorMap* m16 = pl ? &tm_lo_16 : &tm_hi_16;
          tma_load_2d(sK[pl], m128, &tail.k_full, 0, rk);
          tma_load_2d(sK[pl] + 128 * kRow, m128, &tail.k_full, 0, rk + 128);
          tma_load_2d(sK[pl] + 256 * kRow, m16, &tail.k_full, 0, rk + 256);
        }
        mbar_wait(&tail.v_empty, free_par);
        mbar_arrive_expect_tx(&tail.v_full, (uint32_t)(np * kKVPlane));
        for (int pl = 0; pl < np; ++pl) {
          const CUtensorMap* m128 = pl ? &tm_lo_128 : &tm_hi_128;
          const CUtensorMap* m16 = pl ? &tm_lo_16 : &tm_hi_16;
          tma_load_2d(sV[pl], m128, &tail.v_full, 0, rv);
          tma_load_2d(sV[pl] + 128 * kRow, m128, &tail.v_full, 0, rv + 128);
          tma_load_2d(sV[pl] + 256 * kRow, m16, &tail.v_full, 0, rv + 256);
        }
        for (int qt = 1; qt < kQTiles; ++qt) {
          const int buf = qt & 1;
          mbar_wait(&tail.q_empty[buf], free_par);
          mbar_arrive_expect_tx(&tail.q_full[buf], (uint32_t)(np * kQPlane));
          tma_load_2d(sQ + (buf * 2 + 0) * kQPlane, &tm_hi_128, &tail.q_full[buf], 0, rq + qt * 128);
          if (np == 2) tma_load_2d(sQ + (buf * 2 + 1) * kQPlane, &tm_lo_128, &tail.q_full[buf], 0, rq + qt * 128);
        }
      }
    }
  } else if (warp == 1) {
    // ============================== UMMA issuer ==============================
    if (lane == 0) {
      const uint32_t kh = smem_u32(sK[0]), kl = smem_u32(sK[1]), vh = smem_u32(sV[0]), vl = smem_u32(sV[1]);
      int it = 0;
      for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
      const uint32_t item_par = (uint32_t)(it & 1);      // K, V and each Q buffer are filled once per item
      mbar_wait(&tail.k_full, item_par);
      tc_fence_after();
      STAMP(1);
      for (int qt = 0; qt < kQTiles; ++qt) {
        const int buf = qt & 1;
        mbar_wait(&tail.q_full[buf], item_par);
        tc_fence_after();
        const uint32_t qh = smem_u32(sQ + (buf * 2 + 0) * kQPlane), ql = smem_u32(sQ + (buf * 2 + 1) * kQPlane);
        // S = Q K^T : keys [0,256) and [256,272)
#pragma unroll
        for (int pass = 0; pass < 3; ++pass) {
          if (pass < passes) {
            const uint32_t a = pass == 2 ? ql : qh, b = pass == 1 ? kl : kh;
#pragma unroll
            for (int k16 = 0; k16 < 4; ++k16) {
              const uint32_t acc = (pass | k16) != 0 ? 1u : 0u;
              umma_f16(tmem + kColS, umma_desc_kmajor<kRow>(a + k16 * 32), umma_desc_kmajor<kRow>(b + k16 * 32), kIdescS256, acc);
              umma_f16(tmem + kColS + 256, umma_desc_kmajor<kRow>(a + k16 * 32),
                       umma_desc_kmajor<kRow>(b + 256 * kRow + k16 * 32), kIdescS16, acc);
            }
          }
        }
        umma_commit(&tail.q_empty[buf]);               // Q buffer free once these MMAs retire
        if (qt == kQTiles - 1) umma_commit(&tail.k_empty);   // ... and K: the producer may fetch the next item's keys
        umma_commit(&tail.s_full);
        STAMP(2 + 4 * qt);
        // O = P V once the softmax warps have written P
        if (qt == 0) mbar_wait(&tail.v_full, item_par);
        mbar_wait(&tail.p_ready, qt & 1);
        tc_fence_after();
        STAMP(3 + 4 * qt);
#pragma unroll
        for (int j = 0; j < kKeys / 16; ++j) {         // 17 key steps
          const uint32_t ph = tmem + kColS + 32 * (j >> 1) + 8 * (j & 1), pl = tmem + kColPlo + 8 * j;   // keys 16j..16j+15
          const uint64_t dvh = umma_desc_mnmajor_sw128(vh + j * 16 * kRow), dvl = umma_desc_mnmajor_sw128(vl + j * 16 * kRow);
          umma_f16_ts(tmem + kColO, ph, dvh, kIdescPV, j != 0 ? 1u : 0u);
          if (passes == 3) {
            umma_f16_ts(tmem + kColO, ph, dvl, kIdescPV, 1u);
            umma_f16_ts(tmem + kColO, pl, dvh, kIdescPV, 1u);
          }
        }
        umma_commit(&tail.o_full);
        if (qt == kQTiles - 1) umma_commit(&tail.v_empty);
        STAMP(4 + 4 * qt);
      }
      }
    }
  } else if (warp < 2 + kSoftmaxWarps) {
    // ============================== softmax + epilogue (warps 2-9) ==============================
    // warps w and w+4 share a TMEM lane quarter (w & 3): the same 32 query rows, key columns split in two halves
    __shared__ float s_mx[2][128];
    __shared__ float s_sum[2][128];
    const int quarter = warp & 3;                      // TMEM lane quarter this warp may access
    const int half = (warp - 2) >> 2;                  // 0: keys [0,128)   1: keys [128,257)
    const int r = quarter * 32 + lane;                 // query row inside the tile
    const uint32_t lane_base = (uint32_t)(quarter * 32) << 16;
    const uint32_t s_base = tmem + lane_base + kColS + 128 * half;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
    int head, row0, rq_, rk_, rv_;
    coords(item, head, row0, rq_, rk_, rv_);
    // s_full / p_ready / o_full complete twice per item, so their parity is the q-tile index whatever the item
    for (int qt = 0; qt < kQTiles; ++qt) {
      const int tok = qt * 128 + r;
      const bool row_ok = tok < kTok;
      mbar_wait(&tail.s_full, qt & 1);
      tc_fence_after();
      if (warp == 2 && lane == 0) STAMP(12 + 5 * qt);
      // pass 1: maximum of the raw logits over this half's keys (4 chunks of 32 columns; + column 256 in half 1)
      float mx = -INFINITY;
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        uint32_t v[32];
        tmem_ld_32x32(s_base + 32 * c, v);
        tmem_ld_wait_for(v);
#pragma unroll
        for (int j = 0; j < 32; ++j) mx = fmaxf(mx, __uint_as_float(v[j]));
      }
      float tail_logit = -INFINITY;                    // key 256 (columns [256,288): only the first is real)
      if (half == 1) {
        uint32_t tailv[32];
        tmem_ld_32x32(tmem + lane_base + kColS + 256, tailv);
        tmem_ld_wait_for(tailv);
        tail_logit = __uint_as_float(tailv[0]);
        mx = fmaxf(mx, tail_logit);
      }
      s_mx[half][r] = mx;
      named_barrier_sync(1 + quarter, 64);
      mx = fmaxf(mx, s_mx[half ^ 1][r]);
      if (warp == 2 && lane == 0) STAMP(13 + 5 * qt);
      // pass 2: p = exp((s - max) / 8) via ex2; P goes back to TMEM as packed bf16 pairs; row sum in fp32
      float sum4[4] = {0.f, 0.f, 0.f, 0.f};
      auto do_chunk = [&](uint32_t (&v)[32], int c) {   // c = chunk inside this half; keys 128*half + 32c ..
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float pa = ex2_approx((__uint_as_float(v[2 * j]) - mx) * kExpScale);
          const float pb = ex2_approx((__uint_as_float(v[2 * j + 1]) - mx) * kExpScale);
          sum4[j & 3] += pa + pb;
          split_pair(pa, pb, hi[j], lo[j]);
        }
        tmem_st_32x16(s_base + 32 * c, hi);            // first 16 columns of the chunk just read
        tmem_st_32x16(tmem + lane_base + kColPlo + 64 * half + 16 * c, lo);
      };
      {   // software-pipelined: chunk c+1 is in flight while chunk c is processed (the P store of chunk c only touches
          // chunk c's own columns)
        uint32_t va[32], vb[32];
        tmem_ld_32x32(s_base, va);
        tmem_ld_wait_for(va);
#pragma unroll
        for (int c = 0; c < 4; c += 2) {
          tmem_ld_32x32(s_base + 32 * (c + 1), vb);      // in flight during chunk c
          do_chunk(va, c);
          tmem_ld_wait_for(vb);
          if (c + 2 < 4) tmem_ld_32x32(s_base + 32 * (c + 2), va);   // in flight during chunk c+1
          do_chunk(vb, c + 1);
          if (c + 2 < 4) tmem_ld_wait_for(va);
        }
      }
      float sum = (sum4[0] + sum4[1]) + (sum4[2] + sum4[3]);
      if (half == 1) {
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) { hi[j] = 0u; lo[j] = 0u; }
        const float pa = ex2_approx((tail_logit - mx) * kExpScale);
        sum += pa;
        split_pair(pa, 0.f, hi[0], lo[0]);
        tmem_st_32x16(tmem + lane_base + kColS + 256, hi);          // keys 256..287 (271 used)
        tmem_st_32x16(tmem + lane_base + kColPlo + 128, lo);
      }
      s_sum[half][r] = sum;
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tail.p_ready);
      named_barrier_sync(1 + quarter, 64);               // partner's partial sum is in shared memory
      sum += s_sum[half ^ 1][r];
      if (warp == 2 && lane == 0) STAMP(14 + 5 * qt);
      // epilogue: O / sum -> bf16 hi/lo planes; this warp stores output columns [32*half, 32*half + 32)
      mbar_wait(&tail.o_full, qt & 1);
      tc_fence_after();
      if (warp == 2 && lane == 0) STAMP(15 + 5 * qt);
      const float inv = 1.0f / sum;
      {
        const int c = half;
        uint32_t v[32];
        tmem_ld_32x32(tmem + lane_base + kColO + 32 * c, v);
        tmem_ld_wait_for(v);
        if (row_ok) {
          uint32_t hi[16], lo[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            split_pair(__uint_as_float(v[2 * j]) * inv, __uint_as_float(v[2 * j + 1]) * inv, hi[j], lo[j]);
          }
          const size_t o = (size_t)(row0 + tok) * kDim + head * kHd + 32 * c;
          uint4* dh = reinterpret_cast<uint4*>(out_hi + o);
          uint4* dl = reinterpret_cast<uint4*>(out_lo + o);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            dh[j] = make_uint4(hi[4 * j], hi[4 * j + 1], hi[4 * j + 2], hi[4 * j + 3]);
            dl[j] = make_uint4(lo[4 * j], lo[4 * j + 1], lo[4 * j + 2], lo[4 * j + 3]);
          }
        }
      }
      tc_fence_before();                               // O / S reads done before the next tile's MMAs overwrite them
      if (warp == 2 && lane == 0) STAMP(16 + 5 * qt);
    }
    }
  } else {
    // ============================== token 256 on one warp (fp32 FMAs from the smem planes) ==============================
    __shared__ float s_p[kKeys];
    __shared__ float s_q[kHd];
    int it = 0;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
    int head, row0, rq, rk_, rv_;
    coords(item, head, row0, rq, rk_, rv_);
    const uint32_t item_par = (uint32_t)(it & 1);
    __syncwarp();                                      // the previous item's reads of s_q / s_p are done
    // q (64 values): lane loads q[2*lane], q[2*lane+1] straight from the planes and shares them through smem
    const size_t qoff = (size_t)(rq + 256) * kHd + 2 * lane;
    const uint32_t qh = *reinterpret_cast<const uint32_t*>(qkv_hi + qoff);
    const uint32_t ql = passes == 3 ? *reinterpret_cast<const uint32_t*>(qkv_lo + qoff) : 0u;
    s_q[2 * lane] = __uint_as_float(qh << 16) + __uint_as_float(ql << 16);
    s_q[2 * lane + 1] = __uint_as_float(qh & 0xffff0000u) + __uint_as_float(ql & 0xffff0000u);
    __syncwarp();
    mbar_wait(&tail.k_full, item_par);
    if (lane == 0) STAMP(24);
    const uint8_t* klo = passes == 3 ? sK[1] : nullptr;   // bf16 mode: the lo planes are not loaded
    const uint8_t* vlo = passes == 3 ? sV[1] : nullptr;
    // logits: lane handles keys lane, lane+32, ...; one 16-byte chunk (8 channels) of a K row per load
    float sj[9];
    float mx = -INFINITY;
#pragma unroll
    for (int i = 0; i < 9; ++i) {
      const int key = lane + 32 * i;
      float acc = 0.f;
      if (key < kTok) {
#pragma unroll
        for (int ch = 0; ch < 8; ++ch) {
          const uint32_t off = (uint32_t)key * 128u + (((uint32_t)ch ^ ((uint32_t)key & 7u)) << 4);
          const uint4 h4 = *reinterpret_cast<const uint4*>(sK[0] + off);
          const uint4 l4 = klo ? *reinterpret_cast<const uint4*>(klo + off) : make_uint4(0, 0, 0, 0);
          const uint32_t hw[4] = {h4.x, h4.y, h4.z, h4.w}, lw[4] = {l4.x, l4.y, l4.z, l4.w};
#pragma unroll
          for (int w = 0; w < 4; ++w) {
            const float k0 = __uint_as_float(hw[w] << 16) + __uint_as_float(lw[w] << 16);
            const float k1 = __uint_as_float(hw[w] & 0xffff0000u) + __uint_as_float(lw[w] & 0xffff0000u);
            acc = fmaf(s_q[ch * 8 + 2 * w], k0, acc);
            acc = fmaf(s_q[ch * 8 + 2 * w + 1], k1, acc);
          }
        }
      }
      sj[i] = key < kTok ? acc : -INFINITY;
      mx = fmaxf(mx, sj[i]);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < 9; ++i) {
      const int key = lane + 32 * i;
      const float pj = key < kTok ? ex2_approx((sj[i] - mx) * kExpScale) : 0.f;
      sum += pj;
      if (key < kKeys) s_p[key] = pj;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
    __syncwarp();
    if (lane == 0) { STAMP(25); mbar_arrive(&tail.k_empty); }   // every lane's K reads precede the shuffles above
    mbar_wait(&tail.v_full, item_par);
    // output: lane handles d = 2*lane, 2*lane+1 (4 partial accumulators, loads batched by the unroll)
    float o0[4] = {0.f, 0.f, 0.f, 0.f}, o1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 8
    for (int key = 0; key < 256; ++key) {
      const float2 vv = ld_pair_sw128(sV[0], vlo, key, 2 * lane);
      const float pj = s_p[key];
      o0[key & 3] = fmaf(pj, vv.x, o0[key & 3]);
      o1[key & 3] = fmaf(pj, vv.y, o1[key & 3]);
    }
    {
      const float2 vv = ld_pair_sw128(sV[0], vlo, 256, 2 * lane);
      o0[0] = fmaf(s_p[256], vv.x, o0[0]);
      o1[0] = fmaf(s_p[256], vv.y, o1[0]);
    }
    const float o0s = (o0[0] + o0[1]) + (o0[2] + o0[3]), o1s = (o1[0] + o1[1]) + (o1[2] + o1[3]);
    const float inv = 1.0f / sum;
    uint32_t h, l;
    split_pair(o0s * inv, o1s * inv, h, l);
    const size_t oo = (size_t)(row0 + 256) * kDim + head * kHd + 2 * lane;
    *reinterpret_cast<uint32_t*>(out_hi + oo) = h;
    *reinterpret_cast<uint32_t*>(out_lo + oo) = l;
    __syncwarp();                                      // every lane's V reads are done
    if (lane == 0) { STAMP(26); mbar_arrive(&tail.v_empty); }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

cudaError_t read_attention_stamps(long long* host32) {
  return cudaMemcpyFromSymbol(host32, g_attn_stamp, sizeof(long long) * 32);
}

cudaError_t launch_attention_tc(const CUtensorMap& hi128, const CUtensorMap& lo128, const CUtensorMap& hi16,
                                const CUtensorMap& lo16, const uint16_t* qkv_hi, const uint16_t* qkv_lo, uint16_t* out_hi,
                                uint16_t* out_lo, int b, int crop_stride, int passes, cudaStream_t s) {
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(attention_tc_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(attention_tc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
    if (e != cudaSuccess) return e;
    configured = true;
  }
  if (b <= 0) return cudaSuccess;
  static int num_sms = 0;
  if (!num_sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
  }
  const int items = b * kHeads;
  const dim3 grid(items < num_sms ? items : num_sms);
  auto qh = reinterpret_cast<const __nv_bfloat16*>(qkv_hi), ql = reinterpret_cast<const __nv_bfloat16*>(qkv_lo);
  auto oh = reinterpret_cast<__nv_bfloat16*>(out_hi), ol = reinterpret_cast<__nv_bfloat16*>(out_lo);
  if (passes == 3)
    return launch_ex(attention_tc_kernel<3>, grid, dim3(kThreads), kSmem, s, 1, hi128, lo128, hi16, lo16, qh, ql, oh, ol, crop_stride, items);
  return launch_ex(attention_tc_kernel<1>, grid, dim3(kThreads), kSmem, s, 1, hi128, lo128, hi16, lo16, qh, ql, oh, ol, crop_stride, items);
}

}  // namespace gp
