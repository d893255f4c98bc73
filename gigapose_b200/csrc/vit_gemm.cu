// The tcgen05 GEMM of this library: the linear layers of the DINOv2 ViT-L/14 forward (row a1 of SURVEY.md §8; the hub
// module the reference calls at ae_net.py:46 runs them as fp32 cuBLAS GEMMs) and, as implicit GEMMs, the convolutions
// of the IST trunk (row a6, ist_trunk.cu; cuDNN in the reference).
//
// C[M,N] = A[M,K] . W[N,K]^T with both operands stored as bf16 hi/lo planes (x = hi + lo to ~2^-17) and accumulated
// as hi*hi + hi*lo + lo*hi in fp32 TMEM accumulators -- the same fp32-faithful split as the similarity kernel
// (`passes = 1` = plain bf16).  Persistent CTAs, one output tile at a time:
//   warp 0  TMA producer   (32-column k-blocks, SWIZZLE_64B; A rows = 2-D boxes, or 4-D boxes of an NHWC plane when the
//                           GEMM is a convolution: one box per filter tap and 32-channel block, zero fill = padding)
//   warp 1  UMMA issuer    (M=128, N=128..256, K=16), two TMEM accumulators (2 x 256 columns)
//   warp 2  TMEM allocator
//   warps 4-11 epilogue    (TMEM -> registers -> fused bias / GELU / ReLU / LayerScale + residual / shortcut /
//                           positional table -> fp32 rows or bf16 hi/lo planes for the next layer), overlapping the
//                           next tile's MMAs; stores are transposed through shared memory into full 64-byte segments.
// Three tile shapes: <swap=0,pair=0> 128 x bn tiles on one CTA (patch embedding, convolutions); <0,1> 256 x bn tiles on
// a 2-CTA cluster (tcgen05 cta_group::2: the ViT linears and the IST regressor's hidden layers); <1,0> filters as the
// 128-row operand against 256 output pixels (the 128-channel convolutions).
#include "gigapose_kernels.h"
#include "common.cuh"
#include <cuda_bf16.h>
#include <cuda_fp16.h>

namespace gp {

namespace {

constexpr int kBlockK = 32;
constexpr int kRowBytes = kBlockK * 2;            // 64 B rows, SWIZZLE_64B
constexpr int kStages = 4;                        // 48 KB stages; CTA pairs: 6 stages of 32 KB (each CTA holds half of W)
constexpr int kPairStages = 6, kMaxStages = 6;
constexpr int kBM = 128, kBN = 256;
constexpr int kAPlane = kBM * kRowBytes;          // 8 KB
constexpr int kWPlane = kBN * kRowBytes;          // 16 KB
constexpr int kStageBytes = 2 * kAPlane + 2 * kWPlane;   // 48 KB
constexpr int kEpiWarps = 8;
constexpr int kThreads = 4 * 32 + kEpiWarps * 32;

struct __align__(8) GemmSmemTail {
  float bias_s[2][kBN];                           // per-tile bias / LayerScale columns, double buffered with the accumulator
  float gamma_s[2][kBN];
  uint8_t stage_buf[kEpiWarps][32 * 80];          // per-warp transposition buffer: 32 rows x (64 B + 16 B pad)
  uint64_t full_bar[kMaxStages];
  uint64_t empty_bar[kMaxStages];
  uint64_t tmem_full_bar[2];
  uint64_t tmem_empty_bar[2];
  uint32_t tmem_base;
};
constexpr int kSmemBytes = 1024 + kStages * kStageBytes + sizeof(GemmSmemTail);

// Grouped rasterisation: 16 m-tiles x all n-tiles per group, m fastest inside a group.  With plain m-fastest order all
// 148 CTAs stream the same 256-row weight tile at the same moment and serialise on its L2 lines; in a group every
// weight tile is shared by <= 16 CTAs and every activation tile by <= num_n CTAs.
constexpr int kGroupM = 16;
__device__ __forceinline__ void tile_coords(int tile, int num_m, int num_n, int& m_tile, int& n_tile) {
  const int per_group = kGroupM * num_n;
  const int g = tile / per_group, idx = tile - g * per_group;
  const int m_first = g * kGroupM;
  const int gm = min(kGroupM, num_m - m_first);
  n_tile = idx / gm;
  m_tile = m_first + (idx - n_tile * gm);
}

// GELU(x) = 0.5 x (1 + erf(x / sqrt 2)) through erfc(u) = t (a1 + t (a2 + t (a3 + t (a4 + t a5)))) exp(-u^2), t = 1 / (1 + p u)
// (Abramowitz & Stegun 7.1.26, |error| <= 1.5e-7 on erf): 1 + erf = erfc(|u|) for x < 0 (no cancellation) and 2 - erfc(|u|)
// otherwise.  14 instructions per element instead of erff's 25 (fc1 was the one layer whose epilogue was slower than its
// MMAs); against the exact function the result is off by <= 4.2e-7 absolute over [-8, 8] -- the same as the fp32 erff form
// (4.5e-7: both are dominated by the fp32 rounding of the final products).
__device__ __forceinline__ float gelu_erf(float x) {
  const float ax = fabsf(x);
  float t, e;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.231641888f, ax, 1.0f)));          // p / sqrt(2), p = 0.3275911
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * x * -0.72134752f));                   // exp(-x^2 / 2)
  float poly = fmaf(1.061405429f, t, -1.453152027f);
  poly = fmaf(poly, t, 1.421413741f);
  poly = fmaf(poly, t, -0.284496736f);
  poly = fmaf(poly, t, 0.254829592f);
  const float q = poly * t * e;                                                              // erfc(|x| / sqrt 2)
  return 0.5f * x * (x < 0.f ? q : 2.0f - q);
}

__device__ __forceinline__ uint32_t pack_bf16(__nv_bfloat16 a, __nv_bfloat16 b) {
  return (uint32_t)__bfloat16_as_ushort(a) | ((uint32_t)__bfloat16_as_ushort(b) << 16);
}

}  // namespace

// cycle stamps of CTA 0 for the QKV-shaped GEMM (diagnostics: gp_debug_gemm_timeline): [tile][0..3] =
// UMMA start, UMMA issued, epilogue start, epilogue end; [63] = kernel start
__device__ long long g_gemm_stamp[64];
#define GSTAMP(i) do { if (blockIdx.x == 0 && p.N == 3072 && (i) < 64) g_gemm_stamp[i] = clock64(); } while (0)

// kMode (GemmMode) is a template parameter: every layer type gets its own epilogue without the other modes' predicated
// code and registers (the shared runtime-mode epilogue needed 168 registers and ~35 instructions per output element).
// kSwap = false: rows of C are activation rows (tokens / output pixels), columns are output features.
// kSwap = true (convolutions with 128 output channels): the roles are exchanged -- the 128-row UMMA operand is the
// filter bank [128, K] and the 256-row operand is a tile of 256 output pixels, so that the tensor pipe still runs
// M=128 x N=256 instructions (an N=128 instruction re-reads its operands from shared memory twice as often per FLOP
// and is limited by shared-memory bandwidth); the epilogue transposes the [channel, pixel] accumulator back to NHWC.
// kPair = true: two CTAs of a cluster (the two SMs of a TPC) share one 256 x bn tile through `tcgen05.mma.cta_group::2`:
// each CTA stages its own 128 rows of A and bn/2 rows of W, the even CTA issues the M = 256 instructions, every CTA
// drains its own 128 accumulator rows.  Per SM the tensor core then reads 4 KB + 4 KB of operands per 128-cycle
// instruction instead of 4 KB + 8 KB, which is what the shared-memory pipe could not sustain next to the epilogue.
template <bool kSwap, bool kPair, int kMode>
__global__ void __launch_bounds__(kThreads, 1)
vit_gemm_kernel(const __grid_constant__ CUtensorMap tm_a_hi, const __grid_constant__ CUtensorMap tm_a_lo,
                const __grid_constant__ CUtensorMap tm_w_hi, const __grid_constant__ CUtensorMap tm_w_lo, GemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  static_assert(!(kSwap && kPair), "the swapped layers have M = 128 filters: nothing to pair");
  constexpr int kNumStages = kPair ? kPairStages : kStages;
  constexpr int kStageSz = kPair ? 2 * kAPlane + kWPlane : kStageBytes;       // 32 KB / 48 KB
  constexpr int kWLoOff = 2 * kAPlane + (kPair ? kWPlane / 2 : kWPlane);
  constexpr int kTileM = kPair ? 2 * kBM : kBM;
  GemmSmemTail& tail = *reinterpret_cast<GemmSmemTail*>(smem + kStages * kStageBytes);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int passes = p.passes;
  const int bn = p.bn > 0 ? p.bn : kBN;                     // 128 / 192 / 256 output columns per tile
  const uint32_t idesc = umma_idesc_f16(kTileM, bn, p.f16 ? 0 : 1);   // A / B formats: bf16 (1) or fp16 (0) hi / lo planes
  const int M_rows = p.m_dev ? min(*p.m_dev, p.M) : p.M;    // data-dependent row count (IST regressor): read on the device
  const int num_m = (M_rows + kTileM - 1) / kTileM, num_n = p.N / bn;
  const uint32_t rank = kPair ? cluster_ctarank() : 0u;     // 0 = leader of the pair
  const int first_tile = kPair ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int tile_step = kPair ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const int num_tiles = num_m * num_n;
  const int num_kb = p.K / kBlockK;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kNumStages; ++s) { mbar_init(&tail.full_bar[s], 1); mbar_init(&tail.empty_bar[s], 1); }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tail.tmem_full_bar[a], 1);
      mbar_init(&tail.tmem_empty_bar[a], kPair ? 2 * kEpiWarps : kEpiWarps);   // pair: both CTAs' epilogues report to the leader
    }
    fence_barrier_init();
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_a_hi); tma_prefetch_desc(&tm_w_hi);
    if (passes == 3) { tma_prefetch_desc(&tm_a_lo); tma_prefetch_desc(&tm_w_lo); }
  }
  if (warp == 2) { if constexpr (kPair) tmem_alloc_pair(&tail.tmem_base, 512); else tmem_alloc(&tail.tmem_base, 512); }
  tc_fence_before();
  __syncthreads();
  if constexpr (kPair) cluster_sync_all();         // barriers and TMEM of the peer exist before anything reaches across
  tc_fence_after();
  const uint32_t tmem_base = tail.tmem_base;
  if (threadIdx.x == 0) GSTAMP(63);

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      // pair: each CTA loads 128 rows of A + bn/2 rows of W; all bytes of both CTAs are counted on the leader's barrier
      const uint32_t tx = (passes == 3 ? 2 : 1) * (kPair ? 2 * (kAPlane + (bn >> 1) * kRowBytes) : kAPlane + bn * kRowBytes);
      for (int tile = first_tile; tile < num_tiles; tile += tile_step) {
        int mt, nt;
        tile_coords(tile, num_m, num_n, mt, nt);
        const int m0 = mt * kTileM + (int)rank * kBM, n0 = nt * bn + (kPair ? (int)rank * (bn >> 1) : 0);
        int img = 0, y0 = 0;
        if (p.conv) { const int hw = p.Ho * p.Wo, pix0 = kSwap ? n0 : m0; img = pix0 / hw; y0 = (pix0 - img * hw) / p.Wo; }
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&tail.empty_bar[stage], phase ^ 1);
          uint8_t* st = smem + stage * kStageSz;
          if (!kPair || rank == 0) mbar_arrive_expect_tx(&tail.full_bar[stage], tx);
          // the pixel operand (A, or W when kSwap) of a convolution: k-block = (tap ky,kx ; 32-channel block cb), a
          // shifted, strided window of the NHWC plane; the other operand is a plain [rows, K] matrix
          int cb = 0, cx = 0, cy = 0;
          if (p.conv) {
            const int tap = kb / p.cblocks;
            cb = kb - tap * p.cblocks;
            const int ky = tap / p.kw, kx = tap - ky * p.kw;
            cx = kx - p.pad; cy = y0 * p.stride + ky - p.pad;
          }
          auto load2 = [&](void* dst, const CUtensorMap* map, int c0, int c1) {
            if constexpr (kPair) tma_load_2d_pair(dst, map, &tail.full_bar[stage], c0, c1);
            else tma_load_2d(dst, map, &tail.full_bar[stage], c0, c1);
          };
          auto load4 = [&](void* dst, const CUtensorMap* map) {
            if constexpr (kPair) tma_load_4d_pair(dst, map, &tail.full_bar[stage], cb * kBlockK, cx, cy, img);
            else tma_load_4d(dst, map, &tail.full_bar[stage], cb * kBlockK, cx, cy, img);
          };
          if (p.conv && !kSwap) {
            load4(st, &tm_a_hi);
            if (passes == 3) load4(st + kAPlane, &tm_a_lo);
          } else {
            load2(st, &tm_a_hi, kb * kBlockK, m0);
            if (passes == 3) load2(st + kAPlane, &tm_a_lo, kb * kBlockK, m0);
          }
          if (p.conv && kSwap) {
            load4(st + 2 * kAPlane, &tm_w_hi);
            if (passes == 3) load4(st + kWLoOff, &tm_w_lo);
          } else {
            load2(st + 2 * kAPlane, &tm_w_hi, kb * kBlockK, n0);
            if (passes == 3) load2(st + kWLoOff, &tm_w_lo, kb * kBlockK, n0);
          }
          if (++stage == kNumStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && rank == 0) {
      int stage = 0; uint32_t phase = 0, unit = 0;
      for (int tile = first_tile; tile < num_tiles; tile += tile_step, ++unit) {
        const uint32_t acc = unit & 1u;
        mbar_wait(&tail.tmem_empty_bar[acc], ((unit >> 1) & 1u) ^ 1u);
        tc_fence_after();
        GSTAMP(unit * 4 + 0);
        const uint32_t d = tmem_base + acc * 256;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&tail.full_bar[stage], phase);
          tc_fence_after();
          const uint32_t st = smem_u32(smem + stage * kStageSz);
          const uint32_t a_hi = st, a_lo = st + kAPlane, w_hi = st + 2 * kAPlane, w_lo = st + kWLoOff;
#pragma unroll
          for (int pass = 0; pass < 3; ++pass) {
            if (pass < passes) {
              const uint32_t a = (pass == 2 ? a_lo : a_hi), w = (pass == 1 ? w_lo : w_hi);
#pragma unroll
              for (int k16 = 0; k16 < kBlockK / 16; ++k16) {
                const uint64_t da = umma_desc_kmajor<kRowBytes>(a + k16 * 32), dw = umma_desc_kmajor<kRowBytes>(w + k16 * 32);
                const uint32_t accum = (kb | pass | k16) != 0 ? 1u : 0u;
                if constexpr (kPair) umma_f16_pair(d, da, dw, idesc, accum);
                else umma_f16(d, da, dw, idesc, accum);
              }
            }
          }
          if constexpr (kPair) umma_commit_pair(&tail.empty_bar[stage]); else umma_commit(&tail.empty_bar[stage]);
          if (++stage == kNumStages) { stage = 0; phase ^= 1; }
        }
        if constexpr (kPair) umma_commit_pair(&tail.tmem_full_bar[acc]); else umma_commit(&tail.tmem_full_bar[acc]);
        GSTAMP(unit * 4 + 1);
      }
    }
  } else if (warp >= 4) {
    const int e = warp - 4, q = e & 3, ch = e >> 2;
    const int r = q * 32 + lane;
    const int etid = e * 32 + lane;
    uint32_t unit = 0;
    for (int tile = first_tile; tile < num_tiles; tile += tile_step, ++unit) {
      const uint32_t acc = unit & 1u;
      int mt, nt;
      tile_coords(tile, num_m, num_n, mt, nt);
      const int m = mt * kTileM + (int)rank * kBM + r;
      const int ntile0 = nt * bn;
      const int half_cols = bn >> 1;                   // columns per epilogue warp: 64 / 96 / 128
      const int n0 = ntile0 + ch * half_cols;
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * 256 + ch * half_cols;
      // stage the per-column vectors of this tile (256 epilogue threads, one column each)
      if (!kSwap && etid < bn) {
        tail.bias_s[acc][etid] = __ldg(p.bias + ntile0 + etid);
        if (kMode == GEMM_SCALE_RESIDUAL) tail.gamma_s[acc][etid] = __ldg(p.gamma + ntile0 + etid);
      }
      named_barrier_sync(1, kEpiWarps * 32);
      const float* sb = tail.bias_s[acc] + ch * half_cols;
      const float* sg = tail.gamma_s[acc] + ch * half_cols;
      const bool row_ok = m < M_rows;
      size_t out_row = (size_t)m;
      const float* pos_row = nullptr;
      if (kMode == GEMM_PATCH_EMBED) {                // patch row -> token row (CLS first), + positional table
        const int img = m / p.patches_per_img, pp = m - img * p.patches_per_img;
        out_row = (size_t)img * p.tokens_per_img + 1 + pp;
        pos_row = p.pos + (size_t)(1 + pp) * p.N;
      }
      // residual rows are prefetched before the accumulator is ready (GEMM_SCALE_RESIDUAL reads what it overwrites)
      mbar_wait(&tail.tmem_full_bar[acc], (unit >> 1) & 1u);
      tc_fence_after();
      if (e == 0 && lane == 0) GSTAMP(unit * 4 + 2);

      uint8_t* stg = tail.stage_buf[e];
      const unsigned okmask = __ballot_sync(0xffffffffu, row_ok);
      // One warp-wide store instruction of the natural "thread = row" mapping touches 32 different rows with 16 bytes
      // each (32 half-written sectors).  Rows are therefore transposed through a small smem buffer so that 4 (bf16
      // planes) or 4 (fp32, in two 16-column halves) consecutive lanes cover one contiguous 64-byte row segment:
      // every global transaction is a fully written 32-byte sector and an instruction touches 8 rows instead of 32.
      auto store_rows_64B = [&](const uint32_t (&w)[16], uint8_t* base, size_t row_byte_off) {
        uint4* srow = reinterpret_cast<uint4*>(stg + lane * 80);
#pragma unroll
        for (int j = 0; j < 4; ++j) srow[j] = make_uint4(w[4 * j], w[4 * j + 1], w[4 * j + 2], w[4 * j + 3]);
        __syncwarp();
        const uint32_t off_lo = (uint32_t)row_byte_off, off_hi = (uint32_t)(row_byte_off >> 32);
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          const int rr = it * 8 + (lane >> 2), piece = lane & 3;
          const uint4 val = *reinterpret_cast<const uint4*>(stg + rr * 80 + piece * 16);
          const size_t o = ((size_t)__shfl_sync(0xffffffffu, off_hi, rr) << 32) | __shfl_sync(0xffffffffu, off_lo, rr);
          if ((okmask >> rr) & 1u) *reinterpret_cast<uint4*>(base + o + piece * 16) = val;
        }
        __syncwarp();
      };
      auto load_rows_64B = [&](uint32_t (&w)[16], const uint8_t* base, size_t row_byte_off) {
        const uint32_t off_lo = (uint32_t)row_byte_off, off_hi = (uint32_t)(row_byte_off >> 32);
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          const int rr = it * 8 + (lane >> 2), piece = lane & 3;
          const size_t o = ((size_t)__shfl_sync(0xffffffffu, off_hi, rr) << 32) | __shfl_sync(0xffffffffu, off_lo, rr);
          uint4 val = make_uint4(0, 0, 0, 0);
          if ((okmask >> rr) & 1u) val = *reinterpret_cast<const uint4*>(base + o + piece * 16);
          *reinterpret_cast<uint4*>(stg + rr * 80 + piece * 16) = val;
        }
        __syncwarp();
        const uint4* srow = reinterpret_cast<const uint4*>(stg + lane * 80);
#pragma unroll
        for (int j = 0; j < 4; ++j) { const uint4 t = srow[j]; w[4 * j] = t.x; w[4 * j + 1] = t.y; w[4 * j + 2] = t.z; w[4 * j + 3] = t.w; }
        __syncwarp();
      };

      // kSwap: thread = output channel m, the 32 columns of a chunk are 32 consecutive output pixels; every value is
      // transposed through the warp's smem buffer so that a pixel's 32 channels leave as one 64-byte NHWC segment
      auto process_swapped = [&](uint32_t (&v32)[32], int c0) {
        const size_t pix = (size_t)(n0 + c0);
        const size_t cbase = (size_t)(mt * kBM + q * 32);
        const float bias_r = __ldg(p.bias + m);
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(v32[j]) + bias_r;
        auto rows_in = [&](const uint16_t* plane) {          // v[j] += plane[pix + j][channel of this lane]
#pragma unroll
          for (int it = 0; it < 4; ++it) {
            const int rr = it * 8 + (lane >> 2), piece = lane & 3;
            *reinterpret_cast<uint4*>(stg + rr * 80 + piece * 16) =
                *reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(plane) + ((pix + rr) * p.M + cbase) * 2 + piece * 16);
          }
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 32; ++j)
            v[j] += __uint_as_float((uint32_t)*reinterpret_cast<const uint16_t*>(stg + j * 80 + lane * 2) << 16);
          __syncwarp();
        };
        if (kMode == GEMM_PLANES_ADD_RELU) { rows_in(p.res_hi); rows_in(p.res_lo); }
        if (kMode == GEMM_PLANES_RELU || kMode == GEMM_PLANES_ADD_RELU) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
        }
        auto rows_out = [&](uint16_t* plane, bool low) {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const __nv_bfloat16 h = __float2bfloat16_rn(v[j]);
            const __nv_bfloat16 o = low ? __float2bfloat16_rn(v[j] - __bfloat162float(h)) : h;
            *reinterpret_cast<uint16_t*>(stg + j * 80 + lane * 2) = __bfloat16_as_ushort(o);
          }
          __syncwarp();
#pragma unroll
          for (int it = 0; it < 4; ++it) {
            const int rr = it * 8 + (lane >> 2), piece = lane & 3;
            *reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(plane) + ((pix + rr) * p.M + cbase) * 2 + piece * 16) =
                *reinterpret_cast<const uint4*>(stg + rr * 80 + piece * 16);
          }
          __syncwarp();
        };
        rows_out(p.out_hi, false);
        rows_out(p.out_lo, true);
      };

      auto process = [&](uint32_t (&v32)[32], int c0) {
        if constexpr (kSwap) { process_swapped(v32, c0); return; }
        const int n = n0 + c0;
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j)
          v[j] = (p.acc_scale != 0.f ? __uint_as_float(v32[j]) * p.acc_scale : __uint_as_float(v32[j])) + sb[c0 + j];
        if (kMode == GEMM_PLANES || kMode == GEMM_PLANES_GELU || kMode == GEMM_QKV_HEADS || kMode == GEMM_PLANES_RELU ||
            kMode == GEMM_PLANES_ADD_RELU) {
          uint32_t hi[16], lo[16];
          if (kMode == GEMM_PLANES_ADD_RELU) {          // BasicBlock: relu(shortcut + bn2(conv2(.)))   (resnet.py:45-50)
            const size_t rb = (out_row * p.N + n) * 2;
            load_rows_64B(hi, reinterpret_cast<const uint8_t*>(p.res_hi), rb);
            load_rows_64B(lo, reinterpret_cast<const uint8_t*>(p.res_lo), rb);
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              v[2 * j] += __uint_as_float(hi[j] << 16) + __uint_as_float(lo[j] << 16);
              v[2 * j + 1] += __uint_as_float(hi[j] & 0xffff0000u) + __uint_as_float(lo[j] & 0xffff0000u);
            }
          }
#pragma unroll
          for (int j = 0; j < 32; j += 2) {
            float a = v[j], b = v[j + 1];
            if (kMode == GEMM_PLANES_GELU) { a = gelu_erf(a); b = gelu_erf(b); }
            if (kMode == GEMM_PLANES_RELU || kMode == GEMM_PLANES_ADD_RELU) { a = fmaxf(a, 0.f); b = fmaxf(b, 0.f); }
            if (p.f16) {                             // saturating: a value beyond the fp16 range stays finite (and wrong) instead of inf
              a = fminf(fmaxf(a, -65504.f), 65504.f);
              b = fminf(fmaxf(b, -65504.f), 65504.f);
              const __half ah = __float2half_rn(a), bh = __float2half_rn(b);
              hi[j >> 1] = (uint32_t)__half_as_ushort(ah) | ((uint32_t)__half_as_ushort(bh) << 16);
              lo[j >> 1] = (uint32_t)__half_as_ushort(__float2half_rn(a - __half2float(ah))) |
                           ((uint32_t)__half_as_ushort(__float2half_rn(b - __half2float(bh))) << 16);
            } else {
              const __nv_bfloat16 ah = __float2bfloat16_rn(a), bh = __float2bfloat16_rn(b);
              hi[j >> 1] = pack_bf16(ah, bh);
              lo[j >> 1] = pack_bf16(__float2bfloat16_rn(a - __bfloat162float(ah)), __float2bfloat16_rn(b - __bfloat162float(bh)));
            }
          }
          size_t dst = out_row * p.N + n;
          if (kMode == GEMM_QKV_HEADS) {   // head-major: [q|k|v][crop][head][token][64] so that attention tiles are contiguous
            const int which = n >> 10, head = (n & 1023) >> 6, d0 = n & 63;
            const int img = m / p.tokens_per_img, tok = m - img * p.tokens_per_img;
            dst = ((((size_t)which * p.qkv_crop_stride + img) * 16 + head) * p.tokens_per_img + tok) * 64 + d0;
          }
          store_rows_64B(hi, reinterpret_cast<uint8_t*>(p.out_hi), dst * 2);
          store_rows_64B(lo, reinterpret_cast<uint8_t*>(p.out_lo), dst * 2);
        } else if (kMode == GEMM_SCALE_RESIDUAL) {      // x += gamma * (acc + bias)   (blocks: ls1 / ls2 + residual)
          const size_t rowb = (out_row * p.N + n) * 4;
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            uint32_t w[16];
            load_rows_64B(w, reinterpret_cast<const uint8_t*>(p.x), rowb + half * 64);
#pragma unroll
            for (int j = 0; j < 16; ++j)
              w[j] = __float_as_uint(__uint_as_float(w[j]) + sg[c0 + half * 16 + j] * v[half * 16 + j]);
            store_rows_64B(w, reinterpret_cast<uint8_t*>(p.x), rowb + half * 64);
          }
        } else if (kMode == GEMM_ROWS_F32 || kMode == GEMM_ROWS_F32_RELU) {   // plain fp32 rows (last 1x1 convolution of the IST
          const size_t rowb = (out_row * p.N + n) * 4;                          // trunk; second hidden layer of the IST MLP)
          const float floor_v = kMode == GEMM_ROWS_F32_RELU ? 0.f : -INFINITY;
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            uint32_t w[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) w[j] = __float_as_uint(fmaxf(v[half * 16 + j], floor_v));
            store_rows_64B(w, reinterpret_cast<uint8_t*>(p.x), rowb + half * 64);
          }
        } else {                                          // GEMM_PATCH_EMBED
          const size_t rowb = (out_row * p.N + n) * 4;
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            uint32_t w[16];
#pragma unroll
            for (int j = 0; j < 16; ++j)
              w[j] = __float_as_uint(v[half * 16 + j] + (row_ok ? __ldg(pos_row + n + half * 16 + j) : 0.f));
            store_rows_64B(w, reinterpret_cast<uint8_t*>(p.x), rowb + half * 64);
          }
        }
      };

      // software-pipelined TMEM reads: the load of chunk c+1 is in flight while chunk c is processed; the accumulator
      // goes back to the UMMA warp as soon as its last chunk is in registers
      const int nchunks = half_cols >> 5;               // 2, 3 or 4 chunks of 32 columns
      uint32_t va[32], vb[32];
      auto release_acc = [&]() {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if constexpr (kPair) mbar_arrive_cluster(&tail.tmem_empty_bar[acc], 0);
          else mbar_arrive(&tail.tmem_empty_bar[acc]);
        }
      };
      // (a rolled loop over chunk pairs -- `process` instantiated twice instead of six times, SASS 152 -> 64 KB for the GELU
      // kernel -- was measured too: per-kernel times under ncu 7 % WORSE (qkv 101 -> 115 us), step time unchanged; not kept)
      tmem_ld_32x32(taddr, va);
      tmem_ld_wait_for(va);
      tmem_ld_32x32(taddr + 32, vb);
      process(va, 0);
      tmem_ld_wait_for(vb);
      if (nchunks == 2) {
        release_acc();
        process(vb, 32);
      } else {
        tmem_ld_32x32(taddr + 64, va);
        process(vb, 32);
        tmem_ld_wait_for(va);
        if (nchunks == 3) {
          release_acc();
          process(va, 64);
        } else {
          tmem_ld_32x32(taddr + 96, vb);
          process(va, 64);
          tmem_ld_wait_for(vb);
          release_acc();
          process(vb, 96);
        }
      }
      if (e == 0 && lane == 0) GSTAMP(unit * 4 + 3);
    }
  }

  tc_fence_before();
  __syncthreads();
  if constexpr (kPair) cluster_sync_all();         // the leader's UMMAs / commits reach into the peer until here
  if (warp == 2) {
    tc_fence_after();
    if constexpr (kPair) tmem_dealloc_pair(tmem_base, 512); else tmem_dealloc(tmem_base, 512);
  }
}

cudaError_t read_gemm_stamps(long long* host64) { return cudaMemcpyFromSymbol(host64, g_gemm_stamp, sizeof(long long) * 64); }

namespace {
template <bool kSwap, bool kPair, int kMode>
cudaError_t launch_mode(const CUtensorMap& a_hi, const CUtensorMap& a_lo, const CUtensorMap& w_hi, const CUtensorMap& w_lo,
                        const GemmParams& p, int grid, int cluster, cudaStream_t stream) {
  static bool configured = false;                  // one flag per instantiation
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(vit_gemm_kernel<kSwap, kPair, kMode>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
    if (e != cudaSuccess) return e;
    configured = true;
  }
  return launch_ex(vit_gemm_kernel<kSwap, kPair, kMode>, dim3(grid), dim3(kThreads), kSmemBytes, stream, cluster, a_hi, a_lo,
                   w_hi, w_lo, p);
}
}  // namespace

cudaError_t launch_vit_gemm(const CUtensorMap& a_hi, const CUtensorMap& a_lo, const CUtensorMap& w_hi,
                            const CUtensorMap& w_lo, const GemmParams& p, int num_sms, cudaStream_t stream) {
  if (p.M <= 0) return cudaSuccess;
  const int bn = p.bn > 0 ? p.bn : kBN;
  if ((bn != 128 && bn != 192 && bn != 256) || p.N % bn != 0 || p.K % kBlockK != 0) return cudaErrorInvalidValue;
  const int tile_pixels = p.swap ? bn : kBM;
  if (p.conv && (p.Wo <= 0 || tile_pixels % p.Wo != 0 || p.M % kBM != 0 || p.cblocks <= 0)) return cudaErrorInvalidValue;
  if (p.swap && (p.pair || bn != kBN || p.M % kBM != 0)) return cudaErrorInvalidValue;
  // Only the mode / tile-shape combinations some caller launches are instantiated; any other returns
  // cudaErrorInvalidValue.  Pairs: the ViT linears (vit_api.cu) and the IST regressor's hidden layers (api.cu).  1-CTA
  // tiles: the patch embedding and the IST trunk's convolutions (ist_trunk.cu), swapped for the 128-channel layers.
#define GP_GEMM_CASE(SWAP, PAIR, MODE) \
  case MODE: return launch_mode<SWAP, PAIR, MODE>(a_hi, a_lo, w_hi, w_lo, p, grid, PAIR ? 2 : 1, stream);
  if (p.pair) {                                   // one 2-CTA cluster per 256 x bn tile
    if (p.conv && p.M % (2 * kBM) != 0) return cudaErrorInvalidValue;
    const int tiles = ((p.M + 2 * kBM - 1) / (2 * kBM)) * (p.N / bn);
    const int grid = 2 * (tiles < num_sms / 2 ? tiles : num_sms / 2);
    switch (p.mode) {
      GP_GEMM_CASE(false, true, GEMM_QKV_HEADS)
      GP_GEMM_CASE(false, true, GEMM_SCALE_RESIDUAL)
      GP_GEMM_CASE(false, true, GEMM_PLANES_GELU)
      GP_GEMM_CASE(false, true, GEMM_PLANES_RELU)
      GP_GEMM_CASE(false, true, GEMM_ROWS_F32_RELU)
      default: return cudaErrorInvalidValue;
    }
  }
  const int tiles = ((p.M + kBM - 1) / kBM) * (p.N / bn);
  const int grid = tiles < num_sms ? tiles : num_sms;
  if (p.swap) {
    switch (p.mode) {
      GP_GEMM_CASE(true, false, GEMM_PLANES_RELU)
      GP_GEMM_CASE(true, false, GEMM_PLANES_ADD_RELU)
      default: return cudaErrorInvalidValue;
    }
  }
  switch (p.mode) {
    GP_GEMM_CASE(false, false, GEMM_PLANES)
    GP_GEMM_CASE(false, false, GEMM_PATCH_EMBED)
    GP_GEMM_CASE(false, false, GEMM_PLANES_RELU)
    GP_GEMM_CASE(false, false, GEMM_PLANES_ADD_RELU)
    GP_GEMM_CASE(false, false, GEMM_ROWS_F32)
    default: return cudaErrorInvalidValue;
  }
#undef GP_GEMM_CASE
}

}  // namespace gp
