// Per-correspondence scale / in-plane regression (row a5 of SURVEY.md §8; replaces ISTNet.inference
// ist_net.py:97-120, gather utils/batch.py:46-73 and the two Regressor MLP heads ist_net.py:140-155).
//
// For every valid correspondence (b, k, t) a 512-vector cat(query IST descriptor at tar_pt, template IST descriptor at
// src_pt) goes through   scale: 512 -> 512 -> 256 -> 1      in-plane: 512 -> 512 -> 256 -> 2 (tanh).
// The data-dependent row set (boolean-mask indexing + host syncs in the reference) becomes a device-side compaction
// (no host round trip: grids are sized for the worst case and idle tiles exit on the device-side row count).
// This file holds the compaction + gather into the first layer's operand planes and the fp32 output heads; the two
// hidden layers run on tcgen05 through vit_gemm_kernel (launched from gp_ist_mlp, api.cu).
// Their operands are IEEE fp16 hi / lo pairs (not bf16): descriptors, weights and hidden activations of this regressor are
// O(1e-2 .. 1e2), where an fp16 pair carries 22 significant bits -- the regressor outputs then agree with an fp32
// evaluation to 2e-5 (bf16 pairs: 4e-5, which moved a pose component by 1.2e-3 on the parity suite), at the same tensor
// rate.  The downstream RANSAC inlier test (<= 14 px) is a knife edge on these outputs.
#include "gigapose_kernels.h"
#include <cuda_fp16.h>

namespace gp {

namespace {

constexpr int kP = 256;
constexpr int kIstC = 256;

__global__ void __launch_bounds__(256)
mlp_compact_kernel(IstMlpParams p, int total) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= total) return;
  const long long sx = p.src_pts[2 * (size_t)i], sy = p.src_pts[2 * (size_t)i + 1];
  const bool valid = (sx != -1) && (sy != -1);
  p.rel_scale[i] = -1000.0f;                              // ist_net.py:110-113
  p.rel_inplane[2 * (size_t)i] = -1000.0f;
  p.rel_inplane[2 * (size_t)i + 1] = -1000.0f;
  // warp-aggregated append
  const unsigned bal = __ballot_sync(0xffffffffu, valid);
  const int lane = threadIdx.x & 31;
  int base = 0;
  if (lane == 0 && bal) base = atomicAdd(p.row_count, __popc(bal));
  base = __shfl_sync(0xffffffffu, base, 0);
  if (valid) p.row_ids[base + __popc(bal & ((1u << lane) - 1))] = i;
}

// gather the compacted rows into fp16 hi/lo planes (one warp per valid correspondence)
__global__ void __launch_bounds__(256)
mlp_gather_planes_kernel(IstMlpParams p, __half* __restrict__ a_hi, __half* __restrict__ a_lo, int max_rows) {
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= *p.row_count || r >= max_rows) return;
  const int flat = p.row_ids[r];                              // (b, k, t) of this valid correspondence
  const int bk = flat >> 8, b = bk / p.k;
  const long long tx = p.tar_pts[2 * (size_t)flat], ty = p.tar_pts[2 * (size_t)flat + 1];
  const long long sx = p.src_pts[2 * (size_t)flat], sy = p.src_pts[2 * (size_t)flat + 1];
  const long long lid = (p.id_src[bk] - p.id_offset) / p.id_stride;
  const float* q = p.q_ist + ((long long)b * kP + (ty * 16 + tx)) * kIstC;
  const float* t = p.bank_ist + (((long long)p.q_obj[b] * p.T + lid) * kP + (sy * 16 + sx)) * kIstC;
#pragma unroll
  for (int part = 0; part < 2; ++part) {                  // columns [0,256) = query descriptor, [256,512) = template descriptor
    const float* src = part ? t : q;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int c = (lane + 32 * i) * 4;
      const float4 v = *reinterpret_cast<const float4*>(src + c);
      const float x[4] = {v.x, v.y, v.z, v.w};
      // IEEE fp16 hi / lo: 22 significant bits for these O(1) descriptors (bf16 pairs carry 16), same tensor rate
      __half h[4], l[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float xs = fminf(fmaxf(x[j], -65504.f), 65504.f);            // saturate instead of inf
        h[j] = __float2half_rn(xs);
        l[j] = __float2half_rn(xs - __half2float(h[j]));
      }
      const size_t o = (size_t)r * 512 + part * 256 + c;
      *reinterpret_cast<uint2*>(a_hi + o) = make_uint2((uint32_t)__half_as_ushort(h[0]) | ((uint32_t)__half_as_ushort(h[1]) << 16),
                                                       (uint32_t)__half_as_ushort(h[2]) | ((uint32_t)__half_as_ushort(h[3]) << 16));
      *reinterpret_cast<uint2*>(a_lo + o) = make_uint2((uint32_t)__half_as_ushort(l[0]) | ((uint32_t)__half_as_ushort(l[1]) << 16),
                                                       (uint32_t)__half_as_ushort(l[2]) | ((uint32_t)__half_as_ushort(l[3]) << 16));
    }
  }
}

// last layers on the compacted rows: one warp per row, fp32, scattered back to (b,k,t)
__global__ void __launch_bounds__(256)
mlp_head_rows_kernel(IstMlpParams p, IstMlpWeights w, const float* __restrict__ h2s, const float* __restrict__ h2i, int max_rows) {
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= *p.row_count || r >= max_rows) return;
  const float* hs = h2s + (size_t)r * 256;
  const float* hi = h2i + (size_t)r * 256;
  float s = 0.f, c0 = 0.f, c1 = 0.f;
  for (int i = lane; i < 256; i += 32) {
    s = fmaf(hs[i], w.s_w3[i], s);
    const float v = hi[i];
    c0 = fmaf(v, w.i_w3[i], c0);
    c1 = fmaf(v, w.i_w3[256 + i], c1);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, off);
    c0 += __shfl_xor_sync(0xffffffffu, c0, off);
    c1 += __shfl_xor_sync(0xffffffffu, c1, off);
  }
  if (lane == 0) {
    const int flat = p.row_ids[r];
    s += w.s_b3[0];
    c0 += w.i_b3[0];
    c1 += w.i_b3[1];
    if (w.use_tanh) { c0 = tanhf(c0); c1 = tanhf(c1); }
    p.rel_scale[flat] = s;
    p.rel_inplane[2 * (size_t)flat] = c0;
    p.rel_inplane[2 * (size_t)flat + 1] = c1;
  }
}

}  // namespace

cudaError_t launch_mlp_gather_planes(const IstMlpParams& p, uint16_t* a_hi, uint16_t* a_lo, cudaStream_t stream) {
  const int total = p.B * p.k * kP;
  if (total <= 0) return cudaSuccess;
  cudaError_t e = cudaMemsetAsync(p.row_count, 0, sizeof(int), stream);
  if (e != cudaSuccess) return e;
  mlp_compact_kernel<<<(total + 255) / 256, 256, 0, stream>>>(p, total);          // row_ids, row_count, -1000 fill
  mlp_gather_planes_kernel<<<(total + 7) / 8, 256, 0, stream>>>(p, reinterpret_cast<__half*>(a_hi),
                                                               reinterpret_cast<__half*>(a_lo), total);
  return cudaGetLastError();
}

cudaError_t launch_mlp_head_rows(const IstMlpWeights& w, const IstMlpParams& p, const float* h2_scale, const float* h2_inplane,
                                 cudaStream_t stream) {
  const int total = p.B * p.k * kP;
  if (total <= 0) return cudaSuccess;
  mlp_head_rows_kernel<<<(total + 7) / 8, 256, 0, stream>>>(p, w, h2_scale, h2_inplane, total);
  return cudaGetLastError();
}

}  // namespace gp
