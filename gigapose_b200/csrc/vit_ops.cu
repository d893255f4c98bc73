// Non-GEMM pieces of the ViT-L/14 forward (row a1): im2col for the 14x14/14 patch embedding, CLS rows, LayerNorm
// (-> bf16 hi/lo planes, the A operand of the next tcgen05 GEMM) and the fp32 -> hi/lo plane split used to pack weights.
// Attention lives in vit_attention_tc.cu.
#include "gigapose_kernels.h"
#include <cuda_bf16.h>
#include <cuda_fp16.h>

namespace gp {

namespace {

constexpr int kDim = 1024, kHeads = 16, kHd = 64;
constexpr int kTok = 257;

__device__ __forceinline__ void split_store(float v, __nv_bfloat16* hi, __nv_bfloat16* lo, size_t i) {
  const __nv_bfloat16 h = __float2bfloat16_rn(v);
  hi[i] = h;
  lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
}

// ---------------------------------------------------------------- fp32 [rows, K] -> bf16 hi/lo planes [rows, Kpad]
__global__ void split_planes_kernel(const float* __restrict__ x, long long rows, int K, int Kpad,
                                    __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * Kpad) return;
  const long long r = i / Kpad;
  const int k = (int)(i - r * Kpad);
  split_store(k < K ? x[r * K + k] : 0.f, hi, lo, (size_t)i);
}

// same with IEEE fp16 hi / lo (x = hi + lo to ~2^-22 for |x| in [6e-5, 6e4]; smaller values keep 6e-8 absolute)
__global__ void split_planes_f16_kernel(const float* __restrict__ x, long long rows, int K, int Kpad, float pre_scale,
                                        __half* __restrict__ hi, __half* __restrict__ lo) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * Kpad) return;
  const long long r = i / Kpad;
  const int k = (int)(i - r * Kpad);
  // pre_scale (a power of two, exact) lifts small weights into the range where the lo half is a NORMAL fp16 number
  const float v = fminf(fmaxf((k < K ? x[r * K + k] : 0.f) * pre_scale, -65504.f), 65504.f);
  const __half h = __float2half_rn(v);
  hi[i] = h;
  lo[i] = __float2half_rn(v - __half2float(h));
}

// ---------------------------------------------------------------- im2col: [b,3,224,224] -> planes [b*256, 608]
// column = c*196 + ky*14 + kx, the flattening of the conv weight [1024,3,14,14]; columns 588..607 are zero
__global__ void im2col_kernel(const float* __restrict__ img, int b, int Kpad, __nv_bfloat16* __restrict__ hi,
                              __nv_bfloat16* __restrict__ lo) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = (long long)b * 256 * Kpad;
  if (i >= total) return;
  const long long row = i / Kpad;
  const int k = (int)(i - row * Kpad);
  float v = 0.f;
  if (k < 588) {
    const int im = (int)(row >> 8), pidx = (int)(row & 255), py = pidx >> 4, px = pidx & 15;
    const int c = k / 196, rem = k - c * 196, ky = rem / 14, kx = rem - ky * 14;
    v = img[(((size_t)im * 3 + c) * 224 + (py * 14 + ky)) * 224 + px * 14 + kx];
  }
  split_store(v, hi, lo, (size_t)i);
}

// ---------------------------------------------------------------- x[b*257 + 0, :] = cls + pos[0]
__global__ void cls_rows_kernel(const float* __restrict__ cls, const float* __restrict__ pos, int b, float* __restrict__ x) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= b * kDim) return;
  const int im = i / kDim, c = i - im * kDim;
  x[(size_t)im * kTok * kDim + c] = cls[c] + pos[c];
}

// ---------------------------------------------------------------- LayerNorm (eps 1e-6) -> hi/lo planes; warp per row
__global__ void __launch_bounds__(256)
layernorm_planes_kernel(const float* __restrict__ x, int M, const float* __restrict__ w, const float* __restrict__ bsh,
                        float eps, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= M) return;
  const float4* src = reinterpret_cast<const float4*>(x + (size_t)row * kDim);
  float4 v[8];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    v[i] = src[lane + 32 * i];
    s += v[i].x + v[i].y + v[i].z + v[i].w;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
  const float mean = s / kDim;
  float ss = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
    ss += a * a + b * b + c * c + d * d;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, off);
  const float rstd = rsqrtf(ss / kDim + eps);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int c = (lane + 32 * i) * 4;
    const float4 wv = *reinterpret_cast<const float4*>(w + c), bv = *reinterpret_cast<const float4*>(bsh + c);
    const float o[4] = {(v[i].x - mean) * rstd * wv.x + bv.x, (v[i].y - mean) * rstd * wv.y + bv.y,
                        (v[i].z - mean) * rstd * wv.z + bv.z, (v[i].w - mean) * rstd * wv.w + bv.w};
    __nv_bfloat16 h[4], l[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      h[j] = __float2bfloat16_rn(o[j]);
      l[j] = __float2bfloat16_rn(o[j] - __bfloat162float(h[j]));
    }
    const size_t off = (size_t)row * kDim + c;
    *reinterpret_cast<uint2*>(hi + off) = make_uint2((uint32_t)__bfloat16_as_ushort(h[0]) | ((uint32_t)__bfloat16_as_ushort(h[1]) << 16),
                                                     (uint32_t)__bfloat16_as_ushort(h[2]) | ((uint32_t)__bfloat16_as_ushort(h[3]) << 16));
    *reinterpret_cast<uint2*>(lo + off) = make_uint2((uint32_t)__bfloat16_as_ushort(l[0]) | ((uint32_t)__bfloat16_as_ushort(l[1]) << 16),
                                                     (uint32_t)__bfloat16_as_ushort(l[2]) | ((uint32_t)__bfloat16_as_ushort(l[3]) << 16));
  }
}

}  // namespace

cudaError_t launch_split_planes(const float* x, long long rows, int K, int Kpad, uint16_t* hi, uint16_t* lo, cudaStream_t s,
                                bool f16, float pre_scale) {
  const long long total = rows * Kpad;
  if (total <= 0) return cudaSuccess;
  if (f16) {
    split_planes_f16_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(x, rows, K, Kpad, pre_scale, reinterpret_cast<__half*>(hi),
                                                                           reinterpret_cast<__half*>(lo));
    return cudaGetLastError();
  }
  split_planes_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(x, rows, K, Kpad, reinterpret_cast<__nv_bfloat16*>(hi),
                                                                     reinterpret_cast<__nv_bfloat16*>(lo));
  return cudaGetLastError();
}

cudaError_t launch_im2col(const float* img, int b, int Kpad, uint16_t* hi, uint16_t* lo, cudaStream_t s) {
  const long long total = (long long)b * 256 * Kpad;
  if (total <= 0) return cudaSuccess;
  im2col_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(img, b, Kpad, reinterpret_cast<__nv_bfloat16*>(hi),
                                                               reinterpret_cast<__nv_bfloat16*>(lo));
  return cudaGetLastError();
}

cudaError_t launch_cls_rows(const float* cls, const float* pos, int b, float* x, cudaStream_t s) {
  if (b <= 0) return cudaSuccess;
  return launch_ex(cls_rows_kernel, dim3((b * kDim + 255) / 256), dim3(256), 0, s, 1, cls, pos, b, x);
}

cudaError_t launch_layernorm_planes(const float* x, int M, const float* w, const float* b, float eps, uint16_t* hi,
                                    uint16_t* lo, cudaStream_t s) {
  if (M <= 0) return cudaSuccess;
  return launch_ex(layernorm_planes_kernel, dim3((M + 7) / 8), dim3(256), 0, s, 1, x, M, w, b, eps,
                   reinterpret_cast<__nv_bfloat16*>(hi), reinterpret_cast<__nv_bfloat16*>(lo));
}

}  // namespace gp
