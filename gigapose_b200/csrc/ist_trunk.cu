// Native IST trunk (rows a6 / f1 of SURVEY.md §8): the ResNet the reference runs at ist_net.py:62-63 through
// src/models/network/resnet.py:318-381 (bilinear 224 -> 256, 7x7/2 stem, four stages of two BasicBlocks with dims
// 128/192/256/512, 1x1 output convolution to 256 channels at 1/16 resolution), inference form: BatchNorm folded into
// the convolution weights by the caller.
//
// Every convolution is an implicit GEMM on the same tcgen05 kernel as the ViT linears (vit_gemm.cu): activations are
// NHWC bf16 hi/lo planes, one output tile = 128 consecutive output pixels (whole output rows of one image) x all / half
// of the output channels, and the A operand of k-block (ky, kx, 32-channel block) is fetched by ONE 4-D TMA box per
// plane -- a shifted, strided window of the input plane whose out-of-image part TMA zero-fills (the padding).  No
// im2col buffer exists anywhere.  The 3-channel stem reads the resized crop, stored as zero-bordered NHWC planes with 4
// channels, through a tensor map whose rows OVERLAP: row xo of the view is the 8-pixel x 4-channel window starting at
// pixel 2*xo - 4 (16-byte row pitch, 64-byte rows), so that one k-block is one filter row ky (K = 7 x 32 = 224 with
// zero filter entries for the 8th pixel and the 4th channel).
// ReLU, the residual add and the hi/lo split of the next layer's input are the GEMM epilogue.
// The trunk runs on 1-CTA tiles: 2-CTA cluster tiles, which gain 3 % on the ViT linears, were measured 3 % slower here on
// a B200 (96-row filter boxes for the 192-channel layers, 64 pair tiles on 74 clusters in layer4).
#include "../../include/gigapose_b200.h"
#include "gigapose_kernels.h"

#include <cuda_bf16.h>
#include <new>
#include <vector>

extern int gp_internal_fail(int code, const char* fmt, ...);
extern void gp_internal_count_launches(int n);
extern int gp_internal_make_map(CUtensorMap* map, void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows);
extern int gp_internal_make_map_raw(CUtensorMap* map, void* ptr, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                                    const uint32_t* box, const uint32_t* elem_strides);
extern int gp_internal_make_map_nhwc(CUtensorMap* map, void* ptr, uint64_t C, uint64_t W, uint64_t H, uint64_t N,
                                     uint32_t out_w, uint32_t out_h, uint32_t stride);

namespace {

constexpr int kIn = 224, kRes = 256, kStemOut = 128, kStemKPad = 224, kFeat = 256;
constexpr int kPadRows = kRes + 6, kPadCols = kRes + 8;     // resized crop with 3 zero rows above / below, 4 zero pixels left / right
constexpr int kDims[4] = {128, 192, 256, 512};
constexpr int kNumConvs = GP_IST_TRUNK_NUM_CONVS;
constexpr size_t kAlign = 1024;
inline size_t up(size_t x) { return (x + kAlign - 1) / kAlign * kAlign; }

struct Carver {
  uint8_t* base; size_t off = 0;
  explicit Carver(void* b) : base(static_cast<uint8_t*>(b)) {}
  template <typename T> T* take(size_t n) { T* p = base ? reinterpret_cast<T*>(base + off) : nullptr; off += up(n * sizeof(T)); return p; }
};

struct Planes { uint16_t *hi = nullptr, *lo = nullptr; };

struct Conv {
  int cin, cout, k, stride, pad, hin, hout;     // square maps and filters
  int K, Kpad, bn, mode;
  int swap;                                     // 128-channel layers: filters are the 128-row UMMA operand (vit_gemm.cu)
  int in_buf, out_buf, res_buf;                 // activation buffers (-1: stem im2col planes / none)
  Planes w;
  const float* bias;
  CUtensorMap a_hi, a_lo, w_hi, w_lo;
};

// The 21 convolutions in ABI (= execution) order: stem; per BasicBlock conv1, [downsample,] conv2; output convolution.
std::vector<Conv> make_schedule() {
  std::vector<Conv> v;
  auto add = [&](int cin, int cout, int k, int stride, int pad, int hin, int mode, int in_buf, int out_buf, int res_buf) {
    Conv c{};
    c.cin = cin; c.cout = cout; c.k = k; c.stride = stride; c.pad = pad; c.hin = hin; c.hout = hin / stride;
    c.K = k * k * cin; c.Kpad = cin == 3 ? kStemKPad : c.K;
    c.swap = cout == 128 ? 1 : 0;
    c.bn = cout == 192 ? 192 : 256;
    c.mode = mode; c.in_buf = in_buf; c.out_buf = out_buf; c.res_buf = res_buf;
    v.push_back(c);
  };
  add(3, kStemOut, 7, 2, 3, kRes, gp::GEMM_PLANES_RELU, -1, 0, -1);
  int x = 0, width = kStemOut, h = kStemOut;
  for (int st = 0; st < 4; ++st) {
    const int d = kDims[st];
    for (int blk = 0; blk < 2; ++blk) {
      const int stride = (blk == 0 && st > 0) ? 2 : 1;
      int free_buf[3], nf = 0;
      for (int b = 0; b < 4; ++b) if (b != x) free_buf[nf++] = b;
      const int y = free_buf[0];
      const bool ds = stride != 1;
      const int res = ds ? free_buf[1] : x, z = ds ? free_buf[2] : free_buf[1];
      add(width, d, 3, stride, 1, h, gp::GEMM_PLANES_RELU, x, y, -1);                 // relu(bn1(conv1 x))   resnet.py:45
      if (ds) add(width, d, 1, stride, 0, h, gp::GEMM_PLANES, x, res, -1);           // downsample: 1x1/2 conv + bn
      add(d, d, 3, 1, 1, h / stride, gp::GEMM_PLANES_ADD_RELU, y, z, res);            // relu(shortcut + bn2(conv2 .))
      x = z; width = d; h /= stride;
    }
  }
  add(kDims[3], kFeat, 1, 1, 0, h, gp::GEMM_ROWS_F32, x, -1, -1);                     // layer4_outconv   resnet.py:379
  return v;
}

#define GPI_CUDA(expr)                                                                                    \
  do {                                                                                                    \
    cudaError_t _e = (expr);                                                                              \
    if (_e != cudaSuccess) return gp_internal_fail(GP_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(_e)); \
  } while (0)

__device__ __forceinline__ void split_store(float v, __nv_bfloat16* hi, __nv_bfloat16* lo, size_t i) {
  const __nv_bfloat16 h = __float2bfloat16_rn(v);
  hi[i] = h;
  lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
}

// Bilinear 224 -> 256 (align_corners=True, resnet.py:365-368) into zero-bordered NHWC4 hi/lo planes
// [img][262 rows][264 pixels][4]: pixel (y, x) of the resized crop lives at row y + 3, column x + 4.
__global__ void resize_pad_kernel(const float* __restrict__ img, int n, uint2* __restrict__ hi, uint2* __restrict__ lo) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * kRes * kRes) return;
  const int im = i / (kRes * kRes), pix = i - im * kRes * kRes, y = pix / kRes, x = pix - y * kRes;
  const float scale = (float)(kIn - 1) / (float)(kRes - 1);
  const float fy = scale * y, fx = scale * x;
  const int y0 = (int)fy, x0 = (int)fx;
  const int yp = y0 < kIn - 1 ? 1 : 0, xp = x0 < kIn - 1 ? 1 : 0;
  const float ly = fy - y0, lx = fx - x0, hy = 1.f - ly, hx = 1.f - lx;
  uint32_t h[3], l[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float* src = img + ((size_t)im * 3 + c) * kIn * kIn;
    const float v = hy * (hx * src[y0 * kIn + x0] + lx * src[y0 * kIn + x0 + xp]) +
                    ly * (hx * src[(y0 + yp) * kIn + x0] + lx * src[(y0 + yp) * kIn + x0 + xp]);
    const __nv_bfloat16 b = __float2bfloat16_rn(v);
    h[c] = __bfloat16_as_ushort(b);
    l[c] = __bfloat16_as_ushort(__float2bfloat16_rn(v - __bfloat162float(b)));
  }
  const size_t o = ((size_t)im * kPadRows + y + 3) * kPadCols + x + 4;
  hi[o] = make_uint2(h[0] | (h[1] << 16), h[2]);
  lo[o] = make_uint2(l[0] | (l[1] << 16), l[2]);
}

// Stem filter [128, 7, 7, 3] (cout, ky, kx, c) -> [128, 7, 8, 4] = [128, 224] hi/lo planes: window pixel i holds tap
// kx = i - 1 (pixel 0 of a window lies left of the 7 taps), channel 3 does not exist; both get zero weights.
__global__ void pack_stem_filter_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= kStemOut * kStemKPad) return;
  const int co = i / kStemKPad, k = i - co * kStemKPad, ky = k >> 5, px = (k >> 2) & 7, c = k & 3;
  split_store(px >= 1 && c < 3 ? w[((co * 7 + ky) * 7 + (px - 1)) * 3 + c] : 0.f, hi, lo, (size_t)i);
}

__global__ void merge_planes_kernel(const __nv_bfloat16* __restrict__ hi, const __nv_bfloat16* __restrict__ lo, long long n,
                                    float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __bfloat162float(hi[i]) + __bfloat162float(lo[i]);
}

}  // namespace

struct gp_ist_trunk_context {
  int max_crops, passes, num_sms;
  std::vector<Conv> convs;
  Planes act[4];               // NHWC activation planes, each sized for the largest map [max_crops,128,128,128]
  Planes stem;                 // [max_crops, 262, 264, 4] zero-bordered resized crops (NHWC4)
  const float* zero_bias;      // [512] zeros (the output convolution has no bias)
};

namespace {

void carve_weights(Carver& c, gp_ist_trunk_context* h, const std::vector<Conv>& sched) {
  for (size_t i = 0; i < sched.size(); ++i) {
    const size_t n = (size_t)sched[i].cout * sched[i].Kpad;
    uint16_t* a = c.take<uint16_t>(n); uint16_t* b = c.take<uint16_t>(n);
    if (h) { h->convs[i].w.hi = a; h->convs[i].w.lo = b; }
  }
  const float* z = c.take<float>(512);
  if (h) h->zero_bias = z;
}

void carve_workspace(Carver& c, int max_crops, gp_ist_trunk_context* h) {
  const size_t act = (size_t)max_crops * kStemOut * kStemOut * kDims[0];
  for (int b = 0; b < 4; ++b) {
    uint16_t* a = c.take<uint16_t>(act); uint16_t* l = c.take<uint16_t>(act);
    if (h) { h->act[b].hi = a; h->act[b].lo = l; }
  }
  const size_t st = (size_t)max_crops * kPadRows * kPadCols * 4;
  uint16_t* a = c.take<uint16_t>(st); uint16_t* l = c.take<uint16_t>(st);
  if (h) { h->stem.hi = a; h->stem.lo = l; }
}

int run(gp_ist_trunk_context* h, int n, const float* crops, float* feat, int stop_after, float* dump, cudaStream_t s) {
  resize_pad_kernel<<<(n * kRes * kRes + 255) / 256, 256, 0, s>>>(crops, n, reinterpret_cast<uint2*>(h->stem.hi),
                                                                  reinterpret_cast<uint2*>(h->stem.lo));
  GPI_CUDA(cudaGetLastError());
  int launched = 1;
  const int last = stop_after > 0 && stop_after < (int)h->convs.size() ? stop_after : (int)h->convs.size();
  for (int i = 0; i < last; ++i) {
    const Conv& c = h->convs[i];
    gp::GemmParams g{};
    g.passes = h->passes; g.mode = c.mode; g.bn = c.bn;
    g.M = n * c.hout * c.hout; g.N = c.cout; g.K = c.Kpad;
    if (c.swap) { g.swap = 1; g.M = c.cout; g.N = n * c.hout * c.hout; }
    g.bias = c.bias ? c.bias : h->zero_bias;
    if (c.out_buf >= 0) { g.out_hi = h->act[c.out_buf].hi; g.out_lo = h->act[c.out_buf].lo; }
    else g.x = feat;
    if (c.res_buf >= 0) { g.res_hi = h->act[c.res_buf].hi; g.res_lo = h->act[c.res_buf].lo; }
    if (c.in_buf < 0) {          // stem: k-block = filter row ky over the overlapping-window view (x handled by the view)
      g.conv = 1; g.Ho = c.hout; g.Wo = c.hout; g.stride = 2; g.pad = 0; g.kw = 1; g.cblocks = 1;
    } else if (!(c.k == 1 && c.stride == 1)) {
      g.conv = 1; g.Ho = c.hout; g.Wo = c.hout; g.stride = c.stride; g.pad = c.pad; g.kw = c.k; g.cblocks = c.cin / 32;
    }
    if (c.swap) GPI_CUDA(gp::launch_vit_gemm(c.w_hi, c.w_lo, c.a_hi, c.a_lo, g, h->num_sms, s));   // filters take the 128-row slot
    else GPI_CUDA(gp::launch_vit_gemm(c.a_hi, c.a_lo, c.w_hi, c.w_lo, g, h->num_sms, s));
    ++launched;
  }
  if (dump) {
    const Conv& c = h->convs[last - 1];
    if (c.out_buf < 0) return gp_internal_fail(GP_ERR_INVALID, "the last convolution writes `feat` directly; nothing to dump");
    const long long cnt = (long long)n * c.hout * c.hout * c.cout;
    merge_planes_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, s>>>(
        reinterpret_cast<const __nv_bfloat16*>(h->act[c.out_buf].hi), reinterpret_cast<const __nv_bfloat16*>(h->act[c.out_buf].lo),
        cnt, dump);
    GPI_CUDA(cudaGetLastError());
    ++launched;
  }
  gp_internal_count_launches(launched);
  return GP_OK;
}

}  // namespace

extern "C" {

int gp_ist_trunk_query_sizes(int max_crops, size_t* weight_bytes, size_t* workspace_bytes) {
  if (max_crops < 1) return gp_internal_fail(GP_ERR_INVALID, "bad max_crops");
  Carver cw(nullptr), cs(nullptr);
  carve_weights(cw, nullptr, make_schedule());
  carve_workspace(cs, max_crops, nullptr);
  if (weight_bytes) *weight_bytes = cw.off;
  if (workspace_bytes) *workspace_bytes = cs.off;
  return GP_OK;
}

int gp_ist_trunk_create(int device, int max_crops, int precision, const gp_conv_weights_t* w, void* weight_mem,
                        void* workspace_mem, void* stream, gp_ist_trunk_handle_t* out) {
  if (max_crops < 1 || !w || !weight_mem || !workspace_mem || !out) return gp_internal_fail(GP_ERR_INVALID, "bad argument");
  if (precision != GP_PRECISION_FP32_SPLIT && precision != GP_PRECISION_BF16)
    return gp_internal_fail(GP_ERR_INVALID, "unknown precision %d", precision);
  if (((uintptr_t)weight_mem | (uintptr_t)workspace_mem) & (kAlign - 1))
    return gp_internal_fail(GP_ERR_INVALID, "weight and workspace memory must be 1024-byte aligned");
  for (int i = 0; i < kNumConvs; ++i)
    if (!w[i].weight) return gp_internal_fail(GP_ERR_INVALID, "weight pointer %d is null", i);
  GPI_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  GPI_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return gp_internal_fail(GP_ERR_UNSUPPORTED, "device %d is not sm_100", device);
  gp_ist_trunk_context* h = new (std::nothrow) gp_ist_trunk_context();
  if (!h) return gp_internal_fail(GP_ERR_INVALID, "out of host memory");
  h->max_crops = max_crops; h->num_sms = prop.multiProcessorCount;
  h->passes = precision == GP_PRECISION_FP32_SPLIT ? 3 : 1;
  h->convs = make_schedule();
  Carver cw(weight_mem), cs(workspace_mem);
  carve_weights(cw, h, h->convs);
  carve_workspace(cs, max_crops, h);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  cudaError_t ce = cudaMemsetAsync(const_cast<float*>(h->zero_bias), 0, 512 * sizeof(float), s);
  // the zero border (and 4th channel) of the resized-crop planes is written once; resize_pad_kernel fills the interior
  const size_t stem_bytes = (size_t)max_crops * kPadRows * kPadCols * 4 * sizeof(uint16_t);
  if (ce == cudaSuccess) ce = cudaMemsetAsync(h->stem.hi, 0, stem_bytes, s);
  if (ce == cudaSuccess) ce = cudaMemsetAsync(h->stem.lo, 0, stem_bytes, s);
  int e = GP_OK;
  for (int i = 0; i < kNumConvs && !e && ce == cudaSuccess; ++i) {
    Conv& c = h->convs[i];
    c.bias = w[i].bias;
    // weights arrive as [cout, ky, kx, cin] (BatchNorm folded): exactly the [N, K] operand with K = (tap, channel)
    if (c.in_buf < 0) {
      pack_stem_filter_kernel<<<(kStemOut * kStemKPad + 255) / 256, 256, 0, s>>>(
          w[i].weight, reinterpret_cast<__nv_bfloat16*>(c.w.hi), reinterpret_cast<__nv_bfloat16*>(c.w.lo));
      ce = cudaGetLastError();
    } else {
      ce = gp::launch_split_planes(w[i].weight, c.cout, c.K, c.Kpad, c.w.hi, c.w.lo, s);
    }
    if (ce != cudaSuccess) break;
    // rows per TMA box: filters / pixels
    const uint32_t wbox = c.swap ? 128 : c.bn, pix_tile = c.swap ? 256 : 128;
    if ((e = gp_internal_make_map(&c.w_hi, c.w.hi, c.cout, c.Kpad, wbox)) || (e = gp_internal_make_map(&c.w_lo, c.w.lo, c.cout, c.Kpad, wbox)))
      break;
    if (c.in_buf < 0) {
      // stem: {32 elements = 8 pixels x 4 channels, 128 windows at a 16-byte pitch, 262 rows, crops}; a 256-pixel tile
      // is two output rows = every second input row starting at 2*yo + ky
      const uint64_t dims[4] = {32, (uint64_t)kStemOut, (uint64_t)kPadRows, (uint64_t)max_crops};
      const uint64_t strides[3] = {16, (uint64_t)kPadCols * 8, (uint64_t)kPadRows * kPadCols * 8};
      const uint32_t box[4] = {32, (uint32_t)kStemOut, (pix_tile / kStemOut) * 2, 1}, es[4] = {1, 1, 2, 1};
      (e = gp_internal_make_map_raw(&c.a_hi, h->stem.hi, 4, dims, strides, box, es)) ||
          (e = gp_internal_make_map_raw(&c.a_lo, h->stem.lo, 4, dims, strides, box, es));
    } else if (c.k == 1 && c.stride == 1) {               // 1x1/1: the NHWC plane is already the [pixels, cin] operand
      const uint64_t rows = (uint64_t)max_crops * c.hin * c.hin;
      (e = gp_internal_make_map(&c.a_hi, h->act[c.in_buf].hi, rows, c.cin, pix_tile)) ||
          (e = gp_internal_make_map(&c.a_lo, h->act[c.in_buf].lo, rows, c.cin, pix_tile));
    } else {
      const uint32_t ow = c.hout, oh = pix_tile / c.hout;
      (e = gp_internal_make_map_nhwc(&c.a_hi, h->act[c.in_buf].hi, c.cin, c.hin, c.hin, max_crops, ow, oh, c.stride)) ||
          (e = gp_internal_make_map_nhwc(&c.a_lo, h->act[c.in_buf].lo, c.cin, c.hin, c.hin, max_crops, ow, oh, c.stride));
    }
  }
  if (ce != cudaSuccess) { delete h; return gp_internal_fail(GP_ERR_CUDA, "weight packing failed: %s", cudaGetErrorString(ce)); }
  if (e) { delete h; return e; }
  gp_internal_count_launches(kNumConvs);
  *out = h;
  return GP_OK;
}

int gp_ist_trunk_destroy(gp_ist_trunk_handle_t h) {
  delete h;
  return GP_OK;
}

int gp_ist_trunk_forward(gp_ist_trunk_handle_t h, int n, const float* crops, float* feat, void* stream) {
  if (!h || !crops || !feat) return gp_internal_fail(GP_ERR_INVALID, "null argument");
  if (n < 1 || n > h->max_crops) return gp_internal_fail(GP_ERR_INVALID, "batch %d outside [1, %d]", n, h->max_crops);
  return run(h, n, crops, feat, 0, nullptr, static_cast<cudaStream_t>(stream));
}

int gp_debug_ist_trunk(gp_ist_trunk_handle_t h, int n, const float* crops, int num_convs, float* activation, void* stream) {
  if (!h || !crops || !activation) return gp_internal_fail(GP_ERR_INVALID, "null argument");
  if (n < 1 || n > h->max_crops) return gp_internal_fail(GP_ERR_INVALID, "batch %d outside [1, %d]", n, h->max_crops);
  if (num_convs < 1 || num_convs >= kNumConvs) return gp_internal_fail(GP_ERR_INVALID, "num_convs outside [1, %d)", kNumConvs);
  return run(h, n, crops, nullptr, num_convs, activation, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
