// C-ABI of the native DINOv2 ViT-L/14 forward (include/gigapose_b200.h, gp_vit_*): weight packing into bf16 hi/lo
// planes, TMA descriptors, and the per-layer launch sequence.  Geometry is fixed to what the reference uses
// (configs/model/ae_net/dinov2_l.yaml): 224x224 crops, patch 14, dim 1024, 16 heads, MLP 4096; depth is a parameter
// (24 for ViT-L) so that small stacks can be parity-tested quickly.
#include "../../include/gigapose_b200.h"
#include "gigapose_kernels.h"

#include <cstdarg>
#include <cstdio>
#include <new>
#include <string>
#include <vector>

extern int gp_internal_fail(int code, const char* fmt, ...);
extern void gp_internal_count_launches(int n);
extern int gp_internal_make_map(CUtensorMap* map, void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows);
extern int gp_internal_make_map_ex(CUtensorMap* map, void* ptr, uint64_t rows, uint64_t cols, uint32_t box_cols,
                                   uint32_t box_rows, int swizzle_bytes);

namespace {

constexpr int kDim = 1024, kQkv = 3072, kMlp = 4096, kTok = 257, kPatchK = 588, kPatchKPad = 608;
constexpr size_t kAlign = 1024;
inline size_t up(size_t x) { return (x + kAlign - 1) / kAlign * kAlign; }

struct Carver {
  uint8_t* base; size_t off = 0;
  explicit Carver(void* b) : base(static_cast<uint8_t*>(b)) {}
  template <typename T> T* take(size_t n) { T* p = base ? reinterpret_cast<T*>(base + off) : nullptr; off += up(n * sizeof(T)); return p; }
};

struct Planes { uint16_t *hi, *lo; CUtensorMap m_hi, m_lo; };

struct BlockW {
  Planes qkv, proj, fc1, fc2;
  const float *n1w, *n1b, *qkv_b, *proj_b, *ls1, *n2w, *n2b, *fc1_b, *fc2_b, *ls2;
};

#define GPV_CUDA(expr)                                                                                    \
  do {                                                                                                    \
    cudaError_t _e = (expr);                                                                              \
    if (_e != cudaSuccess) return gp_internal_fail(GP_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(_e)); \
  } while (0)

}  // namespace

struct gp_vit_context {
  int depth, max_crops, passes, num_sms;
  Planes patch_w;
  const float *patch_b, *cls, *pos;
  std::vector<BlockW> blocks;
  // workspace
  float* x;                    // [max_crops*257, 1024] residual stream
  Planes ln, qkv, attn, hid, patches;   // activation planes (+ TMA maps for those that feed a GEMM)
  CUtensorMap qkv_hi128, qkv_lo128, qkv_hi16, qkv_lo16;   // attention operand tiles: 64 columns x {128,16} token rows
  size_t workspace_bytes;
};

namespace {

void carve_weights(Carver& c, int depth, gp_vit_context* h) {
  auto planes = [&](Planes* p, size_t n) { uint16_t* a = c.take<uint16_t>(n); uint16_t* b = c.take<uint16_t>(n); if (p) { p->hi = a; p->lo = b; } };
  planes(h ? &h->patch_w : nullptr, (size_t)kDim * kPatchKPad);
  for (int i = 0; i < depth; ++i) {
    BlockW* b = h ? &h->blocks[i] : nullptr;
    planes(b ? &b->qkv : nullptr, (size_t)kQkv * kDim);
    planes(b ? &b->proj : nullptr, (size_t)kDim * kDim);
    planes(b ? &b->fc1 : nullptr, (size_t)kMlp * kDim);
    planes(b ? &b->fc2 : nullptr, (size_t)kDim * kMlp);
  }
}

void carve_workspace(Carver& c, int max_crops, gp_vit_context* h) {
  const size_t M = (size_t)max_crops * kTok;
  auto planes = [&](Planes* p, size_t n) { uint16_t* a = c.take<uint16_t>(n); uint16_t* b = c.take<uint16_t>(n); if (p) { p->hi = a; p->lo = b; } };
  float* x = c.take<float>(M * kDim);
  if (h) h->x = x;
  planes(h ? &h->ln : nullptr, M * kDim);
  planes(h ? &h->qkv : nullptr, M * kQkv);
  planes(h ? &h->attn : nullptr, M * kDim);
  planes(h ? &h->hid : nullptr, M * kMlp);
  planes(h ? &h->patches : nullptr, (size_t)max_crops * 256 * kPatchKPad);
}

int make_maps(Planes* p, uint64_t rows, uint64_t cols, uint32_t box_rows) {
  if (int e = gp_internal_make_map(&p->m_hi, p->hi, rows, cols, box_rows)) return e;
  return gp_internal_make_map(&p->m_lo, p->lo, rows, cols, box_rows);
}

// A linear layer runs on 2-CTA cluster tiles (tcgen05 cta_group::2, 256 x 256): each CTA of a pair stages 128 rows of
// the activations and 128 rows of the weights, so both operands' maps have 128-row boxes.
cudaError_t linear(const gp_vit_context* h, const Planes& a, const Planes& w, gp::GemmParams g, cudaStream_t s) {
  g.pair = 1;
  return gp::launch_vit_gemm(a.m_hi, a.m_lo, w.m_hi, w.m_lo, g, h->num_sms, s);
}

}  // namespace

extern "C" {

int gp_vit_query_sizes(int depth, int max_crops, size_t* weight_bytes, size_t* workspace_bytes) {
  if (depth < 1 || depth > 64 || max_crops < 1) return gp_internal_fail(GP_ERR_INVALID, "bad depth / max_crops");
  Carver cw(nullptr), cs(nullptr);
  carve_weights(cw, depth, nullptr);
  carve_workspace(cs, max_crops, nullptr);
  if (weight_bytes) *weight_bytes = cw.off;
  if (workspace_bytes) *workspace_bytes = cs.off;
  return GP_OK;
}

int gp_vit_create(int device, int depth, int max_crops, int precision, const float* const* w, void* weight_mem,
                  void* workspace_mem, void* stream, gp_vit_handle_t* out) {
  if (depth < 1 || depth > 64 || max_crops < 1 || !w || !weight_mem || !workspace_mem || !out)
    return gp_internal_fail(GP_ERR_INVALID, "bad argument");
  if (precision != GP_PRECISION_FP32_SPLIT && precision != GP_PRECISION_BF16)
    return gp_internal_fail(GP_ERR_INVALID, "unknown precision %d", precision);
  if (((uintptr_t)weight_mem | (uintptr_t)workspace_mem) & (kAlign - 1))
    return gp_internal_fail(GP_ERR_INVALID, "weight and workspace memory must be 1024-byte aligned");
  for (int i = 0; i < 4 + 14 * depth; ++i)
    if (!w[i]) return gp_internal_fail(GP_ERR_INVALID, "weight pointer %d is null", i);
  GPV_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  GPV_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return gp_internal_fail(GP_ERR_UNSUPPORTED, "device %d is not sm_100", device);
  gp_vit_context* h = new (std::nothrow) gp_vit_context();
  if (!h) return gp_internal_fail(GP_ERR_INVALID, "out of host memory");
  h->depth = depth; h->max_crops = max_crops; h->num_sms = prop.multiProcessorCount;
  h->passes = precision == GP_PRECISION_FP32_SPLIT ? 3 : 1;
  h->blocks.resize(depth);
  Carver cw(weight_mem), cs(workspace_mem);
  carve_weights(cw, depth, h);
  carve_workspace(cs, max_crops, h);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  // activation planes start finite: the attention tiles read up to 15 token rows past a crop (masked keys, P = 0),
  // and 0 * NaN from never-written memory would poison the P.V accumulation
  if (cudaMemsetAsync(workspace_mem, 0, cs.off, s) != cudaSuccess) { delete h; return gp_internal_fail(GP_ERR_CUDA, "workspace memset failed"); }

  // pack weights: fp32 [N,K] -> bf16 hi/lo planes (patch embedding padded 588 -> 608 columns)
  h->patch_b = w[1]; h->cls = w[2]; h->pos = w[3];
  cudaError_t ce = gp::launch_split_planes(w[0], kDim, kPatchK, kPatchKPad, h->patch_w.hi, h->patch_w.lo, s);
  int e = ce == cudaSuccess ? make_maps(&h->patch_w, kDim, kPatchKPad, 256) : GP_ERR_CUDA;
  for (int i = 0; i < depth && !e && ce == cudaSuccess; ++i) {
    const float* const* b = w + 4 + 14 * i;
    BlockW& B = h->blocks[i];
    B.n1w = b[0]; B.n1b = b[1]; B.qkv_b = b[3]; B.proj_b = b[5]; B.ls1 = b[6];
    B.n2w = b[7]; B.n2b = b[8]; B.fc1_b = b[10]; B.fc2_b = b[12]; B.ls2 = b[13];
    if ((ce = gp::launch_split_planes(b[2], kQkv, kDim, kDim, B.qkv.hi, B.qkv.lo, s)) != cudaSuccess) break;
    if ((ce = gp::launch_split_planes(b[4], kDim, kDim, kDim, B.proj.hi, B.proj.lo, s)) != cudaSuccess) break;
    if ((ce = gp::launch_split_planes(b[9], kMlp, kDim, kDim, B.fc1.hi, B.fc1.lo, s)) != cudaSuccess) break;
    if ((ce = gp::launch_split_planes(b[11], kDim, kMlp, kMlp, B.fc2.hi, B.fc2.lo, s)) != cudaSuccess) break;
    if ((e = make_maps(&B.qkv, kQkv, kDim, 128)) || (e = make_maps(&B.proj, kDim, kDim, 128)) ||
        (e = make_maps(&B.fc1, kMlp, kDim, 128)) || (e = make_maps(&B.fc2, kDim, kMlp, 128)))
      break;
  }
  const uint64_t M = (uint64_t)max_crops * kTok;
  if (!e && ce == cudaSuccess)
    (e = make_maps(&h->ln, M, kDim, 128)) || (e = make_maps(&h->attn, M, kDim, 128)) || (e = make_maps(&h->hid, M, kMlp, 128)) ||
        (e = make_maps(&h->patches, (uint64_t)max_crops * 256, kPatchKPad, 128)) ||
        (e = gp_internal_make_map_ex(&h->qkv_hi128, h->qkv.hi, 48 * M, 64, 64, 128, 128)) ||   // rows = 3*crops*16*257
        (e = gp_internal_make_map_ex(&h->qkv_lo128, h->qkv.lo, 48 * M, 64, 64, 128, 128)) ||
        (e = gp_internal_make_map_ex(&h->qkv_hi16, h->qkv.hi, 48 * M, 64, 64, 16, 128)) ||
        (e = gp_internal_make_map_ex(&h->qkv_lo16, h->qkv.lo, 48 * M, 64, 64, 16, 128));
  if (ce != cudaSuccess) { delete h; return gp_internal_fail(GP_ERR_CUDA, "weight packing failed: %s", cudaGetErrorString(ce)); }
  if (e) { delete h; return e; }
  gp_internal_count_launches(1 + 4 * depth);
  *out = h;
  return GP_OK;
}

int gp_debug_attention_timeline(long long* stamps32) {
  if (!stamps32) return gp_internal_fail(GP_ERR_INVALID, "null argument");
  GPV_CUDA(cudaDeviceSynchronize());
  GPV_CUDA(gp::read_attention_stamps(stamps32));
  return GP_OK;
}

int gp_debug_gemm_timeline(long long* stamps64) {
  if (!stamps64) return gp_internal_fail(GP_ERR_INVALID, "null argument");
  GPV_CUDA(cudaDeviceSynchronize());
  GPV_CUDA(gp::read_gemm_stamps(stamps64));
  return GP_OK;
}

int gp_vit_destroy(gp_vit_handle_t h) {
  delete h;
  return GP_OK;
}

// diagnostics: the 4 * depth linear layers of one forward over `b` crops, back to back on `stream`, `iters` times,
// between two CUDA events (synchronises the stream).  Operands are whatever the workspace holds (the GEMM does not
// care); the residual stream is clobbered and rebuilt by the next gp_vit_forward.
int gp_vit_time_linears(gp_vit_handle_t h, int b, int iters, float* avg_ms, void* stream) {
  if (!h || !avg_ms || iters < 1) return gp_internal_fail(GP_ERR_INVALID, "bad argument");
  if (b < 1 || b > h->max_crops) return gp_internal_fail(GP_ERR_INVALID, "batch %d outside [1, %d]", b, h->max_crops);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int M = b * kTok;
  auto run = [&]() -> int {
    for (int i = 0; i < h->depth; ++i) {
      const BlockW& B = h->blocks[i];
      gp::GemmParams g{};
      g.passes = h->passes; g.M = M; g.N = kQkv; g.K = kDim; g.mode = gp::GEMM_QKV_HEADS; g.bias = B.qkv_b;
      g.out_hi = h->qkv.hi; g.out_lo = h->qkv.lo; g.tokens_per_img = kTok; g.qkv_crop_stride = h->max_crops;
      GPV_CUDA(linear(h, h->ln, B.qkv, g, s));
      g = gp::GemmParams{}; g.passes = h->passes;
      g.M = M; g.N = kDim; g.K = kDim; g.mode = gp::GEMM_SCALE_RESIDUAL; g.bias = B.proj_b; g.gamma = B.ls1; g.x = h->x;
      GPV_CUDA(linear(h, h->attn, B.proj, g, s));
      g = gp::GemmParams{}; g.passes = h->passes;
      g.M = M; g.N = kMlp; g.K = kDim; g.mode = gp::GEMM_PLANES_GELU; g.bias = B.fc1_b; g.out_hi = h->hid.hi; g.out_lo = h->hid.lo;
      GPV_CUDA(linear(h, h->ln, B.fc1, g, s));
      g = gp::GemmParams{}; g.passes = h->passes;
      g.M = M; g.N = kDim; g.K = kMlp; g.mode = gp::GEMM_SCALE_RESIDUAL; g.bias = B.fc2_b; g.gamma = B.ls2; g.x = h->x;
      GPV_CUDA(linear(h, h->hid, B.fc2, g, s));
    }
    return GP_OK;
  };
  cudaEvent_t e0, e1;
  GPV_CUDA(cudaEventCreate(&e0));
  GPV_CUDA(cudaEventCreate(&e1));
  if (int e = run()) return e;                       // warm-up
  GPV_CUDA(cudaEventRecord(e0, s));
  for (int it = 0; it < iters; ++it)
    if (int e = run()) return e;
  GPV_CUDA(cudaEventRecord(e1, s));
  GPV_CUDA(cudaEventSynchronize(e1));
  float ms = 0.f;
  GPV_CUDA(cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *avg_ms = ms / iters;
  gp_internal_count_launches(4 * h->depth * (iters + 1));
  return GP_OK;
}

int gp_vit_forward(gp_vit_handle_t h, int b, const float* img, float* x_prenorm, void* stream) {
  if (!h || !img || !x_prenorm) return gp_internal_fail(GP_ERR_INVALID, "null argument");
  if (b < 1 || b > h->max_crops) return gp_internal_fail(GP_ERR_INVALID, "batch %d outside [1, %d]", b, h->max_crops);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int M = b * kTok;
  // patch embedding: im2col -> GEMM (+bias +pos) into token rows 1..256 of every crop; CLS rows separately
  GPV_CUDA(gp::launch_im2col(img, b, kPatchKPad, h->patches.hi, h->patches.lo, s));
  gp::GemmParams g{};
  g.passes = h->passes; g.tokens_per_img = kTok; g.patches_per_img = 256;
  g.M = b * 256; g.N = kDim; g.K = kPatchKPad; g.mode = gp::GEMM_PATCH_EMBED; g.bias = h->patch_b; g.pos = h->pos; g.x = h->x;
  GPV_CUDA(gp::launch_vit_gemm(h->patches.m_hi, h->patches.m_lo, h->patch_w.m_hi, h->patch_w.m_lo, g, h->num_sms, s));
  GPV_CUDA(gp::launch_cls_rows(h->cls, h->pos, b, h->x, s));
  for (int i = 0; i < h->depth; ++i) {
    const BlockW& B = h->blocks[i];
    GPV_CUDA(gp::launch_layernorm_planes(h->x, M, B.n1w, B.n1b, 1e-6f, h->ln.hi, h->ln.lo, s));
    g = gp::GemmParams{}; g.passes = h->passes;
    g.M = M; g.N = kQkv; g.K = kDim; g.mode = gp::GEMM_QKV_HEADS; g.bias = B.qkv_b; g.out_hi = h->qkv.hi; g.out_lo = h->qkv.lo;
    g.tokens_per_img = kTok; g.qkv_crop_stride = h->max_crops;
    GPV_CUDA(linear(h, h->ln, B.qkv, g, s));
    GPV_CUDA(gp::launch_attention_tc(h->qkv_hi128, h->qkv_lo128, h->qkv_hi16, h->qkv_lo16, h->qkv.hi, h->qkv.lo,
                                     h->attn.hi, h->attn.lo, b, h->max_crops, h->passes, s));
    g = gp::GemmParams{}; g.passes = h->passes;
    g.M = M; g.N = kDim; g.K = kDim; g.mode = gp::GEMM_SCALE_RESIDUAL; g.bias = B.proj_b; g.gamma = B.ls1; g.x = h->x;
    GPV_CUDA(linear(h, h->attn, B.proj, g, s));
    GPV_CUDA(gp::launch_layernorm_planes(h->x, M, B.n2w, B.n2b, 1e-6f, h->ln.hi, h->ln.lo, s));
    g = gp::GemmParams{}; g.passes = h->passes;
    g.M = M; g.N = kMlp; g.K = kDim; g.mode = gp::GEMM_PLANES_GELU; g.bias = B.fc1_b; g.out_hi = h->hid.hi; g.out_lo = h->hid.lo;
    GPV_CUDA(linear(h, h->ln, B.fc1, g, s));
    g = gp::GemmParams{}; g.passes = h->passes;
    g.M = M; g.N = kDim; g.K = kMlp; g.mode = gp::GEMM_SCALE_RESIDUAL; g.bias = B.fc2_b; g.gamma = B.ls2; g.x = h->x;
    GPV_CUDA(linear(h, h->hid, B.fc2, g, s));
  }
  GPV_CUDA(cudaMemcpyAsync(x_prenorm, h->x, (size_t)M * kDim * sizeof(float), cudaMemcpyDeviceToDevice, s));
  gp_internal_count_launches(3 + 7 * h->depth);
  return GP_OK;
}

}  // extern "C"
