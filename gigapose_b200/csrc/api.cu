// C-ABI layer of libgigapose_b200.so (see include/gigapose_b200.h): handle, memory carving, TMA descriptors and the
// launch sequence for each entry point.  No device memory is allocated here; no call synchronises the host
// (except the explicit diagnostics helper gp_time_sim_kernel).
#include "../../include/gigapose_b200.h"
#include "gigapose_kernels.h"

#include <atomic>
#include <dlfcn.h>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>

int gp_internal_make_map_nhwc(CUtensorMap* map, void* ptr, uint64_t C, uint64_t W, uint64_t H, uint64_t N, uint32_t out_w,
                              uint32_t out_h, uint32_t stride);
int gp_internal_make_map_raw(CUtensorMap* map, void* ptr, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                             const uint32_t* box, const uint32_t* elem_strides);
int gp_internal_make_map_ex(CUtensorMap* map, void* ptr, uint64_t rows, uint64_t cols, uint32_t box_cols, uint32_t box_rows,
                            int swizzle_bytes);
int gp_internal_make_map(CUtensorMap* map, void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows);

namespace {

thread_local std::string g_last_error;
std::atomic<uint64_t> g_launches{0};

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}

#define GP_CUDA(expr)                                                                                     \
  do {                                                                                                    \
    cudaError_t _e = (expr);                                                                              \
    if (_e != cudaSuccess) return fail(GP_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(_e));     \
  } while (0)

constexpr size_t kAlign = 1024;
inline size_t align_up(size_t x) { return (x + kAlign - 1) / kAlign * kAlign; }

// bump allocator over caller memory; with base == nullptr it only measures
struct Carver {
  uint8_t* base;
  size_t off = 0;
  explicit Carver(void* b) : base(static_cast<uint8_t*>(b)) {}
  template <typename T>
  T* take(size_t count) {
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += align_up(count * sizeof(T));
    return p;
  }
};

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

}  // namespace

int gp_internal_fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}
void gp_internal_count_launches(int n) { g_launches += n; }

// generic 2-D bf16 plane map [rows, cols] (cols contiguous) with explicit box and swizzle (64 or 128 = box_cols * 2 bytes)
int gp_internal_make_map_ex(CUtensorMap* map, void* ptr, uint64_t rows, uint64_t cols, uint32_t box_cols, uint32_t box_rows,
                            int swizzle_bytes) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return fail(GP_ERR_UNSUPPORTED, "cuTensorMapEncodeTiled not available from this driver");
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {cols * sizeof(uint16_t)};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(GP_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return GP_OK;
}
// NHWC bf16 plane [N, H, W, C] as a 4-D tensor {C, W, H, N}; box = 32 channels x out_w x out_h output positions taken
// with element stride `stride` along x and y (the traversal box spans out * stride input elements).  Coordinates that
// fall outside [0,W) x [0,H) -- the zero padding of a convolution -- are filled with zeros by TMA.
int gp_internal_make_map_nhwc(CUtensorMap* map, void* ptr, uint64_t C, uint64_t W, uint64_t H, uint64_t N, uint32_t out_w,
                              uint32_t out_h, uint32_t stride) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return fail(GP_ERR_UNSUPPORTED, "cuTensorMapEncodeTiled not available from this driver");
  cuuint64_t dims[4] = {C, W, H, N};
  cuuint64_t strides[3] = {C * sizeof(uint16_t), W * C * sizeof(uint16_t), H * W * C * sizeof(uint16_t)};
  cuuint32_t box[4] = {32, out_w * stride, out_h * stride, 1};
  cuuint32_t estr[4] = {1, stride, stride, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(GP_ERR_CUDA, "cuTensorMapEncodeTiled (NHWC) failed with CUresult %d", (int)r);
  return GP_OK;
}
// bf16 tensor map with caller-chosen dimensions / byte strides (rank <= 5, SWIZZLE_64B): used for views whose rows
// overlap in memory (the stem's sliding 8-pixel windows, ist_trunk.cu)
int gp_internal_make_map_raw(CUtensorMap* map, void* ptr, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                             const uint32_t* box, const uint32_t* elem_strides) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return fail(GP_ERR_UNSUPPORTED, "cuTensorMapEncodeTiled not available from this driver");
  cuuint64_t d[5], st[4];
  cuuint32_t b[5], es[5];
  for (int i = 0; i < rank; ++i) { d[i] = dims[i]; b[i] = box[i]; es[i] = elem_strides[i]; if (i + 1 < rank) st[i] = strides_bytes[i]; }
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, ptr, d, st, b, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(GP_ERR_CUDA, "cuTensorMapEncodeTiled (raw, rank %d) failed with CUresult %d", rank, (int)r);
  return GP_OK;
}
// [rows, cols] plane, box = 32 columns (SWIZZLE_64B) x box_rows
int gp_internal_make_map(CUtensorMap* map, void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows) {
  return gp_internal_make_map_ex(map, ptr, rows, cols, 32, box_rows, 64);
}

namespace {

// k-block-tiled bf16 descriptor plane: [image][32 k-blocks][256 patches][32 channels]; seen by TMA as a 2-D array of
// 64-byte rows [images * 32 * 256, 32]; box = 32 channels (64 B, SWIZZLE_64B) x 128 patches of one k-block slab (the
// half of a query or template slab that one CTA of a similarity pair stages)
int make_plane_map(CUtensorMap* map, void* ptr, uint64_t images) {
  return gp_internal_make_map_ex(map, ptr, images * 32ull * GP_NUM_PATCHES, 32, 32, 128, 64);
}

struct Bank {
  uint16_t *hi, *lo;      // [O*T*256, 1024]
  float* mask16;          // [O*T, 256]
  float* ist;             // [O*T, 256, 256] patch-major
  float *K, *M, *pose;    // [O,9], [O,Tg,9], [O,Tg,16]
};

struct Workspace {
  uint16_t *q_hi, *q_lo;  // [Bm*256, 1024]
  float* q_mask16;        // [Bm,256]
  float* q_ist;           // [Bm,256,256] patch-major
  int *perm, *q_obj;      // [Bm]
  float* sim_avg;         // [Bm,T]
  float* rec_score;       // [Bm,T,256]
  uint8_t *rec_idx, *rec_valid;
  // local candidates
  float* c_score; int* c_id; float* c_pts_score; uint8_t *c_idx, *c_valid;
  // IST MLP scratch: compacted valid rows and the activations of the two hidden layers
  int* row_count; int* row_ids;
  uint16_t *mlp_h1_hi, *mlp_h1_lo;                     // first hidden layer [Bm*k*256, 1024] as fp16 hi / lo planes
  float *mlp_h2_scale, *mlp_h2_inplane;                // second hidden layer of each head [Bm*k*256, 256], fp32 rows
  uint16_t *mlp_a_hi, *mlp_a_lo;                       // gathered inputs [Bm*k*256, 512] as fp16 hi / lo planes
  uint16_t *w1_hi, *w1_lo, *w2s_hi, *w2s_lo, *w2i_hi, *w2i_lo;   // packed regressor weights ([1024,512], [256,512] x 2)
  float* bias1;                                        // [1024] = scale b1 | inplane b1
};

void carve_bank(Carver& c, const gp_config_t& cfg, Bank* b) {
  const size_t OT = (size_t)cfg.num_objects * cfg.num_templates;
  const size_t OTg = (size_t)cfg.num_objects * cfg.num_templates_global;
  Bank tmp;
  tmp.hi = c.take<uint16_t>(OT * GP_NUM_PATCHES * GP_AE_DIM);
  tmp.lo = c.take<uint16_t>(OT * GP_NUM_PATCHES * GP_AE_DIM);
  tmp.mask16 = c.take<float>(OT * GP_NUM_PATCHES);
  tmp.ist = c.take<float>((cfg.ist_bank_global ? OTg : OT) * GP_NUM_PATCHES * GP_IST_DIM);
  tmp.K = c.take<float>((size_t)cfg.num_objects * 9);
  tmp.M = c.take<float>(OTg * 9);
  tmp.pose = c.take<float>(OTg * 16);
  if (b) *b = tmp;
}

void carve_workspace(Carver& c, const gp_config_t& cfg, Workspace* w) {
  const size_t Bm = cfg.max_batch, T = cfg.num_templates, k = cfg.top_k;
  Workspace tmp;
  tmp.q_hi = c.take<uint16_t>(Bm * GP_NUM_PATCHES * GP_AE_DIM);
  tmp.q_lo = c.take<uint16_t>(Bm * GP_NUM_PATCHES * GP_AE_DIM);
  tmp.q_mask16 = c.take<float>(Bm * GP_NUM_PATCHES);
  tmp.q_ist = c.take<float>(Bm * GP_NUM_PATCHES * GP_IST_DIM);
  tmp.perm = c.take<int>(Bm);
  tmp.q_obj = c.take<int>(Bm);
  tmp.sim_avg = c.take<float>(Bm * T);
  tmp.rec_score = c.take<float>(Bm * T * GP_NUM_PATCHES);
  tmp.rec_idx = c.take<uint8_t>(Bm * T * GP_NUM_PATCHES);
  tmp.rec_valid = c.take<uint8_t>(Bm * T * GP_NUM_PATCHES);
  tmp.c_score = c.take<float>(Bm * k);
  tmp.c_id = c.take<int>(Bm * k);
  tmp.c_pts_score = c.take<float>(Bm * k * GP_NUM_PATCHES);
  tmp.c_idx = c.take<uint8_t>(Bm * k * GP_NUM_PATCHES);
  tmp.c_valid = c.take<uint8_t>(Bm * k * GP_NUM_PATCHES);
  tmp.row_count = c.take<int>(1);
  tmp.row_ids = c.take<int>(Bm * k * GP_NUM_PATCHES);
  tmp.mlp_h1_hi = c.take<uint16_t>(Bm * k * GP_NUM_PATCHES * 1024);
  tmp.mlp_h1_lo = c.take<uint16_t>(Bm * k * GP_NUM_PATCHES * 1024);
  tmp.mlp_h2_scale = c.take<float>(Bm * k * GP_NUM_PATCHES * 256);
  tmp.mlp_h2_inplane = c.take<float>(Bm * k * GP_NUM_PATCHES * 256);
  tmp.mlp_a_hi = c.take<uint16_t>(Bm * k * GP_NUM_PATCHES * 512);
  tmp.mlp_a_lo = c.take<uint16_t>(Bm * k * GP_NUM_PATCHES * 512);
  tmp.w1_hi = c.take<uint16_t>(1024 * 512);
  tmp.w1_lo = c.take<uint16_t>(1024 * 512);
  tmp.w2s_hi = c.take<uint16_t>(256 * 512);
  tmp.w2s_lo = c.take<uint16_t>(256 * 512);
  tmp.w2i_hi = c.take<uint16_t>(256 * 512);
  tmp.w2i_lo = c.take<uint16_t>(256 * 512);
  tmp.bias1 = c.take<float>(1024);
  if (w) *w = tmp;
}

int validate(const gp_config_t* cfg) {
  if (!cfg) return fail(GP_ERR_INVALID, "null config");
  if (cfg->abi_version != GP_ABI_VERSION) return fail(GP_ERR_INVALID, "ABI version mismatch: %d vs %d", cfg->abi_version, GP_ABI_VERSION);
  if (cfg->num_objects < 1 || cfg->num_templates < 1 || cfg->max_batch < 1)
    return fail(GP_ERR_INVALID, "num_objects, num_templates and max_batch must be >= 1");
  if (cfg->top_k < 1 || cfg->top_k > 32) return fail(GP_ERR_INVALID, "top_k must be in [1,32]");
  if (cfg->num_templates_global < cfg->num_templates) return fail(GP_ERR_INVALID, "num_templates_global < num_templates");
  if (cfg->num_templates_global < cfg->top_k) return fail(GP_ERR_INVALID, "fewer templates than top_k (torch.topk would raise)");
  if (cfg->template_id_stride < 1 || cfg->template_id_offset < 0) return fail(GP_ERR_INVALID, "bad template id stride/offset");
  if (cfg->patch_size < 1) return fail(GP_ERR_INVALID, "patch_size must be >= 1");
  if (cfg->precision != GP_PRECISION_FP32_SPLIT && cfg->precision != GP_PRECISION_BF16)
    return fail(GP_ERR_INVALID, "unknown precision %d", cfg->precision);
  if (cfg->ist_bank_global != 0 && cfg->ist_bank_global != 1) return fail(GP_ERR_INVALID, "ist_bank_global must be 0 or 1");
  if ((size_t)cfg->num_objects * cfg->num_templates * GP_NUM_PATCHES * 32 >= (1ull << 31))
    return fail(GP_ERR_INVALID, "bank has too many rows for 32-bit TMA coordinates");
  return GP_OK;
}

}  // namespace

struct gp_context {
  gp_config_t cfg;
  int num_sms;
  Bank bank;
  Workspace ws;
  CUtensorMap tm_q_hi, tm_q_lo, tm_t_hi, tm_t_lo;
  CUtensorMap tm_ma_hi, tm_ma_lo;                 // MLP layer 1: gathered rows [rows,512]
  CUtensorMap tm_h1s_hi, tm_h1s_lo, tm_h1i_hi, tm_h1i_lo;   // layer 2: column halves of the first hidden layer [rows,1024]
  CUtensorMap tm_w1_hi, tm_w1_lo, tm_w2s_hi, tm_w2s_lo, tm_w2i_hi, tm_w2i_lo;
  gp::IstMlpWeights mlp;
  bool mlp_set;
  int cur_B;      // batch size staged by gp_set_queries (0 = none)
  void* nccl_comm;   // ncclComm_t bound by gp_comm_init (not owned)
  int rank, world;
};

namespace {
// ncclAllGather(sendbuff, recvbuff, sendcount, datatype, comm, stream), resolved from the libnccl the host process has
// already loaded (torch's bundled libnccl.so.2): the library itself carries no link-time NCCL dependency
typedef int (*NcclAllGatherFn)(const void*, void*, size_t, int, void*, cudaStream_t);
typedef const char* (*NcclErrFn)(int);
NcclAllGatherFn g_allgather = nullptr;
NcclErrFn g_nccl_err = nullptr;
int resolve_nccl() {
  if (g_allgather) return GP_OK;
  void* sym = dlsym(RTLD_DEFAULT, "ncclAllGather");
  void* lib = nullptr;
  if (!sym) {
    lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (lib) sym = dlsym(lib, "ncclAllGather");
  }
  if (!sym) return fail(GP_ERR_UNSUPPORTED, "ncclAllGather not found: load libnccl.so.2 (e.g. import torch) before gp_comm_init");
  g_allgather = reinterpret_cast<NcclAllGatherFn>(sym);
  void* es = dlsym(RTLD_DEFAULT, "ncclGetErrorString");
  if (!es && lib) es = dlsym(lib, "ncclGetErrorString");
  g_nccl_err = reinterpret_cast<NcclErrFn>(es);
  return GP_OK;
}
}  // namespace

extern "C" {

const char* gp_last_error(void) { return g_last_error.c_str(); }
int gp_abi_version(void) { return GP_ABI_VERSION; }
uint64_t gp_launch_count(void) { return g_launches.load(); }

int gp_query_sizes(const gp_config_t* cfg, size_t* bank_bytes, size_t* workspace_bytes) {
  if (int e = validate(cfg)) return e;
  Carver cb(nullptr), cw(nullptr);
  carve_bank(cb, *cfg, nullptr);
  carve_workspace(cw, *cfg, nullptr);
  if (bank_bytes) *bank_bytes = cb.off;
  if (workspace_bytes) *workspace_bytes = cw.off;
  return GP_OK;
}

int gp_create(const gp_config_t* cfg, void* bank_mem, void* workspace_mem, gp_handle_t* out) {
  if (int e = validate(cfg)) return e;
  if (!bank_mem || !workspace_mem || !out) return fail(GP_ERR_INVALID, "null pointer argument");
  if (((uintptr_t)bank_mem | (uintptr_t)workspace_mem) & (kAlign - 1))
    return fail(GP_ERR_INVALID, "bank and workspace must be %zu-byte aligned", kAlign);
  GP_CUDA(cudaSetDevice(cfg->device));
  cudaDeviceProp prop;
  GP_CUDA(cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major != 10)
    return fail(GP_ERR_UNSUPPORTED, "device %d is sm_%d%d; this library contains sm_100a code only", cfg->device,
                prop.major, prop.minor);
  if ((int)prop.sharedMemPerBlockOptin < gp::sim_search_smem_bytes())
    return fail(GP_ERR_UNSUPPORTED, "device offers %zu B of shared memory per block, kernel needs %d",
                prop.sharedMemPerBlockOptin, gp::sim_search_smem_bytes());
  gp_context* h = new (std::nothrow) gp_context();
  if (!h) return fail(GP_ERR_INVALID, "out of host memory");
  h->cfg = *cfg;
  h->num_sms = prop.multiProcessorCount;
  h->mlp_set = false;
  h->cur_B = 0;
  h->nccl_comm = nullptr;
  h->rank = 0;
  h->world = 1;
  Carver cb(bank_mem), cw(workspace_mem);
  carve_bank(cb, *cfg, &h->bank);
  carve_workspace(cw, *cfg, &h->ws);
  const uint64_t bank_rows = (uint64_t)cfg->num_objects * cfg->num_templates;   // images
  const uint64_t q_rows = (uint64_t)cfg->max_batch;
  int e;
  if ((e = make_plane_map(&h->tm_t_hi, h->bank.hi, bank_rows)) || (e = make_plane_map(&h->tm_t_lo, h->bank.lo, bank_rows)) ||
      (e = make_plane_map(&h->tm_q_hi, h->ws.q_hi, q_rows)) || (e = make_plane_map(&h->tm_q_lo, h->ws.q_lo, q_rows))) {
    delete h;
    return e;
  }
  {
    const uint64_t rows = (uint64_t)cfg->max_batch * cfg->top_k * GP_NUM_PATCHES;
    uint16_t *h1_hi = h->ws.mlp_h1_hi, *h1_lo = h->ws.mlp_h1_lo;
    const uint64_t dims[2] = {512, rows}, strides[1] = {1024 * sizeof(uint16_t)};
    const uint32_t box[2] = {32, 128}, estr[2] = {1, 1};
    int e;
    if ((e = gp_internal_make_map(&h->tm_ma_hi, h->ws.mlp_a_hi, rows, 512, 128)) || (e = gp_internal_make_map(&h->tm_ma_lo, h->ws.mlp_a_lo, rows, 512, 128)) ||
        (e = gp_internal_make_map_raw(&h->tm_h1s_hi, h1_hi, 2, dims, strides, box, estr)) ||
        (e = gp_internal_make_map_raw(&h->tm_h1s_lo, h1_lo, 2, dims, strides, box, estr)) ||
        (e = gp_internal_make_map_raw(&h->tm_h1i_hi, h1_hi + 512, 2, dims, strides, box, estr)) ||
        (e = gp_internal_make_map_raw(&h->tm_h1i_lo, h1_lo + 512, 2, dims, strides, box, estr)) ||
        (e = gp_internal_make_map(&h->tm_w1_hi, h->ws.w1_hi, 1024, 512, 128)) || (e = gp_internal_make_map(&h->tm_w1_lo, h->ws.w1_lo, 1024, 512, 128)) ||
        (e = gp_internal_make_map(&h->tm_w2s_hi, h->ws.w2s_hi, 256, 512, 128)) || (e = gp_internal_make_map(&h->tm_w2s_lo, h->ws.w2s_lo, 256, 512, 128)) ||
        (e = gp_internal_make_map(&h->tm_w2i_hi, h->ws.w2i_hi, 256, 512, 128)) || (e = gp_internal_make_map(&h->tm_w2i_lo, h->ws.w2i_lo, 256, 512, 128))) {
      delete h;
      return e;
    }
  }
  *out = h;
  return GP_OK;
}

int gp_destroy(gp_handle_t h) {
  delete h;
  return GP_OK;
}

namespace {
// descriptor rows of one of the three accepted layouts -> normalised bf16 hi/lo planes (k-block-tiled)
int split_features(const float* feat, int feat_layout, long long n_imgs, int norm_passes, uint16_t* hi, uint16_t* lo, cudaStream_t s) {
  const long long rows = n_imgs * GP_NUM_PATCHES;
  cudaError_t e;
  if (feat_layout == GP_LAYOUT_CHANNEL_MAJOR)
    e = gp::launch_split_descriptors(feat, rows, GP_AE_DIM, GP_NUM_PATCHES, (long long)GP_NUM_PATCHES * GP_AE_DIM, 1, GP_NUM_PATCHES,
                                     norm_passes, 1, hi, lo, nullptr, s);
  else if (feat_layout == GP_LAYOUT_PATCH_MAJOR)
    e = gp::launch_split_descriptors(feat, rows, GP_AE_DIM, GP_NUM_PATCHES, (long long)GP_NUM_PATCHES * GP_AE_DIM, GP_AE_DIM, 1,
                                     norm_passes, 1, hi, lo, nullptr, s);
  else if (feat_layout == GP_LAYOUT_VIT_TOKENS)     // [n,257,C]: token 0 (CLS) of every crop is skipped
    e = gp::launch_split_descriptors(feat + GP_AE_DIM, rows, GP_AE_DIM, GP_NUM_PATCHES, (long long)(GP_NUM_PATCHES + 1) * GP_AE_DIM,
                                     GP_AE_DIM, 1, norm_passes, 1, hi, lo, nullptr, s);
  else
    return fail(GP_ERR_INVALID, "unknown feature layout %d", feat_layout);
  if (e != cudaSuccess) return fail(GP_ERR_CUDA, "descriptor split failed: %s", cudaGetErrorString(e));
  return GP_OK;
}
}  // namespace

int gp_normalize_patch_tokens(int b, const float* x_prenorm, float* out, void* stream) {
  if (!x_prenorm || !out || b < 1) return fail(GP_ERR_INVALID, "bad argument");
  GP_CUDA(gp::launch_split_descriptors(x_prenorm + GP_AE_DIM, (long long)b * GP_NUM_PATCHES, GP_AE_DIM, GP_NUM_PATCHES,
                                       (long long)(GP_NUM_PATCHES + 1) * GP_AE_DIM, GP_AE_DIM, 1, 1, 0, nullptr, nullptr, out,
                                       static_cast<cudaStream_t>(stream)));
  g_launches += 1;
  return GP_OK;
}

int gp_bank_write(gp_handle_t h, int obj, int tmpl0, int n, const float* feat, int feat_layout, int norm_passes,
                  const float* mask, int H, int W, const float* ist_feat, void* stream) {
  if (!h) return fail(GP_ERR_INVALID, "null handle");
  const gp_config_t& c = h->cfg;
  if (obj < 0 || obj >= c.num_objects || tmpl0 < 0 || n < 1 || tmpl0 + n > c.num_templates)
    return fail(GP_ERR_INVALID, "template range [%d,%d) of object %d outside the bank (%d x %d)", tmpl0, tmpl0 + n, obj,
                c.num_objects, c.num_templates);
  if (!feat || !mask) return fail(GP_ERR_INVALID, "feat and mask are required");
  if (H < 16 || W < 16) return fail(GP_ERR_INVALID, "mask must be at least 16x16");
  if (norm_passes < 0 || norm_passes > 2) return fail(GP_ERR_INVALID, "norm_passes must be 0, 1 or 2");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t slot = (size_t)obj * c.num_templates + tmpl0;
  const size_t plane_off = slot * GP_NUM_PATCHES * GP_AE_DIM;
  if (int e = split_features(feat, feat_layout, n, norm_passes, h->bank.hi + plane_off, h->bank.lo + plane_off, s)) return e;
  GP_CUDA(gp::launch_sample_mask16(mask, n, H, W, h->bank.mask16 + slot * GP_NUM_PATCHES, s));
  g_launches += 2;
  if (ist_feat) {
    if (c.ist_bank_global) return fail(GP_ERR_INVALID, "cfg.ist_bank_global = 1: write IST features with gp_bank_write_ist (global ids)");
    GP_CUDA(gp::launch_transpose_cp(ist_feat, n, GP_IST_DIM, h->bank.ist + slot * GP_NUM_PATCHES * GP_IST_DIM, s));
    g_launches += 1;
  }
  return GP_OK;
}

int gp_bank_write_ist(gp_handle_t h, int obj, int tmpl0, int n, const float* ist_feat, int ist_layout, void* stream) {
  if (!h || !ist_feat) return fail(GP_ERR_INVALID, "null argument");
  const gp_config_t& c = h->cfg;
  const int Ti = c.ist_bank_global ? c.num_templates_global : c.num_templates;
  if (obj < 0 || obj >= c.num_objects || tmpl0 < 0 || n < 1 || tmpl0 + n > Ti)
    return fail(GP_ERR_INVALID, "IST template range [%d,%d) of object %d outside the bank (%d x %d)", tmpl0, tmpl0 + n, obj,
                c.num_objects, Ti);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  float* dst = h->bank.ist + ((size_t)obj * Ti + tmpl0) * GP_NUM_PATCHES * GP_IST_DIM;
  if (ist_layout == GP_LAYOUT_CHANNEL_MAJOR) {
    GP_CUDA(gp::launch_transpose_cp(ist_feat, n, GP_IST_DIM, dst, s));
    g_launches += 1;
  } else if (ist_layout == GP_LAYOUT_PATCH_MAJOR) {
    GP_CUDA(cudaMemcpyAsync(dst, ist_feat, (size_t)n * GP_NUM_PATCHES * GP_IST_DIM * sizeof(float), cudaMemcpyDeviceToDevice, s));
  } else {
    return fail(GP_ERR_INVALID, "unknown IST feature layout %d", ist_layout);
  }
  return GP_OK;
}

int gp_bank_set_poses(gp_handle_t h, const float* K, const float* M, const float* poses, void* stream) {
  if (!h || !K || !M || !poses) return fail(GP_ERR_INVALID, "null argument");
  const gp_config_t& c = h->cfg;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t OTg = (size_t)c.num_objects * c.num_templates_global;
  GP_CUDA(cudaMemcpyAsync(h->bank.K, K, (size_t)c.num_objects * 9 * sizeof(float), cudaMemcpyDeviceToDevice, s));
  GP_CUDA(cudaMemcpyAsync(h->bank.M, M, OTg * 9 * sizeof(float), cudaMemcpyDeviceToDevice, s));
  GP_CUDA(cudaMemcpyAsync(h->bank.pose, poses, OTg * 16 * sizeof(float), cudaMemcpyDeviceToDevice, s));
  return GP_OK;
}

// The regressor's weights (|w| ~ 0.03) are stored as fp16 pairs of 64 w: the lo half of an unscaled weight would be an fp16
// subnormal (6e-8 absolute precision, i.e. only ~2^-19 of the weight); the GEMM epilogue multiplies by 1/64 (exact).
static constexpr float kMlpWeightScale = 64.0f;

int gp_set_ist_weights(gp_handle_t h, const float* const w[12], int use_tanh, void* stream) {
  if (!h || !w) return fail(GP_ERR_INVALID, "null argument");
  for (int i = 0; i < 12; ++i)
    if (!w[i]) return fail(GP_ERR_INVALID, "IST weight pointer %d is null", i);
  gp::IstMlpWeights& m = h->mlp;
  m.s_w1 = w[0]; m.s_b1 = w[1]; m.s_w2 = w[2]; m.s_b2 = w[3]; m.s_w3 = w[4]; m.s_b3 = w[5];
  m.i_w1 = w[6]; m.i_b1 = w[7]; m.i_w2 = w[8]; m.i_b2 = w[9]; m.i_w3 = w[10]; m.i_b3 = w[11];
  m.use_tanh = use_tanh;
  // both heads' first layers side by side as one [1024,512] operand, fp16 hi / lo planes
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Workspace& ws = h->ws;
  GP_CUDA(gp::launch_split_planes(w[0], 512, 512, 512, ws.w1_hi, ws.w1_lo, s, true, kMlpWeightScale));   // fp16 hi / lo (see ist_mlp.cu)
  GP_CUDA(gp::launch_split_planes(w[6], 512, 512, 512, ws.w1_hi + 512 * 512, ws.w1_lo + 512 * 512, s, true, kMlpWeightScale));
  GP_CUDA(gp::launch_split_planes(w[2], 256, 512, 512, ws.w2s_hi, ws.w2s_lo, s, true, kMlpWeightScale));
  GP_CUDA(gp::launch_split_planes(w[8], 256, 512, 512, ws.w2i_hi, ws.w2i_lo, s, true, kMlpWeightScale));
  GP_CUDA(cudaMemcpyAsync(ws.bias1, w[1], 512 * sizeof(float), cudaMemcpyDeviceToDevice, s));
  GP_CUDA(cudaMemcpyAsync(ws.bias1 + 512, w[7], 512 * sizeof(float), cudaMemcpyDeviceToDevice, s));
  g_launches += 4;
  h->mlp_set = true;
  return GP_OK;
}

int gp_set_queries(gp_handle_t h, int B, const float* q_feat, int feat_layout, int norm_passes, const float* q_mask,
                   int H, int W, const int32_t* q_obj, void* stream) {
  if (!h || !q_feat || !q_mask || !q_obj) return fail(GP_ERR_INVALID, "null argument");
  if (B < 1 || B > h->cfg.max_batch) return fail(GP_ERR_INVALID, "batch %d outside [1, max_batch=%d]", B, h->cfg.max_batch);
  if (H < 16 || W < 16) return fail(GP_ERR_INVALID, "mask must be at least 16x16");
  if (norm_passes < 0 || norm_passes > 2) return fail(GP_ERR_INVALID, "norm_passes must be 0, 1 or 2");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (int e = split_features(q_feat, feat_layout, B, norm_passes, h->ws.q_hi, h->ws.q_lo, s)) return e;
  GP_CUDA(gp::launch_sample_mask16(q_mask, B, H, W, h->ws.q_mask16, s));
  // object ids are clamped into [0, O) on the way in: an out-of-range label must not turn into an out-of-bounds bank
  // address (the host-side callers validate and raise; see GigaPose.retrieve)
  GP_CUDA(gp::launch_object_order(q_obj, B, h->cfg.num_objects, h->ws.q_obj, h->ws.perm, s));
  g_launches += 3;
  h->cur_B = B;
  return GP_OK;
}

static int run_sim(gp_context* h, int B, cudaStream_t s, float* debug_tile = nullptr) {
  gp::SimSearchParams p;
  p.num_items = B * h->cfg.num_templates;
  p.B = B;
  p.T = h->cfg.num_templates;
  p.perm = h->ws.perm;
  p.q_obj = h->ws.q_obj;
  p.q_mask = h->ws.q_mask16;
  p.bank_mask = h->bank.mask16;
  p.sim_threshold = h->cfg.sim_threshold;
  p.patch_threshold = h->cfg.patch_threshold;
  p.passes = h->cfg.precision == GP_PRECISION_FP32_SPLIT ? 3 : 1;
  p.sim_avg = h->ws.sim_avg;
  p.rec_score = h->ws.rec_score;
  p.rec_idx = h->ws.rec_idx;
  p.rec_valid = h->ws.rec_valid;
  p.debug_tile = debug_tile;
  GP_CUDA(gp::launch_sim_search(h->tm_q_hi, h->tm_q_lo, h->tm_t_hi, h->tm_t_lo, p, h->num_sms, s));
  g_launches += 1;
  return GP_OK;
}

int gp_sim_candidates(gp_handle_t h, int B, const gp_candidates_t* out, void* stream) {
  if (!h || !out) return fail(GP_ERR_INVALID, "null argument");
  if (B != h->cur_B) return fail(GP_ERR_STATE, "gp_set_queries staged %d queries, search asked for %d", h->cur_B, B);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (int e = run_sim(h, B, s)) return e;
  gp::TopkSelectParams t;
  t.B = B; t.T = h->cfg.num_templates; t.k = h->cfg.top_k;
  t.id_stride = h->cfg.template_id_stride; t.id_offset = h->cfg.template_id_offset;
  t.sim_avg = h->ws.sim_avg; t.rec_score = h->ws.rec_score; t.rec_idx = h->ws.rec_idx; t.rec_valid = h->ws.rec_valid;
  t.cand_score = out->score; t.cand_id = out->id; t.cand_pts_score = out->pts_score; t.cand_idx = out->idx;
  t.cand_valid = out->valid;
  GP_CUDA(gp::launch_topk_select(t, s));
  g_launches += 1;
  return GP_OK;
}

int gp_topk_merge(gp_handle_t h, int B, int G, const gp_candidates_t* g, size_t rank_stride_bytes,
                  const gp_matches_t* out, float* out_rel_scale, float* out_rel_inplane, void* stream) {
  if (!h || !g || !out) return fail(GP_ERR_INVALID, "null argument");
  if (B < 1 || G < 1 || G * h->cfg.top_k > 64) return fail(GP_ERR_INVALID, "B=%d G=%d: need G*k <= 64", B, G);
  gp::TopkMergeParams m;
  m.B = B; m.k = h->cfg.top_k; m.G = G; m.rank_stride_bytes = rank_stride_bytes;
  m.cand_score = g->score; m.cand_id = g->id; m.cand_pts_score = g->pts_score; m.cand_idx = g->idx; m.cand_valid = g->valid;
  m.cand_rel_scale = g->rel_scale; m.cand_rel_inplane = g->rel_inplane;
  m.out_rel_scale = out_rel_scale; m.out_rel_inplane = out_rel_inplane;
  m.id_src = reinterpret_cast<long long*>(out->id_src); m.score_src = out->score_src; m.score_pts = out->score_pts;
  m.tar_pts = reinterpret_cast<long long*>(out->tar_pts); m.src_pts = reinterpret_cast<long long*>(out->src_pts);
  GP_CUDA(gp::launch_topk_merge_expand(m, static_cast<cudaStream_t>(stream)));
  g_launches += 1;
  return GP_OK;
}

int gp_sim_topk(gp_handle_t h, int B, const gp_matches_t* out, void* stream) {
  if (!h || !out) return fail(GP_ERR_INVALID, "null argument");
  gp_candidates_t c;
  c.score = h->ws.c_score; c.id = h->ws.c_id; c.pts_score = h->ws.c_pts_score; c.idx = h->ws.c_idx; c.valid = h->ws.c_valid;
  c.rel_scale = nullptr; c.rel_inplane = nullptr;
  if (int e = gp_sim_candidates(h, B, &c, stream)) return e;
  return gp_topk_merge(h, B, 1, &c, 0, out, nullptr, nullptr, stream);
}

int gp_ist_mlp(gp_handle_t h, int b0, int n, const float* q_ist, int ist_layout, const gp_matches_t* m, float* rel_scale,
               float* rel_inplane, void* stream) {
  if (!h || !q_ist || !m || !rel_scale || !rel_inplane) return fail(GP_ERR_INVALID, "null argument");
  if (!h->mlp_set) return fail(GP_ERR_STATE, "gp_set_ist_weights has not been called");
  if (b0 < 0 || n < 1 || b0 + n > h->cur_B)
    return fail(GP_ERR_STATE, "gp_set_queries staged %d queries, gp_ist_mlp asked for [%d,%d)", h->cur_B, b0, b0 + n);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const float* q_pm = q_ist;
  if (ist_layout == GP_LAYOUT_CHANNEL_MAJOR) {
    GP_CUDA(gp::launch_transpose_cp(q_ist, n, GP_IST_DIM, h->ws.q_ist, s));
    q_pm = h->ws.q_ist;
    g_launches += 1;
  } else if (ist_layout != GP_LAYOUT_PATCH_MAJOR) {
    return fail(GP_ERR_INVALID, "unknown IST feature layout %d", ist_layout);
  }
  const gp_config_t& c = h->cfg;
  gp::IstMlpParams p;
  p.B = n; p.k = c.top_k;
  if (c.ist_bank_global) { p.T = c.num_templates_global; p.id_stride = 1; p.id_offset = 0; }
  else { p.T = c.num_templates; p.id_stride = c.template_id_stride; p.id_offset = c.template_id_offset; }
  p.id_src = reinterpret_cast<const long long*>(m->id_src);
  p.src_pts = reinterpret_cast<const long long*>(m->src_pts);
  p.tar_pts = reinterpret_cast<const long long*>(m->tar_pts);
  p.q_obj = h->ws.q_obj + b0; p.q_ist = q_pm; p.bank_ist = h->bank.ist;
  p.rel_scale = rel_scale; p.rel_inplane = rel_inplane;
  p.row_count = h->ws.row_count; p.row_ids = h->ws.row_ids;
  // compacted valid rows (device-side count, no host sync) -> 512 -> [512 | 512] -> 256 + 256 -> heads (ist_mlp.cu)
  const int rows = n * c.top_k * GP_NUM_PATCHES;                      // a multiple of 256: whole pair tiles
  float *h2s = h->ws.mlp_h2_scale, *h2i = h->ws.mlp_h2_inplane;
  GP_CUDA(gp::launch_mlp_gather_planes(p, h->ws.mlp_a_hi, h->ws.mlp_a_lo, s));
  gp::GemmParams g{};
  g.passes = 3; g.pair = 1; g.f16 = 1; g.acc_scale = 1.0f / kMlpWeightScale; g.m_dev = h->ws.row_count;
  g.M = rows; g.N = 1024; g.K = 512; g.mode = gp::GEMM_PLANES_RELU; g.bias = h->ws.bias1; g.out_hi = h->ws.mlp_h1_hi; g.out_lo = h->ws.mlp_h1_lo;
  GP_CUDA(gp::launch_vit_gemm(h->tm_ma_hi, h->tm_ma_lo, h->tm_w1_hi, h->tm_w1_lo, g, h->num_sms, s));
  g = gp::GemmParams{};
  g.passes = 3; g.pair = 1; g.f16 = 1; g.acc_scale = 1.0f / kMlpWeightScale; g.m_dev = h->ws.row_count;
  g.M = rows; g.N = 256; g.K = 512; g.mode = gp::GEMM_ROWS_F32_RELU; g.bias = h->mlp.s_b2; g.x = h2s;
  GP_CUDA(gp::launch_vit_gemm(h->tm_h1s_hi, h->tm_h1s_lo, h->tm_w2s_hi, h->tm_w2s_lo, g, h->num_sms, s));
  g.bias = h->mlp.i_b2; g.x = h2i;
  GP_CUDA(gp::launch_vit_gemm(h->tm_h1i_hi, h->tm_h1i_lo, h->tm_w2i_hi, h->tm_w2i_lo, g, h->num_sms, s));
  GP_CUDA(gp::launch_mlp_head_rows(h->mlp, p, h2s, h2i, s));
  g_launches += 6;
  return GP_OK;
}

int gp_ransac(int n, float pixel_threshold, int patch_size, const int64_t* src_pts, const int64_t* tar_pts,
              const float* rel_scale, const float* rel_inplane, const gp_ransac_out_t* out, void* stream) {
  if (!src_pts || !tar_pts || !rel_scale || !rel_inplane || !out || !out->inlier_count || !out->M || !out->failed ||
      !out->inlier_src_pts || !out->inlier_tar_pts || !out->inlier_scores)
    return fail(GP_ERR_INVALID, "null argument");
  if (n < 1) return fail(GP_ERR_INVALID, "n must be >= 1");
  gp::RansacParams p;
  p.n = n; p.pixel_threshold = pixel_threshold; p.patch_size = patch_size;
  p.src_pts = reinterpret_cast<const long long*>(src_pts);
  p.tar_pts = reinterpret_cast<const long long*>(tar_pts);
  p.rel_scale = rel_scale; p.rel_inplane = rel_inplane;
  p.M = out->M; p.failed = out->failed;
  p.in_src = reinterpret_cast<long long*>(out->inlier_src_pts);
  p.in_tar = reinterpret_cast<long long*>(out->inlier_tar_pts);
  p.in_score = reinterpret_cast<long long*>(out->inlier_scores);
  p.in_count = out->inlier_count;
  GP_CUDA(gp::launch_ransac(p, static_cast<cudaStream_t>(stream)));
  g_launches += 1;
  return GP_OK;
}

int gp_pose_recover(int B, int k, int num_templates, const int32_t* q_obj, const float* q_K, const float* q_M,
                    const int64_t* id_src, const float* M, const float* tmpl_K, const float* tmpl_M,
                    const float* tmpl_pose, float* poses, void* stream) {
  if (!q_obj || !q_K || !q_M || !id_src || !M || !tmpl_K || !tmpl_M || !tmpl_pose || !poses)
    return fail(GP_ERR_INVALID, "null argument");
  if (B < 1 || k < 1 || num_templates < 1) return fail(GP_ERR_INVALID, "B, k and num_templates must be >= 1");
  GP_CUDA(gp::launch_pose_only(B * k, k, num_templates, q_obj, q_K, q_M, reinterpret_cast<const long long*>(id_src), M,
                               tmpl_K, tmpl_M, tmpl_pose, poses, static_cast<cudaStream_t>(stream)));
  g_launches += 1;
  return GP_OK;
}

int gp_sort_and_pose(gp_handle_t h, int b0, int n, int sort_by_inliers, const float* q_K, const float* q_M,
                     const gp_matches_t* m, const float* rel_scale, const float* rel_inplane, const gp_ransac_out_t* r,
                     const gp_predictions_t* o, void* stream) {
  if (!h || !q_K || !q_M || !m || !rel_scale || !rel_inplane || !r || !o) return fail(GP_ERR_INVALID, "null argument");
  if (b0 < 0 || n < 1 || b0 + n > h->cur_B)
    return fail(GP_ERR_STATE, "gp_set_queries staged %d queries, gp_sort_and_pose asked for [%d,%d)", h->cur_B, b0, b0 + n);
  gp::PoseParams p;
  p.B = n; p.k = h->cfg.top_k; p.T = h->cfg.num_templates_global;
  p.sort = sort_by_inliers ? 1 : 0;
  p.q_obj = h->ws.q_obj + b0; p.q_K = q_K; p.q_M = q_M;
  p.tmpl_K = h->bank.K; p.tmpl_M = h->bank.M; p.tmpl_pose = h->bank.pose;
  p.in_count = r->inlier_count;
  p.id_src = reinterpret_cast<const long long*>(m->id_src); p.score_src = m->score_src; p.score_pts = m->score_pts;
  p.tar_pts = reinterpret_cast<const long long*>(m->tar_pts); p.src_pts = reinterpret_cast<const long long*>(m->src_pts);
  p.rel_scale = rel_scale; p.rel_inplane = rel_inplane;
  p.M = r->M; p.failed = r->failed;
  p.in_src = reinterpret_cast<const long long*>(r->inlier_src_pts);
  p.in_tar = reinterpret_cast<const long long*>(r->inlier_tar_pts);
  p.in_score = reinterpret_cast<const long long*>(r->inlier_scores);
  p.o_id_src = reinterpret_cast<long long*>(o->matches.id_src); p.o_score_src = o->matches.score_src;
  p.o_score_pts = o->matches.score_pts;
  p.o_tar_pts = reinterpret_cast<long long*>(o->matches.tar_pts); p.o_src_pts = reinterpret_cast<long long*>(o->matches.src_pts);
  p.o_rel_scale = o->rel_scale; p.o_rel_inplane = o->rel_inplane;
  p.o_M = o->ransac.M; p.o_failed = o->ransac.failed;
  p.o_in_src = reinterpret_cast<long long*>(o->ransac.inlier_src_pts);
  p.o_in_tar = reinterpret_cast<long long*>(o->ransac.inlier_tar_pts);
  p.o_in_score = reinterpret_cast<long long*>(o->ransac.inlier_scores);
  p.o_scores = o->scores; p.o_poses = o->poses;
  GP_CUDA(gp::launch_sort_and_pose(p, static_cast<cudaStream_t>(stream)));
  g_launches += 1;
  return GP_OK;
}

int gp_comm_init(gp_handle_t h, void* nccl_comm, int rank, int world) {
  if (!h || !nccl_comm) return fail(GP_ERR_INVALID, "null argument");
  if (world < 1 || rank < 0 || rank >= world) return fail(GP_ERR_INVALID, "rank %d outside [0, world=%d)", rank, world);
  if (world != h->cfg.template_id_stride || rank != h->cfg.template_id_offset)
    return fail(GP_ERR_INVALID, "communicator (rank %d of %d) does not match the shard map of this handle (offset %d, stride %d)",
                rank, world, h->cfg.template_id_offset, h->cfg.template_id_stride);
  if (world * h->cfg.top_k > 64) return fail(GP_ERR_INVALID, "world * top_k = %d exceeds the merge kernel's 64 candidates", world * h->cfg.top_k);
  if (int e = resolve_nccl()) return e;
  h->nccl_comm = nccl_comm;
  h->rank = rank;
  h->world = world;
  return GP_OK;
}

int gp_allgather(gp_handle_t h, const void* send, void* recv, size_t bytes_per_rank, void* stream) {
  if (!h || !send || !recv) return fail(GP_ERR_INVALID, "null argument");
  if (!h->nccl_comm) return fail(GP_ERR_STATE, "gp_comm_init has not been called");
  const int r = g_allgather(send, recv, bytes_per_rank, /*ncclInt8*/ 0, h->nccl_comm, static_cast<cudaStream_t>(stream));
  if (r != 0) return fail(GP_ERR_CUDA, "ncclAllGather failed: %s", g_nccl_err ? g_nccl_err(r) : "?");
  return GP_OK;
}

int gp_topk_allgather_merge(gp_handle_t h, int B, void* packed, size_t rank_stride_bytes, const gp_candidates_t* slot0,
                            const gp_matches_t* out, void* stream) {
  if (!h || !packed || !slot0 || !out) return fail(GP_ERR_INVALID, "null argument");
  if (!h->nccl_comm) return fail(GP_ERR_STATE, "gp_comm_init has not been called");
  if (B != h->cur_B) return fail(GP_ERR_STATE, "gp_set_queries staged %d queries, merge asked for %d", h->cur_B, B);
  uint8_t* base = static_cast<uint8_t*>(packed);
  if (int e = gp_allgather(h, base + (size_t)h->rank * rank_stride_bytes, base, rank_stride_bytes, stream)) return e;
  return gp_topk_merge(h, B, h->world, slot0, rank_stride_bytes, out, nullptr, nullptr, stream);
}

int gp_debug_sim_tiles(gp_handle_t h, int B, float* tiles, void* stream) {
  if (!h || !tiles) return fail(GP_ERR_INVALID, "null argument");
  if (B != h->cur_B) return fail(GP_ERR_STATE, "gp_set_queries staged %d queries, debug asked for %d", h->cur_B, B);
  return run_sim(h, B, static_cast<cudaStream_t>(stream), tiles);
}

int gp_time_sim_kernel(gp_handle_t h, int B, int iters, float* avg_ms, void* stream) {
  if (!h || !avg_ms || iters < 1) return fail(GP_ERR_INVALID, "bad argument");
  if (B != h->cur_B) return fail(GP_ERR_STATE, "gp_set_queries staged %d queries, timing asked for %d", h->cur_B, B);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  cudaEvent_t e0, e1;
  GP_CUDA(cudaEventCreate(&e0));
  GP_CUDA(cudaEventCreate(&e1));
  if (int e = run_sim(h, B, s)) return e;   // warm-up
  GP_CUDA(cudaEventRecord(e0, s));
  for (int i = 0; i < iters; ++i)
    if (int e = run_sim(h, B, s)) return e;
  GP_CUDA(cudaEventRecord(e1, s));
  GP_CUDA(cudaEventSynchronize(e1));
  float ms = 0.f;
  GP_CUDA(cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *avg_ms = ms / iters;
  return GP_OK;
}

}  // extern "C"
