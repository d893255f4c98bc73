// Internal kernel-launch interface shared by the .cu files and the C-ABI layer (api.cu).  Not installed.
#pragma once
#include <cuda_runtime.h>
#include <cuda.h>
#include <stdint.h>

namespace gp {

// Launch helper shared by the .cu files: cluster_x > 1 groups the CTAs into clusters of cluster_x along x.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_ex(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, int cluster_x,
                             Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeClusterDimension;
  attr.val.clusterDim.x = cluster_x; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
  cfg.attrs = &attr; cfg.numAttrs = cluster_x > 1 ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---------------------------------------------------------------- similarity search (sim_search.cu)
struct SimSearchParams {
  int num_items;              // B * T
  int B;                      // queries in this call
  int T;                      // templates per object held by this rank
  const int* perm;            // [B] query order (queries of one object adjacent -> template tiles shared through L2)
  const int* q_obj;           // [B] 0-based object index of every query
  const float* q_mask;        // [B,256]  query mask sampled at the 16x16 patch grid
  const float* bank_mask;     // [O*T,256]
  float sim_threshold;
  float patch_threshold;
  int passes;                 // 3 = hi*hi + hi*lo + lo*hi (fp32-faithful), 1 = hi*hi only (plain bf16)
  float* sim_avg;             // [B,T]      per-template score (matching.py:274-278)
  float* rec_score;           // [B,T,256]  score_tar2src
  uint8_t* rec_idx;           // [B,T,256]  idx_tar2src
  uint8_t* rec_valid;         // [B,T,256]  mask_all != 0
  float* debug_tile;          // nullable [num_items,256,256]: raw fp32 similarity tiles (tests only)
};
// 2-CTA cluster kernel (cta_group::2, one item per pair): every TMA box is 128 rows, the template maps included
cudaError_t launch_sim_search(const CUtensorMap& q_hi, const CUtensorMap& q_lo, const CUtensorMap& t_hi,
                              const CUtensorMap& t_lo, const SimSearchParams& p, int num_sms, cudaStream_t stream);
int sim_search_smem_bytes();

struct TopkSelectParams {
  int B, T, k;
  int id_stride, id_offset;   // global template id = local * id_stride + id_offset (template-interleaved shards)
  const float* sim_avg;
  const float* rec_score;
  const uint8_t* rec_idx;
  const uint8_t* rec_valid;
  float* cand_score;          // [B,k]
  int* cand_id;               // [B,k]
  float* cand_pts_score;      // [B,k,256]
  uint8_t* cand_idx;          // [B,k,256]
  uint8_t* cand_valid;        // [B,k,256]
};
cudaError_t launch_topk_select(const TopkSelectParams& p, cudaStream_t stream);

struct TopkMergeParams {
  int B, k, G;                // G candidate lists; list g of a field starts rank_stride_bytes * g after the field base
  size_t rank_stride_bytes;   // 0 = every field is a dense [G][B][k][...] array
  const float* cand_score;
  const int* cand_id;
  const float* cand_pts_score;
  const uint8_t* cand_idx;
  const uint8_t* cand_valid;
  const float* cand_rel_scale;    // nullable [.,B,k,256]   per-candidate IST outputs computed by the owning shard
  const float* cand_rel_inplane;  // nullable [.,B,k,256,2]
  float* out_rel_scale;           // nullable [B,k,256]
  float* out_rel_inplane;         // nullable [B,k,256,2]
  long long* id_src;          // [B,k]
  float* score_src;           // [B,k]
  float* score_pts;           // [B,k,256]
  long long* tar_pts;         // [B,k,256,2]
  long long* src_pts;         // [B,k,256,2]
};
cudaError_t launch_topk_merge_expand(const TopkMergeParams& p, cudaStream_t stream);

// ---------------------------------------------------------------- descriptor / mask preparation (prep.cu)
// x: n_rows descriptors of `C` channels; element (row r, channel c) at x[(r / rows_per_img) * img_stride +
// (r % rows_per_img) * row_stride + c * chan_stride].  L2-normalises each row `norm_passes` times
// (F.normalize semantics, eps 1e-12) and writes the bf16 hi / lo planes [n_rows, C].
cudaError_t launch_split_descriptors(const float* x, long long n_rows, int C, int rows_per_img, long long img_stride,
                                     long long row_stride, long long chan_stride, int norm_passes,
                                     int tiled /*1: [img][C/32][rows_per_img][32] k-block-tiled planes*/,
                                     uint16_t* hi, uint16_t* lo, float* normalized_out /*nullable [n_rows,C]*/,
                                     cudaStream_t stream);
// nearest-neighbour H x W -> 16 x 16 sampling of float masks (F.interpolate default mode), [n,H,W] -> [n,256]
cudaError_t launch_sample_mask16(const float* mask, long long n, int H, int W, float* out, cudaStream_t stream);
// perm[B] = stable order of the queries by object id, so that tiles sharing a template run back to back
cudaError_t launch_object_order(const int* q_obj, int B, int num_objects, int* q_obj_out, int* perm, cudaStream_t stream);
// [n, C, 256] (channel-major, reference layout) -> [n, 256, C] (patch-major)
cudaError_t launch_transpose_cp(const float* in, long long n, int C, float* out, cudaStream_t stream);

// ---------------------------------------------------------------- IST per-correspondence MLP (ist_mlp.cu)
struct IstMlpWeights {        // fp32, row-major [out,in] exactly as nn.Linear stores them (ist_net.py:140-155)
  const float *s_w1, *s_b1, *s_w2, *s_b2, *s_w3, *s_b3;   // scale head   512->512->256->1
  const float *i_w1, *i_b1, *i_w2, *i_b2, *i_w3, *i_b3;   // inplane head 512->512->256->2 (+tanh)
  int use_tanh;
};
struct IstMlpParams {
  int B, k;
  int T;                      // templates per object held locally (bank row = (obj*T + local_id))
  int id_stride, id_offset;   // local id = (global id - id_offset) / id_stride
  const long long* id_src;    // [B,k] global template ids
  const long long* src_pts;   // [B,k,256,2]
  const long long* tar_pts;   // [B,k,256,2]
  const int* q_obj;           // [B]
  const float* q_ist;         // [B,256(patch),256(ch)]   patch-major query IST features
  const float* bank_ist;      // [O*T,256(patch),256(ch)] patch-major template IST features
  float* rel_scale;           // [B,k,256]   (-1000 where invalid, ist_net.py:110-113)
  float* rel_inplane;         // [B,k,256,2]
  // workspace
  int* row_count;             // [1]
  int* row_ids;               // [B*k*256] flat (b,k,t) of valid rows
};
// The two hidden layers run on tensor cores (vit_gemm_kernel on fp16 hi/lo planes, fp32-faithful 3-pass products):
//  * compact (device-side, no host round trip) + gather: row r = cat(query IST descriptor at tar_pt, template IST descriptor
//    at src_pt) of the r-th valid correspondence -> planes [rows, 512]; *p.row_count rows, the GEMMs read that count
//    on the device (GemmParams::m_dev);
//  * head: scale = h2_s . w3 + b ; (cos, sin) = tanh(h2_i . W3 + b) in fp32, scattered to (b,k,t); -1000 where invalid
//    (ist_net.py:110-113) is written by the compaction pass.
cudaError_t launch_mlp_gather_planes(const IstMlpParams& p, uint16_t* a_hi, uint16_t* a_lo, cudaStream_t stream);
cudaError_t launch_mlp_head_rows(const IstMlpWeights& w, const IstMlpParams& p, const float* h2_scale, const float* h2_inplane,
                                 cudaStream_t stream);

// ---------------------------------------------------------------- RANSAC + scoring + pose lifting (ransac_pose.cu)
struct RansacParams {
  int n;                      // number of (detection, hypothesis) pairs
  float pixel_threshold;      // 14 px (poses.py:18)
  int patch_size;             // 14
  const long long* src_pts;   // [B,k,256,2]
  const long long* tar_pts;
  const float* rel_scale;     // [B,k,256]
  const float* rel_inplane;   // [B,k,256,2]
  float* M;                   // [B,k,3,3]
  uint8_t* failed;            // [B,k]
  long long* in_src;          // [B,k,256,2]
  long long* in_tar;          // [B,k,256,2]
  long long* in_score;        // [B,k,256]
  int* in_count;              // [B,k]
};
cudaError_t launch_ransac(const RansacParams& p, cudaStream_t stream);

struct PoseParams {
  int B, k, T;                // T = GLOBAL templates per object in the pose tables
  int sort;                   // 1: stable re-sort by inlier count (gigaPose.py:590-595); 0: keep the retrieval order
  const int* q_obj;           // [B]
  const float* q_K;           // [B,3,3]
  const float* q_M;           // [B,3,3]
  const float* tmpl_K;        // [O,3,3]
  const float* tmpl_M;        // [O,T,3,3]
  const float* tmpl_pose;     // [O,T,4,4]
  // unsorted inputs (per (b,k))
  const int* in_count;        // [B,k] inlier counts
  const long long* id_src; const float* score_src; const float* score_pts;
  const long long* tar_pts; const long long* src_pts;
  const float* rel_scale; const float* rel_inplane;
  const float* M; const uint8_t* failed;
  const long long* in_src; const long long* in_tar; const long long* in_score;
  // sorted outputs (gigaPose.py:588-604)
  long long* o_id_src; float* o_score_src; float* o_score_pts;
  long long* o_tar_pts; long long* o_src_pts;
  float* o_rel_scale; float* o_rel_inplane;
  float* o_M; uint8_t* o_failed;
  long long* o_in_src; long long* o_in_tar; long long* o_in_score;
  float* o_scores;            // [B,k]
  float* o_poses;             // [B,k,4,4]
};
cudaError_t launch_sort_and_pose(const PoseParams& p, cudaStream_t stream);
cudaError_t launch_pose_only(int n, int k, int T, const int* q_obj, const float* q_K, const float* q_M,
                             const long long* id_src, const float* M, const float* tmpl_K, const float* tmpl_M,
                             const float* tmpl_pose, float* poses, cudaStream_t stream);

// ---------------------------------------------------------------- ViT-L/14 (vit_gemm.cu, vit_ops.cu)
enum GemmMode { GEMM_PLANES = 0, GEMM_PLANES_GELU = 1, GEMM_SCALE_RESIDUAL = 2, GEMM_PATCH_EMBED = 3, GEMM_QKV_HEADS = 4,
                GEMM_PLANES_RELU = 5, GEMM_PLANES_ADD_RELU = 6, GEMM_ROWS_F32 = 7, GEMM_ROWS_F32_RELU = 8 };
struct GemmParams {
  int M, N, K;                // C[M,N] = A[M,K] W[N,K]^T ; N % 256 == 0, K % 32 == 0
  int passes;                 // 3 = hi*hi + hi*lo + lo*hi, 1 = hi*hi
  int mode;                   // GemmMode
  const float* bias;          // [N]
  const float* gamma;         // [N]      LayerScale (GEMM_SCALE_RESIDUAL)
  float* x;                   // fp32 rows (GEMM_SCALE_RESIDUAL: in/out [M,N]; GEMM_PATCH_EMBED: out [imgs*257, N])
  uint16_t *out_hi, *out_lo;  // bf16 planes [M,N] (GEMM_PLANES*)
  const float* pos;           // [257,N] positional table (GEMM_PATCH_EMBED)
  int tokens_per_img, patches_per_img;
  int qkv_crop_stride;        // GEMM_QKV_HEADS: crops per q/k/v section of the head-major planes (= max_crops)
  int bn;                     // output-tile width: 128, 192 or 256 (0 = 256); N % bn == 0
  // implicit-GEMM convolution (conv != 0): A is an NHWC plane read through a 4-D tensor map, one k-block per
  // (filter tap, 32-channel block); a 128-row tile is 128 / Wo whole output rows of one image
  int conv, Ho, Wo, stride, pad, kw, cblocks;
  int pair;                   // 2-CTA clusters: 256 x bn tiles through tcgen05 cta_group::2 (W maps must have bn/2-row boxes)
  int swap;                   // rows of C = output channels (M = cout, a [cout, K] filter bank as the 128-row operand),
                              // columns = output pixels (N); outputs are still written as NHWC planes [N, M]
  const uint16_t *res_hi, *res_lo;   // GEMM_PLANES_ADD_RELU: shortcut planes [M,N]
  const int* m_dev;           // nullable: the row count M lives on the device (data-dependent GEMM size; p.M = upper bound)
  float acc_scale;            // 0 = off; else C = acc * acc_scale + bias (exact power of two undoing a scaled W operand)
  int f16;                    // operand (and output) planes hold IEEE fp16 hi/lo pairs instead of bf16: 22 significant bits
                              // for O(1)-range data (the IST MLP), kind::f16 instruction with fp16 A/B formats
};
cudaError_t launch_vit_gemm(const CUtensorMap& a_hi, const CUtensorMap& a_lo, const CUtensorMap& w_hi,
                            const CUtensorMap& w_lo, const GemmParams& p, int num_sms, cudaStream_t stream);
cudaError_t launch_split_planes(const float* x, long long rows, int K, int Kpad, uint16_t* hi, uint16_t* lo, cudaStream_t s,
                                bool f16 = false, float pre_scale = 1.0f);
cudaError_t launch_im2col(const float* img, int b, int Kpad, uint16_t* hi, uint16_t* lo, cudaStream_t s);
cudaError_t launch_cls_rows(const float* cls, const float* pos, int b, float* x, cudaStream_t s);
cudaError_t launch_layernorm_planes(const float* x, int M, const float* w, const float* b, float eps, uint16_t* hi,
                                    uint16_t* lo, cudaStream_t s);
cudaError_t launch_attention_tc(const CUtensorMap& hi128, const CUtensorMap& lo128, const CUtensorMap& hi16,
                                const CUtensorMap& lo16, const uint16_t* qkv_hi, const uint16_t* qkv_lo, uint16_t* out_hi,
                                uint16_t* out_lo, int b, int crop_stride, int passes, cudaStream_t s);
cudaError_t read_attention_stamps(long long* host32);
cudaError_t read_gemm_stamps(long long* host64);

}  // namespace gp
