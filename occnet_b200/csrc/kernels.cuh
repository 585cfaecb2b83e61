// Launcher declarations shared by the engine (engine.cu) and the C-ABI (capi.cu).
#pragma once
#include "common.cuh"

namespace occ {

// Per-frame camera geometry for the fused spatial cross-attention kernel.
struct ScaParams {
    float cam_mat[8][16];   // lidar2img[c] @ ego2lidar, fp32 row-major (encoder.py:126)
    float zs[8];            // normalised pillar heights linspace(.5, Z-.5, D)/Z (encoder.py:66-67)
    float pc_scale[3];      // pc_range[3+i] - pc_range[i]
    float pc_min[3];        // pc_range[i]
    float img_w, img_h;     // padded image size of batch item 0 (encoder.py:133-134)
    int num_cams, D, bev_h, bev_w;
};

// ---- msda.cu
int launch_msda_forward(const float* value, const int64_t* shapes, const int64_t* lstart, const float* loc,
                        const float* wts, int B, int Nv, int M, int C, int Nq, int L, int P, float* out,
                        cudaStream_t stream);
int launch_msda_backward(const float* value, const int64_t* shapes, const int64_t* lstart, const float* loc,
                         const float* wts, const float* grad_out, int B, int Nv, int M, int C, int Nq, int L, int P,
                         float* grad_value, float* grad_loc, float* grad_attn, cudaStream_t stream);
template <typename T>
int launch_tsa_fused(const T* value_prev, const T* value_cur, const void* qproj, bool qproj_is_half, int bev_h, int bev_w,
                     T* out, cudaStream_t stream);
template <typename T>
int launch_sca_fused(const T* value, const void* qproj, bool qproj_is_half, const ScaParams& sp, const LevelGeom& lg, int Nv,
                     T* out, uint8_t* hits, cudaStream_t stream);
int launch_project_pillars(const ScaParams& sp, float* ref_cam, uint8_t* mask, cudaStream_t stream);

// ---- backbone_kernels.cu (image backbone + neck, channels-last; first version, see the file header)
template <typename T> int launch_nchw_to_nhwc_small(const float* src, T* dst, int N, int C, int H, int W, cudaStream_t stream);
template <typename T>
int launch_im2col_nhwc(const T* in, T* out, int N, int H, int W, int C, int KH, int KW, int stride, int pad, int Ho, int Wo,
                       int Kpad, cudaStream_t stream);
template <typename T> int launch_maxpool3x3s2_nhwc(const T* in, T* out, int N, int H, int W, int C, int Ho, int Wo, cudaStream_t stream);
template <typename T> int launch_add_relu(const T* a, const T* b, T* out, int64_t n, cudaStream_t stream);
template <typename T>
int launch_upsample_add_nhwc(T* fine, const T* coarse, int N, int Hf, int Wf, int Hc, int Wc, int C, cudaStream_t stream);
template <typename T> int launch_nhwc_to_nchw_f32(const T* src, float* dst, int N, int HW, int C, cudaStream_t stream);

// ---- elementwise.cu
// feats level l: [num_cams, C, h, w] f32 (NCHW) -> tokens [num_cams, Nv, C] T, + cams_embeds + level_embeds
// (all levels in one launch; level_embeds [num_levels, C])
// `feats_bf16` != 0: the levels are bf16 [num_cams, C, h, w] (what an on-device backbone / a bf16 host pipeline hands over)
struct PackLevels { const void* feat[8]; int hw[8], start[8], tile_begin[8], num_levels; };
template <typename T>
int launch_pack_levels(const void* const* feats, int feats_bf16, const LevelGeom& lg, const float* cams_embeds,
                       const float* level_embeds, int num_cams, int C, int Nv, T* tokens, cudaStream_t stream);
// same from channels-last bf16 levels [num_cams, h, w, C] (the backbone's native output): an elementwise add, no transpose
template <typename T>
int launch_pack_levels_nhwc(const void* const* feats, const LevelGeom& lg, const float* cams_embeds, const float* level_embeds,
                            int num_cams, int C, int Nv, T* tokens, cudaStream_t stream);
// y = LayerNorm(x) (eps 1e-5); writes fp32 copy (residual stream), T copy (GEMM operand) and T copy of y + pos
template <typename T>
int launch_layernorm(const float* x, const float* gamma, const float* beta, const float* pos, int rows, int C,
                     float* y_f32, T* y_t, T* y_pos_t, cudaStream_t stream);
// bev_queries [Nq,C] f32 -> f32 copy, T copy, T copy + pos (layer-0 input)
template <typename T>
int launch_prepare_query(const float* bev_queries, const float* pos, int64_t n, float* q_f32, T* q_t, T* q_pos_t,
                         int tiled, cudaStream_t stream);
// row-major [rows,256] fp32 <-> "T32" block layout of the tensor-core path's residual stream (see elementwise.cu)
int launch_t32_convert(const float* src, float* dst, int64_t rows, int untile, cudaStream_t stream, int ncols = 256);
// pos[q, :] = cat(col_embed[q % W], row_embed[q / W])     (mmdet LearnedPositionalEncoding)
int launch_bev_pos(const float* row_embed, const float* col_embed, int bev_h, int bev_w, int half, float* pos,
                   cudaStream_t stream);
template <typename T>
int launch_cast(const float* src, T* dst, int64_t n, cudaStream_t stream);
// dst[r] = map[r] >= 0 ? src[map[r]] : 0  (rows of C floats; map == nullptr: identity) -- prev_bev rotation + operand cast
template <typename T>
int launch_gather_rows(const float* src, const int32_t* map, int rows, int C, T* dst, float* dst_f32, cudaStream_t stream);

// ---- decoder_simt.cu
// bev [Nq = H*W, C = mid*Z] f32 -> vox [X=W][Y=H][Z][mid] T with vox[x][y][z][cm] = bev[y*W+x][cm*Z+z]
template <typename T>
int launch_bev_to_voxel(const float* bev, int bev_h, int bev_w, int Z, int mid, T* vox, cudaStream_t stream);
// the same lift from the T32 layout of the residual stream (Z = mid = 16, rows padded to 32), bf16 voxels
int launch_t32_to_voxel(const float* bev_t32, int bev_h, int bev_w, bf16* vox, cudaStream_t stream);
// 3x3x3 conv (pad 1) + folded BatchNorm + ReLU on channels-last [X][Y][Z][Cin] -> [X][Y][Z][Cout=32]
// wfold: [27][Cin][32] f32 (tap = (dz*3+dy)*3+dx), bfold: [32]
template <typename T>
int launch_conv3d_simt(const T* in, const float* wfold, const float* bfold, int X, int Y, int Z, int Cin, T* out,
                       cudaStream_t stream);
// per-voxel heads: occ = W2 softplus(W1 f + b1) + b2 (17), flow = W2' relu(W1' f + b1') + b2' (2), cls = argmax
struct HeadWeights {
    const float *w1, *b1, *w2, *b2;       // predicter:      [64,32],[64],[ncls,64],[ncls]
    const float *fw1, *fb1, *fw2, *fb2;   // flow_predicter: [64,32],[64],[2,64],[2]
    int ncls;
};
template <typename T>
int launch_occ_head(const T* vox, HeadWeights hw, int64_t nvox, float* occ_logits, float* flow, uint8_t* cls_u8,
                    int64_t* cls_i64, cudaStream_t stream);

// ---- raycast.cu
// rows a14/a15: DDA first-hit for T origins x M rays through pred and gt volumes + the 187 counters
int launch_render_forward(const float* sigma, const float* origin, const float* points, const float* tindex,
                          int N, int T, int Z, int Y, int X, int64_t M, float* pred_dist, float* gt_dist,
                          float* coord_index, cudaStream_t stream);
int launch_ray_metric(const uint8_t* sem_pred, const float* flow_pred, const uint8_t* sem_gt, const float* flow_gt,
                      const void* origins, int origin_is_f64, int T, const float* rays, int M, double* counters,
                      float* pcd_pred, float* pcd_gt, cudaStream_t stream);

}  // namespace occ
