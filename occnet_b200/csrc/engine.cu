// Host-side frame engine + C ABI (include/occ_b200.h).  One engine = one model replica on one GPU;
// frames are independent (the reference always runs prev_bev=None, bevformer_occ.py:243-244), so the
// multi-GPU story is one engine per rank and no data-path collective.
//
// Per-frame schedule (reference call stack: SURVEY section 3.1):
//   pack_level x4        transformer_occ.py:207-227   (+cams_embeds, +level_embeds, NCHW -> tokens)
//   per encoder layer    encoder.py:356-404           (self_attn, norm, cross_attn, norm, ffn, norm)
//   bev_to_voxel, conv3d x2, occ_head                 transformer_occ.py:305-319, bevformer_occ_head.py:211-212
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/occ_b200.h"
#include "common.cuh"
#include "conv3d_tc.cuh"
#include "gemm_tc.cuh"
#include "kernels.cuh"

namespace occ {

static thread_local std::string g_last_error;
void set_last_error(const std::string& msg) { g_last_error = msg; }

namespace {

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    int alloc(size_t n) {
        release();
        if (n == 0) return 0;
        OCC_CUDA(cudaMalloc(&p, n));
        bytes = n;
        return 0;
    }
    void release() { if (p) cudaFree(p); p = nullptr; bytes = 0; }
    template <typename U> U* as() const { return reinterpret_cast<U*>(p); }
};

struct LayerW {
    DevBuf tsa_v_w, tsa_v_b, tsa_q_w, tsa_q_b, tsa_o_w, tsa_o_b;
    DevBuf sca_q_w, sca_q_b, sca_v_w, sca_v_b, sca_o_w, sca_o_b;
    DevBuf ffn1_w, ffn1_b, ffn2_w, ffn2_b;
    DevBuf ln_g[3], ln_b[3];
    // bf16 copies for the tensor-core path
    DevBuf tsa_v_wh, tsa_q_wh, tsa_o_wh, sca_q_wh, sca_v_wh, sca_o_wh, ffn1_wh, ffn2_wh;
    // self mode (prev_bev = None): W1 q + W2 (q + pos) + b == (W1 + W2) q + [W2 pos + b]; the bracket depends on parameters
    // only -> an fp32 [Nq,192] constant per layer, added by the GEMM epilogue (K = 256, weight block resident, A read once)
    DevBuf tsa_q_wh_fold, tsa_q_const, tsa_q_const_t32;   // (_t32: the constant in the T32 block layout, TMA-store epilogue)
};

}  // namespace
}  // namespace occ

using namespace occ;

struct occb200_engine {
    occb200_config cfg;
    int Nq = 0, Nv = 0, C = 256;
    LevelGeom lg;
    ScaParams sp;
    bool cameras_set = false, finalized = false, taps = false;
    DevBuf rot_map;                     // occb200_engine_set_prev_rotation: source row of every BEV cell (int32, -1 = outside)
    bool rot_set = false;
    int feats_bf16 = 0;                 // occb200_engine_set_input_dtype: feature levels arrive as bf16 instead of fp32
    std::map<std::string, std::vector<float>> host_params;
    std::vector<LayerW> layers;
    DevBuf bev_queries, pos, pos_t32, cams_embeds, level_embeds;
    DevBuf pos_bf;                      // bev_pos as a bf16 row-major GEMM operand (folded TSA query projection)
    DevBuf qc_f32, qc_t, qc_pos_t;      // parameter-only layer-0 operands (query fp32 T32, bf16 query, bf16 query+pos), built once
    // Self mode (prev_bev = None): layer 0's TemporalSelfAttention + its LayerNorm see only parameters (bev_queries, bev_pos,
    // weights) -- the result is frame-independent and is computed ONCE at finalize by the same kernels (T32 fp32 + bf16 copy)
    DevBuf l0_x_f32, l0_q_t;
    bool l0_ready = false;
    DevBuf conv_w[2], conv_b[2], conv_wh[2];
    DevBuf conv_wh_hi[2], conv_wh_lo[2], vox_split;      // fp32 storage + tensor cores: bf16 hi / lo split of the folded conv weights, [hi | lo] voxel operand
    DevBuf sca_v_all_wh, sca_v_all_b, sca_value_all;     // value_proj of every layer, concatenated (tensor-core path)
    DevBuf hw1, hb1, hw2, hb2, fw1, fb1, fw2, fb2, head_w1h, head_w2h, head_b1c, head_b2c;
    // workspace
    DevBuf tokens, sca_value, q_f32, q_t, q_pos_t, q0_t, prev_t, tsa_value, tsa_value_prev, qproj, attn_out, x_f32,
        ffn_h, vox0, vox1, vox2, hits;
    DevBuf tap_layer, tap_tsa, tap_sca;
    // fp32-grade tensor-core configuration (precision 0 + use_tensor_cores): bf16 [hi | lo] splits of the GEMM operands
    DevBuf split_ws, tokens_split;
    // host-buffer variant
    DevBuf feats_dev[4], occ_i64_dev, flow_dev;
    // pipelined host-buffer variant: 2 slots, copies on their own streams, compute on the caller's stream
    struct Slot {
        DevBuf feats[4], occ, flow;
        cudaEvent_t h2d_done[4] = {nullptr, nullptr, nullptr, nullptr}, compute_done = nullptr, d2h_done = nullptr;
        bool busy = false;
    } slots[2];
    cudaStream_t h2d_stream[4] = {nullptr, nullptr, nullptr, nullptr}, d2h_stream = nullptr;
    int launches = 0;
    // optional per-kernel-category timing (CUDA events on the launch stream)
    bool profiling = false;
    std::vector<std::pair<int, std::pair<cudaEvent_t, cudaEvent_t>>> prof_events;
    std::vector<cudaEvent_t> event_pool;
    size_t event_used = 0;
    size_t elt() const { return cfg.precision ? 2 : 4; }
};

namespace {

int upload(DevBuf& b, const float* src, size_t n)
{
    if (b.alloc(n * sizeof(float))) return 2;
    OCC_CUDA(cudaMemcpy(b.p, src, n * sizeof(float), cudaMemcpyHostToDevice));
    return 0;
}

// [W_hi | W_hi | W_lo] (n x 3k bf16) of an n x k fp32 weight: B operand of gemm_tc_split3
int upload_w3(DevBuf& b, const float* W, size_t n, size_t k)
{
    std::vector<__nv_bfloat16> h(n * 3 * k);
    for (size_t r = 0; r < n; ++r)
        for (size_t j = 0; j < k; ++j) {
            const float w = W[r * k + j];
            const __nv_bfloat16 hi = __float2bfloat16(w);
            const __nv_bfloat16 lo = __float2bfloat16(w - __bfloat162float(hi));
            h[r * 3 * k + j] = hi; h[r * 3 * k + k + j] = hi; h[r * 3 * k + 2 * k + j] = lo;
        }
    if (b.alloc(h.size() * 2)) return 2;
    OCC_CUDA(cudaMemcpy(b.p, h.data(), h.size() * 2, cudaMemcpyHostToDevice));
    return 0;
}

int upload_bf16(DevBuf& b, const float* src, size_t n)
{
    std::vector<__nv_bfloat16> h(n);
    for (size_t i = 0; i < n; ++i) h[i] = __float2bfloat16(src[i]);
    if (b.alloc(n * 2)) return 2;
    OCC_CUDA(cudaMemcpy(b.p, h.data(), n * 2, cudaMemcpyHostToDevice));
    return 0;
}

const std::vector<float>* find(const occb200_engine* e, const std::string& k, size_t numel)
{
    auto it = e->host_params.find(k);
    if (it == e->host_params.end()) { set_last_error("missing parameter: " + k); return nullptr; }
    if (it->second.size() != numel) {
        set_last_error("parameter " + k + " has " + std::to_string(it->second.size()) + " elements, expected " +
                       std::to_string(numel));
        return nullptr;
    }
    return &it->second;
}

#define GETP(var, key, n)                            \
    const std::vector<float>* var = find(e, key, n); \
    if (!var) return 3;

// ---- per-category timing.  Categories: 0 pack/prepare, 1 gemm, 2 tsa gather, 3 sca gather, 4 layernorm,
//      5 bev_to_voxel, 6 conv3d, 7 occ head
enum { CAT_PACK = 0, CAT_GEMM, CAT_TSA, CAT_SCA, CAT_LN, CAT_VOX, CAT_CONV, CAT_HEAD, CAT_COUNT };
struct ProfScope {
    occb200_engine* e; cudaStream_t st; int cat; cudaEvent_t a = nullptr, b = nullptr;
    static cudaEvent_t get(occb200_engine* e) {
        if (e->event_used == e->event_pool.size()) {
            cudaEvent_t ev; cudaEventCreate(&ev); e->event_pool.push_back(ev);
        }
        return e->event_pool[e->event_used++];
    }
    ProfScope(occb200_engine* e_, cudaStream_t st_, int cat_) : e(e_), st(st_), cat(cat_) {
        if (e->profiling) { a = get(e); b = get(e); cudaEventRecord(a, st); }
    }
    ~ProfScope() {
        if (e->profiling) { cudaEventRecord(b, st); e->prof_events.push_back({cat, {a, b}}); }
    }
};

// ---- GEMM dispatch: tensor-core path for bf16 operands when enabled, CUDA-core path otherwise
template <typename TA, typename TC>
int gemm(occb200_engine* e, const TA* A, const TA* A2, int K1, const float* W, const void* Wh, const float* bias,
         const float* residual, TC* C, int M, int N, int K, int act, cudaStream_t st)
{
    e->launches++;
    ProfScope ps(e, st, CAT_GEMM);
    if constexpr (sizeof(TA) == 2) {
        if (e->cfg.use_tensor_cores && Wh != nullptr && gemm_tc_supported(M, N, K, A2 != nullptr ? K1 : K)) {
            return gemm_tc<TC>(reinterpret_cast<const bf16*>(A), reinterpret_cast<const bf16*>(A2), K1,
                               reinterpret_cast<const bf16*>(Wh), bias, residual, C, M, N, K, act, st);
        }
    }
    if constexpr (sizeof(TA) == 4 && std::is_same<TC, float>::value) {
        // fp32 storage + tensor cores: operand split into bf16 hi/lo, weights [W_hi | W_hi | W_lo], three passes in one
        // tcgen05 GEMM (relative error ~2^-16: fp32-grade).  The camera tokens are split once per frame.
        if (e->cfg.use_tensor_cores && e->cfg.precision == 0 && Wh != nullptr && e->split_ws.p != nullptr &&
            gemm_tc_supported(M, N, 3 * K, 2 * K)) {
            const bf16* S = e->split_ws.as<bf16>();
            if ((const void*)A == e->tokens.p && A2 == nullptr && e->tokens_split.p != nullptr) {
                S = e->tokens_split.as<bf16>();
            } else {
                const int Ka = A2 ? K1 : K;
                if (launch_split_bf16(reinterpret_cast<const float*>(A), Ka, reinterpret_cast<const float*>(A2), K - Ka, M,
                                      e->split_ws.as<bf16>(), st)) return 2;
                e->launches++;
            }
            return gemm_tc_split3(S, K, reinterpret_cast<const bf16*>(Wh), bias, residual, C, M, N, act, st);
        }
    }
    if constexpr (std::is_same<TC, __half>::value) {
        OCC_CHECK(false, "gemm: fp16 outputs exist only on the tensor-core path");
    } else {
        const int lda = A2 ? K1 : K;
        return gemm_simt<TA, TC>(A, lda, A2, A2 ? K - K1 : 0, K1, W, bias, residual, N, C, N, M, N, K, act, st);
    }
}

// y = LayerNorm(A.W^T + b + residual): one tcgen05 kernel (GEMM with LayerNorm epilogue) on the tensor-core path
int gemm_ln_fused(occb200_engine* e, const bf16* A, const void* Wh, const float* bias, const float* residual,
                  const float* gamma, const float* beta, const float* pos, float* y_f32, bf16* y_t, bf16* y_pos_t, int M,
                  int K, cudaStream_t st)
{
    e->launches++;
    ProfScope ps(e, st, CAT_GEMM);
    return gemm_tc_ln(A, reinterpret_cast<const bf16*>(Wh), bias, residual, gamma, beta, pos, y_f32, y_t, y_pos_t, M, K, st);
}

enum { MODE_FRAME = 0, MODE_L0_TSA_ONLY = 1 };

template <typename T>
int forward_impl(occb200_engine* e, const float* const* feats, const float* prev_bev, float* bev_embed,
                 float* occ_logits, float* flow, uint8_t* cls_u8, int64_t* cls_i64, cudaStream_t st, int mode = MODE_FRAME)
{
    const occb200_config& c = e->cfg;
    const int Nq = e->Nq, Nv = e->Nv, C = 256, ncam = c.num_cams;
    e->launches = 0;
    T* tokens = e->tokens.as<T>();
    if (mode == MODE_FRAME) {
        ProfScope ps(e, st, CAT_PACK);
        if (e->feats_bf16 == 2) {
            if (launch_pack_levels_nhwc<T>(reinterpret_cast<const void* const*>(feats), e->lg, e->cams_embeds.as<float>(),
                                           e->level_embeds.as<float>(), ncam, C, Nv, tokens, st)) return 2;
        } else if (launch_pack_levels<T>(reinterpret_cast<const void* const*>(feats), e->feats_bf16, e->lg, e->cams_embeds.as<float>(),
                                         e->level_embeds.as<float>(), ncam, C, Nv, tokens, st)) return 2;
        e->launches++;
    }
    if constexpr (sizeof(T) == 4) {
        if (mode == MODE_FRAME && c.use_tensor_cores && e->tokens_split.p != nullptr) {
            ProfScope ps(e, st, CAT_PACK);
            if (launch_split_bf16(reinterpret_cast<const float*>(tokens), C, nullptr, 0, (int64_t)ncam * Nv,
                                  e->tokens_split.as<bf16>(), st)) return 2;
            e->launches++;
        }
    }
    float* q_f32 = e->q_f32.as<float>();
    float* x_f32 = e->x_f32.as<float>();
    T* q_t = e->q_t.as<T>();
    T* q_pos_t = e->q_pos_t.as<T>();
    const float* pos = e->pos.as<float>();
    // tensor-core path: LayerNorm is fused into the GEMM epilogues and the fp32 residual stream lives in the T32 layout
    const bool fuse_ln = sizeof(T) == 2 && c.use_tensor_cores && !e->taps && e->pos_t32.p != nullptr &&
                         e->layers[0].tsa_o_wh.p != nullptr;
    // Layer-0 operands.  On the fused tensor-core path they were built once at finalize (parameters only); the
    // residual stream then rotates through {constant, q_f32, x_f32} without ever writing the constant buffer.
    const bool const_q = fuse_ln && e->qc_f32.p != nullptr;
    const float* cbuf = const_q ? e->qc_f32.as<float>() : nullptr;     // the constant buffer in the rotation (never written)
    float* spare_f32 = nullptr;
    const T* q_in = q_t;                    // bf16/fp32 operand copy of the current query
    const T* q_pos_in = q_pos_t;            // ... of query + pos
    if (const_q) {
        q_in = e->qc_t.as<T>(); q_pos_in = e->qc_pos_t.as<T>();
        spare_f32 = x_f32; x_f32 = q_f32; q_f32 = e->qc_f32.as<float>();     // q_f32 is only READ until advance()
    } else {
        ProfScope ps(e, st, CAT_PACK);
        if (launch_prepare_query<T>(e->bev_queries.as<float>(), pos, (int64_t)Nq * C, q_f32, q_t, q_pos_t, fuse_ln ? 1 : 0,
                                    st)) return 2;
        e->launches++;
    }
    auto advance = [&]() {                  // the LayerNorm output just written to x_f32 becomes the residual stream
        float* old = q_f32;
        q_f32 = x_f32;
        x_f32 = (old == cbuf) ? spare_f32 : old;
    };
    const bool has_prev = prev_bev != nullptr;
    const T* q0_t = nullptr;
    if (has_prev) {
        // encoder.py:204-209: value = stack([prev_bev, bev_query]) built ONCE before the layer loop, so
        // queue 1 keeps seeing the layer-0 query in every layer.
        // (transformer_occ.py:195-205) the rotation of prev_bev about rotate_center is a nearest-neighbour row permutation:
        // applied here, fused with the operand cast, from the index map set by occb200_engine_set_prev_rotation
        if (launch_gather_rows<T>(prev_bev, e->rot_set ? e->rot_map.as<int32_t>() : nullptr, Nq, C, e->prev_t.as<T>(), nullptr, st))
            return 2;
        e->launches++;
        if (const_q) {
            q0_t = e->qc_t.as<T>();
        } else {
            if (launch_cast<T>(e->bev_queries.as<float>(), e->q0_t.as<T>(), (int64_t)Nq * C, st)) return 2;
            e->launches++;
            q0_t = e->q0_t.as<T>();
        }
    }
    // sampling offsets / attention logits: fp16 on the tensor-core path (half the bytes between the projection GEMM and
    // the gather kernel; |offset| is a few pixels, so fp16's 11-bit mantissa keeps locations to < 0.01 px), fp32 otherwise
    const int nq_tsa = 2 * 8 * c.tsa_points * 3;   // offsets (x,y) + logits
    const int nq_sca = 8 * c.num_levels * c.sca_points * 3;
    const bool q_half = sizeof(T) == 2 && c.use_tensor_cores && e->layers[0].tsa_q_wh.p != nullptr &&
                        e->layers[0].sca_q_wh.p != nullptr && gemm_tc_supported(Nq, nq_tsa, 2 * C, C) &&
                        gemm_tc_supported(Nq, nq_sca, C, C);
    void* qproj = e->qproj.p;
    T* attn_out = e->attn_out.as<T>();
    const bool hoist_v = sizeof(T) == 2 && c.use_tensor_cores && e->sca_value_all.p != nullptr;
    // layer-0 TSA + LayerNorm folded into a constant (self mode only; OCC_NO_L0_FOLD=1 recomputes it every frame)
    const bool l0_fold = mode == MODE_FRAME && const_q && !has_prev && e->l0_ready;
    const T* q_t_in = q_t;                  // A operand of the SCA query projection (= the TSA LayerNorm output)
    if (hoist_v && mode == MODE_FRAME) {
        e->launches++;
        ProfScope ps(e, st, CAT_GEMM);
        if (gemm_tc_blocked256((const bf16*)tokens, e->sca_v_all_wh.as<bf16>(), e->sca_v_all_b.as<float>(),
                               e->sca_value_all.as<bf16>(), ncam * Nv, c.num_layers * C, C, st)) return 2;
    }
    for (int l = 0; l < c.num_layers; ++l) {
        LayerW& w = e->layers[l];
        // self mode (prev_bev = None): W1 q + W2 (q + pos) = (W1 + W2) q + W2 pos -- the second operand is the CONSTANT
        // bf16 pos, so no layer has to write (and the FFN LayerNorm epilogue has to read pos for) a bf16 copy of q + pos
        const bool fold_pos = fuse_ln && !has_prev && w.tsa_q_wh_fold.p != nullptr && w.tsa_q_const.p != nullptr && q_half;
        // ---- temporal self-attention (temporal_self_attention.py:177-272)
        if (l == 0 && l0_fold) {
            // precomputed at finalize: residual stream := constant T32 buffer, SCA projection operand := constant bf16 copy
            q_f32 = e->l0_x_f32.as<float>(); x_f32 = e->q_f32.as<float>(); spare_f32 = e->x_f32.as<float>();
            cbuf = q_f32;
            q_t_in = e->l0_q_t.as<T>();
            q_in = q_t; q_pos_in = q_pos_t;
        } else {
        T* v_cur = e->tsa_value.as<T>();
        T* v_prev = v_cur;
        auto value_gemm = [&](const T* a, T* dst) -> int {
            return gemm<T, T>(e, a, nullptr, 0, w.tsa_v_w.as<float>(), w.tsa_v_wh.p, w.tsa_v_b.as<float>(), nullptr, dst, Nq, C, C,
                              ACT_NONE, st);
        };
        // value_proj of every queue entry + the sampling projection are independent GEMMs over [Nq,256] operands: ONE launch on
        // disjoint CTA ranges
        const bool tsa_merge = sizeof(T) == 2 && fuse_ln && q_half && w.tsa_v_wh.p != nullptr;
        if (has_prev) v_prev = e->tsa_value_prev.as<T>();
        if (tsa_merge) {
            if constexpr (sizeof(T) == 2) {
                const bf16* Av[2] = {reinterpret_cast<const bf16*>(has_prev ? q0_t : q_in), e->prev_t.as<bf16>()};
                bf16* Cv[2] = {reinterpret_cast<bf16*>(v_cur), reinterpret_cast<bf16*>(v_prev)};
                e->launches++;
                ProfScope ps(e, st, CAT_GEMM);
                const int rc = fold_pos
                    ? gemm_tc_tsa_inputs(Av, 1, w.tsa_v_wh.as<bf16>(), w.tsa_v_b.as<float>(), Cv, reinterpret_cast<const bf16*>(q_in),
                                         nullptr, C, w.tsa_q_wh_fold.as<bf16>(), nullptr, w.tsa_q_const.as<float>(),
                                         w.tsa_q_const_t32.as<float>(), (__half*)qproj, Nq, nq_tsa, C, st)
                    : gemm_tc_tsa_inputs(Av, has_prev ? 2 : 1, w.tsa_v_wh.as<bf16>(), w.tsa_v_b.as<float>(), Cv,
                                         reinterpret_cast<const bf16*>(has_prev ? e->prev_t.as<T>() : q_in),
                                         reinterpret_cast<const bf16*>(q_pos_in), C, w.tsa_q_wh.as<bf16>(), w.tsa_q_b.as<float>(),
                                         nullptr, nullptr, (__half*)qproj, Nq, nq_tsa, 2 * C, st);
                if (rc) return 2;
            }
        } else {
        if (value_gemm(has_prev ? q0_t : q_in, v_cur)) return 2;
        if (has_prev) {
            if (value_gemm(e->prev_t.as<T>(), v_prev)) return 2;
        }
        if (fold_pos) {
            if (gemm<T, __half>(e, q_in, nullptr, 0, w.tsa_q_w.as<float>(), w.tsa_q_wh_fold.p, nullptr,
                                w.tsa_q_const.as<float>(), (__half*)qproj, Nq, nq_tsa, C, ACT_NONE, st)) return 2;
        } else {
            const T* qa = has_prev ? e->prev_t.as<T>() : q_in;
            const int rc = q_half ? gemm<T, __half>(e, qa, q_pos_in, C, w.tsa_q_w.as<float>(), w.tsa_q_wh.p, w.tsa_q_b.as<float>(),
                                                    nullptr, (__half*)qproj, Nq, nq_tsa, 2 * C, ACT_NONE, st)
                                  : gemm<T, float>(e, qa, q_pos_in, C, w.tsa_q_w.as<float>(), w.tsa_q_wh.p, w.tsa_q_b.as<float>(),
                                                   nullptr, (float*)qproj, Nq, nq_tsa, 2 * C, ACT_NONE, st);
            if (rc) return 2;
        }
        }   // (tsa_merge)
        {
            ProfScope ps(e, st, CAT_TSA);
            if (launch_tsa_fused<T>(v_prev, v_cur, qproj, q_half, c.bev_h, c.bev_w, attn_out, st)) return 2;
        }
        e->launches++;
        if (fuse_ln) {
            float* y32 = mode == MODE_L0_TSA_ONLY ? e->l0_x_f32.as<float>() : x_f32;
            bf16* y16 = mode == MODE_L0_TSA_ONLY ? e->l0_q_t.as<bf16>() : (bf16*)q_t;
            if (gemm_ln_fused(e, (const bf16*)attn_out, w.tsa_o_wh.p, w.tsa_o_b.as<float>(), q_f32, w.ln_g[0].as<float>(),
                              w.ln_b[0].as<float>(), nullptr, y32, y16, nullptr, Nq, C, st)) return 2;
            if (mode == MODE_L0_TSA_ONLY) return 0;
            advance();
            q_in = q_t; q_pos_in = q_pos_t;
        } else {
            if (gemm<T, float>(e, attn_out, nullptr, 0, w.tsa_o_w.as<float>(), w.tsa_o_wh.p, w.tsa_o_b.as<float>(),
                               q_f32, x_f32, Nq, C, C, ACT_NONE, st)) return 2;
            if (e->taps)
                OCC_CUDA(cudaMemcpyAsync(e->tap_tsa.as<float>() + (size_t)l * Nq * C, x_f32, (size_t)Nq * C * 4,
                                         cudaMemcpyDeviceToDevice, st));
            {
                ProfScope ps(e, st, CAT_LN);
                if (launch_layernorm<T>(x_f32, w.ln_g[0].as<float>(), w.ln_b[0].as<float>(), nullptr, Nq, C, q_f32, q_t,
                                        (T*)nullptr, st)) return 2;
            }
            e->launches++;
        }
        }   // (layer-0 TSA fold)
        // ---- spatial cross-attention (spatial_cross_attention.py:128-175, :334-393)
        {
            const int rc = q_half ? gemm<T, __half>(e, q_t_in, nullptr, 0, w.sca_q_w.as<float>(), w.sca_q_wh.p, w.sca_q_b.as<float>(),
                                                    nullptr, (__half*)qproj, Nq, nq_sca, C, ACT_NONE, st)
                                  : gemm<T, float>(e, q_t_in, nullptr, 0, w.sca_q_w.as<float>(), w.sca_q_wh.p, w.sca_q_b.as<float>(),
                                                   nullptr, (float*)qproj, Nq, nq_sca, C, ACT_NONE, st);
            if (rc) return 2;
            q_t_in = q_t;
        }
        const T* sca_val = e->sca_value.as<T>();
        if (hoist_v) {
            sca_val = reinterpret_cast<const T*>(e->sca_value_all.as<bf16>() + (size_t)l * ncam * Nv * C);
        } else if (gemm<T, T>(e, tokens, nullptr, 0, w.sca_v_w.as<float>(), w.sca_v_wh.p, w.sca_v_b.as<float>(), nullptr,
                              e->sca_value.as<T>(), ncam * Nv, C, C, ACT_NONE, st)) return 2;
        {
            ProfScope ps(e, st, CAT_SCA);
            if (launch_sca_fused<T>(sca_val, qproj, q_half, e->sp, e->lg, Nv, attn_out, e->hits.as<uint8_t>(), st)) return 2;
        }
        e->launches++;
        if (fuse_ln) {
            if (gemm_ln_fused(e, (const bf16*)attn_out, w.sca_o_wh.p, w.sca_o_b.as<float>(), q_f32, w.ln_g[1].as<float>(),
                              w.ln_b[1].as<float>(), nullptr, x_f32, (bf16*)q_t, nullptr, Nq, C, st)) return 2;
            advance();
        } else {
            if (gemm<T, float>(e, attn_out, nullptr, 0, w.sca_o_w.as<float>(), w.sca_o_wh.p, w.sca_o_b.as<float>(),
                               q_f32, x_f32, Nq, C, C, ACT_NONE, st)) return 2;
            if (e->taps)
                OCC_CUDA(cudaMemcpyAsync(e->tap_sca.as<float>() + (size_t)l * Nq * C, x_f32, (size_t)Nq * C * 4,
                                         cudaMemcpyDeviceToDevice, st));
            {
                ProfScope ps(e, st, CAT_LN);
                if (launch_layernorm<T>(x_f32, w.ln_g[1].as<float>(), w.ln_b[1].as<float>(), nullptr, Nq, C, q_f32, q_t,
                                        (T*)nullptr, st)) return 2;
            }
            e->launches++;
        }
        // ---- FFN (mmcv FFN: x + W2 relu(W1 x))
        if (gemm<T, T>(e, q_t, nullptr, 0, w.ffn1_w.as<float>(), w.ffn1_wh.p, w.ffn1_b.as<float>(), nullptr,
                       e->ffn_h.as<T>(), Nq, c.ffn_dim, C, ACT_RELU, st)) return 2;
        if (fuse_ln) {
            const bool need_qpos = !fold_pos;                // only the unfolded TSA query projection reads q + pos
            if (gemm_ln_fused(e, e->ffn_h.as<bf16>(), w.ffn2_wh.p, w.ffn2_b.as<float>(), q_f32, w.ln_g[2].as<float>(),
                              w.ln_b[2].as<float>(), need_qpos ? e->pos_t32.as<float>() : nullptr, x_f32, (bf16*)q_t,
                              need_qpos ? (bf16*)q_pos_t : nullptr, Nq, c.ffn_dim, st))
                return 2;
            advance();
        } else {
            if (gemm<T, float>(e, e->ffn_h.as<T>(), nullptr, 0, w.ffn2_w.as<float>(), w.ffn2_wh.p, w.ffn2_b.as<float>(),
                               q_f32, x_f32, Nq, C, c.ffn_dim, ACT_NONE, st)) return 2;
            {
                ProfScope ps(e, st, CAT_LN);
                if (launch_layernorm<T>(x_f32, w.ln_g[2].as<float>(), w.ln_b[2].as<float>(), pos, Nq, C, q_f32, q_t,
                                        q_pos_t, st)) return 2;
            }
            e->launches++;
        }
        if (e->taps)
            OCC_CUDA(cudaMemcpyAsync(e->tap_layer.as<float>() + (size_t)l * Nq * C, q_f32, (size_t)Nq * C * 4,
                                     cudaMemcpyDeviceToDevice, st));
    }
    const int X = c.bev_w, Y = c.bev_h, Z = c.pillar_h, mid = C / Z;
    // the voxel lift reads the T32 residual stream directly when bev_embed itself is not an output (one kernel instead of two)
    const bool lift_from_t32 = fuse_ln && sizeof(T) == 2 && bev_embed == nullptr && Z == 16 && mid == 16;
    if (fuse_ln && !lift_from_t32) {                               // back to row-major for the outputs / voxel decoder
        ProfScope ps(e, st, CAT_PACK);
        if (launch_t32_convert(q_f32, x_f32, Nq, 1, st)) return 2;
        advance();
        e->launches++;
    }
    if (bev_embed)
        OCC_CUDA(cudaMemcpyAsync(bev_embed, q_f32, (size_t)Nq * C * 4, cudaMemcpyDeviceToDevice, st));
    if (!occ_logits && !flow && !cls_u8 && !cls_i64) return 0;
    // ---- voxel decoder + heads
    {
        ProfScope ps(e, st, CAT_VOX);
        if (lift_from_t32) {
            if (launch_t32_to_voxel(q_f32, c.bev_h, c.bev_w, e->vox0.as<bf16>(), st)) return 2;
        } else if (launch_bev_to_voxel<T>(q_f32, c.bev_h, c.bev_w, Z, mid, e->vox0.as<T>(), st)) return 2;
    }
    const bool conv_tc = sizeof(T) == 2 && c.use_tensor_cores && e->conv_wh[0].p && e->conv_wh[1].p && Z == 16;
    // fp32 storage + tensor cores: both convolutions as three bf16-split passes accumulated in fp32
    const bool conv_split = sizeof(T) == 4 && c.use_tensor_cores && e->conv_wh_hi[0].p && e->conv_wh_lo[1].p &&
                            e->vox_split.p && Z == 16 && (mid == 16 || mid == 32) && c.out_dim == 32;
    if (conv_split) {
        const int64_t nv = (int64_t)X * Y * Z;
        ProfScope ps(e, st, CAT_CONV);
        if (launch_split_bf16(e->vox0.as<float>(), mid, nullptr, 0, nv, e->vox_split.as<bf16>(), st)) return 2;
        if (launch_conv3d_tc_split(e->vox_split.as<bf16>(), e->conv_wh_hi[0].as<bf16>(), e->conv_wh_lo[0].as<bf16>(), e->conv_b[0].as<float>(),
                                   X, Y, Z, mid, e->vox1.as<float>(), st)) return 2;
        if (launch_split_bf16(e->vox1.as<float>(), c.out_dim, nullptr, 0, nv, e->vox_split.as<bf16>(), st)) return 2;
        if (launch_conv3d_tc_split(e->vox_split.as<bf16>(), e->conv_wh_hi[1].as<bf16>(), e->conv_wh_lo[1].as<bf16>(), e->conv_b[1].as<float>(),
                                   X, Y, Z, c.out_dim, e->vox2.as<float>(), st)) return 2;
        e->launches += 6;                                       // (+ the 2 counted below = 2 splits + 6 conv passes)
    } else {
    {
        ProfScope ps(e, st, CAT_CONV);
        if (conv_tc) {
            if (launch_conv3d_tc(e->vox0.as<bf16>(), e->conv_wh[0].as<bf16>(), e->conv_b[0].as<float>(), X, Y, Z, mid,
                                 e->vox1.as<bf16>(), st)) return 2;
        } else if (launch_conv3d_simt<T>(e->vox0.as<T>(), e->conv_w[0].as<float>(), e->conv_b[0].as<float>(), X, Y, Z,
                                         mid, e->vox1.as<T>(), st)) return 2;
    }
    {
        ProfScope ps(e, st, CAT_CONV);
        if (conv_tc) {
            if (launch_conv3d_tc(e->vox1.as<bf16>(), e->conv_wh[1].as<bf16>(), e->conv_b[1].as<float>(), X, Y, Z,
                                 c.out_dim, e->vox2.as<bf16>(), st)) return 2;
        } else if (launch_conv3d_simt<T>(e->vox1.as<T>(), e->conv_w[1].as<float>(), e->conv_b[1].as<float>(), X, Y, Z,
                                         c.out_dim, e->vox2.as<T>(), st)) return 2;
    }
    }   // (!conv_split)
    HeadWeights hw{e->hw1.as<float>(), e->hb1.as<float>(), e->hw2.as<float>(), e->hb2.as<float>(),
                   e->fw1.as<float>(), e->fb1.as<float>(), e->fw2.as<float>(), e->fb2.as<float>(), c.num_classes};
    {
        ProfScope ps(e, st, CAT_HEAD);
        if (conv_tc && e->head_w1h.p) {
            if (launch_occ_head_tc(e->vox2.as<bf16>(), e->head_w1h.as<bf16>(), e->head_w2h.as<bf16>(),
                                   e->head_b1c.as<float>(), e->head_b2c.as<float>(), c.num_classes, (int64_t)X * Y * Z,
                                   occ_logits, flow, cls_u8, cls_i64, st)) return 2;
        } else if (launch_occ_head<T>(e->vox2.as<T>(), hw, (int64_t)X * Y * Z, occ_logits, flow, cls_u8, cls_i64, st))
            return 2;
    }
    e->launches += 4;
    return 0;
}

}  // namespace

extern "C" {

const char* occb200_last_error(void) { return g_last_error.c_str(); }
const char* occb200_version(void) { return "occ_b200 0.1 sm_100a"; }

int occb200_ms_deform_attn_forward(const float* value, const int64_t* spatial_shapes, const int64_t* level_start_index,
                                   const float* sampling_loc, const float* attn_weight, int B, int Nv, int M, int C,
                                   int Nq, int L, int P, int im2col_step, float* out, void* stream)
{
    OCC_CHECK(B >= 0 && Nv >= 0 && M > 0 && C > 0 && Nq >= 0 && L > 0 && P > 0, "bad sizes");
    if ((int64_t)B * Nq == 0) return 0;                          // empty query set: nothing to write
    OCC_CHECK(value && spatial_shapes && level_start_index && sampling_loc && attn_weight && out, "null pointer");
    const int step = im2col_step < B ? im2col_step : B;
    OCC_CHECK(B == 0 || (step > 0 && B % step == 0), "batch(" + std::to_string(B) + ") must divide im2col_step(" +
                                                         std::to_string(im2col_step) + ")");
    return launch_msda_forward(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, B, Nv, M, C, Nq, L,
                               P, out, (cudaStream_t)stream);
}

int occb200_ms_deform_attn_backward(const float* value, const int64_t* spatial_shapes, const int64_t* level_start_index,
                                    const float* sampling_loc, const float* attn_weight, const float* grad_output, int B,
                                    int Nv, int M, int C, int Nq, int L, int P, int im2col_step, float* grad_value,
                                    float* grad_sampling_loc, float* grad_attn_weight, void* stream)
{
    OCC_CHECK(B >= 0 && Nv >= 0 && M > 0 && C > 0 && Nq >= 0 && L > 0 && P > 0, "bad sizes");
    if ((int64_t)B * Nq == 0) return 0;
    OCC_CHECK(value && spatial_shapes && level_start_index && sampling_loc && attn_weight && grad_output && grad_value &&
                  grad_sampling_loc && grad_attn_weight, "null pointer");
    const int step = im2col_step < B ? im2col_step : B;
    OCC_CHECK(step > 0 && B % step == 0, "batch(" + std::to_string(B) + ") must divide im2col_step(" +
                                             std::to_string(im2col_step) + ")");
    return launch_msda_backward(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, grad_output, B, Nv, M,
                                C, Nq, L, P, grad_value, grad_sampling_loc, grad_attn_weight, (cudaStream_t)stream);
}

int occb200_engine_create(const occb200_config* cfg, occb200_engine** out)
{
    OCC_CHECK(cfg && out, "null pointer");
    OCC_CHECK(cfg->embed_dims == 256 && cfg->num_heads == 8, "only embed_dims=256, num_heads=8 are supported");
    OCC_CHECK(cfg->num_levels == 4 && cfg->sca_points == 8 && cfg->tsa_points == 4,
              "only num_levels=4, SCA num_points=8, TSA num_points=4 are supported");
    OCC_CHECK(cfg->num_cams >= 1 && cfg->num_cams <= 8, "num_cams must be in [1,8]");
    OCC_CHECK(cfg->num_points_in_pillar >= 1 && cfg->num_points_in_pillar <= 8 && 8 % cfg->num_points_in_pillar == 0,
              "num_points_in_pillar must be 1, 2, 4 or 8");
    OCC_CHECK(cfg->pillar_h == 16 && cfg->out_dim == 32, "only pillar_h=16, out_dim=32 are supported");
    OCC_CHECK(cfg->ffn_dim % 64 == 0 && cfg->num_classes <= 32 && cfg->num_layers >= 1, "bad ffn_dim/num_classes");
    OCC_CHECK(cfg->precision == 0 || cfg->precision == 1, "precision must be 0 (fp32) or 1 (bf16)");
    // the TSA / SCA gathers fetch 2x2 pixel blocks: a side of 1 has none (refused here, not at the first forward)
    OCC_CHECK(cfg->bev_h >= 2 && cfg->bev_w >= 2, "the BEV grid must be at least 2x2");
    for (int l = 0; l < 4; ++l)
        OCC_CHECK(cfg->level_h[l] >= 2 && cfg->level_w[l] >= 2, "every feature level must be at least 2x2");
    int dev_count = 0;
    if (cudaGetDeviceCount(&dev_count) != cudaSuccess || dev_count == 0) {
        set_last_error("no CUDA device: libocc_b200 has no CPU fallback");
        return 4;
    }
    auto* e = new occb200_engine();
    e->cfg = *cfg;
    e->Nq = cfg->bev_h * cfg->bev_w;
    e->lg.num_levels = 4;
    int start = 0;
    for (int l = 0; l < 4; ++l) {
        e->lg.h[l] = cfg->level_h[l]; e->lg.w[l] = cfg->level_w[l]; e->lg.start[l] = start;
        start += cfg->level_h[l] * cfg->level_w[l];
    }
    e->Nv = start;
    e->layers.resize(cfg->num_layers);
    *out = e;
    return 0;
}

void occb200_engine_destroy(occb200_engine* e)
{
    if (!e) return;
    // DevBuf members do not own a destructor on purpose (explicit release keeps teardown order obvious)
    for (auto& w : e->layers) {
        DevBuf* all[] = {&w.tsa_v_w, &w.tsa_v_b, &w.tsa_q_w, &w.tsa_q_b, &w.tsa_o_w, &w.tsa_o_b, &w.sca_q_w, &w.sca_q_b,
                         &w.sca_v_w, &w.sca_v_b, &w.sca_o_w, &w.sca_o_b, &w.ffn1_w, &w.ffn1_b, &w.ffn2_w, &w.ffn2_b,
                         &w.ln_g[0], &w.ln_g[1], &w.ln_g[2], &w.ln_b[0], &w.ln_b[1], &w.ln_b[2], &w.tsa_v_wh,
                         &w.tsa_q_wh, &w.tsa_o_wh, &w.sca_q_wh, &w.sca_v_wh, &w.sca_o_wh, &w.ffn1_wh, &w.ffn2_wh,
                         &w.tsa_q_wh_fold, &w.tsa_q_const, &w.tsa_q_const_t32};
        for (DevBuf* b : all) b->release();
    }
    DevBuf* all[] = {&e->rot_map, &e->split_ws, &e->tokens_split, &e->l0_x_f32, &e->l0_q_t, &e->pos_bf, &e->qc_f32, &e->qc_t, &e->qc_pos_t, &e->bev_queries, &e->pos, &e->pos_t32, &e->cams_embeds, &e->level_embeds, &e->conv_w[0], &e->conv_w[1],
                     &e->conv_b[0], &e->conv_b[1], &e->conv_wh[0], &e->conv_wh[1], &e->conv_wh_hi[0], &e->conv_wh_hi[1], &e->conv_wh_lo[0],
                     &e->conv_wh_lo[1], &e->vox_split, &e->sca_v_all_wh, &e->sca_v_all_b, &e->sca_value_all, &e->hw1, &e->hb1, &e->hw2, &e->hb2,
                     &e->fw1, &e->fb1, &e->fw2, &e->fb2, &e->head_w1h, &e->head_w2h, &e->head_b1c, &e->head_b2c, &e->tokens, &e->sca_value, &e->q_f32, &e->q_t,
                     &e->q_pos_t, &e->q0_t, &e->prev_t, &e->tsa_value, &e->tsa_value_prev, &e->qproj, &e->attn_out,
                     &e->x_f32, &e->ffn_h, &e->vox0, &e->vox1, &e->vox2, &e->hits, &e->tap_layer, &e->tap_tsa,
                     &e->tap_sca, &e->feats_dev[0], &e->feats_dev[1], &e->feats_dev[2], &e->feats_dev[3],
                     &e->occ_i64_dev, &e->flow_dev};
    for (DevBuf* b : all) b->release();
    for (auto& sl : e->slots) {
        for (auto& f : sl.feats) f.release();
        sl.occ.release(); sl.flow.release();
        if (sl.compute_done) {
            for (cudaEvent_t ev : sl.h2d_done) cudaEventDestroy(ev);
            cudaEventDestroy(sl.compute_done); cudaEventDestroy(sl.d2h_done);
        }
    }
    if (e->d2h_stream) {
        for (cudaStream_t hs : e->h2d_stream) cudaStreamDestroy(hs);
        cudaStreamDestroy(e->d2h_stream);
    }
    for (cudaEvent_t ev : e->event_pool) cudaEventDestroy(ev);
    delete e;
}

int occb200_engine_load_param(occb200_engine* e, const char* key, const float* data, int64_t numel)
{
    OCC_CHECK(e && key && data && numel >= 0, "null pointer");
    const std::string k(key);
    static const char* known_prefix[] = {"bev_embedding.", "positional_encoding.", "transformer.level_embeds",
                                         "transformer.cams_embeds", "transformer.encoder.layers.",
                                         "transformer.decoder.", "transformer.predicter.", "transformer.flow_predicter."};
    bool ok = false;
    for (const char* p : known_prefix) ok = ok || k.rfind(p, 0) == 0;
    if (!ok) { set_last_error("unknown parameter key: " + k); return 3; }
    e->host_params[k].assign(data, data + numel);
    e->finalized = false;
    e->l0_ready = false;
    return 0;
}

int occb200_engine_finalize(occb200_engine* e)
{
    OCC_CHECK(e, "null engine");
    const occb200_config& c = e->cfg;
    const int C = 256, Nq = e->Nq, F = c.ffn_dim, od = c.out_dim, mid = C / c.pillar_h;
    const bool tc = c.precision == 1 && c.use_tensor_cores;
    const bool tc32 = c.precision == 0 && c.use_tensor_cores;      // fp32 storage, split-bf16 tensor-core GEMMs
    {
        GETP(bq, "bev_embedding.weight", (size_t)Nq * C);
        if (upload(e->bev_queries, bq->data(), bq->size())) return 2;
        GETP(re, "positional_encoding.row_embed.weight", (size_t)c.bev_h * (C / 2));
        GETP(ce, "positional_encoding.col_embed.weight", (size_t)c.bev_w * (C / 2));
        DevBuf dre, dce;
        if (upload(dre, re->data(), re->size()) || upload(dce, ce->data(), ce->size())) return 2;
        if (e->pos.alloc((size_t)Nq * C * 4)) return 2;
        if (launch_bev_pos(dre.as<float>(), dce.as<float>(), c.bev_h, c.bev_w, C / 2, e->pos.as<float>(), 0)) return 2;
        if (tc) {                                                  // T32 copy of pos for the fused LayerNorm epilogue
            const size_t rows_pad = ((size_t)Nq + 127) / 128 * 128;
            if (e->pos_t32.alloc(rows_pad * C * 4)) return 2;
            OCC_CUDA(cudaMemset(e->pos_t32.p, 0, rows_pad * C * 4));
            if (launch_t32_convert(e->pos.as<float>(), e->pos_t32.as<float>(), Nq, 0, 0)) return 2;
            if (e->pos_bf.alloc((size_t)Nq * C * 2)) return 2;
            if (launch_cast<bf16>(e->pos.as<float>(), e->pos_bf.as<bf16>(), (int64_t)Nq * C, 0)) return 2;
            // bev_queries / pos are parameters: their fp32 (T32) and bf16 operand forms are frame-independent
            if (e->qc_f32.alloc(rows_pad * C * 4) || e->qc_t.alloc((size_t)Nq * C * 2) || e->qc_pos_t.alloc((size_t)Nq * C * 2))
                return 2;
            OCC_CUDA(cudaMemset(e->qc_f32.p, 0, rows_pad * C * 4));
            if (launch_prepare_query<bf16>(e->bev_queries.as<float>(), e->pos.as<float>(), (int64_t)Nq * C, e->qc_f32.as<float>(),
                                           e->qc_t.as<bf16>(), e->qc_pos_t.as<bf16>(), 1, 0)) return 2;
        }
        OCC_CUDA(cudaDeviceSynchronize());
        dre.release(); dce.release();
        GETP(le, "transformer.level_embeds", (size_t)c.num_levels * C);
        GETP(cm, "transformer.cams_embeds", (size_t)c.num_cams * C);
        std::vector<float> cams(*cm);
        if (!c.use_cams_embeds) std::fill(cams.begin(), cams.end(), 0.f);    // transformer_occ.py:214-215: added only if set
        if (upload(e->level_embeds, le->data(), le->size()) || upload(e->cams_embeds, cams.data(), cams.size())) return 2;
    }
    for (int l = 0; l < c.num_layers; ++l) {
        LayerW& w = e->layers[l];
        const std::string pre = "transformer.encoder.layers." + std::to_string(l);
        const std::string a0 = pre + ".attentions.0", a1 = pre + ".attentions.1", d = a1 + ".deformable_attention";
        auto up = [&](DevBuf& wbuf, DevBuf& bbuf, DevBuf* wh, const std::string& name, size_t n, size_t k) -> int {
            const std::vector<float>* W = find(e, name + ".weight", n * k);
            const std::vector<float>* B = find(e, name + ".bias", n);
            if (!W || !B) return 3;
            if (upload(wbuf, W->data(), W->size()) || upload(bbuf, B->data(), B->size())) return 2;
            if (tc && wh && upload_bf16(*wh, W->data(), W->size())) return 2;
            if (tc32 && wh && upload_w3(*wh, W->data(), n, k)) return 2;
            return 0;
        };
        auto up_cat = [&](DevBuf& wbuf, DevBuf& bbuf, DevBuf* wh, const std::string& n1, const std::string& n2,
                          size_t r1, size_t r2, size_t k, DevBuf* fold = nullptr, DevBuf* fold_const = nullptr) -> int {
            const std::vector<float>* W1 = find(e, n1 + ".weight", r1 * k);
            const std::vector<float>* B1 = find(e, n1 + ".bias", r1);
            const std::vector<float>* W2 = find(e, n2 + ".weight", r2 * k);
            const std::vector<float>* B2 = find(e, n2 + ".bias", r2);
            if (!W1 || !B1 || !W2 || !B2) return 3;
            std::vector<float> W(*W1), B(*B1);
            W.insert(W.end(), W2->begin(), W2->end());
            B.insert(B.end(), B2->begin(), B2->end());
            if (upload(wbuf, W.data(), W.size()) || upload(bbuf, B.data(), B.size())) return 2;
            if (tc && wh && upload_bf16(*wh, W.data(), W.size())) return 2;
            if (tc32 && wh && upload_w3(*wh, W.data(), r1 + r2, k)) return 2;
            if (tc && fold) {                                    // k = 2C: (W1 + W2) [r, C] bf16 and the constant W2 pos + b
                const size_t half = k / 2, rows = r1 + r2;
                std::vector<float> Wf(rows * half), W2h(rows * half);
                for (size_t r = 0; r < rows; ++r)
                    for (size_t j = 0; j < half; ++j) {
                        Wf[r * half + j] = W[r * k + j] + W[r * k + half + j];
                        W2h[r * half + j] = W[r * k + half + j];
                    }
                if (upload_bf16(*fold, Wf.data(), Wf.size())) return 2;
                DevBuf w2;
                if (upload(w2, W2h.data(), W2h.size())) return 2;
                if (fold_const->alloc((size_t)Nq * rows * 4)) return 2;
                if (gemm_simt<float, float>(e->pos.as<float>(), (int)half, nullptr, 0, (int)half, w2.as<float>(), bbuf.as<float>(),
                                            nullptr, (int)rows, fold_const->as<float>(), (int)rows, Nq, (int)rows, (int)half,
                                            ACT_NONE, 0)) return 2;
                // the same constant in the T32 block layout (rows padded to 32) for the TMA-store epilogue of the merged launch
                if (rows % 32 == 0) {
                    const size_t rows_pad = ((size_t)Nq + 31) / 32 * 32;
                    if (w.tsa_q_const_t32.alloc(rows_pad * rows * 4)) return 2;
                    OCC_CUDA(cudaMemset(w.tsa_q_const_t32.p, 0, rows_pad * rows * 4));
                    if (launch_t32_convert(fold_const->as<float>(), w.tsa_q_const_t32.as<float>(), Nq, 0, 0, (int)rows)) return 2;
                }
                OCC_CUDA(cudaDeviceSynchronize());
                w2.release();
            }
            return 0;
        };
        int rc;
        const size_t tq_off = 2 * 8 * c.tsa_points * 2, tq_w = 2 * 8 * c.tsa_points;
        const size_t sq_off = 8 * c.num_levels * c.sca_points * 2, sq_w = 8 * c.num_levels * c.sca_points;
        if ((rc = up(w.tsa_v_w, w.tsa_v_b, &w.tsa_v_wh, a0 + ".value_proj", C, C))) return rc;
        if ((rc = up_cat(w.tsa_q_w, w.tsa_q_b, &w.tsa_q_wh, a0 + ".sampling_offsets", a0 + ".attention_weights", tq_off,
                         tq_w, 2 * C, &w.tsa_q_wh_fold, &w.tsa_q_const))) return rc;
        if ((rc = up(w.tsa_o_w, w.tsa_o_b, &w.tsa_o_wh, a0 + ".output_proj", C, C))) return rc;
        if ((rc = up_cat(w.sca_q_w, w.sca_q_b, &w.sca_q_wh, d + ".sampling_offsets", d + ".attention_weights", sq_off,
                         sq_w, C))) return rc;
        if ((rc = up(w.sca_v_w, w.sca_v_b, &w.sca_v_wh, d + ".value_proj", C, C))) return rc;
        if ((rc = up(w.sca_o_w, w.sca_o_b, &w.sca_o_wh, a1 + ".output_proj", C, C))) return rc;
        if ((rc = up(w.ffn1_w, w.ffn1_b, &w.ffn1_wh, pre + ".ffns.0.layers.0.0", F, C))) return rc;
        if ((rc = up(w.ffn2_w, w.ffn2_b, &w.ffn2_wh, pre + ".ffns.0.layers.1", C, F))) return rc;
        for (int n = 0; n < 3; ++n) {
            GETP(g, pre + ".norms." + std::to_string(n) + ".weight", (size_t)C);
            GETP(b, pre + ".norms." + std::to_string(n) + ".bias", (size_t)C);
            if (upload(w.ln_g[n], g->data(), C) || upload(w.ln_b[n], b->data(), C)) return 2;
        }
    }
    if (tc) {
        // SpatialCrossAttention's value_proj input (the camera tokens) does not depend on the layer
        // (spatial_cross_attention.py:334): project once with all layers' weights, [L*256, 256].
        std::vector<float> W, B;
        for (int l = 0; l < c.num_layers; ++l) {
            const std::string d = "transformer.encoder.layers." + std::to_string(l) + ".attentions.1.deformable_attention.value_proj";
            const std::vector<float>* w = find(e, d + ".weight", (size_t)C * C);
            const std::vector<float>* b = find(e, d + ".bias", (size_t)C);
            if (!w || !b) return 3;
            W.insert(W.end(), w->begin(), w->end());
            B.insert(B.end(), b->begin(), b->end());
        }
        if (upload_bf16(e->sca_v_all_wh, W.data(), W.size()) || upload(e->sca_v_all_b, B.data(), B.size())) return 2;
        if (e->sca_value_all.alloc((size_t)c.num_layers * c.num_cams * e->Nv * C * 2)) return 2;
        OCC_CUDA(cudaMemset(e->sca_value_all.p, 0, e->sca_value_all.bytes));
    }
    // decoder: fold BatchNorm3d (eval) into the conv weights; torch layout [Cout][Cin][kz][ky][kx] -> [tap][Cin][Cout]
    for (int i = 0; i < 2; ++i) {
        const int cin = i == 0 ? mid : od;
        const std::string pre = "transformer.decoder." + std::to_string(i);
        GETP(W, pre + ".conv.weight", (size_t)od * cin * 27);
        GETP(g, pre + ".bn.weight", (size_t)od);
        GETP(b, pre + ".bn.bias", (size_t)od);
        GETP(m, pre + ".bn.running_mean", (size_t)od);
        GETP(v, pre + ".bn.running_var", (size_t)od);
        std::vector<float> wf((size_t)27 * cin * od), bf(od);
        for (int co = 0; co < od; ++co) {
            const float s = (*g)[co] / sqrtf((*v)[co] + 1e-5f);
            bf[co] = (*b)[co] - (*m)[co] * s;
            for (int ci = 0; ci < cin; ++ci)
                for (int t = 0; t < 27; ++t)
                    wf[((size_t)t * cin + ci) * od + co] = (*W)[((size_t)co * cin + ci) * 27 + t] * s;
        }
        if (upload(e->conv_w[i], wf.data(), wf.size()) || upload(e->conv_b[i], bf.data(), bf.size())) return 2;
        if (tc) {                                             // tensor-core layout: [tap][cout][cin], K-major rows
            std::vector<float> wt((size_t)27 * od * cin);
            for (int t = 0; t < 27; ++t)
                for (int co = 0; co < od; ++co)
                    for (int ci = 0; ci < cin; ++ci)
                        wt[((size_t)t * od + co) * cin + ci] = wf[((size_t)t * cin + ci) * od + co];
            if (upload_bf16(e->conv_wh[i], wt.data(), wt.size())) return 2;
        }
        if (tc32 && c.pillar_h == 16) {                       // same layout, split into bf16 hi + lo (3-pass fp32-grade convolution)
            std::vector<float> hi((size_t)27 * od * cin), lo(hi.size());
            for (int t = 0; t < 27; ++t)
                for (int co = 0; co < od; ++co)
                    for (int ci = 0; ci < cin; ++ci) {
                        const float w = wf[((size_t)t * cin + ci) * od + co];
                        const float h = __bfloat162float(__float2bfloat16(w));
                        hi[((size_t)t * od + co) * cin + ci] = h;
                        lo[((size_t)t * od + co) * cin + ci] = w - h;
                    }
            if (upload_bf16(e->conv_wh_hi[i], hi.data(), hi.size()) || upload_bf16(e->conv_wh_lo[i], lo.data(), lo.size())) return 2;
        }
    }
    {
        GETP(w1, "transformer.predicter.0.weight", (size_t)2 * od * od);
        GETP(b1, "transformer.predicter.0.bias", (size_t)2 * od);
        GETP(w2, "transformer.predicter.2.weight", (size_t)c.num_classes * 2 * od);
        GETP(b2, "transformer.predicter.2.bias", (size_t)c.num_classes);
        GETP(f1, "transformer.flow_predicter.0.weight", (size_t)2 * od * od);
        GETP(g1, "transformer.flow_predicter.0.bias", (size_t)2 * od);
        GETP(f2, "transformer.flow_predicter.2.weight", (size_t)2 * 2 * od);
        GETP(g2, "transformer.flow_predicter.2.bias", (size_t)2);
        if (upload(e->hw1, w1->data(), w1->size()) || upload(e->hb1, b1->data(), b1->size()) ||
            upload(e->hw2, w2->data(), w2->size()) || upload(e->hb2, b2->data(), b2->size()) ||
            upload(e->fw1, f1->data(), f1->size()) || upload(e->fb1, g1->data(), g1->size()) ||
            upload(e->fw2, f2->data(), f2->size()) || upload(e->fb2, g2->data(), g2->size())) return 2;
        if (tc && od == 32 && c.num_classes + 2 <= 19) {          // tensor-core head: concatenated / block-diagonal weights
            const int H = 2 * od, nc = c.num_classes;
            std::vector<float> w1c((size_t)2 * H * od), b1c(2 * H), w2c((size_t)32 * 2 * H, 0.f), b2c(nc + 2);
            for (int i = 0; i < H * od; ++i) { w1c[i] = (*w1)[i]; w1c[(size_t)H * od + i] = (*f1)[i]; }
            for (int i = 0; i < H; ++i) { b1c[i] = (*b1)[i]; b1c[H + i] = (*g1)[i]; }
            for (int r = 0; r < nc; ++r)
                for (int k = 0; k < H; ++k) w2c[(size_t)r * 2 * H + k] = (*w2)[(size_t)r * H + k];
            for (int r = 0; r < 2; ++r)
                for (int k = 0; k < H; ++k) w2c[(size_t)(nc + r) * 2 * H + H + k] = (*f2)[(size_t)r * H + k];
            for (int i = 0; i < nc; ++i) b2c[i] = (*b2)[i];
            b2c[nc] = (*g2)[0]; b2c[nc + 1] = (*g2)[1];
            if (upload_bf16(e->head_w1h, w1c.data(), w1c.size()) || upload_bf16(e->head_w2h, w2c.data(), w2c.size()) ||
                upload(e->head_b1c, b1c.data(), b1c.size()) || upload(e->head_b2c, b2c.data(), b2c.size())) return 2;
        }
    }
    // workspace
    const size_t es = e->elt();
    const size_t nvox = (size_t)c.bev_w * c.bev_h * c.pillar_h;
    const size_t ntok = (size_t)c.num_cams * e->Nv;
    int maxq = 8 * c.num_levels * c.sca_points * 3;
    const size_t nq_pad = ((size_t)Nq + 127) / 128 * 128;
    if (e->tokens.alloc(ntok * C * es) || e->sca_value.alloc(ntok * C * es) || e->q_f32.alloc(nq_pad * C * 4) ||
        e->q_t.alloc((size_t)Nq * C * es) || e->q_pos_t.alloc((size_t)Nq * C * es) || e->q0_t.alloc((size_t)Nq * C * es) ||
        e->prev_t.alloc((size_t)Nq * C * es) || e->tsa_value.alloc((size_t)Nq * C * es) ||
        e->tsa_value_prev.alloc((size_t)Nq * C * es) || e->qproj.alloc((size_t)Nq * maxq * 4) ||
        e->attn_out.alloc((size_t)Nq * C * es) || e->x_f32.alloc(nq_pad * C * 4) ||
        e->ffn_h.alloc((size_t)Nq * F * es) || e->vox0.alloc(nvox * mid * es) || e->vox1.alloc(nvox * od * es) ||
        e->vox2.alloc(nvox * od * es) || e->hits.alloc(Nq)) return 2;
    OCC_CUDA(cudaMemset(e->q_f32.p, 0, nq_pad * C * 4));
    OCC_CUDA(cudaMemset(e->x_f32.p, 0, nq_pad * C * 4));
    if (tc32) {
        const size_t kmax = (size_t)std::max(2 * C, F);
        if (e->split_ws.alloc((size_t)Nq * 2 * kmax * 2) || e->tokens_split.alloc(ntok * 2 * C * 2)) return 2;
        if (c.pillar_h == 16 && e->vox_split.alloc(nvox * 2 * od * 2)) return 2;
    }
    e->host_params.clear();
    e->l0_ready = false;
    if (tc && e->qc_f32.p != nullptr && getenv("OCC_NO_L0_FOLD") == nullptr) {
        // Layer 0's TemporalSelfAttention (value_proj, query projection over [bev_queries | pos], gather, output_proj) and
        // its LayerNorm depend on parameters only when prev_bev is None: run the frame path's own kernels once, here.
        const size_t rows_pad = ((size_t)Nq + 127) / 128 * 128;
        if (e->l0_x_f32.alloc(rows_pad * C * 4) || e->l0_q_t.alloc((size_t)Nq * C * 2)) return 2;
        OCC_CUDA(cudaMemset(e->l0_x_f32.p, 0, rows_pad * C * 4));
        const bool taps = e->taps;
        e->taps = false;
        const int rc = forward_impl<bf16>(e, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0, MODE_L0_TSA_ONLY);
        e->taps = taps;
        if (rc) return rc;
        OCC_CUDA(cudaDeviceSynchronize());
        e->l0_ready = true;
    }
    e->finalized = true;
    return 0;
}

int occb200_engine_set_cameras(occb200_engine* e, const float* cam_mat, const float* zs, int img_h, int img_w)
{
    OCC_CHECK(e && cam_mat && zs, "null pointer");
    const occb200_config& c = e->cfg;
    memset(&e->sp, 0, sizeof(e->sp));
    for (int i = 0; i < c.num_cams; ++i)
        for (int k = 0; k < 16; ++k) e->sp.cam_mat[i][k] = cam_mat[i * 16 + k];
    for (int i = 0; i < c.num_points_in_pillar; ++i) e->sp.zs[i] = zs[i];
    for (int i = 0; i < 3; ++i) {
        e->sp.pc_scale[i] = (float)((double)c.pc_range[3 + i] - (double)c.pc_range[i]);
        e->sp.pc_min[i] = c.pc_range[i];
    }
    e->sp.img_w = (float)img_w; e->sp.img_h = (float)img_h;
    e->sp.num_cams = c.num_cams; e->sp.D = c.num_points_in_pillar; e->sp.bev_h = c.bev_h; e->sp.bev_w = c.bev_w;
    e->cameras_set = true;
    return 0;
}

int occb200_engine_forward(occb200_engine* e, const float* const* feats, const float* prev_bev, float* bev_embed,
                           float* occ_logits, float* flow, uint8_t* occ_cls_u8, int64_t* occ_cls_i64, void* stream)
{
    OCC_CHECK(e && feats, "null pointer");
    OCC_CHECK(e->finalized, "engine_finalize() has not been called");
    OCC_CHECK(e->cameras_set, "engine_set_cameras() has not been called");
    for (int l = 0; l < e->cfg.num_levels; ++l) OCC_CHECK(feats[l] != nullptr, "null feature level");
    cudaStream_t st = (cudaStream_t)stream;
    if (e->cfg.precision == 0)
        return forward_impl<float>(e, feats, prev_bev, bev_embed, occ_logits, flow, occ_cls_u8, occ_cls_i64, st);
    return forward_impl<bf16>(e, feats, prev_bev, bev_embed, occ_logits, flow, occ_cls_u8, occ_cls_i64, st);
}

int occb200_engine_forward_host(occb200_engine* e, const float* const* feats_host, int64_t* occ_cls_i64_host,
                                float* flow_host, void* stream)
{
    OCC_CHECK(e && feats_host && occ_cls_i64_host && flow_host, "null pointer");
    OCC_CHECK(e->finalized && e->cameras_set, "engine not finalized / cameras not set");
    const occb200_config& c = e->cfg;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t nvox = (size_t)c.bev_w * c.bev_h * c.pillar_h;
    const float* dev_feats[4];
    for (int l = 0; l < 4; ++l) {
        const size_t n = (size_t)c.num_cams * 256 * e->lg.h[l] * e->lg.w[l] * (e->feats_bf16 ? 2 : 4);
        if (e->feats_dev[l].bytes != n && e->feats_dev[l].alloc(n)) return 2;
        OCC_CUDA(cudaMemcpyAsync(e->feats_dev[l].p, feats_host[l], n, cudaMemcpyHostToDevice, st));
        dev_feats[l] = e->feats_dev[l].as<float>();
    }
    if (e->occ_i64_dev.bytes != nvox * 8 && e->occ_i64_dev.alloc(nvox * 8)) return 2;
    if (e->flow_dev.bytes != nvox * 8 && e->flow_dev.alloc(nvox * 8)) return 2;
    int rc = occb200_engine_forward(e, dev_feats, nullptr, nullptr, nullptr, e->flow_dev.as<float>(), nullptr,
                                    e->occ_i64_dev.as<int64_t>(), stream);
    if (rc) return rc;
    OCC_CUDA(cudaMemcpyAsync(occ_cls_i64_host, e->occ_i64_dev.p, nvox * 8, cudaMemcpyDeviceToHost, st));
    OCC_CUDA(cudaMemcpyAsync(flow_host, e->flow_dev.p, nvox * 8, cudaMemcpyDeviceToHost, st));
    OCC_CUDA(cudaStreamSynchronize(st));
    return 0;
}

int occb200_engine_submit_host(occb200_engine* e, int slot, const float* const* feats_host, int64_t* occ_cls_i64_host,
                               float* flow_host, void* stream)
{
    OCC_CHECK(e && feats_host && occ_cls_i64_host && flow_host, "null pointer");
    OCC_CHECK(slot == 0 || slot == 1, "slot must be 0 or 1");
    OCC_CHECK(e->finalized && e->cameras_set, "engine not finalized / cameras not set");
    const occb200_config& c = e->cfg;
    cudaStream_t st = (cudaStream_t)stream;
    occb200_engine::Slot& s = e->slots[slot];
    OCC_CHECK(!s.busy, "slot still in flight: call occb200_engine_wait_host first");
    if (!e->d2h_stream) {
        for (cudaStream_t& hs : e->h2d_stream) OCC_CUDA(cudaStreamCreateWithFlags(&hs, cudaStreamNonBlocking));
        OCC_CUDA(cudaStreamCreateWithFlags(&e->d2h_stream, cudaStreamNonBlocking));
    }
    if (!s.compute_done) {
        for (cudaEvent_t& ev : s.h2d_done) OCC_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        OCC_CUDA(cudaEventCreateWithFlags(&s.compute_done, cudaEventDisableTiming));
        OCC_CUDA(cudaEventCreateWithFlags(&s.d2h_done, cudaEventDisableTiming));
    }
    // Levels larger than 32 MB go up in `nsplit` pieces on separate copy streams: one cudaMemcpyAsync stream reached
    // 46 GB/s of the PCIe link on the test box, two reach 50 GB/s (OCC_H2D_SPLIT = 1..4, default 2).
    static const int nsplit = [] {
        const char* v = getenv("OCC_H2D_SPLIT");
        const int n = v ? atoi(v) : 2;
        return n < 1 ? 1 : (n > 4 ? 4 : n);
    }();
    const size_t nvox = (size_t)c.bev_w * c.bev_h * c.pillar_h;
    const float* dev_feats[4];
    for (int l = 0; l < 4; ++l) {
        const size_t n = (size_t)c.num_cams * 256 * e->lg.h[l] * e->lg.w[l] * (e->feats_bf16 ? 2 : 4);
        if (s.feats[l].bytes != n && s.feats[l].alloc(n)) return 2;
        const int pieces = n >= (32u << 20) ? nsplit : 1;
        const size_t chunk = ((n / pieces) + 255) & ~(size_t)255;
        for (int i = 0; i < pieces; ++i) {
            const size_t o = (size_t)i * chunk, len = o >= n ? 0 : (n - o < chunk ? n - o : chunk);
            if (len) OCC_CUDA(cudaMemcpyAsync((char*)s.feats[l].p + o, (const char*)feats_host[l] + o, len,
                                              cudaMemcpyHostToDevice, e->h2d_stream[i]));
        }
        dev_feats[l] = s.feats[l].as<float>();
    }
    for (int i = 0; i < nsplit; ++i) {                              // compute waits for this frame's features only
        OCC_CUDA(cudaEventRecord(s.h2d_done[i], e->h2d_stream[i]));
        OCC_CUDA(cudaStreamWaitEvent(st, s.h2d_done[i], 0));
    }
    if (s.occ.bytes != nvox * 8 && s.occ.alloc(nvox * 8)) return 2;
    if (s.flow.bytes != nvox * 8 && s.flow.alloc(nvox * 8)) return 2;
    int rc = occb200_engine_forward(e, dev_feats, nullptr, nullptr, nullptr, s.flow.as<float>(), nullptr,
                                    s.occ.as<int64_t>(), stream);
    if (rc) return rc;
    OCC_CUDA(cudaEventRecord(s.compute_done, st));
    OCC_CUDA(cudaStreamWaitEvent(e->d2h_stream, s.compute_done, 0));
    OCC_CUDA(cudaMemcpyAsync(occ_cls_i64_host, s.occ.p, nvox * 8, cudaMemcpyDeviceToHost, e->d2h_stream));
    OCC_CUDA(cudaMemcpyAsync(flow_host, s.flow.p, nvox * 8, cudaMemcpyDeviceToHost, e->d2h_stream));
    OCC_CUDA(cudaEventRecord(s.d2h_done, e->d2h_stream));
    s.busy = true;
    return 0;
}

int occb200_engine_wait_host(occb200_engine* e, int slot)
{
    OCC_CHECK(e && (slot == 0 || slot == 1), "bad arguments");
    occb200_engine::Slot& s = e->slots[slot];
    if (!s.busy) return 0;
    OCC_CUDA(cudaEventSynchronize(s.d2h_done));
    s.busy = false;
    return 0;
}

int occb200_engine_set_prev_rotation(occb200_engine* e, const int32_t* map_host)
{
    OCC_CHECK(e, "null engine");
    if (map_host == nullptr) { e->rot_set = false; return 0; }
    for (int q = 0; q < e->Nq; ++q) OCC_CHECK(map_host[q] >= -1 && map_host[q] < e->Nq, "rotation map entry out of range");
    if (e->rot_map.bytes != (size_t)e->Nq * 4 && e->rot_map.alloc((size_t)e->Nq * 4)) return 2;
    OCC_CUDA(cudaMemcpy(e->rot_map.p, map_host, (size_t)e->Nq * 4, cudaMemcpyHostToDevice));
    e->rot_set = true;
    return 0;
}

int occb200_engine_set_input_dtype(occb200_engine* e, int feats_bf16)
{
    OCC_CHECK(e && feats_bf16 >= 0 && feats_bf16 <= 2, "input dtype must be 0 (fp32 NCHW), 1 (bf16 NCHW) or 2 (bf16 NHWC)");
    e->feats_bf16 = feats_bf16;
    return 0;
}

int occb200_engine_enable_taps(occb200_engine* e, int enable)
{
    OCC_CHECK(e && e->finalized, "engine not finalized");
    e->taps = enable != 0;
    if (e->taps) {
        const size_t n = (size_t)e->cfg.num_layers * e->Nq * 256 * 4;
        if (e->tap_layer.alloc(n) || e->tap_tsa.alloc(n) || e->tap_sca.alloc(n)) return 2;
    }
    return 0;
}

int occb200_engine_copy_tap(occb200_engine* e, int which, int layer, float* dst, void* stream)
{
    OCC_CHECK(e && dst, "null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t n = (size_t)e->Nq * 256;
    if (which >= 0 && which <= 2) {
        OCC_CHECK(e->taps && layer >= 0 && layer < e->cfg.num_layers, "taps not enabled or bad layer");
        const DevBuf& b = which == 0 ? e->tap_layer : (which == 1 ? e->tap_tsa : e->tap_sca);
        OCC_CUDA(cudaMemcpyAsync(dst, b.as<float>() + layer * n, n * 4, cudaMemcpyDeviceToDevice, st));
        return 0;
    }
    if (which == 3) {
        const size_t nv = (size_t)e->cfg.bev_w * e->cfg.bev_h * e->cfg.pillar_h * e->cfg.out_dim;
        if (e->cfg.precision == 0) {
            OCC_CUDA(cudaMemcpyAsync(dst, e->vox2.p, nv * 4, cudaMemcpyDeviceToDevice, st));
            return 0;
        }
        return launch_bf16_to_f32(e->vox2.as<bf16>(), dst, (int64_t)nv, st);
    }
    if (which == 4) {                                            // packed camera tokens [num_cams, Nv, C] (row a9)
        const size_t nt = (size_t)e->cfg.num_cams * e->Nv * 256;
        if (e->cfg.precision == 0) {
            OCC_CUDA(cudaMemcpyAsync(dst, e->tokens.p, nt * 4, cudaMemcpyDeviceToDevice, st));
            return 0;
        }
        return launch_bf16_to_f32(e->tokens.as<bf16>(), dst, (int64_t)nt, st);
    }
    set_last_error("unknown tap");
    return 1;
}

int occb200_engine_project_pillars(occb200_engine* e, float* ref_cam, uint8_t* mask, void* stream)
{
    OCC_CHECK(e && ref_cam && mask && e->cameras_set, "null pointer / cameras not set");
    return launch_project_pillars(e->sp, ref_cam, mask, (cudaStream_t)stream);
}

int occb200_engine_launches_per_frame(const occb200_engine* e) { return e ? e->launches : 0; }

int occb200_engine_profile(occb200_engine* e, int enable)
{
    OCC_CHECK(e, "null engine");
    e->profiling = enable != 0;
    e->prof_events.clear();
    e->event_used = 0;
    return 0;
}

int occb200_engine_profile_read(occb200_engine* e, float* ms_per_category, int* launches_per_category, int n)
{
    OCC_CHECK(e && ms_per_category && launches_per_category && n >= CAT_COUNT, "bad arguments");
    OCC_CUDA(cudaDeviceSynchronize());
    for (int i = 0; i < n; ++i) { ms_per_category[i] = 0.f; launches_per_category[i] = 0; }
    for (auto& pe : e->prof_events) {
        float ms = 0.f;
        OCC_CUDA(cudaEventElapsedTime(&ms, pe.second.first, pe.second.second));
        ms_per_category[pe.first] += ms;
        launches_per_category[pe.first] += 1;
    }
    e->prof_events.clear();
    e->event_used = 0;
    return 0;
}

int occb200_render_forward(const float* sigma, const float* origin, const float* points, const float* tindex, int N,
                           int T, int Z, int Y, int X, int64_t M, float* pred_dist, float* gt_dist, float* coord_index,
                           void* stream)
{
    OCC_CHECK(sigma && origin && points && tindex && pred_dist && gt_dist && coord_index, "null pointer");
    return launch_render_forward(sigma, origin, points, tindex, N, T, Z, Y, X, M, pred_dist, gt_dist, coord_index,
                                 (cudaStream_t)stream);
}

int occb200_ray_metric_accumulate(const uint8_t* sem_pred, const float* flow_pred, const uint8_t* sem_gt,
                                  const float* flow_gt, const void* origins, int origin_is_f64, int T, const float* rays,
                                  int M, double* counters, float* pcd_pred, float* pcd_gt, void* stream)
{
    if (T == 0 || M == 0) return 0;                              // no origins / rays: counters untouched
    OCC_CHECK(sem_pred && flow_pred && sem_gt && flow_gt && origins && rays && counters, "null pointer");
    return launch_ray_metric(sem_pred, flow_pred, sem_gt, flow_gt, origins, origin_is_f64, T, rays, M, counters,
                             pcd_pred, pcd_gt, (cudaStream_t)stream);
}

int occb200_linear_f32(const float* A, const float* W, const float* bias, const float* residual, float* C, int M, int N,
                       int K, int act, void* stream)
{
    OCC_CHECK(A && W && C, "null pointer");
    return gemm_simt<float, float>(A, K, nullptr, 0, K, W, bias, residual, N, C, N, M, N, K, act, (cudaStream_t)stream);
}

int occb200_layernorm_f32(const float* x, const float* gamma, const float* beta, float* y, int rows, int C, void* stream)
{
    OCC_CHECK(x && gamma && beta && y, "null pointer");
    return launch_layernorm<float>(x, gamma, beta, nullptr, rows, C, y, (float*)nullptr, (float*)nullptr,
                                   (cudaStream_t)stream);
}

int occb200_gemm_bf16_tc(const void* A, const void* W, const float* bias, float* C, int M, int N, int K, void* stream)
{
    OCC_CHECK(A && W && C, "null pointer");
    OCC_CHECK(gemm_tc_supported(M, N, K, K), "shape not supported by the tcgen05 GEMM");
    return gemm_tc<float>(reinterpret_cast<const bf16*>(A), nullptr, 0, reinterpret_cast<const bf16*>(W), bias, nullptr,
                          C, M, N, K, ACT_NONE, (cudaStream_t)stream);
}

}  // extern "C"
