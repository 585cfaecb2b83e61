// Multi-scale deformable attention for sm_100a: the operator-boundary kernel (mmcv `_ext` ABI
// semantics) and the two fused BEVFormer variants.
//
//   msda_forward_kernel  <- mmcv._ext.ms_deform_attn_forward, called from
//        bevformer/modules/multi_scale_deformable_attn_function.py:118-124
//   tsa_fused_kernel     <- TemporalSelfAttention.forward, temporal_self_attention.py:206-262
//        (softmax over points, sampling locations, gather, mean over the BEV queue)
//   sca_fused_kernel     <- BEVFormerEncoder.point_sampling (encoder.py:92-151) +
//        SpatialCrossAttention.forward (spatial_cross_attention.py:128-172) +
//        MSDeformableAttention3D.forward (:338-393): camera projection of the pillar points,
//        visibility, softmax, Z-anchor interleave, gather, cross-camera sum and /count --
//        without the reference's nonzero() host sync, rebatch copies and scatter loops.
//
// Mapping (all fused kernels): one warp per BEV query; lane = (head = lane/4, slice = lane%4);
// a lane accumulates 8 of the head's 32 channels, so one warp-wide 128-bit load instruction
// fetches 8 independent 64-byte (bf16) corner rows.  Per-sample scalars (location, weight) are
// prepared by one owner lane per (head, level).
//   sca_fused_kernel (fp32 parity path) / tsa_fused_kernel (both value types): the owner's packed
//        sample is broadcast inside the 4-lane group with shuffles.
//   sca_pipe_kernel (bf16 production path): the owners write 16-byte sample descriptors to shared
//        memory; the gather loop reads them with one broadcast LDS.128 per sample and issues the
//        loads of sample i+1 before the FMAs of sample i.  4 warps per CTA, 6 CTAs per SM.
// Sampling offsets / logits arrive as fp32 or (tensor-core path) fp16.
// Measured bound (ncu, profiles/README.md): the L1 data path -- every 128-bit warp load touches 6-8
// different 128-byte lines and replays once per line -- not HBM (11 % dram) or instruction issue (50 %).
#include <cuda_fp16.h>

#include "common.cuh"
#include "kernels.cuh"

namespace occ {

namespace {

// bilinear gather of 8 channels with zero padding; `base` points at (level start, head, slice),
// consecutive pixels are `pix_stride` elements apart.  Same validity rules as the mmcv kernel.
template <typename T>
__device__ __forceinline__ void bilinear_acc8(const T* __restrict__ base, int H, int W, int pix_stride,
                                              float h_im, float w_im, float wt, float (&acc)[8])
{
    if (!(h_im > -1.f && w_im > -1.f && h_im < (float)H && w_im < (float)W)) return;
    const int h_lo = (int)floorf(h_im), w_lo = (int)floorf(w_im);
    const float lh = h_im - (float)h_lo, lw = w_im - (float)w_lo;
    const float hh = 1.f - lh, hw = 1.f - lw;
    const bool top = h_lo >= 0, bot = h_lo + 1 <= H - 1, lef = w_lo >= 0, rig = w_lo + 1 <= W - 1;
    const T* p = base + ((int64_t)h_lo * W + w_lo) * pix_stride;
    float v1[8], v2[8], v3[8], v4[8];
    const bool b1 = top && lef, b2 = top && rig, b3 = bot && lef, b4 = bot && rig;
    if (b1) load8(p, v1);
    if (b2) load8(p + pix_stride, v2);
    if (b3) load8(p + (int64_t)W * pix_stride, v3);
    if (b4) load8(p + (int64_t)(W + 1) * pix_stride, v4);
    const float w1 = b1 ? wt * (hh * hw) : 0.f, w2 = b2 ? wt * (hh * lw) : 0.f;
    const float w3 = b3 ? wt * (lh * hw) : 0.f, w4 = b4 ? wt * (lh * lw) : 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        float a = acc[i];
        if (b1) a = fmaf(w1, v1[i], a);
        if (b2) a = fmaf(w2, v2[i], a);
        if (b3) a = fmaf(w3, v3[i], a);
        if (b4) a = fmaf(w4, v4[i], a);
        acc[i] = a;
    }
}

// ---- fused-kernel sample pipeline: the owner lane of a (head, level) turns one sampling location into a
// packed descriptor (clamped pixel offset + which neighbours exist) and four pre-multiplied corner weights;
// the four lanes of the head then gather their 8 channels with unconditional, in-bounds 128-bit loads.
struct SamplePrep { int code; float c1, c2, c3, c4; };
constexpr int CODE_VALID = 1 << 30, CODE_OFF_MASK = CODE_VALID - 1;

// The 2x2 block that is fetched always starts at a pixel clamped to [0,H-2] x [0,W-2], so its four addresses are
// base, base+1 pixel, base+1 row, base+1 row+1 pixel with CONSTANT strides (no per-sample border flags, no branches).
// The bilinear corner weights are assigned to the positions of that block that coincide with in-bounds true corners
// (zero padding for the others); for interior samples this is exactly the usual (hh*hw, hh*lw, lh*hw, lh*lw).
__device__ __forceinline__ SamplePrep prep_sample(float h_im, float w_im, float wt, int H, int W, int base_pix = 0)
{
    SamplePrep s;
    const bool valid = h_im > -1.f && w_im > -1.f && h_im < (float)H && w_im < (float)W;   // mmcv kernel's test
    const float hf = valid ? floorf(h_im) : 0.f, wf = valid ? floorf(w_im) : 0.f;
    const int h_lo = (int)hf, w_lo = (int)wf;
    const float lh = h_im - hf, lw = w_im - wf, hh = 1.f - lh, hw = 1.f - lw;
    const int hb = min(max(h_lo, 0), H - 2), wb = min(max(w_lo, 0), W - 2);
    const float rw0 = (h_lo == hb) ? hh : ((h_lo + 1 == hb) ? lh : 0.f);
    const float rw1 = (h_lo == hb + 1) ? hh : ((h_lo == hb) ? lh : 0.f);
    const float cw0 = (w_lo == wb) ? hw : ((w_lo + 1 == wb) ? lw : 0.f);
    const float cw1 = (w_lo == wb + 1) ? hw : ((w_lo == wb) ? lw : 0.f);
    const float g = valid ? wt : 0.f;
    s.c1 = g * (rw0 * cw0); s.c2 = g * (rw0 * cw1); s.c3 = g * (rw1 * cw0); s.c4 = g * (rw1 * cw1);
    s.code = (base_pix + hb * W + wb) | (valid ? CODE_VALID : 0);
    return s;
}

// acc(2 lanes) += a * w using the packed fp32x2 FMA of sm_100
__device__ __forceinline__ void ffma2(float2& acc, float a0, float a1, float w)
{
    unsigned long long d = *reinterpret_cast<unsigned long long*>(&acc);
    const float2 av = make_float2(a0, a1), wv = make_float2(w, w);
    asm("fma.rn.f32x2 %0, %1, %2, %0;"
        : "+l"(d)
        : "l"(*reinterpret_cast<const unsigned long long*>(&av)), "l"(*reinterpret_cast<const unsigned long long*>(&wv)));
    acc = *reinterpret_cast<float2*>(&d);
}

template <typename T>
__device__ __forceinline__ void gather_sample(const T* __restrict__ base, int W, int code, float c1, float c2, float c3,
                                              float c4, float2 (&acc)[4])
{
    if (!(code & CODE_VALID)) return;                            // sample outside the map: contributes nothing
    const T* p = base + (int64_t)(code & CODE_OFF_MASK) * 256;
    float v1[8], v2[8], v3[8], v4[8];
    load8(p, v1); load8(p + 256, v2); load8(p + (int64_t)W * 256, v3); load8(p + (int64_t)W * 256 + 256, v4);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        ffma2(acc[i], v1[2 * i], v1[2 * i + 1], c1);
        ffma2(acc[i], v2[2 * i], v2[2 * i + 1], c2);
        ffma2(acc[i], v3[2 * i], v3[2 * i + 1], c3);
        ffma2(acc[i], v4[2 * i], v4[2 * i + 1], c4);
    }
}

// ---- bf16 value path: Blackwell's mixed-precision FMA (PTX fma.rn.f32.bf16 -> SASS FHFMA.BF16) multiplies two bf16
// operands exactly and accumulates in fp32, and it can read either 16-bit half of a register: the bf16 -> fp32
// unpack disappears.  The four corner weights travel as two packed bf16 pairs (3 shuffles per sample, not 5).
__device__ __forceinline__ float fhfma_lo(float acc, uint32_t v, uint32_t w_lo16)
{
    const unsigned short a = (unsigned short)(v & 0xffffu), b = (unsigned short)(w_lo16 & 0xffffu);
    asm("fma.rn.f32.bf16 %0, %1, %2, %0;" : "+f"(acc) : "h"(a), "h"(b));
    return acc;
}
__device__ __forceinline__ float fhfma_hi(float acc, uint32_t v, uint32_t w_lo16)
{
    const unsigned short a = (unsigned short)(v >> 16), b = (unsigned short)(w_lo16 & 0xffffu);
    asm("fma.rn.f32.bf16 %0, %1, %2, %0;" : "+f"(acc) : "h"(a), "h"(b));
    return acc;
}
__device__ __forceinline__ void fma_word4(float (&acc)[8], const uint4& v, uint32_t w)
{
    acc[0] = fhfma_lo(acc[0], v.x, w); acc[1] = fhfma_hi(acc[1], v.x, w);
    acc[2] = fhfma_lo(acc[2], v.y, w); acc[3] = fhfma_hi(acc[3], v.y, w);
    acc[4] = fhfma_lo(acc[4], v.z, w); acc[5] = fhfma_hi(acc[5], v.z, w);
    acc[6] = fhfma_lo(acc[6], v.w, w); acc[7] = fhfma_hi(acc[7], v.w, w);
}
// accumulator abstraction: bf16 values -> float[8] + FHFMA; fp32 values -> float2[4] + FFMA2
template <typename T> struct Acc;
template <> struct Acc<bf16> {
    float a[8];
    __device__ __forceinline__ void zero() {
#pragma unroll
        for (int i = 0; i < 8; ++i) a[i] = 0.f;
    }
    __device__ __forceinline__ void gather(const bf16* __restrict__ base, int W, int code, uint32_t w12, uint32_t w34) {
        if (!(code & CODE_VALID)) return;                        // sample outside the map (uniform in the 4-lane group)
        const bf16* p = base + (int64_t)(code & CODE_OFF_MASK) * 256;
        const bf16* pr = p + (int64_t)W * 256;
        const uint4 v1 = __ldg(reinterpret_cast<const uint4*>(p)), v2 = __ldg(reinterpret_cast<const uint4*>(p + 256));
        const uint4 v3 = __ldg(reinterpret_cast<const uint4*>(pr)), v4 = __ldg(reinterpret_cast<const uint4*>(pr + 256));
        fma_word4(a, v1, w12); fma_word4(a, v2, w12 >> 16); fma_word4(a, v3, w34); fma_word4(a, v4, w34 >> 16);
    }
    __device__ __forceinline__ void finish(float (&o)[8], float scale, bool divide) const {
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] = divide ? __fdiv_rn(a[i], scale) : a[i] * scale;
    }
};
template <> struct Acc<float> {
    float2 a[4];
    __device__ __forceinline__ void zero() {
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = make_float2(0.f, 0.f);
    }
    __device__ __forceinline__ void gather(const float* __restrict__ base, int W, int code, uint32_t w12, uint32_t w34,
                                           float c1, float c2, float c3, float c4) {
        gather_sample<float>(base, W, code, c1, c2, c3, c4, a);
    }
    __device__ __forceinline__ void finish(float (&o)[8], float scale, bool divide) const {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            o[2 * i] = divide ? __fdiv_rn(a[i].x, scale) : a[i].x * scale;
            o[2 * i + 1] = divide ? __fdiv_rn(a[i].y, scale) : a[i].y * scale;
        }
    }
};
// one sample: broadcast the owner lane's prepared descriptor to the 4 lanes of the head and gather
template <typename T>
__device__ __forceinline__ void shuffle_gather(Acc<T>& acc, const T* __restrict__ base, int W, const SamplePrep& sm, int src)
{
    const unsigned FULLM = 0xffffffffu;
    const int code = __shfl_sync(FULLM, sm.code, src);
    if constexpr (sizeof(T) == 2) {
        const uint32_t w12 = __shfl_sync(FULLM, pack_bf16x2(sm.c1, sm.c2), src);
        const uint32_t w34 = __shfl_sync(FULLM, pack_bf16x2(sm.c3, sm.c4), src);
        acc.gather(base, W, code, w12, w34);
    } else {
        const float c1 = __shfl_sync(FULLM, sm.c1, src), c2 = __shfl_sync(FULLM, sm.c2, src);
        const float c3 = __shfl_sync(FULLM, sm.c3, src), c4 = __shfl_sync(FULLM, sm.c4, src);
        acc.gather(base, W, code, 0u, 0u, c1, c2, c3, c4);
    }
}

// ------------------------------------------------------------------------------------------
// bf16 production path: descriptor-staged, software-pipelined gather.
//   Phase 1: the owner lanes write one 16-byte descriptor per sample {pixel | VALID, w1|w2, w3|w4, -} to shared memory,
//            laid out [sample][head] (one conflict-free 128-byte row per sample).
//   Phase 2: the 4 lanes of a head walk their NS descriptors (one broadcast LDS.128 each, no shuffles); the four
//            128-bit corner loads of sample i+DEPTH are issued BEFORE the 32 FHFMAs of sample i, so every lane keeps
//            4*DEPTH independent loads in flight -- the previous version waited on each sample's loads (ncu: 5.5 of 10
//            stall cycles per issue were long-scoreboard) because the validity branch fenced the loads.
// geom(i, base, W): value pointer (already offset to this lane's head / channel slice) and row pitch of sample i.
// Descriptor slot of (sample i, head): i*8 + (head ^ 2*(i & 3)).  The XOR makes the WRITER conflict-free: the 8 lanes of a
// quarter-warp are (heads 2k, 2k+1) x (levels s = 0..3) and write rows i = 4p + s that are 128 B apart (same banks) -- with the
// plain [sample][head] order that was a 4-way bank conflict (ncu: 16 wavefronts per STS.128 instead of 4, 13 % of the kernel's L1
// data-pipe wavefronts); the reader still sees 8 distinct 16-byte groups of one 128-byte row.
__device__ __forceinline__ int desc_slot(int i, int head) { return i * 8 + (head ^ (2 * (i & 3))); }

template <int NS, int DEPTH, typename Geom>
__device__ __forceinline__ void gather_descs(float (&acc)[8], const uint4* dsm, int head, Geom geom)
{
    uint4 d[DEPTH + 1];
    uint4 v[DEPTH + 1][4];
#pragma unroll
    for (int i = 0; i < NS + DEPTH; ++i) {
        if (i < NS) {
            const int slot = i % (DEPTH + 1);
            d[slot] = dsm[desc_slot(i, head)];
            const bf16* base; int W;
            geom(i, base, W);
            if (d[slot].x & CODE_VALID) {
                const bf16* p = base + (int64_t)(d[slot].x & CODE_OFF_MASK) * 256;
                const bf16* pr = p + (int64_t)W * 256;
                v[slot][0] = __ldg(reinterpret_cast<const uint4*>(p));
                v[slot][1] = __ldg(reinterpret_cast<const uint4*>(p + 256));
                v[slot][2] = __ldg(reinterpret_cast<const uint4*>(pr));
                v[slot][3] = __ldg(reinterpret_cast<const uint4*>(pr + 256));
            }
        }
        if (i >= DEPTH) {
            const int slot = (i - DEPTH) % (DEPTH + 1);
            if (d[slot].x & CODE_VALID) {
                fma_word4(acc, v[slot][0], d[slot].y); fma_word4(acc, v[slot][1], d[slot].y >> 16);
                fma_word4(acc, v[slot][2], d[slot].z); fma_word4(acc, v[slot][3], d[slot].z >> 16);
            }
        }
    }
}

__device__ __forceinline__ void project_point(const float* __restrict__ m, float xs, float ys, float zs,
                                              const ScaParams& sp, float& u, float& v, bool& ok);

// N consecutive query-projection outputs (fp32, or fp16 when the tensor-core GEMM writes them in half precision)
template <int N>
__device__ __forceinline__ void load_q(const float* __restrict__ p, float (&o)[N])
{
    if constexpr (N == 2) {
        const float2 t = __ldg(reinterpret_cast<const float2*>(p));
        o[0] = t.x; o[1] = t.y;
    } else {
#pragma unroll
        for (int i = 0; i < N / 4; ++i) {
            const float4 t = __ldg(reinterpret_cast<const float4*>(p) + i);
            o[4 * i] = t.x; o[4 * i + 1] = t.y; o[4 * i + 2] = t.z; o[4 * i + 3] = t.w;
        }
    }
}
template <int N>
__device__ __forceinline__ void load_q(const __half* __restrict__ p, float (&o)[N])
{
    if constexpr (N == 2) {
        const uint32_t t = __ldg(reinterpret_cast<const uint32_t*>(p));
        const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&t));
        o[0] = f.x; o[1] = f.y;
    } else if constexpr (N == 4) {
        const uint2 t = __ldg(reinterpret_cast<const uint2*>(p));
        const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&t.x));
        const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&t.y));
        o[0] = a.x; o[1] = a.y; o[2] = b.x; o[3] = b.y;
    } else {
#pragma unroll
        for (int i = 0; i < N / 8; ++i) {
            const uint4 t = __ldg(reinterpret_cast<const uint4*>(p) + i);
            const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[j]));
                o[8 * i + 2 * j] = f.x; o[8 * i + 2 * j + 1] = f.y;
            }
        }
    }
}

__device__ __forceinline__ uint4 make_desc(const SamplePrep& sm)
{
    return make_uint4((uint32_t)sm.code, pack_bf16x2(sm.c1, sm.c2), pack_bf16x2(sm.c3, sm.c4), 0u);
}

// bf16 production kernel: one BEV query per warp, CTA b = queries [b*NW, (b+1)*NW) in BEV raster order.
// The body is register-tight (80 = 6 CTAs/SM): getq() RE-DERIVES the query index from blockIdx where it is used instead of
// keeping it live across the gather.
template <typename QT, int DEPTH, int MINB, int NW>
__global__ void __launch_bounds__(NW * 32, MINB)
sca_pipe_kernel(const bf16* __restrict__ value, const QT* __restrict__ qproj, ScaParams sp, LevelGeom lg,
                int Nv, bf16* __restrict__ out, uint8_t* __restrict__ hits)
{
    __shared__ uint4 descs[NW][32 * 8];                          // [warp][sample = point*4 + level][head ^ swizzle]
    auto getq = [] { return (int)(blockIdx.x * NW + (threadIdx.x >> 5)); };
    if (getq() >= sp.bev_h * sp.bev_w) return;
    uint4* dw = descs[threadIdx.x >> 5];                         // this warp's 4 KB descriptor block
    const int lane = threadIdx.x & 31, head = lane >> 2, s = lane & 3;   // s doubles as the owned level
    const unsigned FULL = 0xffffffffu;

    const float xs = __fdiv_rn((float)(getq() % sp.bev_w) + 0.5f, (float)sp.bev_w);
    const float ys = __fdiv_rn((float)(getq() / sp.bev_w) + 0.5f, (float)sp.bev_h);
    float ru[2], rv[2];
    unsigned vis = 0;
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int c = r * 4 + (lane >> 3), z = lane & 7;
        bool ok = false;
        ru[r] = 0.f; rv[r] = 0.f;
        if (c < sp.num_cams && z < sp.D) project_point(sp.cam_mat[c], xs, ys, sp.zs[z], sp, ru[r], rv[r], ok);
        const unsigned b = __ballot_sync(FULL, ok);
#pragma unroll
        for (int k = 0; k < 4; ++k) if ((b >> (8 * k)) & 0xffu) vis |= 1u << (r * 4 + k);
    }
    const int count = __popc(vis);
    if (hits && lane == 0) hits[getq()] = (uint8_t)count;

    float acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.f;
    const int own_W = s == 0 ? lg.w[0] : s == 1 ? lg.w[1] : s == 2 ? lg.w[2] : lg.w[3];
    const int own_H = s == 0 ? lg.h[0] : s == 1 ? lg.h[1] : s == 2 ? lg.h[2] : lg.h[3];
    const int own_start = s == 0 ? lg.start[0] : s == 1 ? lg.start[1] : s == 2 ? lg.start[2] : lg.start[3];
    const float own_w = (float)own_W, own_h = (float)own_H;

    for (int c = 0; c < sp.num_cams; ++c) {
        if (!((vis >> c) & 1u)) continue;                                // warp-uniform
        // ---- phase 1: my (head, level s): 8 offsets + 8 logits -> 8 descriptors.  (Reloaded per visible camera --
        // 1.2 on average -- so that nothing but the accumulators stays live across the gather.)
        {
            const QT* qp = qproj + (int64_t)getq() * 768;
            float off[16], wl[8];
            load_q<16>(qp + head * 64 + s * 16, off);
            load_q<8>(qp + 512 + head * 32 + s * 8, wl);
            float mx = wl[0];
#pragma unroll
            for (int i = 1; i < 8; ++i) mx = fmaxf(mx, wl[i]);
            mx = fmaxf(mx, __shfl_xor_sync(FULL, mx, 1));
            mx = fmaxf(mx, __shfl_xor_sync(FULL, mx, 2));
            float sum = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) { wl[i] = __expf(wl[i] - mx); sum += wl[i]; }
            sum += __shfl_xor_sync(FULL, sum, 1);
            sum += __shfl_xor_sync(FULL, sum, 2);
            const float inv = __fdividef(1.f, sum);
            const int r = c >> 2;
#pragma unroll
            for (int p = 0; p < 8; ++p) {
                const int asrc = (c & 3) * 8 + (p % sp.D);               // Z-anchor interleave (:366-373)
                const float u = __shfl_sync(FULL, r ? ru[1] : ru[0], asrc);
                const float v = __shfl_sync(FULL, r ? rv[1] : rv[0], asrc);
                // (u + dx/W) * W - 0.5 == u*W + dx - 0.5 up to fp32 rounding (bf16 path: not bit-matched to the fp32 one)
                const float w_im = fmaf(u, own_w, off[2 * p] - 0.5f);
                const float h_im = fmaf(v, own_h, off[2 * p + 1] - 0.5f);
                dw[desc_slot(p * 4 + s, head)] = make_desc(prep_sample(h_im, w_im, wl[p] * inv, own_H, own_W, own_start));
            }
        }
        __syncwarp();
        // ---- phase 2
        const bf16* vcam = value + ((int64_t)c * Nv * 8 + head) * 32 + s * 8;
        gather_descs<32, DEPTH>(acc, dw, head, [&](int i, const bf16*& base, int& W) { base = vcam; W = lg.w[i & 3]; });
        __syncwarp();
    }
    const float scale = (float)max(count, 1);
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = __fdiv_rn(acc[i], scale);
    store8(out + (int64_t)getq() * 256 + head * 32 + s * 8, acc);
}

// ------------------------------------------------------------------------------------------
// Operator boundary: value [B,Nv,M,C] f32, loc [B,Nq,M,L,P,2] (x,y), w [B,Nq,M,L,P] -> [B,Nq,M*C]
// One thread per (b, q, head, 8-channel slice) when C % 8 == 0, otherwise per channel.
template <int VEC>
__global__ void msda_forward_kernel(const float* __restrict__ value, const int64_t* __restrict__ shapes,
                                    const int64_t* __restrict__ lstart, const float* __restrict__ loc,
                                    const float* __restrict__ wts, int B, int Nv, int M, int C, int Nq,
                                    int L, int P, float* __restrict__ out)
{
    const int slices = C / VEC;
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t total = (int64_t)B * Nq * M * slices;
    if (idx >= total) return;
    const int s = (int)(idx % slices);
    const int m = (int)((idx / slices) % M);
    const int64_t bq = idx / ((int64_t)slices * M);           // b * Nq + q
    const int b = (int)(bq / Nq);
    const float* lp = loc + (bq * M + m) * (int64_t)L * P * 2;
    const float* wp = wts + (bq * M + m) * (int64_t)L * P;
    float acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.f;
    for (int l = 0; l < L; ++l) {
        const int H = (int)shapes[2 * l], W = (int)shapes[2 * l + 1];
        const float* base = value + (((int64_t)b * Nv + lstart[l]) * M + m) * C + s * VEC;
        for (int p = 0; p < P; ++p) {
            const float w_im = lp[(l * P + p) * 2] * (float)W - 0.5f;
            const float h_im = lp[(l * P + p) * 2 + 1] * (float)H - 0.5f;
            const float wt = wp[l * P + p];
            if constexpr (VEC == 8) {
                bilinear_acc8<float>(base, H, W, M * C, h_im, w_im, wt, acc);
            } else {
                if (!(h_im > -1.f && w_im > -1.f && h_im < (float)H && w_im < (float)W)) continue;
                const int h_lo = (int)floorf(h_im), w_lo = (int)floorf(w_im);
                const float lh = h_im - h_lo, lw = w_im - w_lo, hh = 1.f - lh, hw = 1.f - lw;
                const int64_t st = (int64_t)M * C;
                const float* q = base + ((int64_t)h_lo * W + w_lo) * st;
                float v = 0.f;
                if (h_lo >= 0 && w_lo >= 0) v += hh * hw * q[0];
                if (h_lo >= 0 && w_lo + 1 <= W - 1) v += hh * lw * q[st];
                if (h_lo + 1 <= H - 1 && w_lo >= 0) v += lh * hw * q[(int64_t)W * st];
                if (h_lo + 1 <= H - 1 && w_lo + 1 <= W - 1) v += lh * lw * q[(int64_t)(W + 1) * st];
                acc[0] += wt * v;
            }
        }
    }
    float* o = out + (bq * M + m) * C + s * VEC;
    if constexpr (VEC == 8) store8(o, acc);
    else o[0] = acc[0];
}

// ------------------------------------------------------------------------------------------
// Fused temporal self-attention gather.  qproj [Nq,192] f32 = Linear outputs
//   [0,128):  sampling_offsets viewed (head, queue, level=1, point, xy)   (:206-208)
//   [128,192): attention logits viewed (head, queue, point), softmax over the 4 points (:209-211)
// value_prev / value_cur: [Nq, 8, 32] T (projected values of queue 0 / queue 1).
// out[q] = 0.5 * (MSDA_queue0 + MSDA_queue1)                                (:257-262)
template <typename T, typename QT>
__global__ void __launch_bounds__(256)
tsa_fused_kernel(const T* __restrict__ value_prev, const T* __restrict__ value_cur,
                 const QT* __restrict__ qproj, int bev_h, int bev_w, T* __restrict__ out)
{
    const int q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int Nq = bev_h * bev_w;
    if (q >= Nq) return;
    const int lane = threadIdx.x & 31, head = lane >> 2, s = lane & 3;
    const int qu_own = s >> 1, p0 = (s & 1) * 2;              // owner of samples (queue, p0), (queue, p0+1)
    const QT* qp = qproj + (int64_t)q * 192;
    // offsets of my two samples: index head*16 + queue*8 + p*2 + xy -> 4 consecutive values
    float offv[4], lgv[2];
    load_q<4>(qp + head * 16 + qu_own * 8 + p0 * 2, offv);
    load_q<2>(qp + 128 + head * 8 + qu_own * 4 + p0, lgv);
    const float4 off = make_float4(offv[0], offv[1], offv[2], offv[3]);
    const float2 lg = make_float2(lgv[0], lgv[1]);
    // softmax over the 4 points of (head, queue): my 2 logits + partner lane (s ^ 1)
    float mx = fmaxf(lg.x, lg.y);
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
    const float e0 = expf(lg.x - mx), e1 = expf(lg.y - mx);
    float sum = e0 + e1;
    sum += __shfl_xor_sync(0xffffffffu, sum, 1);
    const float wt0 = e0 / sum, wt1 = e1 / sum;
    // reference point of this query (encoder.py:78-89) and sampling locations (:224-229)
    const float fw = (float)bev_w, fh = (float)bev_h;
    const float rx = __fdiv_rn((float)(q % bev_w) + 0.5f, fw);
    const float ry = __fdiv_rn((float)(q / bev_w) + 0.5f, fh);
    const float wim0 = __fadd_rn(rx, __fdiv_rn(off.x, fw)) * fw - 0.5f;
    const float him0 = __fadd_rn(ry, __fdiv_rn(off.y, fh)) * fh - 0.5f;
    const float wim1 = __fadd_rn(rx, __fdiv_rn(off.z, fw)) * fw - 0.5f;
    const float him1 = __fadd_rn(ry, __fdiv_rn(off.w, fh)) * fh - 0.5f;

    const SamplePrep sa = prep_sample(him0, wim0, wt0, bev_h, bev_w);
    const SamplePrep sb = prep_sample(him1, wim1, wt1, bev_h, bev_w);
    Acc<T> accu;
    accu.zero();
    const int grp = lane & ~3;
#pragma unroll
    for (int o = 0; o < 4; ++o) {                            // owner sub-lane o holds samples (o>>1, (o&1)*2 + {0,1})
        const int src = grp | o;
        const T* base = ((o >> 1) == 0 ? value_prev : value_cur) + head * 32 + s * 8;
        shuffle_gather<T>(accu, base, bev_w, sa, src);
        shuffle_gather<T>(accu, base, bev_w, sb, src);
    }
    float acc[8];
    accu.finish(acc, 0.5f, false);
    store8(out + (int64_t)q * 256 + head * 32 + s * 8, acc);
}

// ------------------------------------------------------------------------------------------
// Camera projection of one pillar point (encoder.py:104-139), fp32, same operation order.
__device__ __forceinline__ void project_point(const float* __restrict__ m /*4x4 row-major*/, float xs, float ys,
                                              float zs, const ScaParams& sp, float& u, float& v, bool& ok)
{
    const float X = __fadd_rn(__fmul_rn(xs, sp.pc_scale[0]), sp.pc_min[0]);
    const float Y = __fadd_rn(__fmul_rn(ys, sp.pc_scale[1]), sp.pc_min[1]);
    const float Z = __fadd_rn(__fmul_rn(zs, sp.pc_scale[2]), sp.pc_min[2]);
    const float cx = fmaf(m[2], Z, fmaf(m[1], Y, fmaf(m[0], X, m[3])));
    const float cy = fmaf(m[6], Z, fmaf(m[5], Y, fmaf(m[4], X, m[7])));
    const float cz = fmaf(m[10], Z, fmaf(m[9], Y, fmaf(m[8], X, m[11])));
    const float eps = 1e-5f;
    const float d = fmaxf(cz, eps);
    u = __fdiv_rn(__fdiv_rn(cx, d), sp.img_w);
    v = __fdiv_rn(__fdiv_rn(cy, d), sp.img_h);
    ok = (cz > eps) && (v > 0.f) && (v < 1.f) && (u < 1.f) && (u > 0.f);
}

// debug / parity kernel for row a2: writes reference_points_cam [cam,Nq,D,2] and bev_mask [cam,Nq,D]
__global__ void project_pillars_kernel(ScaParams sp, float* __restrict__ ref_cam, uint8_t* __restrict__ mask)
{
    const int Nq = sp.bev_h * sp.bev_w;
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)sp.num_cams * Nq * sp.D) return;
    const int z = (int)(idx % sp.D);
    const int q = (int)((idx / sp.D) % Nq);
    const int c = (int)(idx / ((int64_t)sp.D * Nq));
    const float xs = __fdiv_rn((float)(q % sp.bev_w) + 0.5f, (float)sp.bev_w);
    const float ys = __fdiv_rn((float)(q / sp.bev_w) + 0.5f, (float)sp.bev_h);
    float u, v; bool ok;
    project_point(sp.cam_mat[c], xs, ys, sp.zs[z], sp, u, v, ok);
    ref_cam[idx * 2] = u; ref_cam[idx * 2 + 1] = v;
    mask[idx] = ok ? 1 : 0;
}

// Fused spatial cross-attention gather (see file header).
//   value [num_cams, Nv, 8, 32] T;  qproj [Nq, 768] f32 = [offsets (head,level,point,xy) | logits (head, level*point)]
//   out  [Nq, 256] T  = sum_{visible cams} MSDA_cam(q) / max(1, #visible cams)
//   hits (optional) [Nq] u8 = #visible cams (for tests / statistics)
template <typename T>
__global__ void __launch_bounds__(256, 3)
sca_fused_kernel(const T* __restrict__ value, const float* __restrict__ qproj, ScaParams sp, LevelGeom lg,
                 int Nv, T* __restrict__ out, uint8_t* __restrict__ hits)
{
    const int Nq = sp.bev_h * sp.bev_w;
    const int q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (q >= Nq) return;
    const int lane = threadIdx.x & 31, head = lane >> 2, s = lane & 3;   // s doubles as the owned level
    const unsigned FULL = 0xffffffffu;

    // ---- camera projection of the pillar: lane -> (cam = 4*round + lane/8, anchor = lane%8)
    const float xs = __fdiv_rn((float)(q % sp.bev_w) + 0.5f, (float)sp.bev_w);
    const float ys = __fdiv_rn((float)(q / sp.bev_w) + 0.5f, (float)sp.bev_h);
    float ru[2], rv[2];
    unsigned vis = 0;                                                    // bit c: camera c sees the pillar
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int c = r * 4 + (lane >> 3), z = lane & 7;
        bool ok = false;
        ru[r] = 0.f; rv[r] = 0.f;
        if (c < sp.num_cams && z < sp.D) project_point(sp.cam_mat[c], xs, ys, sp.zs[z], sp, ru[r], rv[r], ok);
        const unsigned b = __ballot_sync(FULL, ok);
#pragma unroll
        for (int k = 0; k < 4; ++k) if ((b >> (8 * k)) & 0xffu) vis |= 1u << (r * 4 + k);
    }
    const int count = __popc(vis);
    if (hits && lane == 0) hits[q] = (uint8_t)count;

    Acc<T> accu;
    accu.zero();

    if (count > 0) {
        // ---- owner lane (head, level = s): 8 points x (dx, dy) and 8 logits
        // (static selects instead of lg.w[s]: a dynamically indexed kernel parameter would be copied to local memory)
        const int own_W = s == 0 ? lg.w[0] : s == 1 ? lg.w[1] : s == 2 ? lg.w[2] : lg.w[3];
        const int own_H = s == 0 ? lg.h[0] : s == 1 ? lg.h[1] : s == 2 ? lg.h[2] : lg.h[3];
        const float* qp = qproj + (int64_t)q * 768;
        float offn[16], wl[8];
        {
            const float4* o4 = reinterpret_cast<const float4*>(qp + head * 64 + s * 16);
            const float fw = (float)own_W, fh = (float)own_H;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float4 t = __ldg(o4 + i);
                offn[4 * i + 0] = __fdiv_rn(t.x, fw); offn[4 * i + 1] = __fdiv_rn(t.y, fh);
                offn[4 * i + 2] = __fdiv_rn(t.z, fw); offn[4 * i + 3] = __fdiv_rn(t.w, fh);
            }
            const float4* l4 = reinterpret_cast<const float4*>(qp + 512 + head * 32 + s * 8);
            const float4 a = __ldg(l4), b = __ldg(l4 + 1);
            wl[0] = a.x; wl[1] = a.y; wl[2] = a.z; wl[3] = a.w; wl[4] = b.x; wl[5] = b.y; wl[6] = b.z; wl[7] = b.w;
            // softmax over the head's 32 logits = 4 lanes x 8 (spatial_cross_attention.py:343)
            float mx = wl[0];
#pragma unroll
            for (int i = 1; i < 8; ++i) mx = fmaxf(mx, wl[i]);
            mx = fmaxf(mx, __shfl_xor_sync(FULL, mx, 1));
            mx = fmaxf(mx, __shfl_xor_sync(FULL, mx, 2));
            float sum = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) { wl[i] = expf(wl[i] - mx); sum += wl[i]; }
            sum += __shfl_xor_sync(FULL, sum, 1);
            sum += __shfl_xor_sync(FULL, sum, 2);
#pragma unroll
            for (int i = 0; i < 8; ++i) wl[i] = wl[i] / sum;
        }
        const float own_w = (float)own_W, own_h = (float)own_H;
        const int grp = lane & ~3;
        for (int c = 0; c < sp.num_cams; ++c) {
            if (!((vis >> c) & 1u)) continue;                            // warp-uniform
            const int r = c >> 2;
            const T* vcam = value + ((int64_t)c * Nv * 8 + head) * 32 + s * 8;
#pragma unroll
            for (int p = 0; p < 8; ++p) {
                // sampling location of point p uses pillar anchor p % D (Z-anchor interleave, :366-373)
                const int asrc = (c & 3) * 8 + (p % sp.D);
                const float u = __shfl_sync(FULL, r ? ru[1] : ru[0], asrc);
                const float v = __shfl_sync(FULL, r ? rv[1] : rv[0], asrc);
                const float w_im = __fadd_rn(u, offn[2 * p]) * own_w - 0.5f;
                const float h_im = __fadd_rn(v, offn[2 * p + 1]) * own_h - 0.5f;
                const SamplePrep sm = prep_sample(h_im, w_im, wl[p], own_H, own_W);   // my (head, level s, point p)
#pragma unroll
                for (int l = 0; l < 4; ++l)
                    shuffle_gather<T>(accu, vcam + (int64_t)lg.start[l] * 256, lg.w[l], sm, grp | l);
            }
        }
    }
    float acc[8];
    accu.finish(acc, (float)max(count, 1), true);
    store8(out + (int64_t)q * 256 + head * 32 + s * 8, acc);
}

}  // namespace

// ------------------------------------------------------------------------------------------ launchers
int launch_msda_forward(const float* value, const int64_t* shapes, const int64_t* lstart, const float* loc,
                        const float* wts, int B, int Nv, int M, int C, int Nq, int L, int P, float* out,
                        cudaStream_t stream)
{
    if ((int64_t)B * Nq == 0) return 0;
    if (C % 8 == 0) {
        const int64_t total = (int64_t)B * Nq * M * (C / 8);
        msda_forward_kernel<8><<<ceil_div(total, 256), 256, 0, stream>>>(value, shapes, lstart, loc, wts, B, Nv, M,
                                                                          C, Nq, L, P, out);
    } else {
        const int64_t total = (int64_t)B * Nq * M * C;
        msda_forward_kernel<1><<<ceil_div(total, 256), 256, 0, stream>>>(value, shapes, lstart, loc, wts, B, Nv, M,
                                                                          C, Nq, L, P, out);
    }
    OCC_CUDA(cudaGetLastError());
    return 0;
}

template <typename T>
int launch_tsa_fused(const T* value_prev, const T* value_cur, const void* qproj, bool q_half, int bev_h, int bev_w, T* out,
                     cudaStream_t stream)
{
    OCC_CHECK(bev_h >= 2 && bev_w >= 2, "tsa_fused: the BEV grid must be at least 2x2");
    const int Nq = bev_h * bev_w;
    const dim3 grid(ceil_div(Nq, 8));
    if (q_half) tsa_fused_kernel<T, __half><<<grid, 256, 0, stream>>>(value_prev, value_cur, (const __half*)qproj, bev_h, bev_w, out);
    else        tsa_fused_kernel<T, float><<<grid, 256, 0, stream>>>(value_prev, value_cur, (const float*)qproj, bev_h, bev_w, out);
    OCC_CUDA(cudaGetLastError());
    return 0;
}
template int launch_tsa_fused<float>(const float*, const float*, const void*, bool, int, int, float*, cudaStream_t);
template int launch_tsa_fused<bf16>(const bf16*, const bf16*, const void*, bool, int, int, bf16*, cudaStream_t);

template <typename T>
int launch_sca_fused(const T* value, const void* qproj_v, bool q_half, const ScaParams& sp, const LevelGeom& lg, int Nv,
                     T* out, uint8_t* hits, cudaStream_t stream)
{
    OCC_CHECK(lg.num_levels == 4 && sp.num_cams <= 8 && sp.D <= 8 && sp.D >= 1 && 8 % sp.D == 0,
              "sca_fused: supports 4 levels, <= 8 cameras, pillar anchors in {1,2,4,8}");
    for (int l = 0; l < 4; ++l) OCC_CHECK(lg.h[l] >= 2 && lg.w[l] >= 2, "sca_fused: every level must be at least 2x2");
    const int Nq = sp.bev_h * sp.bev_w;
    if constexpr (sizeof(T) == 2) {
        // production bf16 kernel: descriptor-staged gather, 4 warps per CTA, 6 CTAs per SM (measured variants: profiles/README.md)
        if (q_half) sca_pipe_kernel<__half, 1, 6, 4><<<ceil_div(Nq, 4), 128, 0, stream>>>(value, (const __half*)qproj_v, sp, lg, Nv, out, hits);
        else        sca_pipe_kernel<float, 1, 6, 4><<<ceil_div(Nq, 4), 128, 0, stream>>>(value, (const float*)qproj_v, sp, lg, Nv, out, hits);
    } else {
        OCC_CHECK(!q_half, "sca_fused: the fp32 kernel reads fp32 projections");
        sca_fused_kernel<T><<<ceil_div(Nq, 8), 256, 0, stream>>>(value, (const float*)qproj_v, sp, lg, Nv, out, hits);
    }
    OCC_CUDA(cudaGetLastError());
    return 0;
}
template int launch_sca_fused<float>(const float*, const void*, bool, const ScaParams&, const LevelGeom&, int, float*,
                                     uint8_t*, cudaStream_t);
template int launch_sca_fused<bf16>(const bf16*, const void*, bool, const ScaParams&, const LevelGeom&, int, bf16*,
                                    uint8_t*, cudaStream_t);

int launch_project_pillars(const ScaParams& sp, float* ref_cam, uint8_t* mask, cudaStream_t stream)
{
    const int64_t total = (int64_t)sp.num_cams * sp.bev_h * sp.bev_w * sp.D;
    project_pillars_kernel<<<ceil_div(total, 256), 256, 0, stream>>>(sp, ref_cam, mask);
    OCC_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace occ
