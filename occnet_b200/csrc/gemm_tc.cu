// tcgen05 / TMEM / TMA bf16 GEMM for the dense layers of the encoder (sm_100a):
//     C[M,N] = act(A[M,K] . W[N,K]^T + bias[N]) (+ residual[M,N]),   fp32 accumulation in TMEM.
// Every nn.Linear on the path has this shape (reference: temporal_self_attention.py:99-104,
// spatial_cross_attention.py:67,245-249, mmcv FFN) with K in {256,512}, N in {192,256,512,768}.
//
// Persistent, warp-specialised kernel, one CTA per SM; every CTA owns one n-block and a contiguous range of rows
// (dealt in 32-row blocks so that all CTAs move the same number of bytes):
//   warp 0   TMA producer : the CTA's weight block once (resident, <= 128 KB, one mbarrier per 32 KB k-slice) or a W
//                           k-block per stage; A tiles 128x64 (bf16, 128B swizzle) through a 3-6 stage mbarrier ring
//   warp 1   MMA issuer   : tcgen05.mma.cta_group::1.kind::f16, M=128, N=BN, K=16 x4 per stage;
//                           accumulators double-buffered in TMEM (2 x 256 columns)
//   warps 2-9 epilogue    : tcgen05.ld 32x32b, overlapping the next tile's main loop.  Per-column constants (bias,
//                           gamma, beta) are staged in shared memory once per CTA.  Three variants:
//                           (a) 16-bit output: bias / ReLU -> bf16 or fp16 -> swizzled 2 KB staging -> TMA store;
//                           (b) fused LayerNorm: x = acc + bias + residual written back to TMEM (tcgen05.st), row
//                               statistics exchanged between the two column-half warps, second pass normalises;
//                               fp32 residual stream in the T32 block layout, bf16 operand copy via staging;
//                           (c) fp32 output (+ residual) via swizzled staging, 4 rows x 128 B per store instruction.
// Programmatic dependent launch: the prologue (barriers, TMEM, weights, constants) does not wait for the previous grid.
// The A operand may be the concatenation of two matrices along K (TSA's cat([value, query+pos]),
// temporal_self_attention.py:197) -- two tensor maps, no materialised concat.
#include <cstdlib>
#include <map>
#include <mutex>
#include <tuple>
#include <type_traits>
#include <vector>

#include "gemm_tc.cuh"
#include "tc_common.cuh"

namespace occ {

// ------------------------------------------------------------------------------------------------ host helpers
PFN_encodeTiled get_encode_tiled()
{
    static PFN_encodeTiled fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_encodeTiled>(p);
    });
    return fn;
}

int make_tensor_map_bf16(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                         const uint32_t* box, int swizzle_bytes)
{
    PFN_encodeTiled enc = get_encode_tiled();
    OCC_CHECK(enc != nullptr, "cuTensorMapEncodeTiled is not available from the driver");
    cuuint64_t gdim[5], gstr[5];
    cuuint32_t bdim[5], estr[5];
    for (int i = 0; i < rank; ++i) { gdim[i] = dims[i]; bdim[i] = box[i]; estr[i] = 1; }
    for (int i = 0; i + 1 < rank; ++i) gstr[i] = strides_bytes[i];
    const CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                : swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE;
    const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr,
                           bdim, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    OCC_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed with code " + std::to_string((int)r));
    return 0;
}

int cached_map_2d(const void* base, uint64_t inner, uint64_t rows, uint32_t box_inner, uint32_t box_rows, CUtensorMap* out,
                  uint64_t ld = 0);
int cached_map_out(const void* base, uint64_t cols, uint64_t rows, uint64_t blocks, uint32_t box_cols, CUtensorMap* out);

namespace {

constexpr int BLOCK_M = 128, BLOCK_K = 64, A_TILE_BYTES = BLOCK_M * BLOCK_K * 2;
constexpr int NUM_THREADS = 320;                          // TMA warp, MMA warp, 8 epilogue warps
// shared-memory tail after the operand ring: 8 per-warp staging blocks (4 KB each; 2 KB when a 16-bit output leaves
// through 32-column TMA stores), 256 B of barriers, 2 KB of LayerNorm partials (LN kernels only)
//   + the CTA's per-column constants (bias; gamma, beta for LN) as fp32: 1 KB / 3 KB
constexpr int smem_tail(bool ln, int stg_bytes) { return 8 * stg_bytes + 256 + (ln ? 2048 + 3072 : 1024); }
constexpr int SMEM_MAX = 232448 - 1024;                   // 227 KB opt-in maximum minus alignment slack
constexpr int MAX_STAGES = 6;

struct LnArgs {                                           // fused LayerNorm epilogue (N == BN == 256)
    const float* gamma; const float* beta; const float* pos;
    float* y_f32; bf16* y_bf16; bf16* y_pos_bf16;
};

// One GEMM problem of a launch.  A launch carries up to MAX_PROBS INDEPENDENT problems (e.g. TSA's value projection and
// sampling-offset projection of the same query tensor): the CTAs [cta_begin, cta_begin + cta_count) work on problem p.  These
// GEMMs have only ~2 tiles per CTA on 148 SMs, so their duration is start-up + a latency chain, not bandwidth: two problems on
// 74 + 74 CTAs finish in about the time ONE took on 148.
// w_resident: all nk weight k-blocks of this CTA's n-block stay in shared memory for the CTA's lifetime and the
// ring only carries A tiles; otherwise each stage carries an A tile and a W k-block (v1 behaviour).
constexpr int MAX_PROBS = 3;
struct GemmProb {
    CUtensorMap tmA, tmA2, tmW, tmC, tmC2;                   // (LayerNorm launches: tmC = y_bf16, tmC2 = y_pos_bf16, [M,256] bf16)
    const float* bias; const float* residual; void* C;
    const float* res_t32;                                     // optional fp32 epilogue constant [M,N] in the T32 block layout
                                                              // (TMA-store path: the row-per-thread read is then coalesced)
    long long ldc, nblk_stride;
    int c_tma /* 0: none, 1: [M,N] row-major, 2: n-blocks as separate [M,BN] matrices */;
    int stg_bytes, M, N, BN, nk, nk1, act, w_resident, stages;
    int out_half;                                             // 16-bit outputs as fp16 instead of bf16 (runtime, per problem)
    int cta_begin, cta_count;
};
struct GemmProbs { GemmProb p[MAX_PROBS]; int n; };

template <typename TC, bool LN>
__global__ void __launch_bounds__(NUM_THREADS, 1)          // 10 warps -> 3 on one SMSP -> <= 168 regs (16K per SMSP)
gemm_tc_kernel(const __grid_constant__ GemmProbs probs, LnArgs ln, long long* __restrict__ dbg)
{
    int pi = 0;
    while (pi + 1 < probs.n && (int)blockIdx.x >= probs.p[pi + 1].cta_begin) ++pi;
    const GemmProb& P = probs.p[pi];
    const CUtensorMap& tmA = P.tmA; const CUtensorMap& tmA2 = P.tmA2; const CUtensorMap& tmW = P.tmW; const CUtensorMap& tmC = P.tmC;
    const CUtensorMap& tmC2 = P.tmC2;
    const float* __restrict__ bias = P.bias;
    const float* __restrict__ residual = P.residual;
    const float* __restrict__ res_t32 = P.res_t32;
    TC* __restrict__ C = reinterpret_cast<TC*>(P.C);
    const int c_tma = P.c_tma, stg_bytes = P.stg_bytes, M = P.M, N = P.N, BN = P.BN, nk = P.nk, nk1 = P.nk1, act = P.act;
    const int w_resident = P.w_resident, stages = P.stages;
    const long long ldc = P.ldc, nblk_stride = P.nblk_stride;
    const bool out_half = std::is_same<TC, __half>::value || P.out_half != 0;
    const int bid = (int)blockIdx.x - P.cta_begin, nctas = P.cta_count;
    // optional in-kernel timeline (globaltimer ns): 16 slots per CTA, written by the role that owns the event
    auto stamp = [&](int slot) {
        if (dbg) {
            long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            dbg[(size_t)blockIdx.x * 16 + slot] = t;
        }
    };
    if (threadIdx.x == 0) stamp(0);
    // Programmatic dependent launch: let the next kernel in the stream start its prologue while this grid drains,
    // and (below) only wait for the PREVIOUS grid right before touching data it produced.  Weights, barrier and
    // TMEM setup do not depend on the predecessor.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (tc::smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t w_tile_bytes = BN * BLOCK_K * 2;
    const uint32_t w_region = w_resident ? nk * w_tile_bytes : 0;
    const uint32_t stage_bytes = A_TILE_BYTES + (w_resident ? 0 : w_tile_bytes);
    const uint32_t ring_base = smem_base + w_region;
    const uint32_t stg_base = ring_base + stages * stage_bytes;  // 8 x 4 KB epilogue staging blocks (1024-byte aligned: TMA swizzle)
    const uint32_t bar_base = stg_base + 8 * stg_bytes;
    auto full_bar = [&](int s) { return bar_base + s * 8; };
    auto empty_bar = [&](int s) { return bar_base + (MAX_STAGES + s) * 8; };
    auto tfull_bar = [&](int s) { return bar_base + (2 * MAX_STAGES + s) * 8; };
    auto tempty_bar = [&](int s) { return bar_base + (2 * MAX_STAGES + 2 + s) * 8; };
    // one barrier per resident weight k-block (the last one collects every block >= 7): the first MMA starts as soon
    // as ITS 32 KB slice has landed instead of waiting for the whole 128 KB block
    auto w_bar = [&](int kb) { return bar_base + (2 * MAX_STAGES + 6 + (kb < 7 ? kb : 7)) * 8; };
    const uint32_t tmem_slot = bar_base + (2 * MAX_STAGES + 5) * 8;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_tiles = N / BN;
    // CTA -> (fixed n block, contiguous row range): a resident weight block serves every tile of the CTA, and the
    // rows are dealt out in 32-row blocks so that every CTA gets (almost) the same number of ROWS.  With whole
    // 128-row tiles, 313 tiles on 148 CTAs meant 3 tile-epilogues for some CTAs and 2 for the rest (70 % balance);
    // with row ranges the last tile of a CTA is partial and its (memory-bound) epilogue only touches the rows it owns.
    const int n_blk = bid % n_tiles;
    const int grp = bid / n_tiles, ngrp = nctas / n_tiles;
    const int nb32 = (M + 31) >> 5;
    const int row_begin = (int)(((long long)nb32 * grp) / ngrp) << 5;
    const int row_end = min(M, (int)(((long long)nb32 * (grp + 1)) / ngrp) << 5);

    if (warp == 0 && lane == 0) {
        tc::tma_prefetch_desc(&tmA); tc::tma_prefetch_desc(&tmA2); tc::tma_prefetch_desc(&tmW);
        if (c_tma) tc::tma_prefetch_desc(&tmC);
        for (int s = 0; s < stages; ++s) { tc::mbar_init(full_bar(s), 1); tc::mbar_init(empty_bar(s), 1); }
        for (int s = 0; s < 2; ++s) { tc::mbar_init(tfull_bar(s), 1); tc::mbar_init(tempty_bar(s), 256); }
        for (int kb = 0; kb < 8; ++kb) tc::mbar_init(w_bar(kb), 1);
        tc::mbar_fence_init();
    }
    if (warp == 1) tc::tmem_alloc(tmem_slot, 512);
    float* const cvec = reinterpret_cast<float*>(smem_raw + (bar_base + 256 + (LN ? 2048 : 0) - tc::smem_u32(smem_raw)));
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
    if (threadIdx.x == 0) stamp(1);                              // setup done (barriers, TMEM)

    if (warp == 0) {
        if (lane == 0) {
            if (w_resident) {
                for (int kb = 0; kb < nk && kb < 8; ++kb)
                    tc::mbar_arrive_expect_tx(w_bar(kb), kb < 7 ? w_tile_bytes : (nk - 7) * w_tile_bytes);
                for (int kb = 0; kb < nk; ++kb)
                    tc::tma_load_2d(smem_base + kb * w_tile_bytes, &tmW, w_bar(kb), kb * BLOCK_K, n_blk * BN);
            }
            int s = 0; uint32_t ph = 0;
            asm volatile("griddepcontrol.wait;" ::: "memory");    // A (and residual) come from the previous kernel
            for (int m_row = row_begin; m_row < row_end; m_row += BLOCK_M) {
                for (int kb = 0; kb < nk; ++kb) {
                    tc::mbar_wait(empty_bar(s), ph ^ 1);
                    tc::mbar_arrive_expect_tx(full_bar(s), stage_bytes);
                    const uint32_t a_dst = ring_base + s * stage_bytes;
                    if (kb < nk1) tc::tma_load_2d(a_dst, &tmA, full_bar(s), kb * BLOCK_K, m_row);
                    else          tc::tma_load_2d(a_dst, &tmA2, full_bar(s), (kb - nk1) * BLOCK_K, m_row);
                    if (!w_resident)
                        tc::tma_load_2d(a_dst + A_TILE_BYTES, &tmW, full_bar(s), kb * BLOCK_K, n_blk * BN);
                    if (++s == stages) { s = 0; ph ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc = tc::make_idesc_bf16(BLOCK_M, BN);
            int s = 0; uint32_t ph = 0; int as = 0; uint32_t aph = 0;
            stamp(2);
            int tcount = 0;
            for (int m_row = row_begin; m_row < row_end; m_row += BLOCK_M, ++tcount) {
                tc::mbar_wait(tempty_bar(as), aph ^ 1);
                tc::tc_fence_after();
                for (int kb = 0; kb < nk; ++kb) {
                    if (w_resident && tcount == 0) tc::mbar_wait(w_bar(kb), 0);      // weight slice kb resident
                    tc::mbar_wait(full_bar(s), ph);
                    if (kb == 0 && tcount < 3) stamp(3 + tcount * 3);    // first A k-block of tile landed
                    tc::tc_fence_after();
                    const uint32_t a_addr = ring_base + s * stage_bytes;
                    const uint64_t da = tc::make_smem_desc(a_addr, 128);
                    const uint64_t db = tc::make_smem_desc(w_resident ? smem_base + kb * w_tile_bytes
                                                                      : a_addr + A_TILE_BYTES, 128);
#pragma unroll
                    for (int k = 0; k < BLOCK_K / 16; ++k)       // +32 bytes (>>4 = 2) per UMMA_K step inside the swizzle atom
                        tc::umma_bf16(tmem_base + as * 256, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
                    tc::umma_commit(empty_bar(s));               // frees the smem stage when these MMAs retire
                    if (kb == nk - 1) tc::umma_commit(tfull_bar(as));
                    if (++s == stages) { s = 0; ph ^= 1; }
                }
                if (++as == 2) { as = 0; aph ^= 1; }
            }
        }
    } else {
        // 8 epilogue warps: warp -> (TMEM lane quarter = warp % 4, column half).  tcgen05.ld hands every thread one
        // ROW of the tile; touching global memory in that shape costs 32 separate requests per instruction and is
        // request-rate bound (measured: ~7 us per tile).  So every global access goes through a per-warp 4 KB
        // staging block in shared memory (128-byte rows, 16-byte pieces XOR-swizzled by row) and is issued in the
        // transposed shape: one instruction = 4 rows x 128 contiguous bytes.
        // Per-column constants of this CTA's n-block -> shared memory, once, by the 8 epilogue warps while the first
        // tile is loading.  (Parameters: no dependency on the previous grid.)  Reading them with __ldg inside the
        // epilogue loop exposed one L2 round trip per 32-column chunk -- the streaming residual / output traffic
        // evicts them from L1 between tiles -- which was most of the epilogue time.
        {
            const int t = threadIdx.x - 64;                      // 0..255
            if (t < BN) {
                cvec[t] = bias ? __ldg(bias + n_blk * BN + t) : 0.f;
                if constexpr (LN) { cvec[256 + t] = __ldg(ln.gamma + t); cvec[512 + t] = __ldg(ln.beta + t); }
            }
            asm volatile("bar.sync 5, 256;" ::: "memory");
        }
        const int quarter = warp & 3;
        const int half = (warp - 2) >> 2;
        const int ew = warp - 2;
        const int ncol = BN >> 1;                                // columns owned by this warp
        const int cbeg = half * ncol;
        const uint32_t stg = stg_base + ew * stg_bytes;          // this warp's staging block (shared address)
        float2* part = reinterpret_cast<float2*>(smem_raw + (bar_base + 256 - tc::smem_u32(smem_raw)));   // [2][128]
        const int crow = lane >> 3, cpiece = lane & 7;           // coalesced shape: row 4*i + crow, 16-byte piece cpiece
        // plain C++ accesses through a generic pointer (not volatile asm) so the compiler may overlap the
        // shared-memory round trip with the global stores of the previous rows
        float4* const stg4 = reinterpret_cast<float4*>(smem_raw + (stg - tc::smem_u32(smem_raw)));
        auto sts4 = [&](int r, int piece, float4 v) { stg4[r * 8 + (piece ^ (r & 7))] = v; };
        auto lds4 = [&](int r, int piece) { return stg4[r * 8 + (piece ^ (r & 7))]; };
        int as = 0; uint32_t aph = 0;
        int etile = 0;
        asm volatile("griddepcontrol.wait;" ::: "memory");        // before the first global read / write of this role
        for (int m_row = row_begin; m_row < row_end; m_row += BLOCK_M) {
            const int row0 = m_row + quarter * 32;               // first row of this warp's 32-row block
            const int M = row0 < row_end ? row_end : 0;          // rows >= row_end belong to the next CTA: mask them
            if (M == 0) {                                        // this warp's 32-row block is past the CTA's range
                tc::mbar_wait(tfull_bar(as), aph);               // (warp-uniform; the partner column-half warp skips too)
                tc::tc_fence_before();
                tc::mbar_arrive(tempty_bar(as));
                ++etile;
                if (++as == 2) { as = 0; aph ^= 1; }
                continue;
            }
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + as * 256;
            // coalesced fetch of a [32 rows x 32 cols] fp32 block (rows row0.., columns c..c+31) into registers
            float4 pre[8];
            auto fetch = [&](const float* base, int ld, int c) {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int r = row0 + 4 * i + crow;
                    pre[i] = (base != nullptr && r < M) ? __ldg(reinterpret_cast<const float4*>(base + (size_t)r * ld + c) + cpiece)
                                                        : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            };
            // registers (coalesced shape) -> staging -> this thread's row (v[32])
            auto to_rows = [&](float (&v)[32]) {
#pragma unroll
                for (int i = 0; i < 8; ++i) sts4(4 * i + crow, cpiece, pre[i]);
                __syncwarp();
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float4 t = lds4(lane, j);
                    v[4 * j] = t.x; v[4 * j + 1] = t.y; v[4 * j + 2] = t.z; v[4 * j + 3] = t.w;
                }
                __syncwarp();
            };
            if constexpr (!LN) {
                if (!(sizeof(TC) == 2 && c_tma != 0))
                    fetch(residual, N, n_blk * BN + cbeg);       // independent of the MMA: issue before waiting on it
                tc::mbar_wait(tfull_bar(as), aph);
                if (warp == 2 && lane == 0 && etile < 3) stamp(4 + etile * 3);      // accumulator ready
                tc::tc_fence_after();
            }
            if constexpr (LN) {
                // Residual stream (residual, y_f32) and pos live in the T32 block layout: the thread that owns row
                // `lane` of this warp's 32-row block reads / writes piece j of chunk cb at
                // ((R*8 + cb)*8 + j)*32 + lane  (float4 units) -- 512 contiguous bytes per warp instruction, no
                // shared-memory transpose.  Only the row-major bf16 operand copies go through the staging block.
                const size_t blk4 = (size_t)(row0 >> 5) * 8 * 8 * 32 + lane;          // float4 index of (R, cb=0, j=0, lane)
                auto t32_load = [&](const float* base, int c0, float4 (&dst)[8]) {
                    const float4* p4 = reinterpret_cast<const float4*>(base) + blk4 + (size_t)(c0 >> 5) * 256;
#pragma unroll
                    for (int j = 0; j < 8; ++j) dst[j] = __ldg(p4 + j * 32);
                };
                float sum = 0.f, sumsq = 0.f;
                float4 nxt[8];
                t32_load(residual, cbeg, nxt);
                tc::mbar_wait(tfull_bar(as), aph);
                if (warp == 2 && lane == 0 && etile < 3) stamp(4 + etile * 3);          // accumulator ready
                tc::tc_fence_after();
#pragma unroll
                for (int ci = 0; ci < 4; ++ci) {                 // 128 columns = 4 chunks per warp
                    const int c0 = cbeg + ci * 32;
                    float4 q[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) q[j] = nxt[j];
                    if (ci + 1 < 4) t32_load(residual, c0 + 32, nxt);
                    uint32_t r[32];
                    tc::tmem_ld32(taddr + c0, r);
                    tc::tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float4 b = reinterpret_cast<const float4*>(cvec + c0)[i];
                        const float x0 = __uint_as_float(r[4 * i]) + b.x + q[i].x, x1 = __uint_as_float(r[4 * i + 1]) + b.y + q[i].y;
                        const float x2 = __uint_as_float(r[4 * i + 2]) + b.z + q[i].z, x3 = __uint_as_float(r[4 * i + 3]) + b.w + q[i].w;
                        sum += (x0 + x1) + (x2 + x3);
                        sumsq = fmaf(x0, x0, fmaf(x1, x1, fmaf(x2, x2, fmaf(x3, x3, sumsq))));
                        r[4 * i] = __float_as_uint(x0); r[4 * i + 1] = __float_as_uint(x1);
                        r[4 * i + 2] = __float_as_uint(x2); r[4 * i + 3] = __float_as_uint(x3);
                    }
                    tc::tmem_st32(taddr + c0, r);
                }
                if (ln.y_pos_bf16) t32_load(ln.pos, cbeg, nxt);
                // exchange the half-row statistics with the warp that owns the other 128 columns of these rows
                part[half * 128 + quarter * 32 + lane] = make_float2(sum, sumsq);
                tc::tmem_st_wait();
                asm volatile("bar.sync %0, 64;" ::"r"(1 + quarter) : "memory");
                const float2 other = part[(half ^ 1) * 128 + quarter * 32 + lane];
                const float mean = (sum + other.x) * (1.f / 256.f);
                const float var = fmaxf((sumsq + other.y) * (1.f / 256.f) - mean * mean, 0.f);
                const float rstd = rsqrtf(var + 1e-5f);
#pragma unroll
                for (int ci = 0; ci < 4; ++ci) {
                    const int c0 = cbeg + ci * 32;
                    uint32_t r[32];
                    tc::tmem_ld32(taddr + c0, r);
                    tc::tmem_ld_wait();
                    float4* yo = reinterpret_cast<float4*>(ln.y_f32) + blk4 + (size_t)(c0 >> 5) * 256;
#pragma unroll
                    // bf16 copies: my row -> swizzled staging ([32 rows x 64 B], SWIZZLE_64B: 16-byte piece p of row r at
                    // p ^ ((r >> 1) & 3)) -> one TMA store per [32 x 32] block (was: staging + LDS + per-lane STG.128)
                    if (lane == 0) tc::tma_store_wait_read();
                    __syncwarp();
                    const uint32_t srow = stg + lane * 64, swz = (lane >> 1) & 3;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {                // normalise my row: fp32 straight to T32
                        const float4 g = reinterpret_cast<const float4*>(cvec + 256 + c0)[j];
                        const float4 be = reinterpret_cast<const float4*>(cvec + 512 + c0)[j];
                        float4 y;
                        y.x = (__uint_as_float(r[4 * j]) - mean) * rstd * g.x + be.x;
                        y.y = (__uint_as_float(r[4 * j + 1]) - mean) * rstd * g.y + be.y;
                        y.z = (__uint_as_float(r[4 * j + 2]) - mean) * rstd * g.z + be.z;
                        y.w = (__uint_as_float(r[4 * j + 3]) - mean) * rstd * g.w + be.w;
                        if (ln.y_f32) yo[j * 32] = y;
                        const uint32_t dst = srow + ((((uint32_t)j >> 1) ^ swz) << 4) + (j & 1) * 8;
                        asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(dst), "r"(pack_bf16x2(y.x, y.y)), "r"(pack_bf16x2(y.z, y.w)) : "memory");
                        if (ln.y_pos_bf16) {
                            const float4 p4 = nxt[j];
                            asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(dst + 2048), "r"(pack_bf16x2(y.x + p4.x, y.y + p4.y)),
                                         "r"(pack_bf16x2(y.z + p4.z, y.w + p4.w)) : "memory");
                        }
                    }
                    if (ln.y_pos_bf16 && ci + 1 < 4) t32_load(ln.pos, c0 + 32, nxt);
                    tc::fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) {
                        if (ln.y_bf16) { tc::tma_store_3d(&tmC, stg, c0, row0, 0); tc::tma_store_commit(); }
                        if (ln.y_pos_bf16) { tc::tma_store_3d(&tmC2, stg + 2048, c0, row0, 0); tc::tma_store_commit(); }
                    }
                }
            } else if (sizeof(TC) == 2 && c_tma != 0) {
                // 16-bit outputs: accumulator row -> bias/act -> packed 16-bit -> swizzled staging rows -> ONE TMA store
                // per [32 rows x box] block.  No shared-memory read-back, no per-lane global stores: the LSU only sees
                // the 16-byte STS of each thread's own row (conflict-free under the TMA swizzle).
                constexpr int box = 32;                          // columns per store (= tensor map box; 2 KB staging block per warp)
                for (int c0 = cbeg; c0 < cbeg + ncol; c0 += box) {
                    const int col = n_blk * BN + c0;
                    float4 kq[8];                                // epilogue constant of this thread's row, 32 columns
                    if (res_t32) {
                        const float4* p4 = reinterpret_cast<const float4*>(res_t32) +
                                           ((size_t)(row0 >> 5) * (N >> 5) + (size_t)(col >> 5)) * 256 + lane;
#pragma unroll
                        for (int j = 0; j < 8; ++j) kq[j] = __ldg(p4 + j * 32);
                    }
                    uint32_t r[32];
                    tc::tmem_ld32(taddr + c0, r);
                    tc::tmem_ld_wait();
                    uint32_t pk[16];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {                // 4 columns per step (bias is warp-uniform: broadcast loads)
                        const float4 b4 = reinterpret_cast<const float4*>(cvec + c0)[j];
                        float x0 = __uint_as_float(r[4 * j]) + b4.x, x1 = __uint_as_float(r[4 * j + 1]) + b4.y;
                        float x2 = __uint_as_float(r[4 * j + 2]) + b4.z, x3 = __uint_as_float(r[4 * j + 3]) + b4.w;
                        if (res_t32) { x0 += kq[j].x; x1 += kq[j].y; x2 += kq[j].z; x3 += kq[j].w; }
                        if (act == ACT_RELU) { x0 = fmaxf(x0, 0.f); x1 = fmaxf(x1, 0.f); x2 = fmaxf(x2, 0.f); x3 = fmaxf(x3, 0.f); }
                        if (out_half) {
                            const __half2 a = __floats2half2_rn(x0, x1), b = __floats2half2_rn(x2, x3);
                            pk[2 * j] = *reinterpret_cast<const uint32_t*>(&a); pk[2 * j + 1] = *reinterpret_cast<const uint32_t*>(&b);
                        } else {
                            pk[2 * j] = pack_bf16x2(x0, x1); pk[2 * j + 1] = pack_bf16x2(x2, x3);
                        }
                    }
                    if (lane == 0) tc::tma_store_wait_read();    // the previous store has drained the staging block
                    __syncwarp();
                    // 64-byte rows, SWIZZLE_64B: piece j -> j ^ ((row >> 1) & 3)
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(stg + lane * 64 + ((j ^ ((lane >> 1) & 3)) << 4)),
                                     "r"(pk[4 * j]), "r"(pk[4 * j + 1]), "r"(pk[4 * j + 2]), "r"(pk[4 * j + 3]) : "memory");
                    tc::fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) {
                        if (c_tma == 2) tc::tma_store_3d(&tmC, stg, c0, row0, n_blk);
                        else            tc::tma_store_3d(&tmC, stg, col, row0, 0);
                        tc::tma_store_commit();
                    }
                }
            } else {
                const int nchunk = ncol >> 5;                    // BN/2 is a multiple of 32 for every plan (<= 4 chunks)
#pragma unroll
                for (int ci = 0; ci < 4; ++ci) {
                    if (ci >= nchunk) break;
                    const int c0 = cbeg + ci * 32;
                    const int col = n_blk * BN + c0;
                    uint32_t r[32];
                    tc::tmem_ld32(taddr + c0, r);
                    tc::tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 8; ++j)                  // stage my row of the accumulator
                        sts4(lane, j, make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]),
                                                  __uint_as_float(r[4 * j + 2]), __uint_as_float(r[4 * j + 3])));
                    __syncwarp();
                    const float4 b4 = reinterpret_cast<const float4*>(cvec + c0)[cpiece];
#pragma unroll
                    for (int i = 0; i < 8; ++i) {                // bias / act / residual / store in the coalesced shape
                        const int rr = 4 * i + crow, grow = row0 + rr;
                        float4 v = lds4(rr, cpiece);
                        v.x += b4.x; v.y += b4.y; v.z += b4.z; v.w += b4.w;
                        if (act == ACT_RELU) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
                        if (residual) { const float4 q = pre[i]; v.x += q.x; v.y += q.y; v.z += q.z; v.w += q.w; }
                        if (grow < M) {
                            // default (ldc = N, nblk_stride = BN) is the plain row-major [M,N]; the blocked form
                            // writes each n-block as its own contiguous [M,BN] matrix (per-layer value buffers)
                            const size_t o = (size_t)n_blk * nblk_stride + (size_t)grow * ldc + c0 + cpiece * 4;
                            if constexpr (sizeof(TC) == 4) {
                                *reinterpret_cast<float4*>(reinterpret_cast<float*>(C) + o) = v;
                            } else if (out_half) {
                                const __half2 lo = __floats2half2_rn(v.x, v.y), hi = __floats2half2_rn(v.z, v.w);
                                *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(C) + o) =
                                    make_uint2(*reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
                            } else {
                                *reinterpret_cast<uint2*>(reinterpret_cast<bf16*>(C) + o) =
                                    make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
                            }
                        }
                    }
                    __syncwarp();
                    if (residual && ci + 1 < nchunk) fetch(residual, N, col + 32);
                }
            }
            tc::tc_fence_before();
            tc::mbar_arrive(tempty_bar(as));
            if (warp == 2 && lane == 0 && etile < 3) stamp(5 + etile * 3);          // epilogue of tile done
            ++etile;
            if (++as == 2) { as = 0; aph ^= 1; }
        }
    }
    if ((LN || c_tma != 0) && warp >= 2 && lane == 0) tc::tma_store_wait_all();   // output stores performed before the grid completes
    tc::tc_fence_before();
    __syncthreads();
    if (threadIdx.x == 0) stamp(15);
    if (warp == 1) {
        tc::tc_fence_after();
        tc::tmem_dealloc(tmem_base, 512);
    }
}

// tile-N choice: prefer a weight block that fits resident (<= 128 KB) next to >= 4 A stages
struct Plan { int BN, resident, stages, smem; };

Plan make_plan(int N, int K, bool ln, int stg_bytes = 4096)
{
    const int SMEM_TAIL = smem_tail(ln, stg_bytes), SMEM_LIMIT = SMEM_MAX - SMEM_TAIL;
    Plan p{0, 0, 0, 0};
    const int cands[] = {256, 192, 128, 64};                  // BN/2 must be a multiple of 32 (epilogue column split)
    if (ln) {
        p.BN = 256;
    } else {
        for (int bn : cands) {
            if (N % bn != 0 || bn > N) continue;
            if ((long)bn * K * 2 <= 131072) { p.BN = bn; break; }
        }
        if (K > 512 && p.BN != 0 && p.BN < 128) p.BN = 0;     // split-operand GEMMs (K' = 3K): a 64-wide resident block would
                                                              // re-read A once per 64 columns; stream W with a wide tile instead
        if (p.BN == 0) {                                      // no resident candidate: largest tile that divides N
            for (int bn : cands) if (N % bn == 0 && bn <= N) { p.BN = bn; break; }
        }
        if (p.BN == 0 && N <= 256 && N % 64 == 0) p.BN = N;
    }
    if (p.BN == 0) return p;
    const int w_bytes = p.BN * K * 2;
    p.resident = w_bytes <= 131072;
    const int stage = A_TILE_BYTES + (p.resident ? 0 : p.BN * BLOCK_K * 2);
    const int avail = SMEM_LIMIT - (p.resident ? w_bytes : 0);
    p.stages = avail / stage;
    if (p.stages > MAX_STAGES) p.stages = MAX_STAGES;
    p.smem = 1024 + (p.resident ? w_bytes : 0) + p.stages * stage + SMEM_TAIL;
    return p;
}

struct MapKey {
    const void* p; uint64_t d0, d1, ld; uint32_t b0, b1;
    bool operator<(const MapKey& o) const { return std::tie(p, d0, d1, ld, b0, b1) < std::tie(o.p, o.d0, o.d1, o.ld, o.b0, o.b1); }
};

}  // namespace

// row-major bf16 [rows, inner] with a row pitch of `ld` elements (0 = dense)
int cached_map_2d(const void* base, uint64_t inner, uint64_t rows, uint32_t box_inner, uint32_t box_rows, CUtensorMap* out,
                  uint64_t ld)
{
    static std::map<MapKey, CUtensorMap> cache;
    static std::mutex mu;
    std::lock_guard<std::mutex> g(mu);
    if (ld == 0) ld = inner;
    const MapKey k{base, inner, rows, ld, box_inner, box_rows};
    auto it = cache.find(k);
    if (it == cache.end()) {
        CUtensorMap m;
        const uint64_t dims[2] = {inner, rows}, strides[1] = {ld * 2};
        const uint32_t box[2] = {box_inner, box_rows};
        if (make_tensor_map_bf16(&m, base, 2, dims, strides, box, 128)) return 1;
        if (cache.size() > 4096) cache.clear();
        it = cache.emplace(k, m).first;
    }
    *out = it->second;
    return 0;
}

// output tensor map for the TMA-store epilogue: dims {cols, rows, blocks}, 2-byte elements, box {box_cols, 32, 1}
int cached_map_out(const void* base, uint64_t cols, uint64_t rows, uint64_t blocks, uint32_t box_cols, CUtensorMap* out)
{
    static std::map<std::tuple<const void*, uint64_t, uint64_t, uint64_t, uint32_t>, CUtensorMap> cache;
    static std::mutex mu;
    std::lock_guard<std::mutex> g(mu);
    const auto k = std::make_tuple(base, cols, rows, blocks, box_cols);
    auto it = cache.find(k);
    if (it == cache.end()) {
        CUtensorMap m;
        const uint64_t dims[3] = {cols, rows, blocks}, strides[2] = {cols * 2, rows * cols * 2};
        const uint32_t box[3] = {box_cols, 32, 1};
        if (make_tensor_map_bf16(&m, base, 3, dims, strides, box, (int)box_cols * 2)) return 1;
        if (cache.size() > 4096) cache.clear();
        it = cache.emplace(k, m).first;
    }
    *out = it->second;
    return 0;
}

namespace {

// Fills one problem (tensor maps, plan, CTA share).  ctas = number of CTAs this problem may use (0: all SMs).
template <typename TC, bool LN>
int build_prob(GemmProb& P, int& smem, const bf16* A, const bf16* A2, int K1, const bf16* W, const float* bias, const float* residual,
               TC* C, int M, int N, int K, int act, bool blocked_out, int lda, int lda2, int ctas, int cta_begin)
{
    if (A2 == nullptr) K1 = K;
    // 16-bit outputs without a residual leave through TMA stores of [32 rows x 32 columns]: a 2 KB staging block per warp
    // instead of 4 KB, which buys one or two more operand stages
    const bool use_tma_store = !LN && sizeof(TC) == 2 && residual == nullptr && C != nullptr;
    const int stg_bytes = use_tma_store ? 2048 : 4096;
    const Plan p = make_plan(N, K, LN, stg_bytes);
    OCC_CHECK(p.BN > 0 && p.stages >= 2 && K % 64 == 0 && K1 % 64 == 0 && M > 0, "gemm_tc: unsupported shape");
    if (cached_map_2d(A, (uint64_t)K1, (uint64_t)M, BLOCK_K, BLOCK_M, &P.tmA, (uint64_t)lda)) return 1;
    if (A2) { if (cached_map_2d(A2, (uint64_t)(K - K1), (uint64_t)M, BLOCK_K, BLOCK_M, &P.tmA2, (uint64_t)lda2)) return 1; }
    else P.tmA2 = P.tmA;
    if (cached_map_2d(W, (uint64_t)K, (uint64_t)N, BLOCK_K, (uint32_t)p.BN, &P.tmW)) return 1;
    P.tmC = P.tmW; P.tmC2 = P.tmW;
    P.c_tma = 0;
    if (use_tma_store) {
        const uint32_t box_cols = 32u;
        if (blocked_out) {
            if (cached_map_out(C, (uint64_t)p.BN, (uint64_t)M, (uint64_t)(N / p.BN), box_cols, &P.tmC)) return 1;
            P.c_tma = 2;
        } else {
            if (cached_map_out(C, (uint64_t)N, (uint64_t)M, 1, box_cols, &P.tmC)) return 1;
            P.c_tma = 1;
        }
    }
    if (ctas <= 0) ctas = sm_count_current_device();
    const int m_tiles = (M + BLOCK_M - 1) / BLOCK_M, n_tiles = N / p.BN;
    int per_n = ctas / n_tiles;
    if (per_n > m_tiles) per_n = m_tiles;                        // (row ranges are dealt in 32-row blocks: >= 1 per CTA)
    OCC_CHECK(per_n >= 1, "gemm_tc: fewer CTAs than n-blocks");
    P.bias = bias; P.residual = residual; P.C = C; P.res_t32 = nullptr;
    P.ldc = blocked_out ? (long long)p.BN : (long long)N;
    P.nblk_stride = blocked_out ? (long long)M * p.BN : (long long)p.BN;
    P.stg_bytes = stg_bytes; P.M = M; P.N = N; P.BN = p.BN; P.nk = K / BLOCK_K; P.nk1 = K1 / BLOCK_K; P.act = act;
    P.w_resident = p.resident; P.stages = p.stages;
    P.out_half = std::is_same<TC, __half>::value ? 1 : 0;
    P.cta_begin = cta_begin; P.cta_count = per_n * n_tiles;
    smem = p.smem;
    return 0;
}

template <typename TC, bool LN>
int launch_probs(const GemmProbs& probs, int smem, LnArgs ln, cudaStream_t stream)
{
    // per-device attribute (cheap): a process-wide `static bool` would leave a second device without the opt-in
    OCC_CUDA(cudaFuncSetAttribute(gemm_tc_kernel<TC, LN>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
    const GemmProb& last = probs.p[probs.n - 1];
    const int grid = last.cta_begin + last.cta_count;
    long long* dbg = nullptr;
    static const bool want_dbg = getenv("OCC_GEMM_TIMELINE") != nullptr;
    if (want_dbg) {
        OCC_CUDA(cudaMalloc(&dbg, (size_t)grid * 16 * sizeof(long long)));
        OCC_CUDA(cudaMemsetAsync(dbg, 0, (size_t)grid * 16 * sizeof(long long), stream));
    }
    {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(grid); cfg.blockDim = dim3(NUM_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        OCC_CUDA(cudaLaunchKernelEx(&cfg, gemm_tc_kernel<TC, LN>, probs, ln, dbg));
    }
    OCC_CUDA(cudaGetLastError());
    if (want_dbg) {                                               // development aid: per-CTA timeline in ns
        std::vector<long long> h((size_t)grid * 16);
        OCC_CUDA(cudaStreamSynchronize(stream));
        OCC_CUDA(cudaMemcpy(h.data(), dbg, h.size() * sizeof(long long), cudaMemcpyDeviceToHost));
        cudaFree(dbg);
        long long t0 = h[0];
        for (int b = 0; b < grid; ++b) if (h[(size_t)b * 16] && h[(size_t)b * 16] < t0) t0 = h[(size_t)b * 16];
        for (int q = 0; q < probs.n; ++q)
            fprintf(stderr, "[gemm timeline] problem %d: M=%d N=%d K=%d BN=%d resident=%d stages=%d ctas=%d LN=%d\n", q, probs.p[q].M,
                    probs.p[q].N, probs.p[q].nk * BLOCK_K, probs.p[q].BN, probs.p[q].w_resident, probs.p[q].stages,
                    probs.p[q].cta_count, (int)LN);
        const int show[] = {0, 1, grid / 2, grid - 1};
        for (int b : show) {
            fprintf(stderr, "  cta %3d:", b);
            for (int i = 0; i < 16; ++i) fprintf(stderr, " %6lld", h[(size_t)b * 16 + i] ? h[(size_t)b * 16 + i] - t0 : -1);
            fprintf(stderr, "\n");
        }
    }
    return 0;
}

template <typename TC, bool LN>
int launch(const bf16* A, const bf16* A2, int K1, const bf16* W, const float* bias, const float* residual, TC* C,
           LnArgs ln, int M, int N, int K, int act, cudaStream_t stream, bool blocked_out = false, int lda = 0, int lda2 = 0)
{
    GemmProbs probs;
    probs.n = 1;
    int smem = 0;
    if (build_prob<TC, LN>(probs.p[0], smem, A, A2, K1, W, bias, residual, C, M, N, K, act, blocked_out, lda, lda2, 0, 0))
        return 1;
    return launch_probs<TC, LN>(probs, smem, ln, stream);
}

}  // namespace

bool gemm_tc_supported(int M, int N, int K, int K1)
{
    const Plan p = make_plan(N, K, false);
    return M > 0 && p.BN >= 64 && p.BN % 64 == 0 && p.stages >= 2 && K % 64 == 0 && K1 % 64 == 0 && K1 > 0 && K1 <= K;
}

template <typename TC>
int gemm_tc(const bf16* A, const bf16* A2, int K1, const bf16* W, const float* bias, const float* residual, TC* C,
            int M, int N, int K, int act, cudaStream_t stream)
{
    return launch<TC, false>(A, A2, K1, W, bias, residual, C, LnArgs{}, M, N, K, act, stream);
}

// fp32-grade GEMM on the tensor cores: S = [hi | lo] (bf16 split of an fp32 operand, row pitch 2*Ks), W3 = [W_hi | W_hi | W_lo]
// (N x 3*Ks).  C = hi.W_hi + lo.W_hi + hi.W_lo  (the lo.lo term, 2^-16 relative, is dropped) as ONE GEMM with K' = 3*Ks whose
// A operand is the concatenation [S (2*Ks columns) | first Ks columns of S again] -- two tensor maps over the same buffer.
int gemm_tc_split3(const bf16* S, int Ks, const bf16* W3, const float* bias, const float* residual, float* C, int M, int N,
                   int act, cudaStream_t stream)
{
    return launch<float, false>(S, S, 2 * Ks, W3, bias, residual, C, LnArgs{}, M, N, 3 * Ks, act, stream, false, 2 * Ks, 2 * Ks);
}

int gemm_tc_blocked256(const bf16* A, const bf16* W, const float* bias, bf16* C, int M, int N, int K, cudaStream_t stream)
{
    const Plan p = make_plan(N, K, false);
    OCC_CHECK(p.BN == 256 && N % 256 == 0, "gemm_tc_blocked256: N must be a multiple of 256 with 256-wide tiles");
    return launch<bf16, false>(A, nullptr, 0, W, bias, nullptr, C, LnArgs{}, M, N, K, ACT_NONE, stream, true);
}

// residual, y_f32 and pos are in the T32 block layout (elementwise.cu), rows padded to a multiple of 32
int gemm_tc_ln(const bf16* A, const bf16* W, const float* bias, const float* residual, const float* gamma,
               const float* beta, const float* pos, float* y_f32, bf16* y_bf16, bf16* y_pos_bf16, int M, int K,
               cudaStream_t stream)
{
    OCC_CHECK(bias && residual && gamma && beta, "gemm_tc_ln: bias, residual, gamma, beta are required");
    OCC_CHECK(y_pos_bf16 == nullptr || pos != nullptr, "gemm_tc_ln: pos required for y_pos");
    GemmProbs probs;
    probs.n = 1;
    int smem = 0;
    if (build_prob<float, true>(probs.p[0], smem, A, nullptr, 0, W, bias, residual, (float*)nullptr, M, 256, K, ACT_NONE, false, 0, 0, 0, 0))
        return 1;
    // the bf16 copies of the LayerNorm output leave through TMA stores of [32 rows x 32 columns]
    probs.p[0].tmC2 = probs.p[0].tmC;
    if (y_bf16 && cached_map_out(y_bf16, 256, (uint64_t)M, 1, 32u, &probs.p[0].tmC)) return 1;
    if (y_pos_bf16 && cached_map_out(y_pos_bf16, 256, (uint64_t)M, 1, 32u, &probs.p[0].tmC2)) return 1;
    return launch_probs<float, true>(probs, smem, LnArgs{gamma, beta, pos, y_f32, y_bf16, y_pos_bf16}, stream);
}

// Two (or three) independent 16-bit-output GEMMs in ONE launch: the CTAs are shared out in proportion to N.K.
//   value problems: Cv[i] = Av[i].Wv^T + bv (bf16, [M,256], TMA-store epilogue), i < nv <= 2  (TSA value_proj of each queue entry)
//   projection    : Cq = [Aq | Aq2].Wq^T + bq (+ rq, fp32 [M,Nq]) as fp16                  (sampling offsets + attention logits)
int gemm_tc_tsa_inputs(const bf16* const* Av, int nv, const bf16* Wv, const float* bv, bf16* const* Cv, const bf16* Aq,
                       const bf16* Aq2, int K1q, const bf16* Wq, const float* bq, const float* rq, const float* rq_t32, __half* Cq,
                       int M, int Nq, int Kq, cudaStream_t stream)
{
    OCC_CHECK(nv >= 1 && nv <= 2, "gemm_tc_tsa_inputs: 1 or 2 value problems");
    const int num_sms = sm_count_current_device();
    const double wv = 256.0 * 256.0, wq = (double)Nq * Kq, tot = nv * wv + wq;
    int cq = (int)(num_sms * wq / tot + 0.5);
    const int nq_tiles = Nq / make_plan(Nq, Kq, false, (rq && !rq_t32) ? 4096 : 2048).BN;
    if (cq < nq_tiles) cq = nq_tiles;
    const int cv = (num_sms - cq) / nv;
    OCC_CHECK(cv >= 1, "gemm_tc_tsa_inputs: not enough SMs");
    GemmProbs probs;
    probs.n = nv + 1;
    int smem = 0, sm = 0, begin = 0;
    for (int i = 0; i < nv; ++i) {
        if (build_prob<bf16, false>(probs.p[i], sm, Av[i], nullptr, 0, Wv, bv, nullptr, Cv[i], M, 256, 256, ACT_NONE, false, 0, 0, cv,
                                    begin)) return 1;
        begin += probs.p[i].cta_count;
        smem = sm > smem ? sm : smem;
    }
    // (built through the bf16 instantiation: out_half selects the fp16 packing at run time)
    // rq_t32: the epilogue constant in the T32 layout -> the projection leaves through the TMA-store epilogue as well (the
    // row-major fp32 `rq` forces the staged per-lane epilogue: 4.2-5.5 us per tile instead of 2.1, in-kernel timeline r2 call 8)
    const bool t32 = rq_t32 != nullptr && M % 32 == 0;
    if (build_prob<bf16, false>(probs.p[nv], sm, Aq, Aq2, K1q, Wq, bq, t32 ? nullptr : rq, reinterpret_cast<bf16*>(Cq), M, Nq, Kq,
                                ACT_NONE, false, 0, 0, cq, begin)) return 1;
    probs.p[nv].out_half = 1;
    if (t32) {
        OCC_CHECK(probs.p[nv].c_tma == 1 && probs.p[nv].stg_bytes == 2048, "gemm_tc_tsa_inputs: T32 constant needs the 32-column TMA-store epilogue");
        probs.p[nv].res_t32 = rq_t32;
    }
    smem = sm > smem ? sm : smem;
    return launch_probs<bf16, false>(probs, smem, LnArgs{}, stream);
}

template int gemm_tc<float>(const bf16*, const bf16*, int, const bf16*, const float*, const float*, float*, int, int,
                            int, int, cudaStream_t);
template int gemm_tc<bf16>(const bf16*, const bf16*, int, const bf16*, const float*, const float*, bf16*, int, int, int,
                           int, cudaStream_t);
template int gemm_tc<__half>(const bf16*, const bf16*, int, const bf16*, const float*, const float*, __half*, int, int, int,
                             int, cudaStream_t);

}  // namespace occ
