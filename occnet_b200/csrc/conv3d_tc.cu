// Voxel decoder on the 5th-gen tensor cores (sm_100a): 3x3x3 Conv3d (pad 1, no bias) + folded
// BatchNorm3d + ReLU as an implicit GEMM.   Reference: TransformerOcc.decoder (use_3d),
// projects/mmdet3d_plugin/bevformer/modules/transformer_occ.py:106-131, applied at :305-308.
//
// Tensors are channels-last bf16 [X][Y][Z][C] (see decoder_simt.cu for the layout rationale).
//   M tile  = 128 voxels = 8 (y) x 16 (z, the whole pillar) at one x
//   N       = 32 output channels,  K = 27 taps x Cin
// im2col is done by TMA: one 4-D box load {Cin, 16 z, 8 + 2 y, 1 x} per (plane, dz) with the dz offset in the
// coordinates and a one-row y halo on both sides, so the three dy shifts are SUB-VIEWS of the same shared-memory tile
// (row offset dy * 16, a multiple of the 8-row swizzle atom); out-of-bounds rows are zero-filled by the TMA unit, which
// IS the conv's zero padding (including the z = -1 / z = 16 halo).  All 27 weight tiles stay resident in shared memory.
//   warp 0: TMA producer (8-stage ring)    warp 1: tcgen05.mma issuer (plane-major: each loaded tile feeds the
//   dx = 0/1/2 taps of three neighbouring outputs through ONE N = 96 MMA into adjacent TMEM slots, ring of 8)
//   warps 2-5: epilogue (tcgen05.ld -> +bias -> ReLU -> bf16 -> 64-byte rows, contiguous 8 KB per tile)
#include "common.cuh"
#include "conv3d_tc.cuh"
#include "tc_common.cuh"

namespace occ {

namespace {

constexpr int STAGES = 8, TILE_Y = 8, TILE_Z = 16, BLOCK_M = 128, COUT = 32, TAPS = 27, SLOTS = 8;
constexpr int HALO_ROWS = (TILE_Y + 2) * TILE_Z;          // rows of one staged tile: y0-1 .. y0+8, all 16 z
constexpr int NUM_THREADS = 192;
constexpr int BAR_BYTES = 512;

// Plane-major schedule: an input tile (plane x = p, shift (dz,dy)) is the A operand of three taps -- dx = 0, 1, 2 of
// the outputs x = p+1, p, p-1 -- so it is loaded ONCE (L2->SMEM traffic: ~9 instead of 27 tile loads per output tile)
// and multiplied into the three live accumulators with ONE tcgen05.mma of N = 96: the accumulators of consecutive
// outputs sit in consecutive 32-column TMEM slots (ring of 8), and the weight tiles of a (dz,dy) pair are resident in
// the order dx = 2, 1, 0, i.e. ascending output x.  (The first version issued three N = 32 MMAs per tile: ncu showed
// the single MMA-issuing thread, not TMA or the tensor pipe, was the limiter -- ~64 pipe cycles and ~180 issue-thread
// cycles per tiny MMA.)  Accumulators are zeroed by the epilogue warps when they drain a slot, so every MMA
// accumulates and the issue loop has no per-output special cases.
// Each CTA owns a contiguous range of the (y_tile, x) tile sequence, cut into segments of constant y_tile; a segment
// [xa, xb) streams the planes max(xa-1,0) .. min(xb, X-1).
// The producer / issuer warps run their loops with ALL 32 lanes (lane 0 alone issues the TMA loads, elect.sync picks the lane
// that issues the MMAs and commits): loop counters, stage indices and UMMA descriptors are then warp-uniform values the compiler
// keeps in the uniform datapath, instead of per-lane registers that need an R2UR move in front of every tcgen05.mma operand (ncu
// of a lane-0-only version: 1.8 M R2UR + 1.3 M IMAD around 0.19 M MMAs; the issuing thread, not the tensor pipe, was the limiter).
// EPI: 0 = bf16 out = relu(acc + bias) (the bf16 configuration); fp32-storage configuration, one of three split passes
// (hi.W_hi, lo.W_hi, hi.W_lo of the bf16 split of an fp32 input, relative error ~2^-16 like gemm_tc_split3):
// 1 = out_f32 = acc, 2 = out_f32 += acc, 3 = out_f32 = relu(out_f32 + acc + bias).  Every output row is owned by one thread per
// pass, so the fp32 accumulation across passes needs no atomics.
template <int CIN, int EPI>
__global__ void __launch_bounds__(NUM_THREADS, 1)
conv3d_tc_kernel(const __grid_constant__ CUtensorMap tmIn, const __grid_constant__ CUtensorMap tmW,
                 const float* __restrict__ bias, bf16* __restrict__ out, float* __restrict__ out_f32, int X, int Y)
{
    constexpr int ROW_BYTES = CIN * 2;                       // 32 (SWIZZLE_32B) or 64 (SWIZZLE_64B)
    constexpr int A_BYTES = HALO_ROWS * ROW_BYTES;           // 5 / 10 KB per stage (three dy sub-views of 128 rows)
    constexpr int DY_BYTES = TILE_Z * ROW_BYTES;             // one y row of the tile
    constexpr int W_TAP_BYTES = COUT * ROW_BYTES;            // 1 / 2 KB per tap
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (tc::smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t w_base = smem_base;                                       // 27 weight tiles, resident
    const uint32_t a_base = smem_base + ((TAPS * W_TAP_BYTES + 1023) & ~1023);
    const uint32_t bar_base = a_base + STAGES * A_BYTES;
    auto full_bar = [&](int s) { return bar_base + s * 8; };
    auto empty_bar = [&](int s) { return bar_base + (STAGES + s) * 8; };
    auto tfull_bar = [&](int s) { return bar_base + (2 * STAGES + s) * 8; };
    auto tempty_bar = [&](int s) { return bar_base + (2 * STAGES + SLOTS + s) * 8; };
    const uint32_t w_bar = bar_base + (2 * STAGES + 2 * SLOTS) * 8;
    const uint32_t tmem_slot = bar_base + (2 * STAGES + 2 * SLOTS + 1) * 8;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int y_tiles = (Y + TILE_Y - 1) / TILE_Y;
    const long long total = (long long)X * y_tiles;
    const int t_begin = (int)(total * blockIdx.x / gridDim.x), t_end = (int)(total * (blockIdx.x + 1) / gridDim.x);

    if (warp == 0 && lane == 0) {
        tc::tma_prefetch_desc(&tmIn); tc::tma_prefetch_desc(&tmW);
        for (int s = 0; s < STAGES; ++s) { tc::mbar_init(full_bar(s), 1); tc::mbar_init(empty_bar(s), 1); }
        for (int s = 0; s < SLOTS; ++s) { tc::mbar_init(tfull_bar(s), 1); tc::mbar_init(tempty_bar(s), 128); }
        tc::mbar_init(w_bar, 1);
        tc::mbar_fence_init();
    }
    if (warp == 1) tc::tmem_alloc(tmem_slot, 32 * SLOTS);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

    const bool leader = lane == 0;
    if (warp == 0) {
        if (leader) {
            tc::mbar_arrive_expect_tx(w_bar, TAPS * W_TAP_BYTES);
            for (int t = 0; t < TAPS; ++t)                   // global tap order is (dz,dy,dx); resident order (dz,dy,2-dx)
                tc::tma_load_2d(w_base + ((t / 3) * 3 + (2 - t % 3)) * W_TAP_BYTES, &tmW, w_bar, 0, t * COUT);
        }
        int s = 0; uint32_t ph = 0;
        for (int t = t_begin; t < t_end;) {
            const int yt = t / X, xa = t % X;
            const int xb = min(X, xa + (t_end - t));
            const int y0 = yt * TILE_Y;
            const int p_lo = max(xa - 1, 0), p_hi = min(xb, X - 1);
            for (int p = p_lo; p <= p_hi; ++p) {
                for (int dz = 0; dz < 3; ++dz) {
                    tc::mbar_wait(empty_bar(s), ph ^ 1);
                    if (leader) {
                        tc::mbar_arrive_expect_tx(full_bar(s), A_BYTES);
                        tc::tma_load_4d(a_base + s * A_BYTES, &tmIn, full_bar(s), 0, dz - 1, y0 - 1, p);
                    }
                    if (++s == STAGES) { s = 0; ph ^= 1; }
                }
            }
            t += xb - xa;
        }
    } else if (warp == 1) {
        const uint32_t idesc1 = tc::make_idesc_bf16(BLOCK_M, COUT), idesc2 = tc::make_idesc_bf16(BLOCK_M, 2 * COUT),
                       idesc3 = tc::make_idesc_bf16(BLOCK_M, 3 * COUT);
        auto idesc_of = [&](int outputs) { return outputs == 1 ? idesc1 : (outputs == 2 ? idesc2 : idesc3); };
        const uint64_t da0 = tc::make_smem_desc(a_base, ROW_BYTES), db0 = tc::make_smem_desc(w_base, ROW_BYTES);
        int s = 0; uint32_t ph = 0;
        int n_base = 0;
        tmem_base = __shfl_sync(0xffffffffu, tmem_base, 0);     // (a broadcast from lane 0 is a uniform value to ptxas)
        tc::mbar_wait(w_bar, 0);
        tc::tc_fence_after();
        for (int t = t_begin; t < t_end;) {
            const int xa = t % X;
            const int xb = min(X, xa + (t_end - t));
            const int p_lo = max(xa - 1, 0), p_hi = min(xb, X - 1);
            for (int p = p_lo; p <= p_hi; ++p) {
                const int x_lo = max(p - 1, xa), x_hi = min(p + 1, xb - 1);      // outputs this plane feeds
                const int cnt = x_hi - x_lo + 1, off = x_lo - (p - 1);            // 1..3 outputs, first weight sub-tile
                const int n_lo = n_base + (x_lo - xa), slot_lo = n_lo & (SLOTS - 1);
                const int first = min(cnt, SLOTS - slot_lo);                       // outputs before the ring wraps
                // outputs whose first plane this is: x = p+1 (and x = 0 on plane 0) -- their slot must be drained + zeroed
                for (int x = x_lo; x <= x_hi; ++x) {
                    if (max(x - 1, 0) != p) continue;
                    const int n = n_base + (x - xa);
                    tc::mbar_wait(tempty_bar(n & (SLOTS - 1)), (n / SLOTS) & 1);
                }
                tc::tc_fence_after();
                const uint32_t d0 = tmem_base + slot_lo * COUT;
                const uint32_t i_first = idesc_of(first), i_rest = idesc_of(cnt - first);
                for (int dz = 0; dz < 3; ++dz) {
                    tc::mbar_wait(full_bar(s), ph);
                    tc::tc_fence_after();
                    // warp-uniform control flow: operands stay in the uniform datapath, elect.sync issues from one lane
                    const uint32_t desc_hi = (uint32_t)(da0 >> 32);                    // == high word of db0 (same ROW_BYTES)
                    const uint32_t a_s = (uint32_t)da0 + (uint32_t)((s * A_BYTES) >> 4);
                    const uint32_t b_z = (uint32_t)db0 + (uint32_t)(((dz * 9 + off) * W_TAP_BYTES) >> 4);
                    const uint32_t wrap = first < cnt ? 1u : 0u, b_wrap = (uint32_t)((first * W_TAP_BYTES) >> 4);
                    // one (warp-uniform) branch per STAGE: the 3-output window wraps around the TMEM slot ring for 2 of 8
                    // positions only, and the second MMA's operand set-up costs as much as the first's
                    if (!wrap) {
#pragma unroll
                        for (int dy = 0; dy < 3; ++dy) {
#pragma unroll
                            for (int k = 0; k < CIN / 16; ++k)
                                tc::umma_bf16_acc_elect_lo(d0, a_s + (uint32_t)((dy * DY_BYTES) >> 4) + 2 * k,
                                                           b_z + (uint32_t)((dy * 3 * W_TAP_BYTES) >> 4) + 2 * k, desc_hi, i_first);
                        }
                    } else {
#pragma unroll
                        for (int dy = 0; dy < 3; ++dy) {
#pragma unroll
                            for (int k = 0; k < CIN / 16; ++k) {
                                const uint32_t a_lo = a_s + (uint32_t)((dy * DY_BYTES) >> 4) + 2 * k;
                                const uint32_t b_lo = b_z + (uint32_t)((dy * 3 * W_TAP_BYTES) >> 4) + 2 * k;
                                tc::umma_bf16_acc_elect_lo(d0, a_lo, b_lo, desc_hi, i_first);
                                tc::umma_bf16_acc_elect_lo(tmem_base, a_lo, b_lo + b_wrap, desc_hi, i_rest);
                            }
                        }
                    }
                    __syncwarp();
                    tc::umma_commit_elect(empty_bar(s));
                    __syncwarp();
                    if (++s == STAGES) { s = 0; ph ^= 1; }
                }
                // outputs whose last plane this was: x = p-1 (and x = X-1 on the last plane)
                for (int x = x_lo; x <= x_hi; ++x) {
                    if (min(x + 1, X - 1) != p) continue;
                    tc::umma_commit_elect(tfull_bar((n_base + (x - xa)) & (SLOTS - 1)));
                }
            }
            n_base += xb - xa;
            t += xb - xa;
        }
    } else {
        const int quarter = warp & 3;
        const uint32_t tq = tmem_base + ((uint32_t)(quarter * 32) << 16);
        uint32_t zero[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) zero[i] = 0u;
#pragma unroll
        for (int sl = 0; sl < SLOTS; ++sl) tc::tmem_st32(tq + sl * COUT, zero);      // all accumulators start at zero
        tc::tmem_st_wait();
        tc::tc_fence_before();
#pragma unroll
        for (int sl = 0; sl < SLOTS; ++sl) tc::mbar_arrive(tempty_bar(sl));
        float b[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) b[i] = __ldg(bias + i);
        int n = 0;
        for (int t = t_begin; t < t_end; ++t, ++n) {
            const int x = t % X, y0 = (t / X) * TILE_Y;
            const int slot = n & (SLOTS - 1);
            tc::mbar_wait(tfull_bar(slot), (n / SLOTS) & 1);
            tc::tc_fence_after();
            uint32_t r[32];
            tc::tmem_ld32(tq + slot * COUT, r);
            tc::tmem_ld_wait();
            tc::tmem_st32(tq + slot * COUT, zero);           // accumulator is in registers: re-zero and release the slot
            tc::tmem_st_wait();
            tc::tc_fence_before();
            tc::mbar_arrive(tempty_bar(slot));
            const int row = quarter * 32 + lane;
            const int y = y0 + row / TILE_Z, z = row % TILE_Z;
            if (y < Y) {
                if constexpr (EPI == 0) {
                    uint4* op = reinterpret_cast<uint4*>(out + ((((size_t)x * Y + y) * TILE_Z + z) * COUT));
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        float v[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) v[j] = fmaxf(__uint_as_float(r[8 * i + j]) + b[8 * i + j], 0.f);
                        uint4 u;
                        u.x = pack_bf16x2(v[0], v[1]); u.y = pack_bf16x2(v[2], v[3]);
                        u.z = pack_bf16x2(v[4], v[5]); u.w = pack_bf16x2(v[6], v[7]);
                        op[i] = u;
                    }
                } else {
                    float4* op = reinterpret_cast<float4*>(out_f32 + ((((size_t)x * Y + y) * TILE_Z + z) * COUT));
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        float4 a = make_float4(__uint_as_float(r[4 * i]), __uint_as_float(r[4 * i + 1]), __uint_as_float(r[4 * i + 2]),
                                               __uint_as_float(r[4 * i + 3]));
                        if constexpr (EPI >= 2) { const float4 q = op[i]; a.x += q.x; a.y += q.y; a.z += q.z; a.w += q.w; }
                        if constexpr (EPI == 3) {
                            a.x = fmaxf(a.x + b[4 * i], 0.f); a.y = fmaxf(a.y + b[4 * i + 1], 0.f);
                            a.z = fmaxf(a.z + b[4 * i + 2], 0.f); a.w = fmaxf(a.w + b[4 * i + 3], 0.f);
                        }
                        op[i] = a;
                    }
                }
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc::tc_fence_after();
        tc::tmem_dealloc(tmem_base, 32 * SLOTS);
    }
}

}  // namespace

namespace {
// in_pitch: elements between consecutive voxels of `in` (Cin for a dense tensor, 2*Cin for one half of a [hi | lo] split)
template <int EPI>
int launch_conv3d_tc_impl(const bf16* in, int in_pitch, const bf16* w_tap_major, const float* bias, int X, int Y, int Z, int Cin,
                          bf16* out, float* out_f32, cudaStream_t stream)
{
    OCC_CHECK(Z == TILE_Z && (Cin == 16 || Cin == 32), "conv3d_tc: Z must be 16 and Cin in {16, 32}");
    const int row_bytes = Cin * 2;
    CUtensorMap tmIn, tmW;
    {
        const uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)Z, (uint64_t)Y, (uint64_t)X};
        const uint64_t strides[3] = {(uint64_t)in_pitch * 2, (uint64_t)Z * in_pitch * 2, (uint64_t)Y * Z * in_pitch * 2};
        const uint32_t box[4] = {(uint32_t)Cin, (uint32_t)TILE_Z, (uint32_t)(TILE_Y + 2), 1u};
        if (make_tensor_map_bf16(&tmIn, in, 4, dims, strides, box, row_bytes)) return 1;
    }
    {
        const uint64_t dims[2] = {(uint64_t)Cin, (uint64_t)TAPS * COUT};
        const uint64_t strides[1] = {(uint64_t)Cin * 2};
        const uint32_t box[2] = {(uint32_t)Cin, (uint32_t)COUT};
        if (make_tensor_map_bf16(&tmW, w_tap_major, 2, dims, strides, box, row_bytes)) return 1;
    }
    const int a_bytes = HALO_ROWS * row_bytes, w_bytes = (TAPS * COUT * row_bytes + 1023) & ~1023;
    const int smem = 1024 + w_bytes + STAGES * a_bytes + BAR_BYTES;
    const int num_sms = sm_count_current_device();
    const int tiles = X * ((Y + TILE_Y - 1) / TILE_Y);
    const int grid = tiles < num_sms ? tiles : num_sms;
    const auto kernel = Cin == 16 ? conv3d_tc_kernel<16, EPI> : conv3d_tc_kernel<32, EPI>;
    OCC_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    kernel<<<grid, NUM_THREADS, smem, stream>>>(tmIn, tmW, bias, out, out_f32, X, Y);
    OCC_CUDA(cudaGetLastError());
    return 0;
}
}  // namespace

int launch_conv3d_tc(const bf16* in, const bf16* w_tap_major, const float* bias, int X, int Y, int Z, int Cin,
                     bf16* out, cudaStream_t stream)
{
    return launch_conv3d_tc_impl<0>(in, Cin, w_tap_major, bias, X, Y, Z, Cin, out, nullptr, stream);
}

// fp32-grade convolution on the tensor cores: split = [hi | lo] bf16 halves of the fp32 input ([nvox][2*Cin], launch_split_bf16),
// w_hi / w_lo = bf16 split of the BN-folded fp32 weights ([27][32][Cin] each); out_f32 = relu(hi.W_hi + lo.W_hi + hi.W_lo + bias)
// accumulated in fp32 over three passes of the same kernel (the lo.lo term, 2^-16 relative, is dropped)
int launch_conv3d_tc_split(const bf16* split, const bf16* w_hi, const bf16* w_lo, const float* bias, int X, int Y, int Z, int Cin,
                           float* out_f32, cudaStream_t stream)
{
    if (launch_conv3d_tc_impl<1>(split, 2 * Cin, w_hi, bias, X, Y, Z, Cin, nullptr, out_f32, stream)) return 1;
    if (launch_conv3d_tc_impl<2>(split + Cin, 2 * Cin, w_hi, bias, X, Y, Z, Cin, nullptr, out_f32, stream)) return 1;
    return launch_conv3d_tc_impl<3>(split, 2 * Cin, w_lo, bias, X, Y, Z, Cin, nullptr, out_f32, stream);
}

}  // namespace occ
