// eh_wide_gemm.cuh -- bf16 tcgen05 GEMMs of the wide-hidden-layer path (sm_100a only).
//
// For hidden widths of 256 and more the Dense chain of a hybrid model (prepare_hidden_chain,
// src/models/NNModels.jl:220-231) really is a dense contraction: per optimiser step and hidden layer
//   forward        A_l      = act(A_{l-1} W_l^T + b_l)            [B x H] = [B x H] [H x H]
//   backward data  D_{l-1}  = (D_l W_l) .* act'(A_{l-1})          [B x H] = [B x H] [H x H]
//   weight grad    dW_l     = D_l^T A_{l-1}                       [H x H] = [H x B] [B x H]
// (the Zygote pullback of the chain, SURVEY 10.4).  One kernel template serves the three:
//   * operands travel HBM -> shared memory with TMA (cp.async.bulk.tensor, 128-byte swizzle) through a
//     4-stage mbarrier pipeline filled by one producer thread;
//   * one elected thread issues tcgen05.mma (cta_group::1, kind::f16, 128 x 256 x 16, bf16 in, fp32
//     accumulate); the 128 x 256 accumulator tile lives in tensor memory (256 columns);
//   * four epilogue warps read it back with tcgen05.ld (32 lanes x 32 columns per instruction) and fuse
//     the layer's elementwise tail: bias + activation -> bf16, or .* act'(a) -> bf16, or the fp32
//     split-K partial of a weight gradient (summed later in a fixed order: no atomics).
// The weight-gradient contraction runs over the batch, which is the slow dimension of both of its
// operands: they are fetched as MN-major tiles (64 columns x 64 batch rows per TMA box), so neither
// activations nor deltas are ever transposed in memory.
#pragma once
#include <type_traits>
#include <cuda.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include "eh_device.cuh"

namespace eh {
namespace wide {

constexpr int BM = 128, BK = 64, UMMA_K = 16;
constexpr int WIDE_MAXP = 8;          // chain inputs (all chains together) the kernels of every wide model are built for
constexpr int WIDE_MAXP_X = 12;       // ... and the separate instantiations of models with 9..12 inputs (summed width > 32)
constexpr int BS_BN_OFF = 3 * MAXT;   // == BS_BN of eh_chunk.cuh (per-batch scalar row: input BatchNorm mu / rstd)
constexpr int GEMM_THREADS = 192;            // warp 0: TMA, warp 1: MMA + TMEM alloc, warps 2..5: epilogue
// Tile width and pipeline depth per GEMM kind.
//  * weight gradient: 128 x 256 tiles, 64 k-blocks per CTA, 4 stages of 48 KB, one CTA per SM (main-loop bound);
//  * forward / backward-data: only 8 k-blocks per tile, so the epilogue (TMEM -> bias/activation or act' -> bf16 ->
//    HBM) weighs as much as the main loop.  128 x 128 tiles with 3 stages of 32 KB leave room for TWO CTAs per SM
//    (2 x 97 KB shared memory, 2 x 128 TMEM columns): one CTA's epilogue overlaps the other's main loop without
//    any persistent-scheduler machinery.
__host__ __device__ constexpr int gemm_bn(int mode) { return mode == 2 ? 256 : 128; }
__host__ __device__ constexpr int gemm_stages(int mode) { return mode == 2 ? 4 : 3; }
__host__ __device__ constexpr int gemm_stage_bytes(int mode) { return (BM + gemm_bn(mode)) * BK * 2; }
__host__ __device__ constexpr int gemm_smem(int mode)
{
    return gemm_stages(mode) * gemm_stage_bytes(mode) + 1024 /*alignment slack*/ + 1024 /*barriers, bias*/;
}

enum : int { GEMM_FWD = 0, GEMM_BWD = 1, GEMM_WGRAD = 2 };

struct GemmArgs {
    int M, N, K;             // C is M x N; K = contraction length handled by ONE split
    int ksplits;             // WGRAD: gridDim.z; split z covers K rows [z*K, (z+1)*K)
    int act;                 // ACT_* of the hidden layers
    const float* bias;       // FWD: [N]
    const __nv_bfloat16* aux;  // BWD: A_{l-1} [M x N] (activation whose derivative multiplies the tile)
    __nv_bfloat16* out16;    // FWD / BWD: [M x N] row-major
    float* out32;            // WGRAD: [ksplits][M x N] row-major partials
    // BWD, optional: column sums of the (bf16-rounded) output tile per 32-row slab -> the bias gradient of the layer
    // below, and for the first layer also the x-weighted sums (its weight gradient): [M / 32][(1 + P1) * N]
    float* colsum;
    const float* xb;         // [M x R4] compact batch records (first P1 entries = chain inputs)
    const float* bscal;      // input BatchNorm scalars (mu, rstd per input) when use_bn
    int R4, P1, use_bn;
    // PU instantiations (chains that differ in depth or activation): ACT_* per column of the output (FWD) / of aux
    // (BWD) instead of `act`, [N] bytes
    const uint8_t* uact;
};

// ---- thin PTX wrappers ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
// bounded wait: a broken pipeline must not hang the GPU (returns false after ~1 s)
__device__ __forceinline__ bool mbar_wait(uint32_t bar, uint32_t parity)
{
    for (uint32_t spins = 0; spins < (1u << 24); spins++)
        if (mbar_try_wait(bar, parity)) return true;
    return false;
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map)
{
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// 32 lanes x 32 consecutive fp32 columns of the accumulator -> 32 registers per thread
__device__ __forceinline__ void tc_ld_32x32(uint32_t taddr, uint32_t (&r)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// shared-memory matrix descriptor (SWIZZLE_128B, sm_100 version 1).  K-major tiles: rows of 128 bytes,
// 8-row swizzle atoms 1024 bytes apart (SBO), LBO unused.  MN-major tiles (TMA boxes of 64 columns x BK
// rows): 8 K-rows per atom, atoms 1024 bytes apart along K (SBO), next 64 columns one box further (LBO).
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes)
{
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;   // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;   // SWIZZLE_128B
    return d;
}
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int m, int n, int a_mn_major, int b_mn_major)
{
    return (1u << 4) /* D = f32 */ | (1u << 7) /* A = bf16 */ | (1u << 10) /* B = bf16 */ | ((uint32_t)a_mn_major << 15) |
           ((uint32_t)b_mn_major << 16) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

__device__ __forceinline__ float tanh_fast(float z)
{
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(z));
    return y;
}
// hidden activations of the wide path: the result is rounded to bf16 (8 bits of mantissa) anyway, so one
// MUFU.TANH (2^-11 relative) per element is as good as an exact evaluation and keeps the epilogue short
__device__ __forceinline__ float act1(int act, float z)
{
    if (act == ACT_TANH) return tanh_fast(z);
    if (act == ACT_SIGMOID) return fmaf(0.5f, tanh_fast(0.5f * z), 0.5f);
    if (act == ACT_RELU) return fmaxf(z, 0.f);
    return z;
}
// derivative from the stored output a
__device__ __forceinline__ float dact1(int act, float a)
{
    if (act == ACT_TANH) return fmaf(-a, a, 1.f);
    if (act == ACT_SIGMOID) return a * (1.f - a);
    if (act == ACT_RELU) return a > 0.f ? 1.f : 0.f;
    return 1.f;
}
// per-unit activations: the codes of 32 consecutive columns (16-byte aligned) as eight words, the same in every lane
__device__ __forceinline__ void load_acts32(const uint8_t* uact, uint32_t (&w)[8])
{
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(uact)), b = __ldg(reinterpret_cast<const uint4*>(uact) + 1);
    w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
}
template <int N>
__device__ __forceinline__ int act_at(const uint32_t (&w)[N], int j) { return (int)((w[j >> 2] >> (8 * (j & 3))) & 0xffu); }
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi)
{
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}

// grid: (M / BM, N / BN, ksplits).  FWD / BWD: tmA = [M x K] K-major (box 64 x 128), tmB = [N x K] K-major
// (box 64 x 128).  WGRAD: tmA = deltas [Kall x M], tmB = activations [Kall x N], both MN-major (box 64 x 64).
// PX: chain inputs the backward-data epilogue's input-weighted column sums hold (WIDE_MAXP, or WIDE_MAXP_X in the
// instantiation that serves the layer-1 call of models with more than WIDE_MAXP inputs).  PU: activation per column
// (g.uact), a separate instantiation so that the others keep their code
template <int MODE, int PX = WIDE_MAXP, bool PU = false>
__global__ void __launch_bounds__(GEMM_THREADS, MODE == GEMM_WGRAD ? 1 : 2)
k_wide_gemm(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmArgs g)
{
    constexpr int BN = gemm_bn(MODE);
    constexpr int STAGES = gemm_stages(MODE);
    constexpr int A_STAGE_BYTES = BM * BK * 2, STAGE_BYTES = gemm_stage_bytes(MODE);
    constexpr int BAR_OFF = STAGES * STAGE_BYTES;
    constexpr int TMEM_COLS = BN;                // fp32 accumulator: one column per output column
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;   // swizzle atoms need 1024-byte alignment
    const uint32_t bar0 = base + BAR_OFF;                          // full[STAGES], empty[STAGES], tmem_full, tmem slot
    auto full_bar = [&](int s) { return bar0 + 8u * s; };
    auto empty_bar = [&](int s) { return bar0 + 8u * (STAGES + s); };
    const uint32_t tmem_full_bar = bar0 + 8u * (2 * STAGES);
    const uint32_t tmem_slot = bar0 + 8u * (2 * STAGES + 1);
    uint8_t* gen_base = smem_raw + (base - smem_u32(smem_raw));
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(gen_base + BAR_OFF + 8 * (2 * STAGES + 1));
    float* s_bias = reinterpret_cast<float*>(gen_base + BAR_OFF + 128);   // FWD: bias of the tile's columns

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
    const int kbase = (MODE == GEMM_WGRAD) ? blockIdx.z * g.K : 0;
    const int nkb = g.K / BK;
    constexpr bool MN = (MODE == GEMM_WGRAD);

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        for (int s = 0; s < STAGES; s++) {
            mbar_init(full_bar(s), 1);
            mbar_init(empty_bar(s), 1);
        }
        mbar_init(tmem_full_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"((uint32_t)TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;

    if (warp == 0) {
        if (lane == 0) {
            // ===== TMA producer =====
            for (int kb = 0; kb < nkb; kb++) {
                const int s = kb % STAGES;
                const uint32_t par = ((kb / STAGES) & 1) ^ 1;
                if (!mbar_wait(empty_bar(s), par)) break;
                const uint32_t sa = base + s * STAGE_BYTES, sb = sa + A_STAGE_BYTES;
                mbar_expect_tx(full_bar(s), STAGE_BYTES);
                const int k0 = kbase + kb * BK;
                if (!MN) {
                    tma_load_2d(sa, &tmA, k0, m0, full_bar(s));
                    tma_load_2d(sb, &tmB, k0, n0, full_bar(s));
                } else {
#pragma unroll
                    for (int j = 0; j < BM / 64; j++) tma_load_2d(sa + j * (64 * BK * 2), &tmA, m0 + 64 * j, k0, full_bar(s));
#pragma unroll
                    for (int j = 0; j < BN / 64; j++) tma_load_2d(sb + j * (64 * BK * 2), &tmB, n0 + 64 * j, k0, full_bar(s));
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // ===== MMA issuer =====
            constexpr uint32_t idesc = umma_idesc_bf16(BM, BN, MN ? 1 : 0, MN ? 1 : 0);
            constexpr uint32_t lbo = MN ? 64 * BK * 2 : 0;     // MN-major: next 64 columns = next TMA box
            constexpr uint32_t sbo = 1024;                     // 8 rows (K-major) / 8 K-rows (MN-major) of 128 bytes
            constexpr uint32_t kstep = MN ? UMMA_K * 128 : UMMA_K * 2;  // bytes per UMMA_K along the stage
            bool ok = true;
            for (int kb = 0; kb < nkb && ok; kb++) {
                const int s = kb % STAGES;
                ok = mbar_wait(full_bar(s), (kb / STAGES) & 1);
                tc_fence_after();
                const uint32_t sa = base + s * STAGE_BYTES, sb = sa + A_STAGE_BYTES;
#pragma unroll
                for (int k = 0; k < BK / UMMA_K; k++) {
                    const uint64_t da = umma_desc(sa + k * kstep, lbo, sbo);
                    const uint64_t db = umma_desc(sb + k * kstep, lbo, sbo);
                    tc_mma_bf16(tmem_base, da, db, idesc, (kb | k) ? 1u : 0u);
                }
                tc_commit(empty_bar(s));   // frees the stage once these MMAs have read it
            }
            tc_commit(tmem_full_bar);      // accumulator complete
        }
    } else {
        // ===== epilogue: warps 2..5, TMEM lane quarter = warp % 4 =====
        // A thread owns one accumulator row (TMEM lane), i.e. a 256-byte strip of the bf16 output.  Writing that
        // directly would scatter 16-byte pieces over 32 rows per instruction, so the strip goes through shared
        // memory (the pipeline stages are idle once the accumulator is complete; rows padded to 272 bytes keep
        // the 16-byte accesses conflict-free) and leaves as coalesced 256-byte row segments.
        const int q = warp & 3;
        const int row = m0 + q * 32 + lane;
        constexpr int OPITCH = BN * 2 + 16;
        uint8_t* stg = gen_base + q * (32 * OPITCH);
        // while the main loop runs: fetch what the epilogue needs besides the accumulator
        uint4 auxr[MODE == GEMM_BWD ? BN / 8 : 1];
        if (MODE == GEMM_BWD) {
            const uint4* ap = reinterpret_cast<const uint4*>(g.aux + (size_t)row * g.N + n0);
#pragma unroll
            for (int j = 0; j < BN / 8; j++) auxr[j] = __ldg(ap + j);   // my row of the activation tile, held in registers
        }
        if (MODE == GEMM_FWD) {
            const int t = (warp - 2) * 32 + lane;   // 0..127
            for (int i = t; i < BN; i += 128) s_bias[i] = __ldg(g.bias + n0 + i);
            asm volatile("bar.sync 1, 128;" ::: "memory");   // the four epilogue warps only
        }
        mbar_wait(tmem_full_bar, 0);
        tc_fence_after();
#pragma unroll
        for (int c = 0; c < BN; c += 32) {
            uint32_t r[32];
            tc_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c, r);
            if (MODE == GEMM_WGRAD) {
                float4* dst = reinterpret_cast<float4*>(g.out32 + ((size_t)blockIdx.z * g.M + row) * g.N + n0 + c);
#pragma unroll
                for (int j = 0; j < 8; j++)
                    dst[j] = make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]), __uint_as_float(r[4 * j + 2]),
                                         __uint_as_float(r[4 * j + 3]));
            } else {
                uint32_t o[16];
                uint32_t uw[PU ? 8 : 1];
                if constexpr (PU) load_acts32(g.uact + n0 + c, uw);
                auto act_of = [&](int j) {   // column c + j
                    if constexpr (PU) return act_at(uw, j);
                    else return g.act;
                };
                if (MODE == GEMM_FWD) {
                    const float4* b4 = reinterpret_cast<const float4*>(s_bias + c);
#pragma unroll
                    for (int j = 0; j < 8; j++) {
                        const float4 b = b4[j];
                        o[2 * j] = pack_bf16(act1(act_of(4 * j), __uint_as_float(r[4 * j]) + b.x), act1(act_of(4 * j + 1), __uint_as_float(r[4 * j + 1]) + b.y));
                        o[2 * j + 1] = pack_bf16(act1(act_of(4 * j + 2), __uint_as_float(r[4 * j + 2]) + b.z), act1(act_of(4 * j + 3), __uint_as_float(r[4 * j + 3]) + b.w));
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        const uint4 a = auxr[MODE == GEMM_BWD ? (c >> 3) + j : 0];
                        const uint32_t aw[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
                        for (int e = 0; e < 4; e++) {
                            const __nv_bfloat162 ab = *reinterpret_cast<const __nv_bfloat162*>(&aw[e]);
                            const float2 af = __bfloat1622float2(ab);
                            o[4 * j + e] = pack_bf16(__uint_as_float(r[8 * j + 2 * e]) * dact1(act_of(8 * j + 2 * e), af.x),
                                                     __uint_as_float(r[8 * j + 2 * e + 1]) * dact1(act_of(8 * j + 2 * e + 1), af.y));
                        }
                    }
                }
#pragma unroll
                for (int j = 0; j < 4; j++)
                    *reinterpret_cast<uint4*>(stg + lane * OPITCH + ((c >> 3) + j) * 16) = make_uint4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
            }
        }
        if (MODE == GEMM_BWD && g.colsum != nullptr) {
            // column sums over this warp's 32 rows, straight from the staged bf16 strip: lane l owns columns 4l .. 4l+3
            __syncwarp();
            float cs[4] = {0.f, 0.f, 0.f, 0.f}, cw[PX][4];
            float xr[PX] = {0.f};
#pragma unroll
            for (int p = 0; p < PX; p++) {
                cw[p][0] = cw[p][1] = cw[p][2] = cw[p][3] = 0.f;
                if (p < g.P1) {
                    float x = g.xb[(size_t)row * g.R4 + p];
                    if (g.use_bn) x = (x - g.bscal[BS_BN_OFF + 2 * p]) * g.bscal[BS_BN_OFF + 2 * p + 1];
                    xr[p] = x;
                }
            }
#pragma unroll
            for (int r = 0; r < 32; r++) {
                const uint2 v = *reinterpret_cast<const uint2*>(stg + r * OPITCH + lane * 8);
                const float2 f0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v.x));
                const float2 f1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v.y));
                cs[0] += f0.x; cs[1] += f0.y; cs[2] += f1.x; cs[3] += f1.y;
#pragma unroll
                for (int p = 0; p < PX; p++) {
                    if (p < g.P1) {
                        const float x = __shfl_sync(0xffffffffu, xr[p], r);
                        cw[p][0] = fmaf(f0.x, x, cw[p][0]); cw[p][1] = fmaf(f0.y, x, cw[p][1]);
                        cw[p][2] = fmaf(f1.x, x, cw[p][2]); cw[p][3] = fmaf(f1.y, x, cw[p][3]);
                    }
                }
            }
            // combine the four warps (fixed order) so that one 128-row slab per CTA goes out
            float* s_cs = reinterpret_cast<float*>(gen_base + 4 * (32 * OPITCH));   // [4 warps][1 + PX][BN], behind the strips
            static_assert(4 * 32 * OPITCH + 4 * (1 + PX) * BN * 4 <= STAGES * STAGE_BYTES, "column sums fit the idle stages");
            *reinterpret_cast<float4*>(s_cs + (q * (1 + PX) + 0) * BN + lane * 4) = make_float4(cs[0], cs[1], cs[2], cs[3]);
#pragma unroll
            for (int p = 0; p < PX; p++)
                if (p < g.P1) *reinterpret_cast<float4*>(s_cs + (q * (1 + PX) + 1 + p) * BN + lane * 4) = make_float4(cw[p][0], cw[p][1], cw[p][2], cw[p][3]);
            asm volatile("bar.sync 1, 128;" ::: "memory");
            const int t = (warp - 2) * 32 + lane;   // column of the tile
            for (int p = 0; p <= g.P1; p++) {
                const float v = ((s_cs[(0 * (1 + PX) + p) * BN + t] + s_cs[(1 * (1 + PX) + p) * BN + t]) + s_cs[(2 * (1 + PX) + p) * BN + t]) + s_cs[(3 * (1 + PX) + p) * BN + t];
                g.colsum[((size_t)blockIdx.x * (1 + g.P1) + p) * g.N + n0 + t] = v;
            }
        }
        if (MODE != GEMM_WGRAD) {
            __syncwarp();
            // BN * 2 bytes per row = BN / 8 lanes of 16 bytes: 32 / (BN / 8) rows per instruction
            constexpr int LPR = BN / 8, RPI = 32 / LPR;
#pragma unroll 4
            for (int r0 = 0; r0 < 32; r0 += RPI) {
                const int rr = r0 + lane / LPR, cc = lane % LPR;
                const uint4 v = *reinterpret_cast<const uint4*>(stg + rr * OPITCH + cc * 16);
                *(reinterpret_cast<uint4*>(g.out16 + (size_t)(m0 + q * 32 + rr) * g.N + n0) + cc) = v;
            }
        }
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS) : "memory");
    }
}


// ---- persistent forward / backward-data GEMM -------------------------------------------------------------------------
// One CTA per SM walks the 128 x 256 output tiles (tile t = blockIdx.x + i * gridDim.x).  Two accumulator buffers in
// tensor memory (2 x 256 columns) let the MMA warp start tile i+1 while the SIXTEEN epilogue warps (four per TMEM lane
// quarter, 64 columns each) drain tile i; the TMA producer simply keeps the 3-stage ring full across tile borders.
// The epilogue is a chain of dependent long-latency steps (tcgen05.ld -> math -> STS -> LDS -> STG); with two warps per
// scheduler (the first form: eight warps of 128 columns) it, not the tensor pipe, set the pace: 6.4 us per tile against
// 2.2 us of MMAs.  PG_EPI_WARPS = 8 keeps that form for comparison.
// Barriers: full/empty per stage (TMA <-> MMA), tmem_full/tmem_empty per accumulator buffer (MMA <-> epilogue).
#ifndef PG_EPI_WARPS
#define PG_EPI_WARPS 16
#endif
constexpr int PG_BN = 256, PG_STAGES = 3, PG_THREADS = (2 + PG_EPI_WARPS) * 32;   // warp 0 TMA, warp 1 MMA, then the epilogue warps
constexpr int PG_EPI_THREADS = PG_EPI_WARPS * 32;
constexpr int PG_CW = PG_BN / (PG_EPI_WARPS / 4);              // output columns of one epilogue warp (64)
constexpr int PG_STAGE_BYTES = (BM + PG_BN) * BK * 2;          // 48 KB
constexpr int PG_OPITCH = PG_CW * 2 + 16;                      // staged row of one epilogue warp: PG_CW bf16 + pad
constexpr int PG_STG_BYTES = PG_EPI_WARPS * 32 * PG_OPITCH;    // 73 728
constexpr int PG_SIDE_BYTES = PG_EPI_WARPS * PG_CW * 4;         // bias values, one private copy per epilogue warp
constexpr int PG_SMEM = PG_STAGES * PG_STAGE_BYTES + PG_STG_BYTES + PG_SIDE_BYTES + 1024 + 256;
static_assert(PG_SMEM <= 232448, "persistent GEMM: shared memory");

__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// cluster forms: the TMA box lands at the same shared-memory offset of every CTA in `mask` and completes bytes on the
// barrier at the same offset there; the commit arrives on the barrier at the same offset of every CTA in `mask`
__device__ __forceinline__ void tma_load_2d_mc(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar, uint16_t mask)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "h"(mask)
        : "memory");
}
__device__ __forceinline__ void tc_commit_mc(uint32_t bar, uint16_t mask)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"(mask)
                 : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// CL = 2: clusters of two CTAs work on two row tiles of the SAME column tile at a time; each CTA fetches one half of the
// weight tile of a stage (128 of the 256 rows) and multicasts it into both, so a tile costs 256 KB of L2 reads instead of
// 384 KB -- the kernel runs at the L2 throughput limit (about 12 TB/s), not at the tensor pipe's.  A stage is reusable
// when BOTH CTAs' MMAs have read it (the commits arrive on both empty barriers).  tmB: box of BN rows for CL = 1, BN / 2 for CL = 2.
// PX: as for k_wide_gemm (the staged strip of a warp, 32 x PG_OPITCH bytes, holds the (1 + PX) x PG_CW parked sums).
// PU: as for k_wide_gemm
template <int MODE, int CL, int PX = WIDE_MAXP, bool PU = false>
__global__ void __launch_bounds__(PG_THREADS, 1)
k_wide_gemm_p(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmArgs g)
{
    static_assert(MODE == GEMM_FWD || MODE == GEMM_BWD, "persistent form serves forward and backward-data");
    static_assert(CL == 1 || CL == 2, "cluster of one or two CTAs");
    static_assert((1 + PX) * PG_CW * 4 <= 32 * PG_OPITCH, "parked column sums fit the staged strip");
    constexpr int BN = PG_BN, STAGES = PG_STAGES, STAGE_BYTES = PG_STAGE_BYTES, A_STAGE_BYTES = BM * BK * 2;
    constexpr int STG_OFF = STAGES * STAGE_BYTES, SIDE_OFF = STG_OFF + PG_STG_BYTES, BAR_OFF = SIDE_OFF + PG_SIDE_BYTES;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* gen_base = smem_raw + (base - smem_u32(smem_raw));
    const uint32_t bar0 = base + BAR_OFF;
    auto full_bar = [&](int s) { return bar0 + 8u * s; };
    auto empty_bar = [&](int s) { return bar0 + 8u * (STAGES + s); };
    auto tfull_bar = [&](int b) { return bar0 + 8u * (2 * STAGES + b); };
    auto tempty_bar = [&](int b) { return bar0 + 8u * (2 * STAGES + 2 + b); };
    const uint32_t tmem_slot = bar0 + 8u * (2 * STAGES + 4);
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(gen_base + BAR_OFF + 8 * (2 * STAGES + 4));
    float* s_bias = reinterpret_cast<float*>(gen_base + SIDE_OFF);                 // [epilogue warp][PG_CW]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int num_n = g.N / BN;
    const int nkb = g.K / BK;
    // work units: (row-tile group of CL tiles, column tile); cluster cid walks units cid, cid + ncl, ...; CTA `crank` of
    // the cluster takes row tile mp * CL + crank of the group
    const int crank = CL > 1 ? (int)cluster_ctarank() : 0;
    const int cid = blockIdx.x / CL, ncl = gridDim.x / CL;
    const int num_units = (g.M / BM / CL) * num_n;
    auto unit_m0 = [&](int u) { return ((u / num_n) * CL + crank) * BM; };
    auto unit_n0 = [&](int u) { return (u % num_n) * BN; };

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        for (int s = 0; s < STAGES; s++) {
            mbar_init(full_bar(s), 1);
            mbar_init(empty_bar(s), CL);
        }
        for (int b = 0; b < 2; b++) {
            mbar_init(tfull_bar(b), 1);
            mbar_init(tempty_bar(b), PG_EPI_WARPS);   // one arrival per epilogue warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    if (CL > 1) cluster_sync_all();   // the peer's barriers exist before anything arrives on them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;

    if (warp == 0) {
        if (lane == 0) {
            // ===== TMA producer: one continuous ring over all tiles of this CTA =====
            constexpr int B_HALF_BYTES = (BN / 2) * BK * 2;
            int kbc = 0;
            bool pok = true;
            for (int u = cid; u < num_units && pok; u += ncl) {
                const int m0 = unit_m0(u), n0 = unit_n0(u);
                for (int kb = 0; kb < nkb && pok; kb++, kbc++) {
                    const int s = kbc % STAGES;
                    pok = mbar_wait(empty_bar(s), ((kbc / STAGES) & 1) ^ 1);
                    if (!pok) break;
                    const uint32_t sa = base + s * STAGE_BYTES, sb = sa + A_STAGE_BYTES;
                    mbar_expect_tx(full_bar(s), STAGE_BYTES);
                    tma_load_2d(sa, &tmA, kb * BK, m0, full_bar(s));
                    if (CL > 1) {
                        tma_load_2d_mc(sb + crank * B_HALF_BYTES, &tmB, kb * BK, n0 + crank * (BN / 2), full_bar(s), (uint16_t)3);
                    } else {
                        tma_load_2d(sb, &tmB, kb * BK, n0, full_bar(s));   // one box of BN rows
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // ===== MMA issuer =====
            constexpr uint32_t idesc = umma_idesc_bf16(BM, BN, 0, 0);
            int kbc = 0, it = 0;
            bool ok = true;
            for (int u = cid; u < num_units && ok; u += ncl, it++) {
                const int ab = it & 1;
                ok = mbar_wait(tempty_bar(ab), ((it >> 1) & 1) ^ 1);   // the epilogue has drained this accumulator buffer
                tc_fence_after();
                const uint32_t acc = tmem_base + (uint32_t)(ab * BN);
                for (int kb = 0; kb < nkb && ok; kb++, kbc++) {
                    const int s = kbc % STAGES;
                    ok = mbar_wait(full_bar(s), (kbc / STAGES) & 1);
                    tc_fence_after();
                    const uint32_t sa = base + s * STAGE_BYTES, sb = sa + A_STAGE_BYTES;
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; k++)
                        tc_mma_bf16(acc, umma_desc(sa + k * UMMA_K * 2, 0, 1024), umma_desc(sb + k * UMMA_K * 2, 0, 1024), idesc,
                                    (kb | k) ? 1u : 0u);
                    if (CL > 1) tc_commit_mc(empty_bar(s), (uint16_t)3);
                    else tc_commit(empty_bar(s));
                }
                tc_commit(tfull_bar(ab));
            }
        }
    } else {
        // ===== epilogue: warps 2..; TMEM lane quarter q = warp % 4, column slice h = (warp - 2) / 4 of PG_CW columns =====
        constexpr int CW = PG_CW, NCC = CW / 32;
        constexpr int LPR = CW / 8, RPI = 32 / LPR;        // 16-byte lanes per staged row, rows per warp-wide instruction
        constexpr int NAUX = 32 / RPI;                     // 16-byte pieces of the activation strip per thread
        const int q = warp & 3, h = (warp - 2) >> 2;
        uint8_t* stg = gen_base + STG_OFF + (warp - 2) * (32 * PG_OPITCH);
        const int prow = lane / LPR, pc16 = lane % LPR;    // this lane's place in the coalesced strip walk
        // BWD: the activation strip (32 rows x CW columns of A_{l-1}) of the NEXT tile travels in registers while this
        // tile is worked on, read in the coalesced pattern (full 16-byte lanes of consecutive row pieces)
        uint4 apre[MODE == GEMM_BWD ? NAUX : 1];
        auto load_aux = [&](int u) {
            const int m0 = unit_m0(u), n0 = unit_n0(u);
            const uint4* ap = reinterpret_cast<const uint4*>(g.aux + (size_t)(m0 + q * 32 + prow) * g.N + n0 + h * CW) + pc16;
#pragma unroll
            for (int i = 0; i < NAUX; i++) apre[i] = __ldg(ap + (size_t)i * RPI * (g.N / 8));
        };
        if (MODE == GEMM_BWD && cid < num_units) load_aux(cid);
        int it = 0;
        for (int u = cid; u < num_units; u += ncl, it++) {
            const int ab = it & 1;
            const int m0 = unit_m0(u), n0 = unit_n0(u);
            const int row = m0 + q * 32 + lane;
            const int ncol0 = n0 + h * CW;                // first output column of this warp
            float* bias = s_bias + (warp - 2) * CW;      // this warp's own copy: no CTA-wide barrier per tile
            if (MODE == GEMM_FWD) {
                __syncwarp();
#pragma unroll
                for (int k = 0; k < CW / 32; k++) bias[k * 32 + lane] = __ldg(g.bias + ncol0 + k * 32 + lane);
                __syncwarp();
            } else {
#pragma unroll
                for (int i = 0; i < NAUX; i++) *reinterpret_cast<uint4*>(stg + (i * RPI + prow) * PG_OPITCH + pc16 * 16) = apre[i];
                __syncwarp();
                if (u + ncl < num_units) load_aux(u + ncl);
            }
            mbar_wait(tfull_bar(ab), (it >> 1) & 1);
            tc_fence_after();
#pragma unroll
            for (int cc = 0; cc < NCC; cc++) {
                const int c = cc * 32;
                uint32_t r[32];
                uint32_t uw[PU ? 8 : 1];
                if constexpr (PU) load_acts32(g.uact + ncol0 + c, uw);
                auto act_of = [&](int j) {   // column ncol0 + c + j
                    if constexpr (PU) return act_at(uw, j);
                    else return g.act;
                };
                tc_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(ab * BN + h * CW + c), r);
                uint32_t o[16];
                if (MODE == GEMM_FWD) {
                    const float4* b4 = reinterpret_cast<const float4*>(bias + c);
#pragma unroll
                    for (int j = 0; j < 8; j++) {
                        const float4 b = b4[j];
                        o[2 * j] = pack_bf16(act1(act_of(4 * j), __uint_as_float(r[4 * j]) + b.x), act1(act_of(4 * j + 1), __uint_as_float(r[4 * j + 1]) + b.y));
                        o[2 * j + 1] = pack_bf16(act1(act_of(4 * j + 2), __uint_as_float(r[4 * j + 2]) + b.z), act1(act_of(4 * j + 3), __uint_as_float(r[4 * j + 3]) + b.w));
                    }
                } else {
                    // this thread's own row of the activation strip; the result goes back to the same bytes
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        const uint4 cur = *reinterpret_cast<const uint4*>(stg + lane * PG_OPITCH + ((c >> 3) + j) * 16);
                        const uint32_t aw[4] = {cur.x, cur.y, cur.z, cur.w};
#pragma unroll
                        for (int e = 0; e < 4; e++) {
                            const float2 af = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&aw[e]));
                            o[4 * j + e] = pack_bf16(__uint_as_float(r[8 * j + 2 * e]) * dact1(act_of(8 * j + 2 * e), af.x),
                                                     __uint_as_float(r[8 * j + 2 * e + 1]) * dact1(act_of(8 * j + 2 * e + 1), af.y));
                        }
                    }
                }
#pragma unroll
                for (int j = 0; j < 4; j++)
                    *reinterpret_cast<uint4*>(stg + lane * PG_OPITCH + ((c >> 3) + j) * 16) = make_uint4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
            }
            // this warp is done with the accumulator buffer: hand it back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty_bar(ab));
            // BWD: column sums over this warp's 32 rows, straight from the staged strip (lane l owns columns NCC l .. NCC l + NCC - 1)
            // (the input-weighted sums exist for the layer-1 call only; the loop is specialised on their count -- unrolled over
            // WIDE_MAXP with a run-time bound it cost 1 000 mostly predicated-off instructions per tile and warp)
            float cs[NCC], cw[PX][NCC];
            const bool want_cs = MODE == GEMM_BWD && g.colsum != nullptr;
            if (want_cs) {
#pragma unroll
                for (int k = 0; k < NCC; k++) cs[k] = 0.f;
#pragma unroll
                for (int p = 0; p < PX; p++)
#pragma unroll
                    for (int k = 0; k < NCC; k++) cw[p][k] = 0.f;
                auto colsums = [&](auto pn_c) {
                    constexpr int PN = decltype(pn_c)::value;
                    float xr[PN > 0 ? PN : 1];
#pragma unroll
                    for (int p = 0; p < PN; p++) {
                        xr[p] = 0.f;
                        if (p < g.P1) {
                            float x = g.xb[(size_t)row * g.R4 + p];
                            if (g.use_bn) x = (x - g.bscal[BS_BN_OFF + 2 * p]) * g.bscal[BS_BN_OFF + 2 * p + 1];
                            xr[p] = x;
                        }
                    }
#pragma unroll 8
                    for (int r2 = 0; r2 < 32; r2++) {
                        float f[NCC];
#pragma unroll
                        for (int k = 0; k < NCC; k += 2) {
                            const uint32_t v = *reinterpret_cast<const uint32_t*>(stg + r2 * PG_OPITCH + lane * (2 * NCC) + 2 * k);
                            const float2 ff = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v));
                            f[k] = ff.x; f[k + 1] = ff.y;
                        }
#pragma unroll
                        for (int k = 0; k < NCC; k++) cs[k] += f[k];
#pragma unroll
                        for (int p = 0; p < PN; p++) {
                            const float x = __shfl_sync(0xffffffffu, xr[p], r2);
#pragma unroll
                            for (int k = 0; k < NCC; k++) cw[p][k] = fmaf(f[k], x, cw[p][k]);
                        }
                    }
                };
                if constexpr (PX > WIDE_MAXP) {
                    colsums(std::integral_constant<int, PX>{});   // (launched for layer 1 of a model with > WIDE_MAXP inputs)
                } else {
                    if (g.P1 == 0) colsums(std::integral_constant<int, 0>{});
                    else if (g.P1 == 1) colsums(std::integral_constant<int, 1>{});
                    else if (g.P1 == 2) colsums(std::integral_constant<int, 2>{});
                    else if (g.P1 <= 4) colsums(std::integral_constant<int, 4>{});
                    else colsums(std::integral_constant<int, WIDE_MAXP>{});
                }
            }
            __syncwarp();
            // CW bf16 per row = LPR lanes of 16 bytes: RPI rows per instruction
#pragma unroll 4
            for (int r0 = 0; r0 < 32; r0 += RPI) {
                const int rr = r0 + prow;
                const uint4 v = *reinterpret_cast<const uint4*>(stg + rr * PG_OPITCH + pc16 * 16);
                *(reinterpret_cast<uint4*>(g.out16 + (size_t)(m0 + q * 32 + rr) * g.N + ncol0) + pc16) = v;
            }
            __syncwarp();
            if (want_cs) {
                // the strip is free now: park this warp's sums in it, combine the four lane-quarter warps of each
                // column slice in a fixed order, one 128-row slab per tile goes out
                float* mine = reinterpret_cast<float*>(stg);
#pragma unroll
                for (int k = 0; k < NCC; k++) mine[lane * NCC + k] = cs[k];
#pragma unroll
                for (int p = 0; p < PX; p++)
                    if (p < g.P1) {
#pragma unroll
                        for (int k = 0; k < NCC; k++) mine[(1 + p) * CW + lane * NCC + k] = cw[p][k];
                    }
                // (only the four warps of this column slice meet: named barrier 2 + h, 128 threads)
                asm volatile("bar.sync %0, 128;" ::"r"(2 + h) : "memory");
                const int ti = ((warp - 2) & 3) * 32 + lane;   // 0..127 among the warps of the slice
                if (ti < CW) {
                    for (int p = 0; p <= g.P1; p++) {
                        float v = 0.f;
#pragma unroll
                        for (int qq = 0; qq < 4; qq++) {
                            const int wi = 4 * h + ((qq + 2) & 3);   // epilogue warp with lane quarter qq of this column slice
                            v += reinterpret_cast<const float*>(gen_base + STG_OFF + wi * (32 * PG_OPITCH))[p * CW + ti];
                        }
                        g.colsum[((size_t)(m0 / BM) * (1 + g.P1) + p) * g.N + n0 + h * CW + ti] = v;
                    }
                }
                asm volatile("bar.sync %0, 128;" ::"r"(2 + h) : "memory");   // the strips are rewritten by the next tile
            }
            __syncwarp();   // the strip is rewritten by the next tile
        }
    }
    __syncthreads();
    if (CL > 1) cluster_sync_all();   // no multicast write or remote arrival may find this CTA gone
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

}  // namespace wide
}  // namespace eh
