// eh_wide_kernels.cuh -- the non-GEMM kernels of the wide-hidden-layer training step (sm_100a).
//
// One optimiser step of a hybrid model whose Dense chain is  P -> H -> ... -> H -> NOUT  with H >= 256
// (BASELINE config 5: 3 x 512) is a sequence of launches on one stream:
//   k_wide_gather    batch records (AoS, gathered through the index stream) -> compact batch
//   k_wide_first     layer 1 (fan-in P is tiny: elementwise)          A_1 = act(W_1 x + b_1)        bf16
//   gemm_fwd  x(NH-1)  tcgen05                                          A_l = act(A_{l-1} W_l^T + b_l)  bf16
//   k_wide_head      output layer (fan-out NOUT is tiny), parameter squashing, process model, masked loss
//                    seeds, analytic backward into D_NH, gradient of the output layer and of phi
//   per hidden layer l = NH .. 2:   gemm_wgrad (dW_l partials), gemm_bwd (D_{l-1}; its epilogue also emits the column sums = db)
//   k_wide_wreduce   split-K partials -> flat gradient (fixed order)
//   k_wide_gradfin   remaining gradient entries (W_1, biases, output layer, phi) and the loss value
//   k_wide_gradpost  (single-target rmse, weight_l2) rmse factor of the hidden weight blocks, weight_l2 term and its loss
//   k_wide_update    optimiser over the flat vector, bf16 weight images for the next step
// Prediction-statistics losses (rmse over several targets, pearsonLoss, kgeLoss, pbkgeLoss: LOSS_AFFINE targets) put two
// launches between the forward GEMMs and the training head: k_wide_head in its statistics mode over A_NH (sufficient
// statistics of the batch's predictions per CTA) and k_stat_seeds (eh_stat_seeds.cuh: seed coefficients and loss value
// into the batch's scalar row).
// Replaces Lux.Training.single_train_step! (src/training/epoch.jl:20-26) for wide chains; formulas: SURVEY 10.2-10.5.
#pragma once
#include <cuda_bf16.h>
#include "eh_chunk.cuh"
#include "eh_wide_gemm.cuh"
#include "eh_wide.h"

namespace eh {
namespace wide {

static_assert(BS_BN_OFF == BS_BN, "per-batch scalar row layout");

// partial vector written by one CTA of k_wide_head (floats): [NOUT][H] dWo, [NOUT] dbo(pad 4), [H] db_NH,
// [MAXT] loss sums, [MAXPS] phi sums
__host__ __device__ constexpr int head_off_dbo(int H, int NOUT) { return NOUT * H; }
__host__ __device__ constexpr int head_off_dbh(int H, int NOUT) { return NOUT * H + 4; }
__host__ __device__ constexpr int head_off_loss(int H, int NOUT) { return NOUT * H + 4 + H; }
__host__ __device__ constexpr int head_off_phi(int H, int NOUT) { return head_off_loss(H, NOUT) + MAXT; }
__host__ __device__ constexpr int head_npart(int H, int NOUT) { return head_off_phi(H, NOUT) + MAXPS; }

// Shape of the EMBEDDED chain the tensor-core path trains.  A model with several Dense chains (MultiNNHybridModel,
// src/models/GenericHybridModel.jl:169-189: one chain per neural parameter) is embedded block-diagonally: chain c owns
// the units [off_c, off_c + h_c) of every hidden layer, weights between units of different chains (and everything beyond
// the real widths, up to the padded width H) are zeros in the bf16 / fp32 images and never receive an update, because
// the optimiser only walks the flat parameter vector.  `ParamMap` says where a flat entry lives in the images.
struct WideDims {
    int P, H, NH, NOUT, R4;      // total chain inputs, padded hidden width (256 / 512), hidden layers, chain outputs, floats per record
    int nflat, ntheta;
};
// kinds: WK_* (eh_wide.h)
struct ParamMap {                // one per flat entry (reference ComponentArray order)
    int kind;                    // WK_*
    int l;                       // layer (1-based) for WK_W1 / WK_WH / WK_B
    int r, c;                    // image row (output unit / chain output) and column (input unit / chain input / hidden unit)
};

// ---- gather: rec[idx[b]] -> xb[b] ---------------------------------------------------------------------------
// (rows past `Bvalid` -- padding of a batch up to a multiple of 128 -- repeat the batch's first record; the head
// kernel masks them; rows past `nrec` of a contiguous evaluation chunk repeat the last record)
__global__ void __launch_bounds__(256) k_wide_gather(const float4* rec, const int* idx, long long rec_base, long long nrec, int B,
                                                     int Bvalid, int R4q, float4* xb)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const int bs = b < Bvalid ? b : 0;
    long long i = idx ? (long long)idx[bs] : rec_base + bs;
    if (i >= nrec) i = nrec - 1;
    for (int q = 0; q < R4q; q++) xb[(size_t)b * R4q + q] = __ldg(rec + i * R4q + q);
}

__device__ __forceinline__ float act_bf16(int act, float z) { return act1(act, z); }
__device__ __forceinline__ float dact_out(int act, float a) { return dact1(act, a); }
__device__ __forceinline__ uint32_t pack2(float lo, float hi) { return pack_bf16(lo, hi); }

// ---- layer 1: A1[b][o] = act(b1[o] + sum_p xn[b][p] W1[o][p]) ----
// W1img [P][H] / b1img [H]: fp32 images of the embedded first layer (zeros where a unit does not see an input).
// A thread owns 8 consecutive outputs (their weights stay in registers) and walks FIRST_ROWS rows of the batch;
// a CTA covers the whole width for 256 / (H / 8) row groups.
constexpr int FIRST_ROWS = 16;
// PMAX: compile-time bound on the chain inputs (2 / 4 / 8) -- the weights a thread keeps in registers.  Rows go four at
// a time with their inputs loaded first: the kernel is a stream of 16-byte stores (H bf16 per row) and must not wait for
// one L2 round trip per row.
template <int PMAX>
__global__ void __launch_bounds__(256) k_wide_first(const float* __restrict__ xb, const float* __restrict__ W1img,
                                                    const float* __restrict__ b1img, const float* __restrict__ bscal, int use_bn,
                                                    WideDims d, int B, int act, __nv_bfloat16* __restrict__ A1)
{
    const int per_row = d.H / 8;                       // threads across the width
    const int groups = 256 / per_row;                  // row groups per CTA
    const int o0 = (threadIdx.x % per_row) * 8;
    const int r0 = (blockIdx.x * groups + threadIdx.x / per_row) * FIRST_ROWS;
    float bias[8], w[PMAX][8], mu[PMAX], rs[PMAX];
#pragma unroll
    for (int j = 0; j < 8; j++) bias[j] = __ldg(b1img + o0 + j);
#pragma unroll
    for (int p = 0; p < PMAX; p++) {
        mu[p] = (use_bn && p < d.P) ? bscal[BS_BN + 2 * p] : 0.f;
        rs[p] = (use_bn && p < d.P) ? bscal[BS_BN + 2 * p + 1] : 1.f;
#pragma unroll
        for (int j = 0; j < 8; j++) w[p][j] = p < d.P ? __ldg(W1img + (size_t)p * d.H + o0 + j) : 0.f;
    }
    for (int b0 = r0; b0 < r0 + FIRST_ROWS && b0 < B; b0 += 4) {
        float x[4][PMAX];
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
            for (int p = 0; p < PMAX; p++)
                x[i][p] = (b0 + i < B && p < d.P) ? (__ldg(xb + (size_t)(b0 + i) * d.R4 + p) - mu[p]) * rs[p] : 0.f;
#pragma unroll
        for (int i = 0; i < 4; i++) {
            float z[8];
#pragma unroll
            for (int j = 0; j < 8; j++) z[j] = bias[j];
#pragma unroll
            for (int p = 0; p < PMAX; p++)
#pragma unroll
                for (int j = 0; j < 8; j++) z[j] = fmaf(x[i][p], w[p][j], z[j]);
            uint4 o;
            o.x = pack2(act_bf16(act, z[0]), act_bf16(act, z[1]));
            o.y = pack2(act_bf16(act, z[2]), act_bf16(act, z[3]));
            o.z = pack2(act_bf16(act, z[4]), act_bf16(act, z[5]));
            o.w = pack2(act_bf16(act, z[6]), act_bf16(act, z[7]));
            if (b0 + i < B) *reinterpret_cast<uint4*>(A1 + (size_t)(b0 + i) * d.H + o0) = o;
        }
    }
}

// the pieces of StepCfg that resolve_params / the process-model functors look at.  AFF: the training mode knows LOSS_AFFINE
// seeds (a separate instantiation: the kernel runs at its register limit, and the extra case must not cost the others)
template <class PM_, int NOUT_, bool SCALE_, bool AFF_ = false>
struct HeadCfg {
    using PM = PM_;
    static constexpr int NOUT = NOUT_, NPS = PM_::NPS, T = PM_::NT, F = PM_::NF;
    static constexpr bool SCALE = SCALE_, AFF = AFF_;
};

struct HeadArgs {
    const __nv_bfloat16* A;    // [B x H] last hidden activation
    const float* xb;           // [B x R4] compact batch records
    const float* pblock;       // flat theta/phi + tail
    const float* WOimg;        // [NOUT][H] fp32 image of the embedded output layer
    const float* BOimg;        // [4] its bias
    const float* bscal;        // per-batch scalar row
    __nv_bfloat16* D;          // out [B x H] delta of the last hidden layer
    float* partial;            // out [gridDim.x][head_npart]
    float* yhat;               // eval mode: nullable [T][ldy] predictions
    float* parout;             // eval mode: nullable [NPS][ldy] neural parameter values
    long long ldy, row0;       // eval mode: row offset of this batch inside yhat / parout
    double* evalstat;          // eval mode: nullable [gridDim.x][T * 8] sufficient statistics (EVAL_NSTAT layout)
    float shift_y[MAXT];
    WideDims d;
    int B, act, train;
    int Bvalid;                // rows that really exist (eval chunks are padded to a multiple of 128)
    int loss_kind[MAXT];
    PSlot slot[MAXPS];
    float pmc[4];
    const PmProgData* prog;    // device copy of the traced program (PmProgram heads), else NULL
    int nf, nt;                // real forcing / target counts (PmProgram heads; the built-in forms know theirs)
};

// ---- output layer + physics + loss seeds + backward into D_NH; one warp per sample row, 8 warps per CTA ----
// H / 256 chunks of 8 consecutive features per lane (16-byte bf16 accesses).
template <class HC, int HCH>
__global__ void __launch_bounds__(256, 3) k_wide_head(const HeadArgs a)
{
    using PM = typename HC::PM;
    constexpr int NOUT = HC::NOUT, T = HC::T, F = HC::F, NPS = HC::NPS;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int H = a.d.H, P = a.d.P;
    __shared__ float s_pms[MAXPS * PMS_PER_SLOT + MAXPS];
    __shared__ float s_red[8][64];
    __shared__ PmProgData s_prog;
    if (threadIdx.x < MAXPS * PMS_PER_SLOT + MAXPS) s_pms[threadIdx.x] = a.pblock[a.d.nflat + threadIdx.x];
    if (PM::DYNAMIC) {
        const int* src = reinterpret_cast<const int*>(a.prog);
        int* dst = reinterpret_cast<int*>(&s_prog);
        for (int i = threadIdx.x; i < (int)(sizeof(PmProgData) / 4); i += blockDim.x) dst[i] = src[i];
    }
    __syncthreads();
    // real forcing / target counts: compile-time for the built-in forms, from the program otherwise
    const int nf = PM::DYNAMIC ? a.nf : F, nt = PM::DYNAMIC ? a.nt : T;
    // s_pms: [0..8) uniform slot values, [8..40) derived scalars -- same order as the parameter block tail
    PmCtx cx;
    cx.pms = s_pms + MAXPS;
    cx.c = a.pmc;
    cx.prog = &s_prog;
    cx.scale_rt = HC::SCALE ? 1 : 0;
    cx.uniform_mask = 0;
    cx.phi_flag = nullptr;
    cx.phi_want = 0;
#pragma unroll
    for (int s = 0; s < MAXPS; s++)
        if (s >= NPS || a.slot[s].role != ROLE_NEURAL) cx.uniform_mask |= 1u << s;

    // output-layer weights: a CTA copy in shared memory behind the warps' scratch ([NOUT][H]); a lane reads the eight of
    // its features where it needs them (registers are what limits the number of resident warps here, and with it how well
    // the long per-row dependency chain is hidden)
    extern __shared__ float s_vec[];   // [8][(NOUT + 1) * H] reduction scratch / row rings, then [NOUT][H] weights
    float* s_w = s_vec + 8 * (NOUT + 1) * H;
    // lane-major: float4 number ((o * HCH + c) * 2 + half) * 32 + lane holds features (c * 32 + lane) * 8 + 4 half .. + 3 of
    // output o, so that a warp's LDS.128 walks consecutive 16-byte words (feature-major it was a 2-way bank conflict and the
    // shared-memory pipe, at 64 % busy, set the pace of the kernel)
    for (int i = threadIdx.x; i < NOUT * H; i += blockDim.x) {
        const int o = i / H, f = i % H, c = f >> 8, ln = (f >> 3) & 31, half = (f >> 2) & 1, e = f & 3;
        s_w[((((o * HCH + c) * 2 + half) * 32 + ln) << 2) + e] = a.WOimg[i];
    }
    __syncthreads();
    float bout[NOUT];
#pragma unroll
    for (int o = 0; o < NOUT; o++) bout[o] = a.BOimg[o];

    float gW[NOUT][HCH][8], gB[NOUT], gDb[HCH][8], lsum[MAXT], gphi[MAXPS];
    // eval mode: sufficient statistics per warp, kept in shared memory (32 registers the training loop needs for its row prefetch)
    __shared__ double s_e[8][MAXT * 8];
    if (lane == 0)
        for (int i = 0; i < MAXT * 8; i++) s_e[warp][i] = 0.0;
#pragma unroll
    for (int o = 0; o < NOUT; o++) {
        gB[o] = 0.f;
#pragma unroll
        for (int c = 0; c < HCH; c++)
#pragma unroll
            for (int e = 0; e < 8; e++) gW[o][c][e] = 0.f;
    }
#pragma unroll
    for (int c = 0; c < HCH; c++)
#pragma unroll
        for (int e = 0; e < 8; e++) gDb[c][e] = 0.f;
#pragma unroll
    for (int t = 0; t < MAXT; t++) lsum[t] = 0.f;
#pragma unroll
    for (int q = 0; q < MAXPS; q++) gphi[q] = 0.f;

    // The activations of a warp's next FOUR rows are in flight (cp.async into a ring in shared memory) while the current row
    // is worked on: the row's chain of dependent steps -- dot product, warp sum, process model, delta -- is long, and with one
    // row in flight per warp the kernel was bound by memory-level parallelism (16 KB per SM: 3 TB/s).  The ring aliases the
    // warp's own slice of the reduction scratch, which is only written after the loop.
    constexpr int DEPTH = 4;
    const int bend = a.train ? a.B : a.Bvalid, bstep = gridDim.x * 8;
    const uint32_t ring = (uint32_t)__cvta_generic_to_shared(s_vec) + (uint32_t)(warp * (NOUT + 1) * H * 4);
    const int row_bytes = H * 2;
    auto fetch_row = [&](int brow, int slot) {
        if (brow < bend) {
#pragma unroll
            for (int c = 0; c < HCH; c++)
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(ring + (uint32_t)(slot * row_bytes + (c * 32 + lane) * 16)),
                             "l"(a.A + (size_t)brow * H + (c * 32 + lane) * 8)
                             : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");   // (an empty group keeps the count uniform)
    };
#pragma unroll
    for (int dd = 0; dd < DEPTH; dd++) fetch_row(blockIdx.x * 8 + warp + dd * bstep, dd);
    int it = 0;
    for (int b = blockIdx.x * 8 + warp; b < bend; b += bstep, it++) {
        const bool rowvalid = b < a.Bvalid;   // rows beyond: padding of the batch up to a multiple of 128 (train mode)
        float zo[NOUT];
#pragma unroll
        for (int o = 0; o < NOUT; o++) zo[o] = 0.f;
        const int slot = it & (DEPTH - 1);
        asm volatile("cp.async.wait_group %0;" ::"n"(DEPTH - 1) : "memory");   // this row has landed (each lane reads its own 16 bytes)
        // my eight activations of chunk c, from the ring (read again in the delta loop instead of living in registers)
        auto load_av = [&](int c, float (&av)[8]) {
            uint4 raw;
            asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                         : "=r"(raw.x), "=r"(raw.y), "=r"(raw.z), "=r"(raw.w)
                         : "r"(ring + (uint32_t)(slot * row_bytes + (c * 32 + lane) * 16))
                         : "memory");
            const uint32_t rw[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
            for (int e = 0; e < 4; e++) {
                const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&rw[e]));
                av[2 * e] = f.x;
                av[2 * e + 1] = f.y;
            }
        };
        auto load_w = [&](int o, int c, float (&w)[8]) {
            const float4 w0 = reinterpret_cast<const float4*>(s_w)[((o * HCH + c) * 2 + 0) * 32 + lane];
            const float4 w1 = reinterpret_cast<const float4*>(s_w)[((o * HCH + c) * 2 + 1) * 32 + lane];
            w[0] = w0.x; w[1] = w0.y; w[2] = w0.z; w[3] = w0.w; w[4] = w1.x; w[5] = w1.y; w[6] = w1.z; w[7] = w1.w;
        };
#pragma unroll
        for (int c = 0; c < HCH; c++) {
            float av[8];
            load_av(c, av);
#pragma unroll
            for (int o = 0; o < NOUT; o++) {
                float w[8];
                load_w(o, c, w);
#pragma unroll
                for (int e = 0; e < 8; e++) zo[o] = fmaf(av[e], w[e], zo[o]);
            }
        }
#pragma unroll
        for (int o = 0; o < NOUT; o++) zo[o] = warp_sum(zo[o]) + bout[o];

        // every lane evaluates the (cheap) per-sample scalar part redundantly: no broadcast needed afterwards
        float f[F > 0 ? F : 1], y[T], pv[NPS], sg[NPS], yh[T], sv[PM::NSV], gy[T], gp[NPS], dz[NOUT];
        const float* r = a.xb + (size_t)b * a.d.R4;
#pragma unroll
        for (int k = 0; k < F; k++) f[k] = k < nf ? r[P + k] : 0.f;
#pragma unroll
        for (int k = 0; k < T; k++) y[k] = k < nt ? r[P + nf + k] : __int_as_float(0x7fc00000);   // absent target = masked
        resolve_params<HC>(a.slot, s_pms, zo, pv, sg, cx);
        PM::fwd(pv, f, cx, yh, sv);
        if (!a.train) {
            if (lane == 0) {
#pragma unroll
                for (int t = 0; t < T; t++) {
                    if (a.yhat && t < nt) a.yhat[(size_t)t * a.ldy + a.row0 + b] = yh[t];
                    if (y[t] == y[t]) {
                        const double yy = (double)y[t] - a.shift_y[t], hh = (double)yh[t] - a.shift_y[t], rr = (double)yh[t] - y[t];
                        double* e8 = &s_e[warp][t * 8];
                        e8[0] += 1.0; e8[1] += yy; e8[2] += hh; e8[3] += yy * yy;
                        e8[4] += hh * hh; e8[5] += yy * hh; e8[6] += rr * rr; e8[7] += fabs(rr);
                    }
                }
                if (a.parout) {
#pragma unroll
                    for (int q = 0; q < NPS; q++)
                        if (a.slot[q].role == ROLE_NEURAL) a.parout[(size_t)q * a.ldy + a.row0 + b] = pv[q];
                }
            }
            __syncwarp();
            fetch_row(b + DEPTH * bstep, slot);
            continue;
        }
#pragma unroll
        for (int t = 0; t < T; t++) {
            const bool m = rowvalid && (y[t] == y[t]);   // valid_mask = !isnan(y), src/training/train.jl:221-232
            const float rr = m ? yh[t] - y[t] : 0.f;
            const float c = a.bscal[BS_C + t];
            if (a.loss_kind[t] == LOSS_MAE) {
                lsum[t] += fabsf(rr);
                gy[t] = rr > 0.f ? c : (rr < 0.f ? -c : 0.f);
            } else if (HC::AFF && a.loss_kind[t] == LOSS_AFFINE) {
                // dL/dyhat = sa + sb yhat + sc y (k_stat_seeds): the coefficients carry the aggregation weight, the loss value
                // is in the scalar row already
                gy[t] = m ? fmaf(a.bscal[BS_AFF + 2 * MAXT + t], y[t], fmaf(a.bscal[BS_AFF + MAXT + t], yh[t], a.bscal[BS_AFF + t])) : 0.f;
            } else {
                lsum[t] = fmaf(rr, rr, lsum[t]);
                gy[t] = 2.f * c * rr;
            }
        }
        PM::bwd(pv, f, cx, yh, sv, gy, gp);
#pragma unroll
        for (int o = 0; o < NOUT; o++) dz[o] = 0.f;
#pragma unroll
        for (int q = 0; q < NPS; q++) {
            const PSlot sl = a.slot[q];
            if (sl.role == ROLE_NEURAL) {
                float g = gp[q];
                if (HC::SCALE) g *= sl.span * sg[q] * (1.f - sg[q]);
#pragma unroll
                for (int o = 0; o < NOUT; o++)
                    if (sl.idx == o) dz[o] += g;
            } else if (sl.role == ROLE_GLOBAL) {
                gphi[q] += gp[q];
            }
        }
#pragma unroll
        for (int o = 0; o < NOUT; o++) gB[o] += dz[o];
        // delta of the last hidden layer for my features, its column sums, and the output-layer gradient
#pragma unroll
        for (int c = 0; c < HCH; c++) {
            float dv[8], av[8], sacc[8];
            load_av(c, av);
#pragma unroll
            for (int e = 0; e < 8; e++) sacc[e] = 0.f;
#pragma unroll
            for (int o = 0; o < NOUT; o++) {
                float w[8];
                load_w(o, c, w);
#pragma unroll
                for (int e = 0; e < 8; e++) {
                    sacc[e] = fmaf(dz[o], w[e], sacc[e]);
                    gW[o][c][e] = fmaf(dz[o], av[e], gW[o][c][e]);
                }
            }
#pragma unroll
            for (int e = 0; e < 8; e++) {
                // round first: db must be the column sum of the very deltas the weight-gradient GEMM reads
                dv[e] = __bfloat162float(__float2bfloat16_rn(sacc[e] * dact_out(a.act, av[e])));
                gDb[c][e] += dv[e];
            }
            uint4 o4;
            o4.x = pack2(dv[0], dv[1]); o4.y = pack2(dv[2], dv[3]); o4.z = pack2(dv[4], dv[5]); o4.w = pack2(dv[6], dv[7]);
            *reinterpret_cast<uint4*>(a.D + (size_t)b * H + (c * 32 + lane) * 8) = o4;
        }
        __syncwarp();
        fetch_row(b + DEPTH * bstep, slot);   // the slot is free now
    }

    if (!a.train) {
        if (a.evalstat) {
            __syncthreads();
            if (threadIdx.x < nt * 8) {
                double s = 0.0;
                for (int wv = 0; wv < 8; wv++) s += s_e[wv][threadIdx.x];
                a.evalstat[(size_t)blockIdx.x * (nt * 8) + threadIdx.x] = s;
            }
        }
        return;
    }
    // CTA reduction in a fixed order: per-feature vectors through shared memory, warp by warp
    float* out = a.partial + (size_t)blockIdx.x * head_npart(H, NOUT);
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncwarp();
    const int VS = (NOUT + 1) * H;
#pragma unroll
    for (int c = 0; c < HCH; c++)
#pragma unroll
        for (int e = 0; e < 8; e++) {
            const int i = (c * 32 + lane) * 8 + e;
#pragma unroll
            for (int o = 0; o < NOUT; o++) s_vec[warp * VS + o * H + i] = gW[o][c][e];
            s_vec[warp * VS + NOUT * H + i] = gDb[c][e];
        }
    if (lane == 0) {
#pragma unroll
        for (int o = 0; o < NOUT; o++) s_red[warp][o] = gB[o];
#pragma unroll
        for (int t = 0; t < MAXT; t++) s_red[warp][4 + t] = lsum[t];
#pragma unroll
        for (int q = 0; q < MAXPS; q++) s_red[warp][8 + q] = gphi[q];
    }
    __syncthreads();
    for (int i = threadIdx.x; i < VS; i += blockDim.x) {
        float s = 0.f;
        for (int wv = 0; wv < 8; wv++) s += s_vec[wv * VS + i];
        // s_vec order: [NOUT][H] dWo then [H] db_NH ; partial order: dWo, dbo(4), db_NH
        out[i < NOUT * H ? i : i + 4] = s;
    }
    if (threadIdx.x < 4 + MAXT + MAXPS) {
        float s = 0.f;
        for (int wv = 0; wv < 8; wv++) s += s_red[wv][threadIdx.x];
        const int q = threadIdx.x;
        if (q < 4) out[head_off_dbo(H, NOUT) + q] = q < NOUT ? s : 0.f;
        else out[head_off_loss(H, NOUT) + (q - 4)] = s;   // loss sums then phi sums are contiguous
    }
}

// ---- split-K partials [S][H(o)][H(i)] -> flat gradient of one hidden weight block (index o + i * hout), fixed order ----
// The block is the hout x hin matrix of one chain at layer l; it sits at rows o_off.., columns i_off.. of the H x H
// product.  grid = (ceil(hin / 32), ceil(hout / 32)).
__global__ void __launch_bounds__(256) k_wide_wreduce(const float* partial, int S, int H, int hout, int hin, int o_off, int i_off,
                                                      float* grad_w)
{
    __shared__ float tile[32][33];
    const int i0 = blockIdx.x * 32, o0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
    for (int r = ty; r < 32; r += 8) {
        float t[16];
        const bool in = o0 + r < hout && i0 + tx < hin;
#pragma unroll
        for (int z = 0; z < 16; z++)
            t[z] = (z < S && in) ? __ldcs(partial + ((size_t)z * H + (o_off + o0 + r)) * H + i_off + i0 + tx) : 0.f;
        float s = 0.f;
#pragma unroll
        for (int z = 0; z < 16; z++) s += t[z];   // fixed order
        tile[r][tx] = s;   // [o][i]
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8)
        if (i0 + r < hin && o0 + tx < hout) grad_w[(size_t)(i0 + r) * hout + o0 + tx] = tile[tx][r];
}

struct FinArgs {
    WideDims d;
    const ParamMap* map;                          // [nflat]
    const int* small; int n_small;                // flat indices this kernel produces: everything but the hidden weight blocks
    const float* head_partial; int n_head;        // [n_head][head_npart]
    const float* colsum[8]; int n_slab;           // per hidden layer l < NH (index l-1): [n_slab][(1 + P1) * H], P1 = P for l = 1
    const float* bscal;
    const float* theta;
    float* grad;                                  // in/out flat gradient (hidden weight blocks already there)
    float* stats;                                 // out [MAXT] loss sums, [MAXT] the loss value (read by k_wide_gradpost)
    float* loss_out;                              // nullable
    int T, agg_mean;
    int loss_kind[MAXT];
    PSlot slot[MAXPS];
    const int* slot_of_flat;
    int* skip_out;                                // 1: all-masked batch (epoch.jl:17-19)
    int dp;                                       // data parallel: the sums are per-rank; write the loss sums behind the
                                                  // gradient (grad[nflat + t]) and leave loss / skip to k_wide_allreduce
};

// ---- everything of the gradient that is not a hidden weight block, plus the loss value ----
// 8 threads per entry walk the partial vectors (128-row slabs of the backward-data epilogues / CTAs of k_wide_head) with
// a stride of 8 and combine in a fixed shuffle order: deterministic, and the dependent-load chains are 8x shorter.
__global__ void __launch_bounds__(256) k_wide_gradfin(const FinArgs a)
{
    const int H = a.d.H, NOUT = a.d.NOUT, NH = a.d.NH, P = a.d.P;
    const int HP = head_npart(H, NOUT);
    // loss sums of the head CTAs: all 256 threads fetch (one 16-byte load per head CTA), fixed combination order
    __shared__ float s_loss[MAXT];
    __shared__ float s_lw[8][MAXT];
    {
        static_assert(MAXT == 4, "one float4 of loss sums per head CTA");
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int g = threadIdx.x; g < a.n_head; g += 256) {
            const float4 v = *reinterpret_cast<const float4*>(a.head_partial + (size_t)g * HP + head_off_loss(H, NOUT));
            acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
        acc.x = warp_sum(acc.x); acc.y = warp_sum(acc.y); acc.z = warp_sum(acc.z); acc.w = warp_sum(acc.w);
        if ((threadIdx.x & 31) == 0) {
            float* d4 = s_lw[threadIdx.x >> 5];
            d4[0] = acc.x; d4[1] = acc.y; d4[2] = acc.z; d4[3] = acc.w;
        }
        __syncthreads();
        if (threadIdx.x < MAXT) {
            float t8 = 0.f;
            for (int wv = 0; wv < 8; wv++) t8 += s_lw[wv][threadIdx.x];
            s_loss[threadIdx.x] = t8;
        }
    }
    __syncthreads();
    float post = 1.f, ntot = 0.f, L = 0.f;
    for (int t = 0; t < a.T; t++) {
        const float n = a.bscal[BS_N + t], ss = a.bscal[BS_SS + t], acc = s_loss[t];
        ntot += n;
        if (a.loss_kind[t] == LOSS_RMSE) post = 1.f / (2.f * sqrtf(acc / n));
        L += (a.loss_kind[t] == LOSS_NSELOSS)  ? acc / ss
             : (a.loss_kind[t] == LOSS_RMSE)   ? sqrtf(acc / n)
             : (a.loss_kind[t] == LOSS_AFFINE) ? a.bscal[BS_AFF + 3 * MAXT + t]   // value left by k_stat_seeds
                                               : acc / n;
    }
    if (a.agg_mean) L /= (float)a.T;
    if (a.dp) post = 1.f;   // rmse is refused in data-parallel mode
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        if (a.dp) {
            for (int t = 0; t < MAXT; t++) a.grad[a.d.nflat + t] = s_loss[t];
        } else {
            if (a.loss_out) *a.loss_out = ntot == 0.f ? __int_as_float(0x7fc00000) : L;
            *a.skip_out = ntot == 0.f;
            for (int t = 0; t < MAXT; t++) a.stats[t] = s_loss[t];
            a.stats[MAXT] = L;
        }
    }
    const int q = blockIdx.x * 32 + (threadIdx.x >> 3), zl = threadIdx.x & 7;
    const bool live = q < a.n_small;
    int p = 0, cnt = 0, phi_slot = -1;
    size_t stride = 0;
    const float* src = nullptr;
    bool is_phi = false;
    if (live) {
        p = a.small[q];
        const ParamMap m = a.map[p];
        if (m.kind == WK_W1) {            // W_1[r][c]: x-weighted column sums of D_1 live at (1 + c) H + r
            src = a.colsum[0] + (size_t)(1 + m.c) * H + m.r; stride = (size_t)(1 + P) * H; cnt = a.n_slab;
        } else if (m.kind == WK_B) {      // b_l[r]: column sums of D_l
            if (m.l == NH) { src = a.head_partial + head_off_dbh(H, NOUT) + m.r; stride = HP; cnt = a.n_head; }
            else { src = a.colsum[m.l - 1] + m.r; stride = (size_t)(m.l == 1 ? 1 + P : 1) * H; cnt = a.n_slab; }
        } else if (m.kind == WK_WO) {
            src = a.head_partial + (size_t)m.r * H + m.c; stride = HP; cnt = a.n_head;
        } else if (m.kind == WK_BO) {
            src = a.head_partial + head_off_dbo(H, NOUT) + m.r; stride = HP; cnt = a.n_head;
        } else {                          // phi_raw
            is_phi = true;
            phi_slot = a.slot_of_flat[p];
            src = a.head_partial + head_off_phi(H, NOUT) + (phi_slot >= 0 ? phi_slot : 0);
            stride = HP; cnt = phi_slot >= 0 ? a.n_head : 0;
        }
    }
    float s = 0.f;
    {
        // four independent loads in flight per thread (the partial vectors are L2-resident: latency, not bandwidth)
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
        int z = zl;
        for (; z + 24 < cnt; z += 32) {
            s0 += src[(size_t)z * stride];
            s1 += src[(size_t)(z + 8) * stride];
            s2 += src[(size_t)(z + 16) * stride];
            s3 += src[(size_t)(z + 24) * stride];
        }
        for (; z < cnt; z += 8) s0 += src[(size_t)z * stride];
        s = (s0 + s1) + (s2 + s3);
    }
    s += __shfl_xor_sync(0xffffffffu, s, 4);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    if (live && zl == 0) {
        if (is_phi && phi_slot >= 0) {
            // phi_raw: chained through the sigmoid squash (SURVEY 10.4)
            const float sg = 1.f / (1.f + expf(-a.theta[p]));
            s *= a.slot[phi_slot].span * sg * (1.f - sg);
        }
        a.grad[p] = s * post;
    }
}

struct PostArgs {
    const ParamMap* map; int nflat;
    const float* theta;                           // parameters before this step's update
    float* grad;                                  // in/out flat gradient (complete after k_wide_gradfin)
    const float* stats;                           // [MAXT] loss sums, [MAXT] loss value (k_wide_gradfin)
    const float* bscal;
    int T;
    int loss_kind[MAXT];
    const float* l2coef;                          // nullable [nflat]: 2 l2_loss_coef on the weight_l2 entries, else 0
    float l2_aggw, l2_loss_coef;
    float* l2part;                                // [gridDim.x] CTA sums of theta^2 over the weight_l2 entries
    unsigned* ticket;                             // CTAs done (zero between launches)
    float* loss_out;                              // nullable
};

// ---- the last pass over the flat gradient, for the loss terms that need all of it (exact path: k_update) ----
// single-target rmse: the hidden weight blocks come straight from the GEMM partials, without the 1 / (2 rmse) that
// k_wide_gradfin applies to every other entry.  weight_l2: g <- l2_aggw (g + l2coef[p] theta[p]) for every entry, and the
// loss l2_aggw (L + l2_loss_coef sum theta^2) -- the sum over the flagged entries in a fixed order: per CTA (thread stride,
// warp tree, warps in order), then the CTA sums in order by the CTA that finishes last.
__global__ void __launch_bounds__(256) k_wide_gradpost(const PostArgs a)
{
    float post = 1.f;
    for (int t = 0; t < a.T; t++)
        if (a.loss_kind[t] == LOSS_RMSE) post = 1.f / (2.f * sqrtf(a.stats[t] / a.bscal[BS_N + t]));
    float s = 0.f;
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < a.nflat; p += gridDim.x * blockDim.x) {
        float g = a.grad[p];
        if (post != 1.f && a.map[p].kind == WK_WH) g *= post;
        if (a.l2coef) {
            const float th = a.theta[p], c = a.l2coef[p];
            if (c != 0.f) s = fmaf(th, th, s);
            g = a.l2_aggw * fmaf(c, th, g);
        }
        a.grad[p] = g;
    }
    if (!a.l2coef) return;
    __shared__ float s_w[8];
    __shared__ bool s_last;
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        float cta = 0.f;
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) cta += s_w[w];
        a.l2part[blockIdx.x] = cta;
        __threadfence();   // the CTA sum is visible before the ticket says so
        s_last = atomicAdd(a.ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last || threadIdx.x != 0) return;
    __threadfence();
    float S = 0.f, ntot = 0.f;
    for (int g = 0; g < (int)gridDim.x; g++) S += __ldcg(a.l2part + g);
    for (int t = 0; t < a.T; t++) ntot += a.bscal[BS_N + t];
    if (a.loss_out) *a.loss_out = ntot == 0.f ? __int_as_float(0x7fc00000) : a.l2_aggw * (a.stats[MAXT] + a.l2_loss_coef * S);
    *a.ticket = 0u;
}

// ---- data parallel (one process per GPU): gradient all-reduce over NVLink peer memory ----
// Every rank exposes [2 parities][xlen] floats (flat gradient, then MAXT loss sums) and two flags through CUDA IPC.
// A rank publishes "my vector of step `tag` is complete" with a system-scope release store of its flag; every CTA
// waits for all ranks' flags, then sums its slice of the vector over the ranks IN RANK ORDER straight out of the
// peers' memory (bit-identical result everywhere, no NCCL, no second pass).  Double buffering by step parity is
// enough: a rank can publish step s+2 only after it has seen every peer's step s+1 flag, which a peer raises after
// it has finished reading step s.
struct AllredArgs {
    float* peer[EH_MAX_WORLD];   // rank r's exchange block as mapped here
    int world, rank, par;
    int xlen, nflat;
    unsigned tag;
    float* grad_out;             // [nflat] summed gradient
    float* stats;                // [MAXT] summed loss sums
    float* loss_out;             // nullable
    int* skip_out;
    const float* bscal;          // row of the GLOBAL batch
    int T, agg_mean;
    int loss_kind[MAXT];
    unsigned* err;
};
__device__ __forceinline__ unsigned* allred_flag(float* block, int xlen, int par)
{
    return reinterpret_cast<unsigned*>(block + 2 * (size_t)xlen) + 16 * par;
}
__global__ void __launch_bounds__(256) k_wide_allreduce(const AllredArgs a)
{
    if (threadIdx.x == 0) {
        if (blockIdx.x == 0) {
            __threadfence_system();   // this rank's gradient kernels have completed: make their writes visible to peers
            asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(allred_flag(a.peer[a.rank], a.xlen, a.par)), "r"(a.tag) : "memory");
        }
        for (int r = 0; r < a.world; r++) {
            const unsigned* f = allred_flag(a.peer[r], a.xlen, a.par);
            unsigned v, spins = 0;
            do {
                asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
                if (v != a.tag && ++spins > (1u << 24)) { *a.err = 1; break; }
            } while (v != a.tag);
        }
    }
    __syncthreads();
    const size_t off = (size_t)a.par * a.xlen;
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < a.nflat; p += gridDim.x * blockDim.x) {
        float s = 0.f;
        for (int r = 0; r < a.world; r++) s += __ldcv(a.peer[r] + off + p);
        a.grad_out[p] = s;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        float L = 0.f, ntot = 0.f;
        for (int t = 0; t < a.T; t++) {
            float acc = 0.f;
            for (int r = 0; r < a.world; r++) acc += __ldcv(a.peer[r] + off + a.nflat + t);
            a.stats[t] = acc;
            const float n = a.bscal[BS_N + t], ss = a.bscal[BS_SS + t];
            ntot += n;
            L += (a.loss_kind[t] == LOSS_NSELOSS) ? acc / ss : acc / n;
        }
        if (a.agg_mean) L /= (float)a.T;
        if (a.loss_out) *a.loss_out = ntot == 0.f ? __int_as_float(0x7fc00000) : L;
        *a.skip_out = ntot == 0.f;
    }
}

struct WUpdArgs {
    WideDims d;
    const ParamMap* map;
    float* theta; float* m; float* v; OptState* ost;
    const float* grad;
    const int* skip;
    int opt_kind, adamw_coupled;
    float eta, beta1, beta2, eps, lambda;
    // images of the embedded chain, all zero outside the real entries
    float* W1img;              // [P][H] fp32
    __nv_bfloat16* Wf[8];      // [l-1], l = 2..NH: W_l as [out][in]  (B operand of the forward GEMM)
    __nv_bfloat16* Wb[8];      //                  W_l as [in][out]  (B operand of the backward-data GEMM)
    float* Bp[8];              // [l-1], l = 1..NH: b_l padded to H floats
    float* WOimg;              // [NOUT][H] fp32
    float* BOimg;              // [4]
    int apply;                 // 0: only refresh the images from theta
};

// ---- optimiser over the flat vector (Optimisers.jl rules, SURVEY 10.5) + images for the next step ----
__global__ void __launch_bounds__(256) k_wide_update(const WUpdArgs a)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= a.d.nflat) return;
    const ParamMap mp = a.map[p];
    float th = a.theta[p];
    if (a.apply && !*a.skip) {
        const float g = a.grad[p];
        const float b1t = a.ost->b1t, b2t = a.ost->b2t;
        float dx;
        if (a.opt_kind == OPT_ADAM || a.opt_kind == OPT_ADAMW) {
            const float mt = a.beta1 * a.m[p] + (1.f - a.beta1) * g;
            const float vt = a.beta2 * a.v[p] + (1.f - a.beta2) * g * g;
            a.m[p] = mt;
            a.v[p] = vt;
            dx = mt / (1.f - b1t) / (sqrtf(vt / (1.f - b2t)) + a.eps) * a.eta;
            if (a.opt_kind == OPT_ADAMW) dx += (a.adamw_coupled ? a.eta * a.lambda : a.lambda) * th;
        } else if (a.opt_kind == OPT_RMSPROP) {
            const float qv = a.beta2 * a.v[p] + (1.f - a.beta2) * g * g;
            a.v[p] = qv;
            dx = g * a.eta / (sqrtf(qv) + a.eps);
        } else {
            dx = a.eta * g;
        }
        th -= dx;
        a.theta[p] = th;
    }
    const int H = a.d.H;
    if (mp.kind == WK_WH) {
        const __nv_bfloat16 hb = __float2bfloat16_rn(th);
        a.Wb[mp.l - 1][(size_t)mp.c * H + mp.r] = hb;
        a.Wf[mp.l - 1][(size_t)mp.r * H + mp.c] = hb;
    } else if (mp.kind == WK_W1) {
        a.W1img[(size_t)mp.c * H + mp.r] = th;
    } else if (mp.kind == WK_B) {
        a.Bp[mp.l - 1][mp.r] = th;
    } else if (mp.kind == WK_WO) {
        a.WOimg[(size_t)mp.r * H + mp.c] = th;
    } else if (mp.kind == WK_BO) {
        a.BOimg[mp.r] = th;
    }
}
// step counters advance once per applied step (after k_wide_update of that step)
__global__ void k_wide_advance(OptState* ost, const int* skip, float beta1, float beta2, int apply)
{
    if (!apply) return;
    if (*skip) { ost->skipped++; return; }
    ost->b1t *= beta1;
    ost->b2t *= beta2;
    ost->t++;
}

}  // namespace wide
}  // namespace eh
