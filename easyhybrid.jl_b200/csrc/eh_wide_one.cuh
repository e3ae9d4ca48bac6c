// eh_wide_one.cuh -- one training step of a chain with ONE wide hidden layer (33..512 units), exact fp32, one kernel (sm_100a).
//
// With one hidden layer there is no H x H contraction: layer 1 has fan-in P <= 12 and the output layer fan-out NOUT <= 4,
// so the whole forward, the loss seeds, the backward and the gradient sums are per-sample work on CUDA cores.  k_wide_one
// does all of it on-chip and reads nothing per step but the batch records; it replaces k_wide_gather, k_wide_first, the
// forward / backward GEMMs and k_wide_head of the NH >= 2 path.  What follows it is the wide path's unchanged tail:
// k_wide_gradfin (reads the partials below), k_wide_gradpost, k_wide_allreduce, k_wide_update, k_wide_advance.
//
// Mapping.  The padded width H is a multiple of 64.  A GROUP of H / 2 threads covers the width, a thread owns two adjacent
// units (its W1 columns, b1 entries and output-layer weights stay in registers as float2: FFMA2 over the unit pair); a CTA
// holds G = 256 / (H / 2) groups (1 at H = 512, 8 at H = 64).  Rows go in tiles of G x ONE_R (group g takes rows
// [g ONE_R, (g + 1) ONE_R) of the tile); per tile:
//   1. forward of the owned units for the group's rows; a, act'(z) kept in registers; the output-layer partial sums
//      transpose-reduced across the warp (8 rows per pass) into shared memory
//   2. __syncthreads; one thread per row adds its group's warps (fixed order) -> zo, then the per-sample scalar part of
//      k_wide_head: input BatchNorm (from the batch's scalar row), resolve_params / PM::fwd / PM::bwd, MAE / squared-error /
//      LOSS_AFFINE seeds, NaN-target and padding masks, scale_nn_outputs -> dz into shared memory
//   3. __syncthreads; delta = act'(z) sum_o Wo[o][h] dz_o accumulated into dW1, db1 and dWo in registers
// The batch records of the next tile are loaded (through the index stream) while the current one is worked on, into one of
// three buffers.  Activations are the exact path's (eh_device.cuh: act_fwd2 / act_bwd2, swish included), not the
// tanh.approx of the GEMM epilogues.
//
// Partials (one row per CTA, no atomics), in the layouts k_wide_gradfin reads for NH = 1:
//   head_partial [CTA][head_npart(H, NOUT)]: dWo [NOUT][H], dbo (4), db1 at head_off_dbh, loss sums, phi sums
//   colsum       [CTA][(1 + P) H]:          dW1[u][p] at (1 + p) H + u   (the first H floats are not written: db1 is above)
// The CTA count and every CTA's tiles (tile = CTA + k * CTAs) depend on the shape and B only, and all sums run in a fixed
// order: a step is bit-reproducible.
// Modes: ONE_TRAIN (the above), ONE_STATS (forward only: per-CTA sufficient statistics of the predictions in the EVAL_NSTAT
// layout, for k_stat_seeds), ONE_EVAL (yhat, parout, evalstat).
#pragma once
#include "eh_wide_kernels.cuh"

namespace eh {
namespace wide {

constexpr int ONE_THREADS = 256;   // CTA size at H = 64 / 128 / 256 / 512 (fewer where H / 2 does not divide 256)
constexpr int ONE_R = 16;          // rows per group and tile
constexpr int ONE_FY = 8;          // forcing + target floats of a record kept per row (PmProgram: NF + NT <= 6)
enum : int { ONE_TRAIN = 0, ONE_STATS = 1, ONE_EVAL = 2 };

__host__ __device__ constexpr int one_group_threads(int H) { return H / 2; }
__host__ __device__ constexpr int one_block(int H) { return ONE_THREADS / (H / 2) * (H / 2); }
__host__ __device__ constexpr int one_tile_rows(int H) { return ONE_THREADS / (H / 2) * ONE_R; }
// chain inputs an instantiation holds: WIDE_MAXP, or WIDE_MAXP_X for models with 9..12 inputs (their own instantiations:
// the weights and gradient accumulators of 12 inputs do not fit the register budget of the 8-input kernel)
__host__ __device__ constexpr int one_px(int P) { return P > WIDE_MAXP ? WIDE_MAXP_X : WIDE_MAXP; }
// dynamic shared memory: three record buffers [3][tile rows][PX + ONE_FY], reused after the row loop for the CTA
// reduction of the unit accumulators [groups][NOUT + 1 + P][H]
__host__ __device__ constexpr int one_smem(int H, int P, int NOUT)
{
    return 4 * (3 * one_tile_rows(H) * (one_px(P) + ONE_FY) > (ONE_THREADS / (H / 2)) * (NOUT + 1 + P) * H
                    ? 3 * one_tile_rows(H) * (one_px(P) + ONE_FY)
                    : (ONE_THREADS / (H / 2)) * (NOUT + 1 + P) * H);
}

struct OneArgs {
    const float* rec;          // batch records [.][R4]: row b is rec[idx[b]], or rec[rec_base + b] (clamped to nrec - 1) without idx
    const int* idx;
    long long rec_base, nrec;
    const float* pblock;       // flat theta/phi + tail
    const float* W1img;        // [P][H] fp32 images of the embedded chain (zeros outside the real entries)
    const float* b1img;        // [H]
    const float* WOimg;        // [NOUT][H]
    const float* BOimg;        // [4]
    const float* bscal;        // per-batch scalar row
    float* partial;            // train: [gridDim.x][head_npart(H, NOUT)]
    float* colsum;             // train: [gridDim.x][(1 + P) H]
    float* yhat;               // eval: nullable [T][ldy]
    float* parout;             // eval: nullable [NPS][ldy]
    long long ldy, row0;       // eval: row offset of this chunk inside yhat / parout
    double* evalstat;          // statistics / eval: nullable [gridDim.x][nt * 8] (EVAL_NSTAT layout)
    float shift_y[MAXT];
    WideDims d;
    int B;                     // rows
    int act, mode, use_bn;
    int loss_kind[MAXT];
    PSlot slot[MAXPS];
    float pmc[4];
    const PmProgData* prog;    // PmProgram: device copy of the traced program
    int nf, nt;
};

// v[i]: this lane's partial of row i of an 8-row pass.  Returns the warp's sum of row (lane >> 2) & 7 (transpose-reduce:
// 4 + 2 + 1 exchanges halve the rows a lane carries, two butterflies finish the sum).  Fixed order: deterministic.
__device__ __forceinline__ float one_xsum8(float (&v)[8], int lane)
{
    const unsigned FULL = 0xffffffffu;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const bool up = lane & 16;
        const float s = __shfl_xor_sync(FULL, up ? v[i] : v[i + 4], 16);
        v[i] = (up ? v[i + 4] : v[i]) + s;
    }
#pragma unroll
    for (int i = 0; i < 2; i++) {
        const bool up = lane & 8;
        const float s = __shfl_xor_sync(FULL, up ? v[i] : v[i + 2], 8);
        v[i] = (up ? v[i + 2] : v[i]) + s;
    }
    {
        const bool up = lane & 4;
        const float s = __shfl_xor_sync(FULL, up ? v[0] : v[1], 4);
        v[0] = (up ? v[1] : v[0]) + s;
    }
    v[0] += __shfl_xor_sync(FULL, v[0], 2);
    v[0] += __shfl_xor_sync(FULL, v[0], 1);
    return v[0];
}

// forward of a thread's two units over its group's ONE_R rows.  xs: the group's rows of the tile, [ONE_R][PX]
// normalised inputs (zero beyond P); s_pw: this warp's [NO][ONE_R] output-layer sums (NO = max(NOUT, 2))
template <int ACT, int PMAX, int NOUT, int PX, int NO>
__device__ __forceinline__ void one_forward(const float* xs, const float2 (&w1)[PX], float2 b1, const float2 (&wo)[NO],
                                            float2 (&A)[ONE_R], float2 (&Gd)[ONE_R], float* s_pw, int lane)
{
#pragma unroll
    for (int c = 0; c < ONE_R / 8; c++) {
        float part[NOUT][8];
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const int r = c * 8 + i;
            float x[PMAX];
#pragma unroll
            for (int q = 0; q < PMAX; q += 2) {
                const float2 v = *reinterpret_cast<const float2*>(xs + r * PX + q);
                x[q] = v.x;
                if (q + 1 < PMAX) x[q + 1] = v.y;
            }
            float2 z = b1;
#pragma unroll
            for (int p = 0; p < PMAX; p++) z = fma2s(w1[p], x[p], z);
            float2 aux = f2s(0.f);
            const float2 av = act_fwd2<ACT>(z, aux);
            A[r] = av;
            Gd[r] = act_bwd2<ACT>(av, aux);
#pragma unroll
            for (int o = 0; o < NOUT; o++) part[o][i] = fmaf(av.y, wo[o].y, av.x * wo[o].x);
        }
#pragma unroll
        for (int o = 0; o < NOUT; o++) {
            const float s = one_xsum8(part[o], lane);
            if ((lane & 3) == 0) s_pw[o * ONE_R + c * 8 + (lane >> 2)] = s;
        }
    }
}

template <int ACT, int NOUT, int PX, int NO>
__device__ __forceinline__ void one_forward_p(int P, const float* xs, const float2 (&w1)[PX], float2 b1, const float2 (&wo)[NO],
                                              float2 (&A)[ONE_R], float2 (&Gd)[ONE_R], float* s_pw, int lane)
{
    if constexpr (PX > WIDE_MAXP) {
        one_forward<ACT, PX, NOUT, PX, NO>(xs, w1, b1, wo, A, Gd, s_pw, lane);   // (9..12 inputs)
    } else {
        if (P <= 2) one_forward<ACT, 2, NOUT, PX, NO>(xs, w1, b1, wo, A, Gd, s_pw, lane);
        else if (P <= 4) one_forward<ACT, 4, NOUT, PX, NO>(xs, w1, b1, wo, A, Gd, s_pw, lane);
        else one_forward<ACT, 8, NOUT, PX, NO>(xs, w1, b1, wo, A, Gd, s_pw, lane);
    }
}

// backward of a thread's two units over its group's rows: delta = act'(z) sum_o Wo[o] dz_o -> dW1, db1, dWo
template <int PMAX, int NOUT, int PX, int NO>
__device__ __forceinline__ void one_backward(const float* xs, const float* s_dzg, const float2 (&wo)[NO], const float2 (&A)[ONE_R],
                                             const float2 (&Gd)[ONE_R], float2 (&gW1)[PX], float2& gb, float2 (&gWo)[NO])
{
#pragma unroll
    for (int r = 0; r < ONE_R; r++) {
        float dz[NOUT];
#pragma unroll
        for (int o = 0; o < NOUT; o++) dz[o] = s_dzg[o * (ONE_THREADS / 32 * ONE_R) + r];
        float2 s = f2s(0.f);
#pragma unroll
        for (int o = 0; o < NOUT; o++) s = fma2s(wo[o], dz[o], s);
        const float2 dl = mul2(s, Gd[r]);
        gb = add2(gb, dl);
#pragma unroll
        for (int q = 0; q < PMAX; q += 2) {
            const float2 v = *reinterpret_cast<const float2*>(xs + r * PX + q);
            gW1[q] = fma2s(dl, v.x, gW1[q]);
            if (q + 1 < PMAX) gW1[q + 1] = fma2s(dl, v.y, gW1[q + 1]);
        }
#pragma unroll
        for (int o = 0; o < NOUT; o++) gWo[o] = fma2s(A[r], dz[o], gWo[o]);
    }
}

// PX: chain inputs held (one_px).  The instantiations of 9..12 inputs or 3..4 outputs (traced process models) keep more
// weights and accumulators in registers than the 128 of two resident CTAs allow: they run at one CTA per SM.
template <class HC, int PX = WIDE_MAXP>
__global__ void __launch_bounds__(ONE_THREADS, (PX > WIDE_MAXP || HC::NOUT > 2) ? 1 : 2) k_wide_one(const OneArgs a)
{
    using PM = typename HC::PM;
    constexpr int NOUT = HC::NOUT, T = HC::T, F = HC::F, NPS = HC::NPS;
    constexpr int NO = NOUT > 2 ? NOUT : 2;            // output-layer registers / shared rows (two for one output, as before)
    constexpr int NPRE = (PX + ONE_FY) / 2;            // record floats a thread fetches per tile, at most (16 R4 / (H / 2))
    constexpr int MAXRT = ONE_THREADS / 32 * ONE_R;   // tile rows at most (H = 64)
    const int H = a.d.H, P = a.d.P, R4 = a.d.R4;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int NTg = H / 2, RT = (int)blockDim.x / NTg * ONE_R, wpg = NTg / 32;
    const int grp = tid / NTg, u0 = 2 * (tid - grp * NTg);   // my group, my two units
    __shared__ float s_pms[MAXPS * PMS_PER_SLOT + MAXPS];
    __shared__ PmProgData s_prog;
    __shared__ float s_bn[2 * PX];
    __shared__ float s_part[ONE_THREADS / 32][NO * ONE_R];  // per warp: output-layer sums of its group's rows
    __shared__ float s_dz[NO * MAXRT];                       // [NOUT][tile rows] output-layer deltas
    __shared__ double s_e[ONE_THREADS / 32][MAXT * 8];      // statistics / eval: sufficient statistics per warp
    __shared__ float s_red[ONE_THREADS / 32][16];
    extern __shared__ float s_dyn[];                         // [3][tile rows][PX + ONE_FY] records, then the reduction
    float* s_x = s_dyn;                                      // [3][RT][PX] normalised chain inputs (zero beyond P)
    float* s_fy = s_dyn + 3 * RT * PX;                       // [3][RT][ONE_FY] forcings then targets
    for (int i = tid; i < MAXPS * PMS_PER_SLOT + MAXPS; i += blockDim.x) s_pms[i] = a.pblock[a.d.nflat + i];
    if (PM::DYNAMIC) {
        const int* src = reinterpret_cast<const int*>(a.prog);
        int* dst = reinterpret_cast<int*>(&s_prog);
        for (int i = tid; i < (int)(sizeof(PmProgData) / 4); i += blockDim.x) dst[i] = src[i];
    }
    if (tid < 2 * PX) s_bn[tid] = (a.use_bn && tid < 2 * P) ? a.bscal[BS_BN + tid] : ((tid & 1) ? 1.f : 0.f);
    for (int i = tid; i < ONE_THREADS / 32 * MAXT * 8; i += blockDim.x) (&s_e[0][0])[i] = 0.0;
    for (int i = tid; i < 3 * RT * PX; i += blockDim.x) s_x[i] = 0.f;
    const int nf = PM::DYNAMIC ? a.nf : F, nt = PM::DYNAMIC ? a.nt : T;
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

    // my units' weights (registers) and the accumulators of their gradient
    float2 w1[PX], wo[NO], gW1[PX], gWo[NO];
    const float2 b1 = f2(__ldg(a.b1img + u0), __ldg(a.b1img + u0 + 1));
    float2 gb = f2s(0.f);
#pragma unroll
    for (int p = 0; p < PX; p++) {
        w1[p] = p < P ? f2(__ldg(a.W1img + (size_t)p * H + u0), __ldg(a.W1img + (size_t)p * H + u0 + 1)) : f2s(0.f);
        gW1[p] = f2s(0.f);
    }
#pragma unroll
    for (int o = 0; o < NO; o++) {
        wo[o] = o < NOUT ? f2(__ldg(a.WOimg + (size_t)o * H + u0), __ldg(a.WOimg + (size_t)o * H + u0 + 1)) : f2s(0.f);
        gWo[o] = f2s(0.f);
    }
    float bout[NOUT], gB[NOUT], lsum[MAXT], gphi[MAXPS];   // (row threads)
#pragma unroll
    for (int o = 0; o < NOUT; o++) { bout[o] = __ldg(a.BOimg + o); gB[o] = 0.f; }
#pragma unroll
    for (int t = 0; t < MAXT; t++) lsum[t] = 0.f;
#pragma unroll
    for (int q = 0; q < MAXPS; q++) gphi[q] = 0.f;

    // records of a tile: up to NPRE floats per thread in flight (16 R4 / (H / 2) <= 8 / 10), stored after the forward of the tile before
    const int ntiles = (a.B + RT - 1) / RT, nrec_el = RT * R4;
    float pre[NPRE];
    auto fetch = [&](int tile) {
#pragma unroll
        for (int k = 0; k < NPRE; k++) {
            const int i = tid + k * (int)blockDim.x;
            pre[k] = 0.f;
            if (tile < ntiles && i < nrec_el) {
                const int r = i / R4, b = tile * RT + r;
                if (b < a.B) {
                    long long ri = a.idx ? (long long)__ldg(a.idx + b) : a.rec_base + b;
                    if (ri >= a.nrec) ri = a.nrec - 1;
                    pre[k] = __ldg(a.rec + ri * R4 + (i - r * R4));
                }
            }
        }
    };
    auto store = [&](int buf) {
#pragma unroll
        for (int k = 0; k < NPRE; k++) {
            const int i = tid + k * (int)blockDim.x;
            if (i < nrec_el) {
                const int r = i / R4, j = i - r * R4;
                if (j < P) s_x[(buf * RT + r) * PX + j] = (pre[k] - s_bn[2 * j]) * s_bn[2 * j + 1];
                else if (j - P < ONE_FY) s_fy[(buf * RT + r) * ONE_FY + j - P] = pre[k];
            }
        }
    };
    __syncthreads();   // s_bn, s_x zeros
    fetch(blockIdx.x);
    store(0);
    __syncthreads();

    float2 A[ONE_R], Gd[ONE_R];
    int it = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, it++) {
        const int buf = it % 3;
        fetch(tile + gridDim.x);
        const float* xs = s_x + (buf * RT + grp * ONE_R) * PX;
        switch (a.act) {
        case ACT_TANH: one_forward_p<ACT_TANH, NOUT, PX, NO>(P, xs, w1, b1, wo, A, Gd, s_part[warp], lane); break;
        case ACT_SIGMOID: one_forward_p<ACT_SIGMOID, NOUT, PX, NO>(P, xs, w1, b1, wo, A, Gd, s_part[warp], lane); break;
        case ACT_RELU: one_forward_p<ACT_RELU, NOUT, PX, NO>(P, xs, w1, b1, wo, A, Gd, s_part[warp], lane); break;
        case ACT_SWISH: one_forward_p<ACT_SWISH, NOUT, PX, NO>(P, xs, w1, b1, wo, A, Gd, s_part[warp], lane); break;
        default: one_forward_p<ACT_IDENTITY, NOUT, PX, NO>(P, xs, w1, b1, wo, A, Gd, s_part[warp], lane); break;
        }
        store((it + 1) % 3);
        __syncthreads();

        // ---- per-sample scalar part: one thread per row of the tile (whole warps enter: warp sums below) ----
        if (warp * 32 < RT) {
            const int rt = tid, b = tile * RT + rt;
            const bool live = rt < RT && b < a.B;
            float y[T], yh[T];
#pragma unroll
            for (int t = 0; t < T; t++) { y[t] = __int_as_float(0x7fc00000); yh[t] = 0.f; }
            if (live) {
                const int g = rt / ONE_R, rr = rt - g * ONE_R;
                float zo[NOUT];
#pragma unroll
                for (int o = 0; o < NOUT; o++) {
                    float s = 0.f;
                    for (int w = 0; w < wpg; w++) s += s_part[g * wpg + w][o * ONE_R + rr];
                    zo[o] = s + bout[o];
                }
                const float* fy = s_fy + (buf * RT + rt) * ONE_FY;
                float f[F > 0 ? F : 1], pv[NPS], sg[NPS], sv[PM::NSV], gy[T], gp[NPS];
#pragma unroll
                for (int k = 0; k < F; k++) f[k] = k < nf ? fy[k] : 0.f;
#pragma unroll
                for (int k = 0; k < T; k++) y[k] = k < nt ? fy[nf + k] : __int_as_float(0x7fc00000);   // absent target = masked
                resolve_params<HC>(a.slot, s_pms, zo, pv, sg, cx);
                PM::fwd(pv, f, cx, yh, sv);
                if (a.mode == ONE_EVAL) {
                    const long long row = a.row0 + b;
#pragma unroll
                    for (int t = 0; t < T; t++)
                        if (a.yhat && t < nt) a.yhat[(size_t)t * a.ldy + row] = yh[t];
                    if (a.parout) {
#pragma unroll
                        for (int q = 0; q < NPS; q++)
                            if (a.slot[q].role == ROLE_NEURAL) a.parout[(size_t)q * a.ldy + row] = pv[q];
                    }
                } else if (a.mode == ONE_TRAIN) {
#pragma unroll
                    for (int t = 0; t < T; t++) {
                        const bool m = y[t] == y[t];   // valid_mask = !isnan(y), src/training/train.jl:221-232
                        const float rr2 = m ? yh[t] - y[t] : 0.f;
                        const float c = a.bscal[BS_C + t];
                        if (a.loss_kind[t] == LOSS_MAE) {
                            lsum[t] += fabsf(rr2);
                            gy[t] = rr2 > 0.f ? c : (rr2 < 0.f ? -c : 0.f);
                        } else if (a.loss_kind[t] == LOSS_AFFINE) {
                            // dL/dyhat = sa + sb yhat + sc y (k_stat_seeds; the loss value is in the scalar row already)
                            gy[t] = m ? fmaf(a.bscal[BS_AFF + 2 * MAXT + t], y[t], fmaf(a.bscal[BS_AFF + MAXT + t], yh[t], a.bscal[BS_AFF + t])) : 0.f;
                        } else {
                            lsum[t] = fmaf(rr2, rr2, lsum[t]);
                            gy[t] = 2.f * c * rr2;
                        }
                    }
                    PM::bwd(pv, f, cx, yh, sv, gy, gp);
#pragma unroll
                    for (int o = 0; o < NOUT; o++) zo[o] = 0.f;   // (now: dz)
#pragma unroll
                    for (int q = 0; q < NPS; q++) {
                        const PSlot sl = a.slot[q];
                        if (sl.role == ROLE_NEURAL) {
                            float gq = gp[q];
                            if (HC::SCALE) gq *= sl.span * sg[q] * (1.f - sg[q]);
#pragma unroll
                            for (int o = 0; o < NOUT; o++)
                                if (sl.idx == o) zo[o] += gq;
                        } else if (sl.role == ROLE_GLOBAL) {
                            gphi[q] += gp[q];
                        }
                    }
#pragma unroll
                    for (int o = 0; o < NOUT; o++) {
                        gB[o] += zo[o];
                        s_dz[o * MAXRT + rt] = zo[o];
                    }
                }
            }
            if (a.mode == ONE_TRAIN && !live && rt < RT) {
#pragma unroll
                for (int o = 0; o < NOUT; o++) s_dz[o * MAXRT + rt] = 0.f;   // padding rows of the last tile
            }
            if (a.mode != ONE_TRAIN && a.evalstat) {
                for (int t = 0; t < nt; t++) {
                    const bool m = live && y[t] == y[t];
                    const double yy = m ? (double)y[t] - a.shift_y[t] : 0.0, hh = m ? (double)yh[t] - a.shift_y[t] : 0.0;
                    const double rr2 = m ? (double)yh[t] - y[t] : 0.0;
                    const double e8[8] = {m ? 1.0 : 0.0, yy, hh, yy * yy, hh * hh, yy * hh, rr2 * rr2, fabs(rr2)};
#pragma unroll
                    for (int k = 0; k < 8; k++) {
                        const double s = warp_sum_d(e8[k]);
                        if (lane == 0) s_e[warp][t * 8 + k] += s;
                    }
                }
            }
        }
        __syncthreads();
        if (a.mode != ONE_TRAIN) continue;
        // ---- backward of my units over my group's rows ----
        const float* dzg = s_dz + grp * ONE_R;
        if constexpr (PX > WIDE_MAXP) {
            one_backward<PX, NOUT, PX, NO>(xs, dzg, wo, A, Gd, gW1, gb, gWo);
        } else {
            if (P <= 2) one_backward<2, NOUT, PX, NO>(xs, dzg, wo, A, Gd, gW1, gb, gWo);
            else if (P <= 4) one_backward<4, NOUT, PX, NO>(xs, dzg, wo, A, Gd, gW1, gb, gWo);
            else one_backward<8, NOUT, PX, NO>(xs, dzg, wo, A, Gd, gW1, gb, gWo);
        }
    }

    if (a.mode != ONE_TRAIN) {
        if (a.evalstat) {
            __syncthreads();
            if (tid < nt * 8) {
                double s = 0.0;
                for (int wv = 0; wv < ONE_THREADS / 32; wv++) s += s_e[wv][tid];
                a.evalstat[(size_t)blockIdx.x * (nt * 8) + tid] = s;
            }
        }
        return;
    }
    // ---- CTA reduction in a fixed order: unit accumulators group by group through shared memory ----
    __syncthreads();   // the record buffers are free
    const int G = (int)blockDim.x / NTg, NQ = NOUT + 1 + P;   // per unit: dWo[o], db1, dW1[p]
    float* s_acc = s_dyn;                                     // [G][NQ][H]
    {
        float* mine = s_acc + (size_t)grp * NQ * H + u0;
#pragma unroll
        for (int o = 0; o < NOUT; o++) { mine[o * H] = gWo[o].x; mine[o * H + 1] = gWo[o].y; }
        mine[NOUT * H] = gb.x;
        mine[NOUT * H + 1] = gb.y;
#pragma unroll
        for (int p = 0; p < PX; p++)
            if (p < P) { mine[(NOUT + 1 + p) * H] = gW1[p].x; mine[(NOUT + 1 + p) * H + 1] = gW1[p].y; }
    }
    // row-thread scalars: dbo, loss sums, phi sums (warp tree, then warps in order)
    {
        float v[16];
#pragma unroll
        for (int q = 0; q < 4; q++) v[q] = q < NOUT ? gB[q < NOUT ? q : 0] : 0.f;
#pragma unroll
        for (int t = 0; t < MAXT; t++) v[4 + t] = lsum[t];
#pragma unroll
        for (int q = 0; q < MAXPS; q++) v[8 + q] = gphi[q];
#pragma unroll
        for (int q = 0; q < 4 + MAXT + MAXPS; q++) {
            const float s = warp_sum(v[q]);
            if (lane == 0) s_red[warp][q] = s;
        }
    }
    __syncthreads();
    float* out = a.partial + (size_t)blockIdx.x * head_npart(H, NOUT);
    float* cs = a.colsum + (size_t)blockIdx.x * (1 + P) * H;
    for (int i = tid; i < NQ * H; i += blockDim.x) {
        float s = 0.f;
        for (int g = 0; g < G; g++) s += s_acc[(size_t)g * NQ * H + i];
        const int q = i / H, u = i - q * H;
        if (q < NOUT) out[i] = s;                              // dWo[o][u]
        else if (q == NOUT) out[head_off_dbh(H, NOUT) + u] = s; // db1[u]
        else cs[(size_t)(q - NOUT) * H + u] = s;                // dW1[u][p] at (1 + p) H + u
    }
    if (tid < 4 + MAXT + MAXPS) {
        float s = 0.f;
        for (int wv = 0; wv < (int)(blockDim.x >> 5); wv++) s += s_red[wv][tid];
        if (tid < 4) out[head_off_dbo(H, NOUT) + tid] = s;
        else out[head_off_loss(H, NOUT) + (tid - 4)] = s;      // loss sums then phi sums are contiguous
    }
}

}  // namespace wide
}  // namespace eh
