// eh_eval_kernel.cuh -- K5: test-mode forward over a whole split with on-device
// sufficient statistics for every loss type of src/losses/loss_fn.jl:58-179.
// Replaces evaluate_acc (src/training/train.jl:347-355) as used by evaluate_epoch
// (src/training/epoch.jl:53-66): forward + all loss_types on train and val per epoch.
// This kernel is HBM-streaming: 4(P+F+T) bytes read and 4 T (+ 4 per NEURAL slot)
// written per sample when predictions are requested, nothing written otherwise.
#pragma once
#include "eh_step_kernel.cuh"
#include "eh_stat_seeds.cuh"

namespace eh {

struct EvalArgs {
    const float4* rec;
    const int* idx;        // optional: sample i of the pass is record idx[i] (training batches); NULL: rec_base + i
    long long rec_base;
    long long N;
    const float* pblock;
    int nflat;
    const int* wsrc;
    const float* bscal;    // test-mode BN row (running mean / rstd) or NULL
    int use_bn;
    PSlot slot[MAXPS];
    float pmc[4];
    float shift_y[MAXT];
    float* yhat;           // nullable [T][N]
    float* parout;         // nullable [NPS][N] (NEURAL slots only)
    double* partial;       // [gridDim.x][T * EVAL_NSTAT]
    const PmProgData* prog;   // traced process model (PmProgram variants), device memory
    int scale_rt;             // PmProgram variants: scale_nn_outputs
    unsigned pass_mask[3];    // PmProgram variants: pass-through units per hidden layer (PmCtx::pass)
};

template <class C>
__global__ void __launch_bounds__(256) k_eval(const EvalArgs a)
{
    constexpr int P = C::P, NOUT = C::NOUT, T = C::T, F = C::F, NPS = C::NPS, HP = C::H / 2;
    using PM = typename C::PM;
    extern __shared__ float4 smem4[];
    float* sW = reinterpret_cast<float*>(smem4);
    float* sS = sW + rup4(C::NW);
    __shared__ double shd[8][MAXT * EVAL_NSTAT];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;

    load_weights_and_scalars<C>(a.pblock, a.nflat, a.wsrc, a.bscal, a.use_bn, sW, sS);
    __syncthreads();
    PmCtx cx;
    cx.pms = sS + SS_PMS;
    cx.c = a.pmc;
    cx.prog = a.prog;
    cx.scale_rt = a.scale_rt;
    for (int l = 0; l < 3; l++) cx.pass[l] = a.pass_mask[l];
    cx.uniform_mask = 0;
    cx.phi_flag = nullptr;
    cx.phi_want = 0;
#pragma unroll
    for (int s = 0; s < MAXPS; s++)
        if (s >= NPS || a.slot[s].role != ROLE_NEURAL) cx.uniform_mask |= 1u << s;

    double st[T][EVAL_NSTAT];
#pragma unroll
    for (int t = 0; t < T; t++)
#pragma unroll
        for (int q = 0; q < EVAL_NSTAT; q++) st[t][q] = 0.0;

    const long long nchunks = (a.N + CHUNK - 1) / CHUNK;
    for (long long chunk = (long long)blockIdx.x * nwarps + warp; chunk < nchunks; chunk += (long long)gridDim.x * nwarps) {
        const long long s0 = chunk * CHUNK + lane;
        const bool v0 = s0 < a.N;
        float4 r[C::R4 / 4];
#pragma unroll
        for (int q = 0; q < C::R4 / 4; q++)
            r[q] = v0 ? __ldg(a.rec + (a.idx ? (long long)a.idx[s0] : a.rec_base + s0) * (C::R4 / 4) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
        const float* p0 = reinterpret_cast<const float*>(r);
        float x[P], f[F > 0 ? F : 1], y[T];
#pragma unroll
        for (int k = 0; k < P; k++) x[k] = (p0[k] - sS[SS_BN + 2 * k]) * sS[SS_BN + 2 * k + 1];
#pragma unroll
        for (int k = 0; k < F; k++) f[k] = p0[P + k];
#pragma unroll
        for (int k = 0; k < T; k++) y[k] = p0[P + F + k];

        float2 hp[HP];
        float zo[NOUT], pv[NPS], sg[NPS], yh[T], sv[PM::NSV];
        chain_forward<C, false>(sW, nullptr, lane, x, hp, zo, cx.pass);
        resolve_params<C>(a.slot, sS, zo, pv, sg, cx);
        PM::fwd(pv, f, cx, yh, sv);

#pragma unroll
        for (int t = 0; t < T; t++) {
            if (a.yhat && v0) a.yhat[(size_t)t * a.N + s0] = yh[t];   // consecutive lanes: coalesced
            if (v0 && y[t] == y[t]) {
                const double sh = a.shift_y[t];
                double dy = (double)y[t] - sh, dh = (double)yh[t] - sh, rr = (double)yh[t] - (double)y[t];
                st[t][0] += 1.0; st[t][1] += dy; st[t][2] += dh;
                st[t][3] += dy * dy; st[t][4] += dh * dh; st[t][5] += dy * dh;
                st[t][6] += rr * rr; st[t][7] += fabs(rr);
            }
        }
        if (a.parout && v0) {
#pragma unroll
            for (int s = 0; s < NPS; s++)
                if (a.slot[s].role == ROLE_NEURAL) a.parout[(size_t)s * a.N + s0] = pv[s];
        }
    }
#pragma unroll
    for (int t = 0; t < T; t++)
#pragma unroll
        for (int q = 0; q < EVAL_NSTAT; q++) {
            double v = warp_sum_d(st[t][q]);
            if (lane == 0) shd[warp][t * EVAL_NSTAT + q] = v;
        }
    __syncthreads();
    if (threadIdx.x < T * EVAL_NSTAT) {
        double s = 0.0;
        for (int w = 0; w < nwarps; w++) s += shd[w][threadIdx.x];
        a.partial[(size_t)blockIdx.x * (T * EVAL_NSTAT) + threadIdx.x] = s;
    }
}

}  // namespace eh
