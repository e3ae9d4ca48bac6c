// eh_stat_seeds.cuh -- seeds of the prediction-statistics losses from per-CTA sufficient statistics of a batch.
// Shared by the exact-fp32 path (pre-pass k_eval over the batch, eh_lib.cu) and the tensor-core path (statistics pass of
// k_wide_head over the last hidden activation, eh_wide.cu): one implementation of the seed formulas.
#pragma once
#include "eh_chunk.cuh"

namespace eh {

constexpr int EVAL_NSTAT = 8;  // n, Sy, Sh, Syy, Shh, Syh, SSE, SAE  (y, yhat shifted by shift_y)

// ---- seeds of the prediction-statistics losses ----
// rmse over several targets, pearsonLoss, kgeLoss, pbkgeLoss (loss_fn.jl:58-60, 75-77, 104-127, 160-174) are functions of
// n, sum yhat, sum yhat^2, sum y yhat and the data statistics of the batch -- exactly what k_eval (and the statistics mode
// of k_wide_head) leave in their partials.
// One thread per target sums the partials in a fixed order, evaluates the loss and the coefficients of its seeds
//   dL/dyhat_i = sa + sb yhat_i + sc y_i        (times the aggregation weight)
// and writes them into the batch's scalar row (BS_AFF..), where the step kernel (LOSS_AFFINE) and k_update pick them up.
struct StatSeedArgs {
    const double* partial;   // [nparts][Tk * EVAL_NSTAT] as written by k_eval over the batch
    int nparts, Tk;          // Tk = targets of the compiled variant (row length of the partials)
    int T;                   // targets of the model
    int kind[MAXT];          // ABI loss kind per target (LOSS_RMSE, LOSS_PEARSONLOSS, ...); other kinds are left alone
    float shift_y[MAXT];
    int agg_mean;
    float* bscal;            // the batch's scalar row
};
static __global__ void k_stat_seeds(const StatSeedArgs a)
{
    const int t = threadIdx.x;
    if (t >= a.T) return;
    const int k = a.kind[t];
    if (!(k == LOSS_RMSE || k == LOSS_PEARSONLOSS || k == LOSS_KGELOSS || k == LOSS_PBKGELOSS)) return;
    double s[EVAL_NSTAT];
    for (int q = 0; q < EVAL_NSTAT; q++) {
        double v = 0.0;
        for (int g = 0; g < a.nparts; g++) v += a.partial[(size_t)g * a.Tk * EVAL_NSTAT + t * EVAL_NSTAT + q];
        s[q] = v;
    }
    const double n = s[0], Sy = s[1], Sh = s[2], Syy = s[3], Shh = s[4], Syh = s[5], sse = s[6];
    const double aggw = a.agg_mean ? 1.0 / a.T : 1.0, sh = (double)a.shift_y[t];
    double sa = 0.0, sb = 0.0, sc = 0.0, L = 0.0;
    if (n > 0) {
        if (k == LOSS_RMSE) {
            L = sqrt(sse / n);
            sb = 1.0 / (n * L);
            sc = -sb;
        } else {
            const double mu_s = sh + Sh / n, mu_o = sh + Sy / n;
            const double Qs = Shh - Sh * Sh / n, Qo = Syy - Sy * Sy / n, Qso = Syh - Sh * Sy / n;
            const double D = sqrt(Qs * Qo), r = Qso / D, alpha = sqrt(Qs / Qo), beta = mu_s / mu_o;
            // d r / d yhat_i = (y_i - mu_o) / D - r (yhat_i - mu_s) / Qs;  d alpha = (yhat_i - mu_s) / D;  d beta = 1 / (n mu_o)
            const double r0 = -mu_o / D + r * mu_s / Qs, rh = -r / Qs, ry = 1.0 / D;
            const double a0 = -mu_s / D, ah = 1.0 / D, b0 = 1.0 / (n * mu_o);
            if (k == LOSS_PEARSONLOSS) {
                L = 1.0 - r;
                sa = -r0; sb = -rh; sc = -ry;
            } else {
                const bool kge = k == LOSS_KGELOSS;
                const double K = sqrt((r - 1) * (r - 1) + (kge ? (alpha - 1) * (alpha - 1) : 0.0) + (beta - 1) * (beta - 1));
                L = K;
                sa = ((r - 1) * r0 + (kge ? (alpha - 1) * a0 : 0.0) + (beta - 1) * b0) / K;
                sb = ((r - 1) * rh + (kge ? (alpha - 1) * ah : 0.0)) / K;
                sc = ((r - 1) * ry) / K;
            }
        }
    }
    a.bscal[BS_AFF + t] = (float)(sa * aggw);
    a.bscal[BS_AFF + MAXT + t] = (float)(sb * aggw);
    a.bscal[BS_AFF + 2 * MAXT + t] = (float)(sc * aggw);
    a.bscal[BS_AFF + 3 * MAXT + t] = (float)L;
}

}  // namespace eh
