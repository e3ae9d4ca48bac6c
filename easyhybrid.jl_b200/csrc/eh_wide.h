// eh_wide.h -- host interface of the wide-hidden-layer (bf16 tcgen05) path, shared by eh_wide.cu and eh_lib.cu
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace eh {
namespace wide {

bool make_map_bf16(CUtensorMap* map, const void* ptr, uint64_t inner, uint64_t rows, uint64_t pitch_elems, uint32_t box_rows);
cudaError_t gemm_prepare();
cudaError_t gemm_fwd(const CUtensorMap& tmA, const CUtensorMap& tmW, int M, int N, int K, const float* bias, int act,
                     __nv_bfloat16* out, cudaStream_t st);
cudaError_t gemm_bwd(const CUtensorMap& tmD, const CUtensorMap& tmWt, int M, int N, int K, const __nv_bfloat16* aux, int act,
                     __nv_bfloat16* out, cudaStream_t st, float* colsum, const float* xb, const float* bscal, int R4, int P1,
                     int use_bn);
cudaError_t gemm_wgrad(const CUtensorMap& tmD, const CUtensorMap& tmA, int M, int N, int Kall, int ksplits, float* partial,
                       cudaStream_t st);

// where a flat parameter lives in the images of the embedded chain (== the WK_* enum of eh_wide_kernels.cuh)
enum : int { WK_W1 = 0, WK_WH = 1, WK_B = 2, WK_WO = 3, WK_BO = 4, WK_PHI = 5 };

struct WideDp {             // data-parallel state handed to WideNet::step
    int world, rank;
    float* peer[8];         // exchange blocks of all ranks as mapped in this process (own block at [rank])
    unsigned tag;           // absolute step tag (grows by one per exchanged step, never reused)
    unsigned* err;          // device flag raised when a peer never arrived
};

struct PSlotH { int role, idx; float lo, span, fixedv; };   // == eh::PSlot (kept POD here: this header is host-only)

struct WideModel {          // filled by eh_lib's planner from the model descriptor
    int P, H, NH, NOUT, R4, nflat, ntheta;   // embedded chain: total inputs, padded hidden width (256 / 512), ...
    const int* h_map;                        // [nflat][4] host: {kind, layer, image row, image column} per flat entry
    int n_blocks;                            // hidden weight blocks (one per chain and hidden layer l >= 2)
    struct { int l, flat_off, hout, hin, o_off, i_off; } blocks[32];
    int act, scale, pm, T, F, NPS, use_bn, agg_mean;
    int loss_kind[4];                        // LOSS_AFFINE for the prediction-statistics losses (seeds from a statistics pass)
    int loss_kind_abi[4];                    // the descriptor's loss kind per target (what k_stat_seeds evaluates)
    PSlotH slot[8];
    float pmc[4];
    int opt_kind, adamw_coupled;
    float eta, beta1, beta2, eps, lambda;
    const int* d_slot_of_flat;
    // native extra loss lambda * weight_l2 (d_l2coef NULL: none): loss l2_aggw (L + l2_loss_coef sum theta^2 over the flagged
    // entries), gradient l2_aggw (g + l2coef[p] theta[p])
    const float* d_l2coef;
    float l2_aggw, l2_loss_coef;
    int nsm;
    // traced process model (pm == PM_PROGRAM): eh_pm_instr fields, value ids of the targets
    int prog_len;
    short prog_op[48], prog_a[48], prog_b[48];
    float prog_imm[48];
    int prog_out[4];
};

// the wide-chain training step: owns activations / deltas / bf16 weight images / partial buffers
class WideNet {
public:
    // hmax: widest embedded hidden layer (padded up to 256 or 512 inside)
    static bool supported(int P, int hmax, int NH, int NOUT, int act, int pm);
    static int padded_width(int hmax) { return hmax <= 256 ? 256 : 512; }
    static WideNet* create(const WideModel& m, char* err, size_t errlen);
    ~WideNet();
    // any batch size: rows are padded up to a multiple of 128 inside and masked
    static bool batch_ok(long long B) { return B > 0 && B < (1ll << 30); }
    // bf16 weight images from the fp32 master parameters (after eh_set_params)
    cudaError_t refresh_images(float* pblock, float* m, float* v, void* ost, cudaStream_t st);
    // one optimiser step (apply = 1) or loss + gradient only (apply = 0) on `B` samples rec[idx[.]];
    // grad: [nflat] device buffer receiving dL/dflat; loss_out: device (or pinned host) float.  bscal: the batch's scalar
    // row (device); the statistics pass of the LOSS_AFFINE targets writes their seed coefficients into it.  shift_y: the
    // train split's target shifts (read for LOSS_AFFINE targets only)
    cudaError_t step(const float* rec, const int* idx, long long rec_base, int B, float* bscal, float* pblock, float* m,
                     float* v, void* ost, float* grad, float* loss_out, int apply, cudaStream_t st, const WideDp* dp = nullptr,
                     const float* shift_y = nullptr);
    // launches step() adds to the base sequence: statistics pass + seeds (LOSS_AFFINE targets), gradient epilogue
    // (single-target rmse, weight_l2)
    int extra_launches() const { return (affine_ ? 2 : 0) + (post_ ? 1 : 0); }
    // bytes of the exchange block a rank exposes in data-parallel mode: [2][xlen] floats + flags
    size_t dp_block_bytes() const { return (size_t)2 * dp_xlen() * sizeof(float) + 256; }
    int dp_xlen() const { return (m_.nflat + 16 + 31) / 32 * 32; }
    // test-mode forward of rows [row0, row0 + B) of a split: yhat / parout nullable device buffers with leading
    // dimension ldy; evalstat_dev: [T * 8] doubles, ACCUMULATED into (caller zeroes)
    cudaError_t eval_rows(const float* rec, long long nrec, long long row0, int Bvalid, const float* bscal, const float* pblock,
                          float* yhat, float* parout, long long ldy, double* evalstat_dev, const float* shift_y, cudaStream_t st);
    const char* error() const { return err_; }
    int eval_chunk() const { return 16384; }

private:
    WideNet() {}
    cudaError_t ensure(int B);
    cudaError_t forward(const float* rec, const int* idx, long long rec_base, long long nrec, int B, int Bvalid,
                        const float* bscal, const float* pblock, cudaStream_t st);
    WideModel m_{};
    int cap_ = 0, mapB_ = 0, n_head_ = 0, n_slab_ = 0, ksplit_ = 1;
    bool persist_ = true;
    bool affine_ = false;      // some target is LOSS_AFFINE: statistics pass of the head kernel + k_stat_seeds per step
    bool post_ = false;        // single-target rmse or weight_l2: k_wide_gradpost finishes the flat gradient
    float* xb_ = nullptr;
    __nv_bfloat16* A_[8] = {nullptr};
    __nv_bfloat16* D_[2] = {nullptr, nullptr};
    __nv_bfloat16* Wf_[8] = {nullptr};
    __nv_bfloat16* Wb_[8] = {nullptr};
    float* Bp_[8] = {nullptr};
    float* W1img_ = nullptr;
    float* WOimg_ = nullptr;
    float* BOimg_ = nullptr;
    void* d_map_ = nullptr;    // ParamMap[nflat]
    int* d_small_ = nullptr;   // flat indices assembled by k_wide_gradfin
    int n_small_ = 0;
    void* d_prog_ = nullptr;   // PmProgData on the device
    float* partial_ = nullptr;
    // the split-K reductions (latency-bound, a few CTAs) run on a side stream next to the backward-data GEMM of their layer
    cudaStream_t side_ = nullptr;
    cudaEvent_t ev_wgrad_ = nullptr, ev_wred_ = nullptr;
    float* colsum_[8] = {nullptr};
    float* head_partial_ = nullptr;
    float* stats_ = nullptr;
    double* evalpart_ = nullptr;
    float* l2part_ = nullptr;      // [gradpost CTAs] partial sums of theta^2 over the weight_l2 entries
    unsigned* ticket_ = nullptr;   // CTAs of k_wide_gradpost that have finished (the last one writes the loss)
    int* skip_ = nullptr;
    CUtensorMap tmA_k_[8], tmA_mn_[8], tmD_k_[2], tmD_mn_[2], tmWf_[8], tmWb_[8];
    char err_[256] = {0};
};

}  // namespace wide
}  // namespace eh
