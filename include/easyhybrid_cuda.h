/*
 * easyhybrid_cuda.h -- C ABI of libeasyhybrid_cuda.so
 *
 * The drop-in boundary for EasyHybrid.jl's hybrid training step
 * (forward Dense chain -> process model -> masked loss -> analytic backward
 * -> optimiser update), implemented as hand-written sm_100a CUDA.
 *
 * Everything here is plain C: opaque handle, host pointers + sizes, int32/
 * int64/float scalars.  No torch / CUDA types cross the boundary.  A Julia
 * host reaches it with `ccall` (see INTEGRATION.md, julia/EasyHybridCUDA.jl);
 * this repo's tests and bench reach it with `ctypes`.
 *
 * Conventions
 *   - every entry point returns eh_status and never throws/aborts; the text
 *     for the last failure on a ctx is eh_last_error(ctx) (ctx==NULL: the
 *     text of the last failed eh_create on this thread).
 *   - all pointers are HOST pointers owned by the caller; the library copies
 *     during the call and retains nothing (Julia: GC.@preserve for the call).
 *   - index arrays are Julia 1-based int64 and converted inside.
 *   - "flat" parameter vectors use the reference's ComponentArray order
 *     (src/training/initialization.jl:42-44 `ps |> ComponentArray`;
 *      src/models/GenericHybridModel.jl:236-256 initialparameters):
 *       [chain 1: layer_1.weight (out x in, column-major), layer_1.bias, ...,
 *        chain 2: ..., phi_raw[g] for g in global_param_names]
 *   - a ctx is single-owner (not thread-safe); calls are synchronous unless
 *     stated otherwise.
 *   - there is NO CPU fallback: without a usable sm_100 device eh_create
 *     fails with EH_ECUDA.
 *
 * Reference interfaces replaced (paths relative to the EasyHybrid.jl tree):
 *   eh_create        <- constructHybridModel (src/models/GenericHybridModel.jl:89-232)
 *                       + TrainConfig fields   (src/config/TrainingConfig.jl:9-160)
 *                       + init_model_state     (src/training/initialization.jl:17-51)
 *   eh_upload        <- prepare_data output layout (src/data/prepare_data.jl:3-10),
 *                       `|> cfg.gdev` staging  (src/training/train.jl:114-116)
 *   eh_set/get_params<- train_state.parameters (src/training/epoch.jl:29-30)
 *   eh_step          <- Lux.Training.single_train_step! call site
 *                       (src/training/epoch.jl:20-26) on DataLoader batch k
 *   eh_step_host     <- collect_dim_data + `|> cfg.gdev` + single_train_step!
 *                       (src/training/epoch.jl:1-11, 20-26)
 *   eh_loss_grad     <- Zygote.pullback of compute_loss (src/losses/compute_loss.jl:20-35)
 *   eh_epoch         <- run_epoch! (src/training/epoch.jl:13-33)
 *   eh_eval          <- evaluate_acc / evaluate_epoch (src/training/train.jl:347-355,
 *                       src/training/epoch.jl:53-66)
 */
#ifndef EASYHYBRID_CUDA_H
#define EASYHYBRID_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EH_ABI_VERSION 2   /* 2: the weight_l2 fields at the end of eh_model_desc (a version-1 descriptor is still accepted) */

typedef struct eh_ctx eh_ctx; /* opaque; one per training run */

typedef enum {
    EH_OK = 0,
    EH_EINVAL = 1,       /* bad argument / inconsistent descriptor            */
    EH_ENOMEM = 2,       /* host or device allocation failed                  */
    EH_ECUDA = 3,        /* CUDA runtime error or no sm_100 device            */
    EH_ENCCL = 4,        /* NCCL / peer-memory error                          */
    EH_EUNSUPPORTED = 5  /* valid model, but no fused kernel for it (caller   */
                         /* may fall back to the stock Lux path explicitly)   */
} eh_status;

/* activation of the hidden Dense layers (src/models/NNModels.jl:225-230) */
typedef enum {
    EH_ACT_IDENTITY = 0, EH_ACT_TANH = 1, EH_ACT_SIGMOID = 2,
    EH_ACT_RELU = 3, EH_ACT_SWISH = 4
} eh_activation;

/* role of one process-model parameter (GenericHybridModel.jl:127, 377-414) */
typedef enum { EH_ROLE_NEURAL = 0, EH_ROLE_GLOBAL = 1, EH_ROLE_FIXED = 2 } eh_role;

/* per-target loss (src/losses/loss_fn.jl:58-81) */
/* training losses of src/losses/loss_fn.jl:58-179.  The last three (and rmse over more than one target) depend on
 * statistics of the batch's PREDICTIONS (mean, variance, covariance with the observations): on the exact-fp32 kernels
 * their steps run a forward pre-pass over the batch first and take the one-launch-pair-per-step path (no persistent
 * kernel), on the tensor-core path (chains wider than 32) a statistics pass of the head kernel; single GPU on both.   */
typedef enum {
    EH_LOSS_MSE = 0, EH_LOSS_RMSE = 1, EH_LOSS_MAE = 2, EH_LOSS_NSELOSS = 3,
    EH_LOSS_PEARSONLOSS = 4, /* 1 - cor(yhat, y)                                                loss_fn.jl:75-77   */
    EH_LOSS_KGELOSS = 5,     /* sqrt((r-1)^2 + (sigma_s/sigma_o - 1)^2 + (mu_s/mu_o - 1)^2)     loss_fn.jl:104-127 */
    EH_LOSS_PBKGELOSS = 6    /* sqrt((r-1)^2 + (mu_s/mu_o - 1)^2)                               loss_fn.jl:160-174 */
} eh_loss;

/* agg over targets (src/config/TrainingConfig.jl:77; compute_loss.jl:50-53) */
typedef enum { EH_AGG_SUM = 0, EH_AGG_MEAN = 1 } eh_agg;

/* Optimisers.jl rules routed by train (src/training/train.jl:20-22) */
typedef enum { EH_OPT_ADAM = 0, EH_OPT_ADAMW = 1, EH_OPT_RMSPROP = 2, EH_OPT_DESCENT = 3 } eh_opt;

/* built-in process-model forms (SURVEY.md section 8 a9).  Argument binding
 * for each form is given by eh_model_desc.pm_args (see below).            */
typedef enum {
    EH_PM_RBQ10 = 0,    /* y0 = rb * Q10^(0.1*(ta - tref));  args: rb, Q10, ta ; consts: tref */
    EH_PM_EXPO = 1,     /* y0 = Resp0 * exp(k * T);          args: Resp0, k, T               */
    EH_PM_LINEAR = 2,   /* y0 = a * x + b;                   args: a, b, x                   */
    EH_PM_LINEAR2 = 3,  /* y0 = a*x + b ; y1 = 2a*x + b;     args: a, b, x (test_compute_loss.jl:209-211) */
    EH_PM_EXPO2 = 4,    /* y0 = Resp0*exp(k*T) ; y1 = 2*y0;   args: Resp0, k, T (two-target form of the Expo model) */
    EH_PM_PROGRAM = 100 /* traced straight-line program, see eh_pm_instr                      */
} eh_process_model;

/* one argument of a built-in process model: where its value comes from */
typedef struct {
    int32_t kind;  /* 0 = process parameter (index into the parameter table), 1 = forcing column */
    int32_t index;
} eh_pm_arg;

/* Straight-line SSA program for EH_PM_PROGRAM: instruction i defines value i.
 * Produced by tracing the user's `mechanistic_model(; forcings..., params...)`
 * with a symbolic number type on the host side.                             */
typedef enum {
    EH_OP_CONST = 0, EH_OP_FORCING = 1, EH_OP_PARAM = 2,
    EH_OP_ADD = 10, EH_OP_SUB = 11, EH_OP_MUL = 12, EH_OP_DIV = 13, EH_OP_POW = 14,
    EH_OP_MIN = 15, EH_OP_MAX = 16,
    EH_OP_NEG = 20, EH_OP_EXP = 21, EH_OP_LOG = 22, EH_OP_SQRT = 23, EH_OP_TANH = 24,
    EH_OP_SIGMOID = 25, EH_OP_ABS = 26, EH_OP_SIN = 27, EH_OP_COS = 28
} eh_pm_op;

typedef struct {
    int32_t op;   /* eh_pm_op                                   */
    int32_t a, b; /* operand value ids, or column / parameter index for FORCING / PARAM */
    float imm;    /* EH_OP_CONST value                          */
} eh_pm_instr;

/* One Dense chain (prepare_hidden_chain, src/models/NNModels.jl:220-231):
 *   Chain(identity|BatchNorm(affine=false), Dense(in,h1,act), ..., Dense(hk,out))
 * SingleNNHybridModel has one chain with n_out = #neural params;
 * MultiNNHybridModel has one chain per neural param, each with n_out = 1.   */
typedef struct {
    int32_t n_in;             /* predictors feeding this chain                        */
    const int32_t* in_cols;   /* [n_in] indices into the predictor columns of a record */
    int32_t n_hidden;         /* number of hidden layers (>= 1)                        */
    const int32_t* hidden;    /* [n_hidden] widths                                     */
    int32_t n_out;            /* output width                                          */
    int32_t activation;       /* eh_activation of the hidden layers                    */
    int32_t input_batchnorm;  /* 0/1: BatchNorm(n_in, affine=false) in front           */
} eh_chain_desc;

typedef struct {
    int32_t abi_version; /* = EH_ABI_VERSION */

    /* record layout: predictors, forcings, targets (prepare_data.jl:3-10) */
    int32_t n_pred, n_forc, n_targ;

    /* Dense chains */
    int32_t n_chains;
    const eh_chain_desc* chains;

    /* process parameters, ParameterContainer order (helpers_for_HybridModel.jl:95-102) */
    int32_t n_params;
    const int32_t* role;        /* [n_params] eh_role                                     */
    const int32_t* role_index;  /* NEURAL: chain*65536 + output row; GLOBAL: position in   */
                                /* global_param_names (= position in the flat vector tail) */
    const float* deflt;         /* [n_params] */
    const float* lower;         /* [n_params] */
    const float* upper;         /* [n_params] */
    int32_t scale_nn_outputs;   /* GenericHybridModel.jl:394-401 */

    /* process model */
    int32_t process_model;      /* eh_process_model */
    int32_t n_pm_args;
    const eh_pm_arg* pm_args;   /* built-ins: canonical argument order of the form         */
    float pm_consts[4];         /* built-ins: e.g. tref for RBQ10                          */
    const eh_pm_instr* pm_prog; /* EH_PM_PROGRAM */
    int32_t pm_len;
    const int32_t* pm_outputs;  /* [n_targ] value ids of the targets                       */

    /* loss: training_loss (one per target; the same value repeated unless PerTarget) */
    const int32_t* loss_per_target; /* [n_targ] eh_loss */
    int32_t agg;                    /* eh_agg */

    /* optimiser (one rule over the whole flat vector, phi included) */
    int32_t opt_kind;               /* eh_opt */
    float eta, beta1, beta2, eps, lambda; /* rho of RMSProp travels in beta2 */
    int32_t adamw_decay_coupled_eta;  /* 1: theta -= eta*lambda*theta (Optimisers >= 0.4); 0: lambda*theta */

    /* device / data parallel */
    int32_t device;                 /* CUDA device ordinal for this ctx */
    int32_t flags;                  /* EH_FLAG_* */

    /* ---- ABI version 2 ----
     * native extra loss: the reference's documented use of TrainConfig.extra_loss,
     *     extra_loss = (yhat, ps) -> (; l2 = lambda * weight_l2(ps.<branch>; normalize),)
     * (src/utils/extract_weights.jl:55-91, hook: src/losses/compute_loss.jl:31-34), as ONE extra term over the `weight`
     * arrays (not the biases) of the selected chains:  E = lambda * sum(w^2) [/ number of weights],  loss = agg([L, E])
     * with the TrainConfig's agg (sum: L + E; mean: (L + E) / 2).  Steps then take the one-launch-pair-per-step path.  */
    float l2_lambda;                /* 0: no extra loss */
    int32_t l2_normalize;           /* weight_l2(...; normalize = true) */
    uint32_t l2_chain_mask;         /* bit k: chain k takes part; 0 = every chain */
} eh_model_desc;

#define EH_FLAG_NO_GRAPH 1u   /* launch every step individually (debug / profiling) */
#define EH_FLAG_NO_PDL   2u   /* no programmatic dependent launch                   */
#define EH_FLAG_NO_PERSIST 4u /* never use the persistent multi-step kernel         */
#define EH_FLAG_TENSOR_PIPE 16u /* hidden-layer contractions on the tensor pipe (HMMA, 3xTF32 split:
                                  fp32-level accuracy) where a variant exists; default is the exact-fp32
                                  FFMA2 engine */

#define EH_FLAG_JIT 32u       /* traced process model (EH_PM_PROGRAM) on the exact-fp32 path: compile the program into the
                                  kernels at eh_create (NVRTC, a few seconds, cached on disk under $EH_JIT_CACHE or
                                  ~/.cache/easyhybrid_b200) instead of interpreting it per sample.  eh_create fails with
                                  EH_EUNSUPPORTED if NVRTC is not available; models that take another path ignore it.
                                  Shapes without a compiled-in generic variant -- 9..12 chain inputs, 3 or 4 chain outputs
                                  or chains that differ in activation -- are compiled this way WITHOUT the flag (EH_JIT=0 in the
                                  environment forbids it) */

enum { EH_SPLIT_TRAIN = 0, EH_SPLIT_VAL = 1 };

/* number of doubles written per target by eh_eval (sufficient statistics, see DESIGN.md):
 *  n, sum_y, sum_yhat, sum_yy, sum_hh, sum_yh, sse, sae    -- sums are shifted by the
 *  per-split target mean estimate that is written in slot 8 (shift), so callers
 *  compute mse/rmse/mae/r2/nse/pearson/kge from them without cancellation. */
#define EH_EVAL_STATS 9

eh_status eh_create(eh_ctx** out, const eh_model_desc* desc);
void eh_destroy(eh_ctx* ctx);
const char* eh_last_error(const eh_ctx* ctx);

/* number of entries of the flat parameter vector (theta then phi) */
int64_t eh_num_params(const eh_ctx* ctx);

/* Stage one split on the device, once.  X is n_pred x N column-major (each
 * sample's predictors contiguous, Julia Matrix{Float32} P x N), forc/targ are
 * arrays of n_forc / n_targ pointers to N-vectors; NaN target = missing
 * (valid_mask, src/training/train.jl:221-232, is derived on the device).    */
eh_status eh_upload(eh_ctx* ctx, int32_t split, int64_t N, const float* X,
                    const float* const* forc, const float* const* targ);

eh_status eh_set_params(eh_ctx* ctx, const float* flat, int64_t n);
eh_status eh_get_params(eh_ctx* ctx, float* flat, int64_t n);
/* optimiser state: m, v (Adam/AdamW; RMSProp uses v only), step count t */
eh_status eh_set_opt_state(eh_ctx* ctx, const float* m, const float* v, int64_t n, int64_t t);
eh_status eh_get_opt_state(eh_ctx* ctx, float* m, float* v, int64_t n, int64_t* t);
/* input-BatchNorm running statistics of chain c (Lux `st`): mean, var [n_in] */
eh_status eh_set_bn_state(eh_ctx* ctx, int32_t chain, const float* mean, const float* var, int32_t n);
eh_status eh_get_bn_state(eh_ctx* ctx, int32_t chain, float* mean, float* var, int32_t n);

/* loss and gradient of the training objective on batch idx1 of the TRAIN split,
 * no update (parity hook; grad_out has eh_num_params entries, may be NULL)   */
eh_status eh_loss_grad(eh_ctx* ctx, const int64_t* idx1, int64_t B, float* loss_out, float* grad_out);

/* one optimiser step on batch idx1 (1-based indices into the TRAIN split).
 * An all-masked batch is skipped (src/training/epoch.jl:17-19): *loss_out = NaN,
 * parameters and step count unchanged.                                       */
eh_status eh_step(eh_ctx* ctx, const int64_t* idx1, int64_t B, float* loss_out, float* grad_out);

/* same, on a batch handed over as host arrays laid out like eh_upload's
 * (collect_dim_data |> gdev, src/training/epoch.jl:1-11); the H2D copy is
 * part of the call.                                                          */
eh_status eh_step_host(eh_ctx* ctx, int64_t B, const float* X, const float* const* forc,
                       const float* const* targ, float* loss_out);

/* Pipelined form of eh_step_host for streaming callers: enqueue the transfer
 * and the step asynchronously and return; *loss_slot is filled by eh_sync,
 * which waits for everything enqueued so far.  Page-locked arrays
 * (eh_host_alloc, cudaHostAlloc / cudaHostRegister, CUDA.pin) are read IN
 * PLACE over PCIe by a packer kernel -- no staging copy -- and the steps of up
 * to 16 consecutive batches of equal size run inside one persistent launch
 * (issued when the group is full, at eh_sync, or by any other entry point of
 * this ctx); pageable arrays are staged through the copy engine, one launch
 * pair per batch.  Either way the arrays must stay valid and unchanged until
 * eh_sync returns (the rule cudaMemcpyAsync imposes).  Steps are applied in
 * call order.                                                                */
eh_status eh_step_host_async(eh_ctx* ctx, int64_t B, const float* X, const float* const* forc,
                             const float* const* targ, float* loss_slot);
eh_status eh_sync(eh_ctx* ctx);

/* run_epoch!: batches k = perm1[(k-1)B+1 : min(kB,n)] in order, one step each,
 * last batch partial; losses (nullable) receives ceil(n/B) per-step losses.  */
eh_status eh_epoch(eh_ctx* ctx, const int64_t* perm1, int64_t n, int64_t B, float* losses);

/* same, with the index stream already resident (set once with eh_set_perm):
 * runs steps [first_step, first_step + n_steps); step s trains on batch
 * s mod ceil(n/B), i.e. steps past one pass start another pass over the same
 * permutation.  Whole passes are replayed as one CUDA graph.                 */
eh_status eh_set_perm(eh_ctx* ctx, const int64_t* perm1, int64_t n);
eh_status eh_run_steps(eh_ctx* ctx, int64_t B, int64_t first_step, int64_t n_steps, float* losses);

/* test-mode forward on a whole split (evaluate_acc): yhat (nullable) is
 * n_targ x N row-major-by-target (target t at yhat + t*N); stats (nullable) is
 * n_targ x EH_EVAL_STATS doubles.  nn_out (nullable) is n_params x N: the
 * scaled per-sample value of every NEURAL parameter (rows of other roles are
 * left untouched) -- the `parameters` entry of the reference forward output. */
eh_status eh_eval(eh_ctx* ctx, int32_t split, float* yhat, double* stats, float* nn_out);

/* ---- data parallel (one process per GPU of one NVLink / NVSwitch box) --------
 * Every rank owns a shard of the samples (its own eh_upload + eh_set_perm); global
 * batch k is the union of the ranks' local batches k, which must have the same
 * size on every rank (see eh_dp_batch_moments for losses that need batch statistics).  Per step the ranks exchange ONE vector (loss-scaled
 * gradient + loss sums) inside the persistent kernel: rank r's CTA 0 stores it
 * into every peer's inbox through NVLink peer memory and raises a flag, all CTAs
 * sum the rank vectors in rank order and apply the optimiser redundantly, so
 * parameters and optimiser state stay replicated bit-identically.  No NCCL.
 * Setup: each rank calls eh_comm_id on its ctx (allocates the inbox, returns an
 * EH_COMM_ID_BYTES blob = a CUDA IPC handle), the caller all-gathers the blobs
 * with its own plumbing (torch.distributed / MPI / files) and hands all of them
 * (rank order) to eh_comm_init.  world <= 8.  In data-parallel mode only
 * eh_run_steps / eh_epoch train; configurations that need per-batch data
 * statistics (NaN targets, nseLoss, input BatchNorm) answer EH_EUNSUPPORTED.   */
#define EH_COMM_ID_BYTES 128
eh_status eh_comm_id(eh_ctx* ctx, void* id_out);
eh_status eh_comm_init(eh_ctx* ctx, int32_t rank, int32_t world, const void* ids /* world x EH_COMM_ID_BYTES */);

/* Data-parallel runs whose loss needs per-batch DATA statistics (valid-target counts with NaN targets, SS_tot of
 * nseLoss, batch moments of the input BatchNorm): those are statistics of the GLOBAL batch.  After eh_set_perm every
 * rank calls eh_dp_batch_moments (raw sums of its local batches, EH_DP_MOMENTS doubles per batch, taken with the
 * same zero shift on every rank), the caller adds the arrays over the ranks with its own plumbing (the same one that
 * carried the comm ids) and hands the sums to eh_dp_set_batch_moments on every rank; eh_run_steps then trains with
 * them.  NaN-free mse / mae / rmse runs without BatchNorm do not need this.                                      */
#define EH_DP_MOMENTS 37
eh_status eh_dp_batch_moments(eh_ctx* ctx, int64_t B, double* out /* [ceil(n/B)][EH_DP_MOMENTS] */);
eh_status eh_dp_set_batch_moments(eh_ctx* ctx, int64_t B, const double* summed /* same shape */);

/* page-locked host buffers for callers that stream batches (eh_step_host_async reads them in
 * place over PCIe; pageable memory also works, through the copy engine and synchronously) */
eh_status eh_host_alloc(void** out, size_t bytes);
eh_status eh_host_free(void* p);

/* timing hook: device time in ms of the last eh_epoch / eh_run_steps call,
 * measured with CUDA events on the stream the kernels ran on; kernel launches
 * made by that call; and the accumulated device time of the fused step kernel
 * alone when profiling is enabled with eh_set_profiling(ctx, 1).             */
eh_status eh_last_timing(eh_ctx* ctx, float* total_ms, int64_t* launches, float* step_kernel_ms);
eh_status eh_set_profiling(eh_ctx* ctx, int32_t on);

/* which compiled kernel family serves this ctx (static string, never NULL), e.g.
 * "ffma2/PmRbQ10/P2/NH2/H16/O1/ACT_TANH/scale=true" (exact-fp32 register-tile kernels, specialised form),
 * "ffma2/PmProgram/..." (same kernels, process model interpreted per sample) or "wide/bf16-tcgen05".
 * The reference has no counterpart; callers use it to report / assert the path a model took.          */
const char* eh_kernel_variant(const eh_ctx* ctx);
/* Plans `desc` as eh_create would and compiles its traced process model with NVRTC (EH_FLAG_JIT implied) WITHOUT touching a
 * device: EH_OK and a one-line description ("nvrtc/PmTraced#<hash>/... cubin=<bytes> cached=<0|1> seconds=<s>") in `info`,
 * or the planner's / compiler's error through eh_last_error(NULL).  For build checks and for warming the disk cache.
 * The reference has no counterpart (Julia compiles the user's closure itself, GenericHybridModel.jl:425). */
eh_status eh_jit_check(const eh_model_desc* desc, char* info, size_t info_bytes);
/* ... and the family that serves the PERSISTENT launches (eh_epoch / eh_run_steps) at batch size `batch`: the same as above,
 * or "tcgen05/..." where the tensor engine (hidden-layer products on tcgen05 with TMEM operands) takes large batches.     */
const char* eh_epoch_variant(const eh_ctx* ctx, int64_t batch);

/* diagnostics: runs one tcgen05 GEMM of the wide-hidden-layer path on host matrices (bf16 bit patterns) so that a
 * test harness can check the kernels in isolation.  mode 0: out = act(A B^T + bias), A [M x K], B [N x K];
 * mode 1: out = (A B^T) .* act'(aux), aux [M x N]; both write bf16 [M x N].  modes 3 / 4: the persistent forms of 0 / 1.  mode 2: out[z] = A_z^T B_z for the
 * `ksplits` row slices of A [K x M], B [K x N]; writes fp32 [ksplits][M x N].  ms_out (nullable): device time.  */
eh_status eh_selftest_wide_gemm(int32_t mode, int32_t M, int32_t N, int32_t K, int32_t ksplits, int32_t act,
                                const uint16_t* A, const uint16_t* B, const float* bias, const uint16_t* aux,
                                void* out, int32_t device, float* ms_out);

#ifdef __cplusplus
}
#endif
#endif /* EASYHYBRID_CUDA_H */
