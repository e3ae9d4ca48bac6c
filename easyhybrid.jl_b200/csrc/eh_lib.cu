// eh_lib.cu -- C ABI of libeasyhybrid_cuda.so (see include/easyhybrid_cuda.h).
//
// Host-side runtime of the fused training path: descriptor -> kernel variant +
// layout tables, device-resident datasets (packed once), per-epoch index stream,
// step launch sequence (K1 fused step, K2 reduce+update, chained with programmatic
// dependent launch), evaluation, timing hooks.  No PyTorch, no CPU fallback.
#include "eh_ctx.h"
#include "eh_update_kernel.cuh"

namespace eh {
namespace rt {
thread_local std::string g_create_error;
eh_status fail(eh_ctx* c, eh_status s, const char* fmt, ...)
{
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (c) c->err = buf;
    else g_create_error = buf;
    return s;
}
void set_create_error(const std::string& s) { g_create_error = s; }
}  // namespace rt
}  // namespace eh

namespace {

template <class T>
cudaError_t dalloc(T** p, size_t n)
{
    return cudaMalloc((void**)p, std::max<size_t>(n, 1) * sizeof(T));
}

// n_valid-independent per-batch rows when no data statistics are needed:
// c_t = agg_w / B_k, n_t = B_k (no NaN targets anywhere in the split)
__global__ void k_fill_bscal(float* bscal, int nb, long long n, int Bfull, int T, int agg_mean, int world)
{
    int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nb) return;
    long long rem = n - (long long)b * Bfull;
    float bk = (float)(rem < Bfull ? rem : Bfull) * (float)world;  // data parallel: the global batch
    float* o = bscal + (size_t)b * BS_STRIDE;
    float aggw = agg_mean ? 1.f / (float)T : 1.f;
    for (int t = 0; t < MAXT; t++) {
        o[BS_C + t] = t < T ? aggw / bk : 0.f;
        o[BS_N + t] = t < T ? bk : 0.f;
        o[BS_SS + t] = 0.f;
    }
    for (int k = 0; k < MAXP; k++) { o[BS_BN + 2 * k] = 0.f; o[BS_BN + 2 * k + 1] = 1.f; }
}

// host-step path: c_t from the valid-target counts produced by the packer
// (also re-zeroes the counters for the next batch that uses this staging slot)
__global__ void k_bscal_from_counts(float* bscal, int* cnt, int T, int agg_mean)
{
    int t = threadIdx.x;
    if (t >= MAXT) return;
    float aggw = agg_mean ? 1.f / (float)T : 1.f;
    float n = t < T ? (float)cnt[t] : 0.f;
    cnt[t] = 0;
    bscal[BS_C + t] = t < T ? aggw / n : 0.f;
    bscal[BS_N + t] = n;
    bscal[BS_SS + t] = 0.f;
    if (t == 0)
        for (int k = 0; k < MAXP; k++) { bscal[BS_BN + 2 * k] = 0.f; bscal[BS_BN + 2 * k + 1] = 1.f; }
}

// packer variant that also counts valid targets (integer atomics: deterministic)
__global__ void __launch_bounds__(256) k_pack_count(const PackArgs a, int T, int ycol0, int* cnt)
{
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    int valid[MAXT] = {0, 0, 0, 0};
    if (i < a.N) {
        float* r = a.rec + (a.rec_base + i) * a.R4;
        for (int c = 0; c < a.R4; c++) {
            float v = 0.f;
            if (c < a.ncols) v = pack_load(a, c, i);
            r[c] = v;
            int t = c - ycol0;
            if (t >= 0 && t < T && v == v) valid[t] = 1;
        }
    }
    for (int t = 0; t < T; t++) {
        unsigned m = __ballot_sync(0xffffffffu, valid[t]);
        if ((threadIdx.x & 31) == 0 && m) atomicAdd(&cnt[t], __popc(m));
    }
}

// Zero-copy packer of the host-batch path: the caller's page-locked arrays are read straight over PCIe
// (UVA device pointers of pinned host memory) and leave as packed records in HBM -- one launch on the copy
// stream replaces the three cudaMemcpyAsync + the packer + the per-batch-scalar kernel.  Packers rotate
// over EH_NPACK streams (the ramp-up / drain of one overlaps the others: 37 GB/s with one stream, 44 with two,
// 49 with four, measured on 1 MiB batches; a 256 MiB cudaMemcpy reaches 55 GB/s on the same box, 1 MiB ones
// 33 GB/s) and together are kept to EH_PACK_HOST_CTAS
// big CTAs, so that they only ever occupy that many SMs next to a running step / persistent kernel
// (step_geometry and the 128-CTA persistent grid leave them free); measured insensitive to the grid between
// 16 x 1024 and 296 x 256 threads.  The last CTA to finish (ticket) turns the valid-target counts into the
// batch's scalar row, like k_bscal_from_counts.
constexpr int EH_PACK_HOST_CTAS = 16;
constexpr int EH_PACK_MAXPLANES = 24;
struct PackHostArgs {
    const float* X;                         // [N][P_raw], host memory mapped into the device address space
    const float* plane[EH_PACK_MAXPLANES];  // forcings then targets, each [N], mapped host memory
    long long N;
    int P_raw, ncols, R4;
    int x_pair;                             // columns 0,1 of a record are X[2i], X[2i+1] (one 8-byte load)
    int src_kind[24], src_idx[24];
    float* rec;                             // [N][R4] device
    int T, ycol0, agg_mean;
    int world;                              // data parallel: the scalar row describes the GLOBAL batch of world * N rows
                                            // (NaN-free targets are a precondition of host batches in that mode)
    int* cnt;                               // [MAXT + 1] valid-target counters + ticket (all zero between launches)
    float* bscal;                           // per-batch scalar row to fill (NULL: K0 computes it from the records)
    // consumer mode (the persistent kernel of a burst is already running, eh_epoch_kernel.cuh): the slot may only be
    // overwritten once the step that last trained on it has retired (*wait_done >= wait_min), and the kernel picks the
    // batch up as soon as *ready == ready_val
    const unsigned* wait_done;
    unsigned wait_min;
    unsigned* ready;
    unsigned ready_val;
};

__device__ __forceinline__ float pack_host_load(const PackHostArgs& a, int c, long long i)
{
    if (c >= a.ncols) return 0.f;
    const int k = a.src_kind[c];
    if (k >= 2) return k == 2 ? 0.f : __int_as_float(0x7fc00000);   // padding columns of the generic variants: zero / NaN
    return k == 0 ? __ldg(a.X + i * a.P_raw + a.src_idx[c]) : __ldg(a.plane[a.src_idx[c]] + i);
}

__global__ void __launch_bounds__(1024) k_pack_host(const PackHostArgs a)
{
    if (a.wait_done) {
        if (threadIdx.x == 0)
            while ((int)(*reinterpret_cast<const volatile unsigned*>(a.wait_done) - a.wait_min) < 0) {}
        __syncthreads();
    }
    int valid[MAXT] = {0, 0, 0, 0};
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long first = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (a.R4 == 4) {
        // two samples per thread and trip: eight independent loads in flight before the first store
        for (long long i = first; i < a.N; i += 2 * stride) {
            const long long j = i + stride;
            const bool two = j < a.N;
            float r0[4], r1[4] = {0.f, 0.f, 0.f, 0.f};
            int c0 = 0;
            if (a.x_pair) {
                const float2 x0 = __ldg(reinterpret_cast<const float2*>(a.X) + i);
                r0[0] = x0.x; r0[1] = x0.y;
                if (two) { const float2 x1 = __ldg(reinterpret_cast<const float2*>(a.X) + j); r1[0] = x1.x; r1[1] = x1.y; }
                c0 = 2;
            }
#pragma unroll
            for (int c = 0; c < 4; c++)
                if (c >= c0) {
                    r0[c] = pack_host_load(a, c, i);
                    if (two) r1[c] = pack_host_load(a, c, j);
                }
            reinterpret_cast<float4*>(a.rec)[i] = make_float4(r0[0], r0[1], r0[2], r0[3]);
            if (two) reinterpret_cast<float4*>(a.rec)[j] = make_float4(r1[0], r1[1], r1[2], r1[3]);
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const int t = c - a.ycol0;
                if (t >= 0 && t < a.T) {
                    if (r0[c] == r0[c]) valid[t]++;
                    if (two && r1[c] == r1[c]) valid[t]++;
                }
            }
        }
    } else {
        for (long long i = first; i < a.N; i += stride) {
            float* r = a.rec + i * a.R4;
            for (int c = 0; c < a.R4; c++) {
                const float v = pack_host_load(a, c, i);
                r[c] = v;
                const int t = c - a.ycol0;
                if (t >= 0 && t < a.T && v == v) valid[t]++;
            }
        }
    }
    if (!a.bscal) return;
    for (int t = 0; t < a.T; t++) {
        const int s = __reduce_add_sync(0xffffffffu, valid[t]);
        if ((threadIdx.x & 31) == 0 && s) atomicAdd(&a.cnt[t], s);   // integer atomics: deterministic
    }
    __shared__ int s_last;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = atomicAdd(&a.cnt[MAXT], 1) == (int)gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    if (threadIdx.x < MAXT) {
        const int t = threadIdx.x;
        const float aggw = a.agg_mean ? 1.f / (float)a.T : 1.f;
        float n = t < a.T ? (float)atomicExch(&a.cnt[t], 0) : 0.f;   // read and re-arm for the next launch
        if (a.world > 1 && t < a.T) n = (float)a.N * (float)a.world;
        a.bscal[BS_C + t] = t < a.T ? aggw / n : 0.f;
        a.bscal[BS_N + t] = n;
        a.bscal[BS_SS + t] = 0.f;
    }
    if (threadIdx.x == MAXT) atomicExch(&a.cnt[MAXT], 0);
    if (threadIdx.x >= 32 && threadIdx.x < 32 + MAXP) {
        const int k = threadIdx.x - 32;
        a.bscal[BS_BN + 2 * k] = 0.f;
        a.bscal[BS_BN + 2 * k + 1] = 1.f;
    }
    if (a.ready) {
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();   // records (all CTAs, ordered by the ticket) and the scalar row before the flag
            *reinterpret_cast<volatile unsigned*>(a.ready) = a.ready_val;
        }
    }
}

// device-visible address of a page-locked host array (cudaHostAlloc / cudaHostRegister), NULL for anything else
const float* mapped_host_ptr(const float* p)
{
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    if (at.type != cudaMemoryTypeHost || !at.devicePointer) return nullptr;
    return static_cast<const float*>(at.devicePointer);
}

struct Geom {
    int grid, nwarps;
    size_t smem;
};

// which compiled variant serves a batch of B samples.  The two-samples-per-lane form halves the
// shared-memory operand traffic but also the number of warps; measured at 65 536 samples per step it is
// 15 % slower than one sample per lane (8 vs 16 warps per SM: the step is latency- not LSU-bound), so it is
// only used on request (EH_USE_X2=1) until large-batch measurements say otherwise.
const Variant* pick_variant(const eh_ctx* c, int64_t B)
{
    if (c->var2 && getenv("EH_USE_X2") && B >= (int64_t)c->nsm * 4 * c->var2->chunk) return c->var2;
    return c->var;
}

// launchers: compiled-in variants bring their own (eh_variant_impl.cuh); the run-time compiled one goes through its handles
static bool is_jit(const eh_ctx* c, const Variant* v) { return c->jit_on && v == &c->jit_var; }
static cudaError_t vlaunch_step(const eh_ctx* c, const Variant* v, const StepArgs& a, int grid, int nwarps, size_t smem, cudaStream_t st, bool pdl)
{
    if (is_jit(c, v)) return jit_launch(c->jit.k_step, &a, grid, nwarps * 32, smem, st, pdl);
    return v->launch_step(a, grid, nwarps, smem, st, pdl);
}
static cudaError_t vlaunch_eval(const eh_ctx* c, const Variant* v, const EvalArgs& a, int grid, int nwarps, size_t smem, cudaStream_t st)
{
    if (is_jit(c, v)) return jit_launch(c->jit.k_eval, &a, grid, nwarps * 32, smem, st, false);
    return v->launch_eval(a, grid, nwarps, smem, st);
}
static cudaError_t vlaunch_epoch(const eh_ctx* c, const Variant* v, const EpochArgs& a, int grid, int nwarps, size_t smem, cudaStream_t st)
{
    if (is_jit(c, v)) return jit_launch_cooperative(c->jit.k_epoch, &a, grid, nwarps * 32, smem, st);
    return v->launch_epoch(a, grid, nwarps, smem, st);
}
static cudaError_t vepoch_max_grid(const eh_ctx* c, const Variant* v, int nwarps, size_t smem, int* max_ctas)
{
    if (is_jit(c, v)) return jit_max_grid(c->jit.k_epoch, nwarps * 32, smem, max_ctas);
    return v->epoch_max_grid(nwarps, smem, max_ctas);
}

// ... and which one serves a persistent launch: the tensor engine pays off once every SM has a few 128-sample tiles per
// step (EH_TC_MIN_BATCH overrides the threshold)
// 0: the tensor engine is opt-in (EH_TC_MIN_BATCH=<batch size from which it serves the persistent launches>)
constexpr long long EH_TC_DEFAULT_MIN_BATCH = 0;
const Variant* pick_epoch_variant(const eh_ctx* c, int64_t B)
{
    const Variant* v = pick_variant(c, B);
    if (c->var_tc && v == c->var) {
        const char* e = getenv("EH_TC_MIN_BATCH");   // (read per call: tests switch it)
        const long long tc_min = e ? atoll(e) : EH_TC_DEFAULT_MIN_BATCH;
        if (tc_min > 0 && B >= tc_min) v = c->var_tc;
    }
    return v;
}

Geom step_geometry(const eh_ctx* c, int64_t B, int reserve_sms = 0)
{
    const Variant* v = pick_variant(c, B);
    const int nsm = std::max(1, c->nsm - reserve_sms);  // SMs left to a concurrently running zero-copy packer
    size_t fixed = (size_t)(rup4(v->NW) + SS_FLOATS) * 4;
    size_t stage = (size_t)std::max(v->stage_floats, v->NPART) * 4;  // staging tile, later one row of the reduction scratch
    int wmax = (int)std::min<size_t>((size_t)v->max_warps, (c->smem_optin - fixed - 8192) / stage);
    if (wmax < 1) wmax = 1;
    int64_t nchunks = (B + v->chunk - 1) / v->chunk;
    Geom g;
    if (nchunks <= (int64_t)nsm * wmax) {
        int w = (int)((nchunks + nsm - 1) / nsm);
        w = std::max(1, std::min(w, wmax));
        g.nwarps = w;
        g.grid = (int)((nchunks + w - 1) / w);
    } else {
        g.nwarps = wmax;
        g.grid = nsm;
    }
    if (g.grid < 1) g.grid = 1;
    g.smem = fixed + (size_t)g.nwarps * stage;
    return g;
}

void fill_step_args(const eh_ctx* c, StepArgs& a)
{
    memset(&a, 0, sizeof a);
    a.pblock = c->d_theta;
    a.nflat = c->nflat;
    a.wsrc = c->d_wsrc;
    a.partial = c->d_partial;
    a.npart = c->var->NPART;
    for (int t = 0; t < MAXT; t++) a.loss_kind[t] = c->loss_kind[t];
    for (int s = 0; s < MAXPS; s++) a.slot[s] = c->slots[s];
    for (int i = 0; i < 4; i++) a.pmc[i] = c->pmc[i];
    a.use_bn = c->use_bn;
    a.prog = c->d_prog;
    a.scale_rt = c->scale_rt;
    for (int l = 0; l < 3; l++) a.pass_mask[l] = c->pass_mask[l];
}

void fill_update_args(const eh_ctx* c, UpdateArgs& u)
{
    memset(&u, 0, sizeof u);
    u.partial = c->d_partial;
    u.npart = c->var->NPART;
    u.npart_dw = c->var->off_stats;
    u.gvec = c->d_gvec;
    u.mode = UPD_FULL;
    u.apply = 1;
    u.nflat = c->nflat;
    u.ntheta = c->ntheta;
    u.pmap = c->d_pmap;
    u.pspan = c->d_pspan;
    u.theta = c->d_theta;
    u.m = c->d_m;
    u.v = c->d_v;
    u.ost = c->d_ost;
    u.T = c->n_targ;
    u.agg_mean = c->agg_mean;
    for (int t = 0; t < MAXT; t++) u.loss_kind[t] = c->loss_kind[t];
    u.opt_kind = c->opt_kind;
    u.adamw_coupled = c->adamw_coupled;
    u.l2coef = c->l2_on ? c->d_l2coef : nullptr; u.l2_aggw = c->l2_aggw; u.l2_loss_coef = c->l2_loss_coef;
    u.eta = c->eta; u.beta1 = c->beta1; u.beta2 = c->beta2; u.eps = c->eps; u.lambda = c->lambda;
    u.slot_of_flat = c->d_slot_of_flat;
    for (int s = 0; s < MAXPS; s++) u.slot[s] = c->slots[s];
    u.pm_id = c->pm_id;
}

// refresh the tail of the parameter block (uniform slot values + derived scalars) from phi
cudaError_t refresh_tail(const eh_ctx* c)
{
    TailArgs t;
    memset(&t, 0, sizeof t);
    t.pblock = c->d_theta; t.nflat = c->nflat; t.ntheta = c->ntheta; t.pm_id = c->pm_id;
    t.slot_of_flat = c->d_slot_of_flat;
    for (int s = 0; s < MAXPS; s++) t.slot[s] = c->slots[s];
    k_param_tail<<<1, 64, 0, c->stream>>>(t);
    return cudaGetLastError();
}

cudaError_t launch_update(const UpdateArgs& u, cudaStream_t st, bool pdl)
{
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(1);
    cfg.blockDim = dim3(512);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, k_update, u);
}

eh_status ensure_loss_cap(eh_ctx* c, size_t n)
{
    if (n <= c->loss_cap) return EH_OK;
    if (c->d_loss) cudaFree(c->d_loss);
    if (c->h_loss) cudaFreeHost(c->h_loss);
    c->d_loss = nullptr; c->h_loss = nullptr; c->loss_cap = 0;
    size_t cap = std::max<size_t>(n, 1024);
    CK(dalloc(&c->d_loss, cap));
    CK(cudaMallocHost((void**)&c->h_loss, cap * sizeof(float)));
    c->loss_cap = cap;
    return EH_OK;
}

eh_status ensure_idx_cap(eh_ctx* c, size_t n)
{
    if (n <= c->idx_cap) return EH_OK;
    if (c->d_idx) cudaFree(c->d_idx);
    if (c->d_idx64) cudaFree(c->d_idx64);
    c->d_idx = nullptr; c->d_idx64 = nullptr; c->idx_cap = 0;
    CK(dalloc(&c->d_idx, n));
    CK(dalloc(&c->d_idx64, n));
    c->idx_cap = n;
    return EH_OK;
}

// records [off, off + cnt) of the resident index stream -> d_stage, enqueued on `st`
eh_status stage_range(eh_ctx* c, int64_t n_total, int64_t off, int64_t cnt, cudaStream_t st)
{
    const Split& sp = c->split[EH_SPLIT_TRAIN];
    const int R4 = c->var->R4;
    if ((size_t)n_total > c->stage_cap) {
        CK(cudaStreamSynchronize(c->stream));
        if (c->d_stage) cudaFree(c->d_stage);
        c->d_stage = nullptr; c->stage_cap = 0;
        CK(dalloc(&c->d_stage, (size_t)n_total * R4));
        c->stage_cap = (size_t)n_total;
    }
    k_stage_records<<<(unsigned)((cnt + 255) / 256), 256, 0, st>>>(reinterpret_cast<const float4*>(sp.rec), c->d_idx + off,
                                                                     reinterpret_cast<float4*>(c->d_stage) + (size_t)off * (R4 / 4), cnt, R4 / 4);
    CK(cudaGetLastError());
    return EH_OK;
}

eh_status ensure_bscal_cap(eh_ctx* c, size_t nb)
{
    if (nb > c->bscal_cap) {
        if (c->d_bscal) cudaFree(c->d_bscal);
        c->d_bscal = nullptr; c->bscal_cap = 0;
        CK(dalloc(&c->d_bscal, nb * BS_STRIDE));
        c->bscal_cap = nb;
    }
    if (c->use_bn && nb > c->bn_batch_cap) {
        if (c->d_bn_batch) cudaFree(c->d_bn_batch);
        c->d_bn_batch = nullptr; c->bn_batch_cap = 0;
        CK(dalloc(&c->d_bn_batch, nb * 2 * MAXP));
        c->bn_batch_cap = nb;
    }
    return EH_OK;
}

// upload a 1-based int64 index stream and convert to 0-based int32 on the device
eh_status upload_indices(eh_ctx* c, const int64_t* idx1, int64_t n, int64_t nmax)
{
    eh_status s = ensure_idx_cap(c, (size_t)n);
    if (s != EH_OK) return s;
    c->idx_gen++;
    CK(cudaMemsetAsync(c->d_err, 0, sizeof(int), c->stream));
    CK(cudaMemcpyAsync(c->d_idx64, idx1, (size_t)n * sizeof(int64_t), cudaMemcpyHostToDevice, c->stream));
    k_idx_convert<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(c->d_idx64, c->d_idx, n, nmax, c->d_err);
    CK(cudaGetLastError());
    int herr = 0;
    CK(cudaMemcpyAsync(&herr, c->d_err, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    if (herr) return fail(c, EH_EINVAL, "index out of range 1..%lld in batch / permutation", (long long)nmax);
    return EH_OK;
}

bool needs_data_stats(const eh_ctx* c)
{
    if (c->use_bn || c->split[EH_SPLIT_TRAIN].has_nan) return true;
    for (int t = 0; t < c->n_targ; t++)
        if (c->loss_kind[t] == LOSS_NSELOSS) return true;
    return false;
}

// per-batch scalar rows for batches [b0, b1) of size B over the index stream d_idx[0..n), enqueued on c->stream
eh_status prepare_batch_rows_range(eh_ctx* c, int64_t n, int64_t B, int64_t b0, int64_t b1)
{
    int64_t nb = (n + B - 1) / B;
    eh_status s = ensure_bscal_cap(c, (size_t)nb);
    if (s != EH_OK) return s;
    const Split& sp = c->split[EH_SPLIT_TRAIN];
    const int64_t off = b0 * B;
    if (needs_data_stats(c) && c->world > 1)
        return fail(c, EH_EUNSUPPORTED,
                    "data-parallel mode with NaN targets, nseLoss or input BatchNorm: per-batch statistics are global -- call "
                    "eh_dp_batch_moments, add the result over the ranks and hand it to eh_dp_set_batch_moments after eh_set_perm");
    if (needs_data_stats(c)) {
        StatArgs a;
        memset(&a, 0, sizeof a);
        a.rec = sp.rec;
        a.R4 = c->var->R4;
        a.idx = c->d_idx + off;
        a.n = std::min<int64_t>(n, b1 * B) - off;
        a.Bfull = (int)B;
        a.P = c->var->P; a.F = c->var->F; a.T = c->n_targ;
        for (int t = 0; t < MAXT; t++) { a.shift_y[t] = sp.shift_y[t]; a.loss_kind[t] = c->loss_kind[t]; }
        for (int k = 0; k < MAXP; k++) a.shift_x[k] = sp.shift_x[k];
        a.agg_mean = c->agg_mean;
        a.use_bn = c->use_bn;
        a.bscal = c->d_bscal + (size_t)b0 * BS_STRIDE;
        a.bn_batch = c->use_bn ? c->d_bn_batch + (size_t)b0 * 2 * c->var->P : nullptr;
        k_batch_stats<<<(unsigned)(b1 - b0), 256, 0, c->stream>>>(a);
    } else {
        k_fill_bscal<<<(unsigned)((b1 - b0 + 127) / 128), 128, 0, c->stream>>>(c->d_bscal + (size_t)b0 * BS_STRIDE, (int)(b1 - b0),
                                                                               std::min<int64_t>(n, b1 * B) - off, (int)B,
                                                                               c->n_targ, c->agg_mean, c->world);
    }
    CK(cudaGetLastError());
    return EH_OK;
}

eh_status prepare_batch_rows(eh_ctx* c, int64_t n, int64_t B) { return prepare_batch_rows_range(c, n, B, 0, (n + B - 1) / B); }

// enqueue the K1/K2 launches of batches [b0, b1) of the resident index stream; the loss of
// batch b goes to loss_base[b - b0]
// Pre-pass of the prediction-statistics losses (rmse over several targets, pearsonLoss, kgeLoss, pbkgeLoss): forward over the
// batch with the CURRENT parameters and the batch's own scalar row (train-mode BatchNorm), sufficient statistics per
// target (k_eval), then the seed coefficients and the loss value into the row (k_stat_seeds).
eh_status enqueue_stat_prepass(eh_ctx* c, const float* rec, const int* idx, int64_t B, float* bscal_row)
{
    const Variant* v = c->var;
    const Split& sp = c->split[EH_SPLIT_TRAIN];
    const int nwarps = 8;
    const int64_t nchunks = (B + CHUNK - 1) / CHUNK;
    int grid = (int)std::min<int64_t>((nchunks + nwarps - 1) / nwarps, (int64_t)c->nsm * 2);
    if (grid < 1) grid = 1;
    if (grid > c->statpart_cap) {
        if (c->d_statpart) cudaFree(c->d_statpart);
        c->d_statpart = nullptr; c->statpart_cap = 0;
        CK(dalloc(&c->d_statpart, (size_t)c->nsm * 2 * MAXT * EVAL_NSTAT));
        c->statpart_cap = c->nsm * 2;
    }
    EvalArgs a;
    memset(&a, 0, sizeof a);
    a.rec = reinterpret_cast<const float4*>(rec);
    a.idx = idx; a.rec_base = 0; a.N = B; a.pblock = c->d_theta; a.nflat = c->nflat; a.wsrc = c->d_wsrc;
    a.use_bn = c->use_bn; a.bscal = bscal_row; a.prog = c->d_prog; a.scale_rt = c->scale_rt;
    for (int l = 0; l < 3; l++) a.pass_mask[l] = c->pass_mask[l];
    for (int s = 0; s < MAXPS; s++) a.slot[s] = c->slots[s];
    for (int i = 0; i < 4; i++) a.pmc[i] = c->pmc[i];
    for (int t = 0; t < MAXT; t++) a.shift_y[t] = sp.shift_y[t];
    a.partial = c->d_statpart;
    CK(vlaunch_eval(c, v, a, grid, nwarps, (size_t)(rup4(v->NW) + SS_FLOATS) * 4, c->stream));
    StatSeedArgs z;
    memset(&z, 0, sizeof z);
    z.partial = c->d_statpart; z.nparts = grid; z.Tk = v->T; z.T = c->n_targ; z.agg_mean = c->agg_mean; z.bscal = bscal_row;
    for (int t = 0; t < MAXT; t++) { z.kind[t] = c->loss_kind[t] == LOSS_AFFINE ? c->loss_kind_abi[t] : -1; z.shift_y[t] = sp.shift_y[t]; }
    k_stat_seeds<<<1, 32, 0, c->stream>>>(z);
    CK(cudaGetLastError());
    return EH_OK;
}

eh_status enqueue_steps(eh_ctx* c, int64_t n, int64_t B, int64_t b0, int64_t b1, float* loss_base, int apply,
                        bool want_grad, bool pdl, bool profile, int64_t prof_off)
{
    const Split& sp = c->split[EH_SPLIT_TRAIN];
    StepArgs a;
    fill_step_args(c, a);
    a.rec = reinterpret_cast<const float4*>(sp.rec);
    UpdateArgs u;
    fill_update_args(c, u);
    u.apply = apply;
    u.grad_out = want_grad ? c->d_grad : nullptr;
    for (int64_t b = b0; b < b1; b++) {
        int64_t Bk = std::min<int64_t>(B, n - b * B);
        Geom g = step_geometry(c, Bk);
        a.idx = c->d_idx + b * B;
        a.B = (int)Bk;
        a.bscal = c->d_bscal + (size_t)b * BS_STRIDE;
        if (c->stat_loss) {
            eh_status ps = enqueue_stat_prepass(c, sp.rec, a.idx, Bk, c->d_bscal + (size_t)b * BS_STRIDE);
            if (ps != EH_OK) return ps;
        }
        if (profile) CK(cudaEventRecord(c->prof_ev[2 * (prof_off + b - b0)], c->stream));
        CK(vlaunch_step(c, pick_variant(c, Bk), a, g.grid, g.nwarps, g.smem, c->stream, pdl));
        if (profile) CK(cudaEventRecord(c->prof_ev[2 * (prof_off + b - b0) + 1], c->stream));
        u.G = g.grid;
        u.bscal = a.bscal;
        u.loss_out = loss_base + (b - b0);
        CK(launch_update(u, c->stream, pdl));
    }
    return EH_OK;
}

void drop_graph(eh_ctx* c)
{
    if (c->gexec) cudaGraphExecDestroy(c->gexec);
    c->gexec = nullptr;
    c->g_n = c->g_B = 0;
}

// One whole pass over the resident permutation as a CUDA graph (2 kernel nodes per batch, chained
// with programmatic-dependent-launch edges): the per-step CPU launch cost leaves the critical path.
eh_status ensure_pass_graph(eh_ctx* c, int64_t n, int64_t B, bool pdl)
{
    if (c->gexec && c->g_n == n && c->g_B == B && c->g_pdl == (int)pdl && c->g_idx == c->d_idx &&
        c->g_bscal == c->d_bscal && c->g_loss == c->d_loss)
        return EH_OK;
    drop_graph(c);
    const int64_t nb = (n + B - 1) / B;
    for (int attempt = 0; attempt < 2; attempt++) {
        bool use_pdl = pdl && attempt == 0;
        cudaGraph_t graph = nullptr;
        CK(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
        eh_status s = enqueue_steps(c, n, B, 0, nb, c->d_loss, 1, false, use_pdl, false, 0);
        cudaError_t e = cudaStreamEndCapture(c->stream, &graph);
        if (s == EH_OK && e == cudaSuccess) e = cudaGraphInstantiate(&c->gexec, graph, 0);
        if (graph) cudaGraphDestroy(graph);
        if (s == EH_OK && e == cudaSuccess) {
            c->g_n = n; c->g_B = B; c->g_pdl = (int)pdl; c->g_idx = c->d_idx; c->g_bscal = c->d_bscal; c->g_loss = c->d_loss;
            c->g_has_pdl = use_pdl;
            return EH_OK;
        }
        cudaGetLastError();  // clear, retry without PDL edges
        c->gexec = nullptr;
        if (attempt == 1) return fail(c, EH_ECUDA, "CUDA graph capture of the epoch failed: %s", cudaGetErrorString(e));
    }
    return EH_OK;
}

// Persistent path: all nsteps optimiser steps in ONE launch (eh_epoch_kernel.cuh).
// Geometry: grid G (all co-resident, at most one CTA per SM; `reserve_sms` SMs are left to concurrently running
// packer kernels), w compute warps + one service warp per CTA.
// enqueue only (no host synchronisation): rec/idx/bscal select the data source, per-step loss sums go to
// c->d_stats and the losses to loss_out (device)
struct StreamLaunch {   // consumer mode (EpochArgs: ready .. batch_stride)
    const unsigned* ready; unsigned ready_base; unsigned* done; const int* host_total; float* loss_stream; long long batch_stride;
};

eh_status enqueue_persistent(eh_ctx* c, const float* rec, const int* idx, const float* bscal, float* loss_out, int64_t n,
                             int64_t B, int64_t first, int64_t nsteps, bool* used, long long** dbg_out, int reserve_sms = 0,
                             const StreamLaunch* sl = nullptr)
{
    *used = false;
    const Variant* v = pick_epoch_variant(c, B);
    const int64_t nb = (n + B - 1) / B;
    const int npartp = rup4(v->NPART);
    const size_t fixed = (size_t)(rup4(v->NW) + SS_FLOATS) * 4;
    const size_t stage = (size_t)std::max(v->stage_floats, v->NPART) * 4;
    const size_t eng_bytes = v->eng_bytes ? (size_t)v->eng_bytes + 128 : 0;   // engine-private region at the end (128-byte aligned)
    auto extra_of = [&](int tile_floats) { return (size_t)epoch_extra_floats(npartp, c->nflat, tile_floats, c->nsm) * 4 + 64 + eng_bytes; };
    const size_t smem_cap = c->smem_optin - 256;
    const int wpc = std::max(1, v->wpc);
    if (fixed + extra_of(0) + (size_t)wpc * stage > smem_cap) return EH_OK;  // does not fit: two-kernel path
    const int64_t nchunks = (B + v->chunk - 1) / v->chunk;
    const char* ew = getenv("EH_EPOCH_WARPS");
    const char* eg = getenv("EH_EPOCH_GRID");
    // the geometry only depends on (variant, batch size, reserved SMs, gather / contiguous): the occupancy query behind it
    // costs ~100 us of host time
    const int mode = (idx ? 1 : 0) | (reserve_sms << 1);
    if (!(c->geo_var == v && c->geo_B == B && c->geo_mode == mode)) {
        // at most 15 compute warps: with the service warp the CTA has 512 threads (128 registers each)
        int wcap = (int)std::min<size_t>((size_t)std::min(v->max_warps, wpc > 1 ? 16 : 15), (smem_cap - fixed - extra_of(0)) / stage);
        if (ew) wcap = std::max(1, std::min(atoi(ew), wcap));
        wcap -= wcap % wpc;
        if (wcap < wpc) return EH_OK;
        int max_ctas = 0;
        if (vepoch_max_grid(c, v, wcap + 1, fixed + extra_of(0) + (size_t)wcap * stage, &max_ctas) != cudaSuccess) { cudaGetLastError(); return EH_OK; }
        max_ctas = std::min(max_ctas, std::max(1, c->nsm - reserve_sms));
        if (eg) max_ctas = std::max(1, std::min(max_ctas, atoi(eg)));
        if (max_ctas < 1) return EH_OK;
        int w, G;
        if (wpc > 1) {
            // tile engines: `wpc` warps per tile; fewest rounds, then the fewest tile slots per CTA (at least two), then the
            // smallest grid that covers the batch
            const int ucap = wcap / wpc;
            const int64_t per_cta = (nchunks + max_ctas - 1) / max_ctas;
            const int64_t rounds = (per_cta + ucap - 1) / ucap;
            const int u = ew ? ucap : (int)std::min<int64_t>(ucap, std::max<int64_t>(2, (per_cta + rounds - 1) / rounds));
            w = u * wpc;
            G = (int)std::max<int64_t>(1, std::min<int64_t>(max_ctas, (nchunks + (int64_t)u * rounds - 1) / ((int64_t)u * rounds)));
        } else if (!ew && nchunks <= 8 && wcap >= 8) {
            // a batch of <= 256 samples runs in ONE CTA of 8 compute warps and needs no grid-wide exchange at all
            w = 8; G = 1;
        } else {
            // fewest rounds over the batch first; then the fewest warps per CTA that keep that round count -- but not
            // fewer than 8: below that the per-step exchange and the optimiser (one element per thread and trip) dominate
            // (tools/geom_sweep.py); then the smallest grid that covers the batch
            const int64_t per_cta = (nchunks + max_ctas - 1) / max_ctas;
            const int64_t rounds = (per_cta + wcap - 1) / wcap;
            w = ew ? wcap : (int)std::min<int64_t>(wcap, std::max<int64_t>(8, (per_cta + rounds - 1) / rounds));
            G = (int)std::min<int64_t>(max_ctas, (nchunks + (int64_t)w * rounds - 1) / ((int64_t)w * rounds));
            if (G < 1) G = 1;
        }
        // record tiles (TMA): batch-contiguous records only; two buffers of the largest per-CTA sample range
        int tile_floats = 0;
        if (!idx && !getenv("EH_NO_TILES")) {
            const int64_t per_cta = (nchunks + G - 1) / G;
            const size_t tf = (size_t)per_cta * v->chunk * v->R4;
            if (fixed + extra_of((int)tf) + (size_t)w * stage <= smem_cap) tile_floats = (int)tf;
        }
        int pg = 0;
        while (pg < 4 && (2 << pg) <= G) pg++;   // lanes per element pair in the slice reduction: min(16, pow2floor(G))
        c->geo_var = v; c->geo_B = B; c->geo_mode = mode; c->geo_G = G; c->geo_w = w; c->geo_tile = tile_floats; c->geo_pg = pg;
    }
    const int G = c->geo_G, w = c->geo_w, tile_floats = c->geo_tile;
    const size_t smem = fixed + extra_of(tile_floats) + (size_t)w * stage;
    if ((size_t)nsteps > c->stats_cap) {
        if (c->d_stats) cudaFree(c->d_stats);
        c->d_stats = nullptr; c->stats_cap = 0;
        CK(dalloc(&c->d_stats, (size_t)nsteps * MAXT));
        c->stats_cap = (size_t)nsteps;
    }
    EpochArgs a;
    memset(&a, 0, sizeof a);
    a.rec = reinterpret_cast<const float4*>(rec);
    a.idx = idx; a.n = n; a.B = (int)B; a.first_step = first; a.nsteps = (int)nsteps; a.nb = (int)nb;
    a.pblock = c->d_theta; a.nflat = c->nflat; a.ntheta = c->ntheta;
    a.m = c->d_m; a.v = c->d_v; a.ost = c->d_ost;
    a.wsrc = c->d_wsrc; a.pmap = c->d_pmap; a.cells = c->d_cells; a.pspan = c->d_pspan; a.slot_of_flat = c->d_slot_of_flat;
    a.bscal = bscal; a.pbuf = reinterpret_cast<uint2*>(c->d_pbuf); a.pbuf_rows = c->nsm + EH_PBUF_EXTRA_ROWS; a.tag_base = c->epoch_tag; a.stats_out = c->d_stats;
    a.npartp = npartp; a.work_floats = (int)((size_t)w * stage / 4); a.wcomp = w; a.pg_log2 = c->geo_pg; a.tile_floats = tile_floats;
    a.T = c->n_targ; a.agg_mean = c->agg_mean;
    for (int t = 0; t < MAXT; t++) a.loss_kind[t] = c->loss_kind[t];
    for (int s = 0; s < MAXPS; s++) a.slot[s] = c->slots[s];
    for (int i = 0; i < 4; i++) a.pmc[i] = c->pmc[i];
    a.use_bn = c->use_bn; a.pm_id = c->pm_id; a.prog = c->d_prog; a.scale_rt = c->scale_rt;
    for (int l = 0; l < 3; l++) a.pass_mask[l] = c->pass_mask[l];
    a.opt_kind = c->opt_kind; a.adamw_coupled = c->adamw_coupled;
    a.eta = c->eta; a.beta1 = c->beta1; a.beta2 = c->beta2; a.eps = c->eps; a.lambda = c->lambda;
    a.world = c->world; a.rank = c->rank; a.step_base = c->dp_steps; a.err = c->d_dperr;
    {
        const int stagger = getenv("EH_TC_STAGGER_NS") ? atoi(getenv("EH_TC_STAGGER_NS")) : 0;
        a.stagger_ns = wpc > 1 ? stagger : 0;
    }
    a.eng_off = v->eng_bytes ? (int)((smem - (size_t)v->eng_bytes) & ~(size_t)127) : 0;
    if (getenv("EH_DEBUG_GEOM"))
        fprintf(stderr, "[eh] persistent launch: %s G=%d warps=%d+1 smem=%zu (fixed %zu, per-warp %zu, tile %d floats) eng_off=%d eng_bytes=%d steps=%lld\n",
                v->name, G, w, smem, fixed, stage, tile_floats, a.eng_off, v->eng_bytes, (long long)nsteps);
    if (sl) {
        if (!tile_floats) return EH_OK;   // the consumer mode hands batches over through the record tiles
        a.ready = sl->ready; a.ready_base = sl->ready_base; a.done = sl->done; a.host_total = sl->host_total;
        a.loss_stream = sl->loss_stream; a.batch_stride = sl->batch_stride;
    }
    for (int r = 0; r < c->world && c->world > 1; r++) {
        a.inbox_peer[r] = reinterpret_cast<uint2*>(c->dp_peer[r]);
    }
    long long* d_dbg = nullptr;
    if (dbg_out && getenv("EH_EPOCH_DEBUG") && nsteps <= 64) {
        CK(dalloc(&d_dbg, (size_t)nsteps * G * 32));
        CK(cudaMemsetAsync(d_dbg, 0, (size_t)nsteps * G * 32 * sizeof(long long), c->stream));
        a.dbg = d_dbg;
        *dbg_out = d_dbg;
    }
    bool launched = false;
    if (!c->pg_off && !getenv("EH_NO_COOP")) {
        void* kargs[] = {(void*)&a};
        cudaKernelNodeParams kp{};
        kp.func = const_cast<void*>(v->epoch_func);
        kp.gridDim = dim3((unsigned)G); kp.blockDim = dim3((unsigned)((w + 1) * 32));
        kp.sharedMemBytes = (unsigned)smem; kp.kernelParams = kargs; kp.extra = nullptr;
        cudaError_t ge = cudaSuccess;
        if (!c->pg_exec || c->pg_func != v->epoch_func || c->pg_G != G || c->pg_threads != (w + 1) * 32 || c->pg_smem != smem) {
            if (c->pg_exec) cudaGraphExecDestroy(c->pg_exec);
            if (c->pg_graph) cudaGraphDestroy(c->pg_graph);
            c->pg_exec = nullptr; c->pg_graph = nullptr;
            cudaGraphNode_t n0 = nullptr, n2 = nullptr;
            ge = cudaGraphCreate(&c->pg_graph, 0);
            if (ge == cudaSuccess) ge = cudaGraphAddEventRecordNode(&n0, c->pg_graph, nullptr, 0, c->ev0);
            if (ge == cudaSuccess) ge = cudaGraphAddKernelNode(&c->pg_knode, c->pg_graph, &n0, 1, &kp);
            if (ge == cudaSuccess) {
                cudaLaunchAttributeValue av;
                memset(&av, 0, sizeof av);
                av.cooperative = 1;
                ge = cudaGraphKernelNodeSetAttribute(c->pg_knode, cudaLaunchAttributeCooperative, &av);
            }
            if (ge == cudaSuccess) ge = cudaGraphAddEventRecordNode(&n2, c->pg_graph, &c->pg_knode, 1, c->ev1);
            if (ge == cudaSuccess) ge = cudaGraphInstantiate(&c->pg_exec, c->pg_graph, 0);
            if (ge == cudaSuccess) { c->pg_func = v->epoch_func; c->pg_G = G; c->pg_threads = (w + 1) * 32; c->pg_smem = smem; }
        } else {
            ge = cudaGraphExecKernelNodeSetParams(c->pg_exec, c->pg_knode, &kp);
        }
        if (ge == cudaSuccess) ge = cudaGraphLaunch(c->pg_exec, c->stream);
        if (ge == cudaSuccess) {
            launched = true;
        } else {
            cudaGetLastError();
            if (c->pg_exec) cudaGraphExecDestroy(c->pg_exec);
            if (c->pg_graph) cudaGraphDestroy(c->pg_graph);
            c->pg_exec = nullptr; c->pg_graph = nullptr;
            c->pg_off = true;   // this driver / device does not take the graph form: plain stream launches from now on
        }
    }
    if (!launched) {
        CK(cudaEventRecord(c->ev0, c->stream));
        cudaError_t le = vlaunch_epoch(c, v, a, G, w + 1, smem, c->stream);
        if (le != cudaSuccess) {
            // e.g. cooperative launch refused: fall back to the two-kernel path
            cudaGetLastError();
            c->err = std::string("persistent launch refused: ") + cudaGetErrorString(le);
            return EH_OK;
        }
        CK(cudaEventRecord(c->ev1, c->stream));
    }
    c->epoch_tiles = tile_floats > 0; c->epoch_grid = G; c->epoch_warps = w;
    if (c->world > 1) c->dp_steps += (unsigned)nsteps;
    c->epoch_tag += (unsigned)nsteps;
    if (!sl) {   // (the consumer mode writes its losses itself, step by step)
        k_losses_from_stats<<<(unsigned)((nsteps + 127) / 128), 128, 0, c->stream>>>(c->d_stats, bscal, first, (int)nb,
                                                                                     (int)nsteps, c->n_targ, c->agg_mean,
                                                                                     c->d_losskind, loss_out);
        CK(cudaGetLastError());
    }
    *used = true;
    return EH_OK;
}

// Persistent path: all nsteps optimiser steps of the resident index stream in ONE launch, synchronous
eh_status run_persistent(eh_ctx* c, int64_t n, int64_t B, int64_t first, int64_t nsteps, bool* used)
{
    long long* d_dbg = nullptr;
    const bool staged = c->stage_on && !c->wide;
    if (staged && c->stage_gen != c->idx_gen) {
        eh_status ss = stage_range(c, n, 0, n, c->stream);
        if (ss != EH_OK) return ss;
        c->stage_gen = c->idx_gen;
    }
    eh_status s = enqueue_persistent(c, staged ? c->d_stage : c->split[EH_SPLIT_TRAIN].rec, staged ? nullptr : c->d_idx, c->d_bscal,
                                     c->d_loss, n, B, first, nsteps, used, &d_dbg);
    if (s != EH_OK || !*used) return s;
    CK(cudaMemcpyAsync(c->h_loss, c->d_loss, (size_t)nsteps * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    unsigned herr = 0;
    CK(cudaMemcpyAsync(&herr, c->d_dperr, sizeof(unsigned), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    if (herr) {
        cudaMemset(c->d_dperr, 0, sizeof(unsigned));
        return fail(c, EH_ENCCL, "persistent kernel gave up waiting (a CTA or a data-parallel peer never arrived)");
    }
    CK(cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1));
    if (d_dbg) {
        const int G = c->epoch_grid;
        std::vector<long long> h((size_t)nsteps * G * 32);
        CK(cudaMemcpy(h.data(), d_dbg, h.size() * sizeof(long long), cudaMemcpyDeviceToHost));
        cudaFree(d_dbg);
        if (FILE* f = fopen(getenv("EH_EPOCH_DEBUG"), "wb")) {
            long long hdr[4] = {nsteps, G, c->epoch_warps, c->epoch_tiles};
            fwrite(hdr, sizeof hdr, 1, f);
            fwrite(h.data(), sizeof(long long), h.size(), f);
            fclose(f);
        }
    }
    c->last_launches = 1;
    c->last_step_ms = c->last_ms;
    return EH_OK;
}

// one host batch's moments into the running statistics (same rule as update_bn_running); skipped batches excluded
void fold_bn_host_batch(eh_ctx* c, const float* mom, int64_t B, float loss)
{
    if (std::isnan(loss)) return;
    const int P = c->var->P;
    for (int i = 0; i < P; i++) {
        const float mu = mom[2 * i], var = mom[2 * i + 1];
        const float unb = B > 1 ? var * (float)B / (float)(B - 1) : var;
        c->bn_mean[i] = 0.9f * c->bn_mean[i] + 0.1f * mu;
        c->bn_var[i] = 0.9f * c->bn_var[i] + 0.1f * unb;
    }
}

// Lux BatchNorm running statistics (momentum 0.1, unbiased variance) after steps [first, first+nsteps) whose
// losses sit in c->h_loss[0..nsteps); skipped batches excluded
eh_status update_bn_running(eh_ctx* c, int64_t n, int64_t B, int64_t first, int64_t nsteps)
{
    const int64_t nb = (n + B - 1) / B;
    const int P = c->var->P;
    std::vector<float> bb((size_t)nb * 2 * P);
    CK(cudaMemcpy(bb.data(), c->d_bn_batch, bb.size() * sizeof(float), cudaMemcpyDeviceToHost));
    for (int64_t k = 0; k < nsteps; k++) {
        if (std::isnan(c->h_loss[k])) continue;
        int64_t b = (first + k) % nb;
        int64_t Bk = std::min<int64_t>(B, n - b * B) * c->world;  // rows of the global batch
        for (int i = 0; i < P; i++) {
            float mu = bb[(size_t)b * 2 * P + 2 * i], var = bb[(size_t)b * 2 * P + 2 * i + 1];
            float unb = Bk > 1 ? var * (float)Bk / (float)(Bk - 1) : var;
            c->bn_mean[i] = 0.9f * c->bn_mean[i] + 0.1f * mu;
            c->bn_var[i] = 0.9f * c->bn_var[i] + 0.1f * unb;
        }
    }
    return EH_OK;
}

// the step loop of the wide path: one sequence of launches per step on c->stream (eh_wide.cu)
eh_status wide_run_steps(eh_ctx* c, int64_t n, int64_t B, int64_t first, int64_t nsteps, float* losses, int apply,
                         float* grad_out_host)
{
    const Split& sp = c->split[EH_SPLIT_TRAIN];
    const int64_t nb = (n + B - 1) / B;
    if (c->world > 1) {
        if (!apply || grad_out_host) return fail(c, EH_EUNSUPPORTED, "data-parallel mode trains through eh_run_steps / eh_epoch only");
        for (int t = 0; t < c->n_targ; t++)
            if (c->loss_kind[t] == LOSS_RMSE) return fail(c, EH_EUNSUPPORTED, "rmse is not available in data-parallel mode on the wide path");
    }
    for (int64_t b = 0; b < nb; b++)
        if (!eh::wide::WideNet::batch_ok(std::min<int64_t>(B, n - b * B)))
            return fail(c, EH_EUNSUPPORTED, "wide path: batch size out of range (got %lld)",
                        (long long)std::min<int64_t>(B, n - b * B));
    CK(cudaEventRecord(c->ev0, c->stream));
    for (int64_t k = 0; k < nsteps; k++) {
        const int64_t b = (first + k) % nb;
        const int64_t Bk = std::min<int64_t>(B, n - b * B);
        eh::wide::WideDp dp;
        memset(&dp, 0, sizeof dp);
        if (c->world > 1) {
            dp.world = c->world; dp.rank = c->rank; dp.tag = ++c->dp_steps; dp.err = c->d_dperr;
            for (int r = 0; r < c->world; r++) dp.peer[r] = reinterpret_cast<float*>(c->dp_peer[r]);
        }
        cudaError_t e = c->wide->step(sp.rec, c->d_idx + b * B, 0, (int)Bk, c->d_bscal + (size_t)b * BS_STRIDE, c->d_theta, c->d_m,
                                      c->d_v, c->d_ost, c->d_grad, c->d_loss + k, apply, c->stream, c->world > 1 ? &dp : nullptr,
                                      sp.shift_y);
        if (e != cudaSuccess) return fail(c, EH_ECUDA, "wide path: %s", c->wide->error());
        if (apply) CK(refresh_tail(c));
    }
    CK(cudaEventRecord(c->ev1, c->stream));
    CK(cudaMemcpyAsync(c->h_loss, c->d_loss, (size_t)nsteps * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    if (grad_out_host)
        CK(cudaMemcpyAsync(grad_out_host, c->d_grad, (size_t)c->nflat * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    unsigned herr = 0;
    CK(cudaMemcpyAsync(&herr, c->d_dperr, sizeof(unsigned), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    if (herr) {
        cudaMemset(c->d_dperr, 0, sizeof(unsigned));
        return fail(c, EH_ENCCL, "wide path: a data-parallel peer never published its gradient");
    }
    CK(cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1));
    c->last_launches = nsteps * (3 + 5 * (int64_t)(c->var->NH - 1) + 4 + c->wide->extra_launches());
    c->last_step_ms = c->last_ms;
    if (losses) memcpy(losses, c->h_loss, (size_t)nsteps * sizeof(float));
    if (c->use_bn && apply) return update_bn_running(c, n, B, first, nsteps);
    return EH_OK;
}

// the step loop: steps [first, first+nsteps) of the resident index stream; step s trains on batch
// s mod nb (steps beyond one pass start another pass over the same permutation)
eh_status run_steps(eh_ctx* c, int64_t n, int64_t B, int64_t first, int64_t nsteps, float* losses, int apply,
                    float* grad_out_host)
{
    const Split& sp = c->split[EH_SPLIT_TRAIN];
    if (!sp.rec) return fail(c, EH_EINVAL, "train split not uploaded");
    const int64_t nb = (n + B - 1) / B;
    if (first < 0 || nsteps < 0) return fail(c, EH_EINVAL, "step range out of bounds");
    eh_status s = ensure_loss_cap(c, (size_t)std::max<int64_t>(nsteps, nb));
    if (s != EH_OK) return s;
    if (c->wide) return wide_run_steps(c, n, B, first, nsteps, losses, apply, grad_out_host);
    const bool profile = c->profiling != 0;
    // (steps with a statistics pre-pass are launched one by one: no PDL chaining, no pass graph)
    const bool pdl = !(c->flags & EH_FLAG_NO_PDL) && !profile && !c->stat_loss;
    const bool use_graph = !(c->flags & EH_FLAG_NO_GRAPH) && !profile && apply && !grad_out_host && nsteps >= nb && nb >= 4 && !c->stat_loss;
    if (profile) {
        while ((int64_t)c->prof_ev.size() < 2 * nsteps) {
            cudaEvent_t e;
            CK(cudaEventCreate(&e));
            c->prof_ev.push_back(e);
        }
    }
    bool persisted = false;
    if (c->world > 1) {
        // data parallel: the exchange lives in the persistent kernel
        if (!apply || grad_out_host || profile || !c->persist_ok)
            return fail(c, EH_EUNSUPPORTED, "data-parallel mode trains through eh_run_steps / eh_epoch only");
        s = run_persistent(c, n, B, first, nsteps, &persisted);
        if (s != EH_OK) return s;
        if (!persisted) return fail(c, EH_EUNSUPPORTED, "persistent kernel unavailable for this shape: %s", c->err.c_str());
    } else if (c->persist_ok && !(c->flags & EH_FLAG_NO_PERSIST) && !profile && apply && !grad_out_host && nsteps >= 2 &&
               nsteps < (1 << 30)) {
        s = run_persistent(c, n, B, first, nsteps, &persisted);
        if (s != EH_OK) return s;
    }
    if (use_graph && !persisted) {
        s = ensure_pass_graph(c, n, B, pdl);
        if (s != EH_OK) return s;
    }
    if (!persisted) CK(cudaEventRecord(c->ev0, c->stream));
    int64_t done = persisted ? nsteps : 0, launches = 0;
    while (done < nsteps) {
        int64_t b0 = (first + done) % nb;
        int64_t cnt = std::min<int64_t>(nb - b0, nsteps - done);
        if (use_graph && b0 == 0 && cnt == nb) {
            CK(cudaGraphLaunch(c->gexec, c->stream));
            CK(cudaMemcpyAsync(c->h_loss + done, c->d_loss, (size_t)nb * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
        } else {
            // direct launches write their losses behind the graph's slots
            s = enqueue_steps(c, n, B, b0, b0 + cnt, c->d_loss, apply, grad_out_host != nullptr, pdl, profile, done);
            if (s != EH_OK) return s;
            CK(cudaMemcpyAsync(c->h_loss + done, c->d_loss, (size_t)cnt * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
        }
        launches += 2 * cnt;
        done += cnt;
    }
    if (!persisted) {
        CK(cudaEventRecord(c->ev1, c->stream));
        if (grad_out_host)
            CK(cudaMemcpyAsync(grad_out_host, c->d_grad, (size_t)c->nflat * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        CK(cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1));
        c->last_launches = launches;
        c->last_step_ms = 0.f;
    }
    if (profile) {
        float tot = 0.f;
        for (int64_t k = 0; k < nsteps; k++) {
            float ms = 0.f;
            CK(cudaEventElapsedTime(&ms, c->prof_ev[2 * k], c->prof_ev[2 * k + 1]));
            tot += ms;
        }
        c->last_step_ms = tot;
    }
    if (losses) memcpy(losses, c->h_loss, (size_t)nsteps * sizeof(float));
    if (c->use_bn && apply) return update_bn_running(c, n, B, first, nsteps);
    return EH_OK;
}

// run_epoch! with the host permutation streamed in: the 8-byte indices of segment k+1 travel host->device
// (copy stream) and are converted while segment k trains (persistent kernel, compute stream).  Used for long
// epochs; *used = false leaves everything untouched and the caller takes the plain path.
eh_status epoch_pipelined(eh_ctx* c, const int64_t* perm1, int64_t n, int64_t B, float* losses, bool* used)
{
    *used = false;
    const int64_t nb = (n + B - 1) / B;
    // (the 8-byte host permutation is the largest transfer of this path: 8 B per sample against 11 us of training per 65 536
    // samples -- it is streamed in segments behind the training for every epoch of 8 or more batches)
    if (nb < 8 || !c->persist_ok || (c->flags & EH_FLAG_NO_PERSIST) || c->profiling) return EH_OK;
    const Split& sp = c->split[EH_SPLIT_TRAIN];
    if (!sp.rec) return fail(c, EH_EINVAL, "train split not uploaded");
    if (needs_data_stats(c) && c->world > 1) return EH_OK;  // the plain path reports it
    eh_status s = ensure_idx_cap(c, (size_t)n);
    if (s != EH_OK) return s;
    s = ensure_bscal_cap(c, (size_t)nb);
    if (s != EH_OK) return s;
    s = ensure_loss_cap(c, (size_t)nb);
    if (s != EH_OK) return s;
    // snapshot of the trainable state: an out-of-range index is only known once its segment has been converted,
    // and a failed call must leave the ctx as it found it
    if (!c->d_snap) CK(dalloc(&c->d_snap, (size_t)3 * c->nflat + PARAM_TAIL + 16));
    float* snap = c->d_snap;
    CK(cudaMemcpyAsync(snap, c->d_theta, ((size_t)c->nflat + PARAM_TAIL) * sizeof(float), cudaMemcpyDeviceToDevice, c->stream));
    CK(cudaMemcpyAsync(snap + c->nflat + PARAM_TAIL, c->d_m, (size_t)c->nflat * sizeof(float), cudaMemcpyDeviceToDevice, c->stream));
    CK(cudaMemcpyAsync(snap + 2 * c->nflat + PARAM_TAIL, c->d_v, (size_t)c->nflat * sizeof(float), cudaMemcpyDeviceToDevice, c->stream));
    static_assert(sizeof(OptState) <= 16 * sizeof(float), "snapshot tail too small");
    CK(cudaMemcpyAsync(snap + 3 * c->nflat + PARAM_TAIL, c->d_ost, sizeof(OptState), cudaMemcpyDeviceToDevice, c->stream));
    const std::vector<float> bn_mean0 = c->bn_mean, bn_var0 = c->bn_var;

    const int64_t seg = std::max<int64_t>(nb >= 256 ? 32 : 4, (nb + 7) / 8);  // steps per segment
    const int64_t nseg = (nb + seg - 1) / seg;
    while ((int64_t)c->seg_ev.size() < nseg) {
        cudaEvent_t e;
        CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        c->seg_ev.push_back(e);
    }
    cudaStream_t cs = c->copy_stream;
    const bool staged = c->stage_on && !c->wide;
    c->idx_gen++;
    if (staged && (size_t)n > c->stage_cap) {
        CK(cudaStreamSynchronize(c->stream));
        if (c->d_stage) cudaFree(c->d_stage);
        c->d_stage = nullptr; c->stage_cap = 0;
        CK(dalloc(&c->d_stage, (size_t)n * c->var->R4));
        c->stage_cap = (size_t)n;
    }
    CK(cudaMemsetAsync(c->d_err, 0, sizeof(int), c->stream));
    CK(cudaEventRecord(c->ev2, c->stream));
    CK(cudaStreamWaitEvent(cs, c->ev2, 0));  // earlier work on the compute stream may still read d_idx
    auto copy_seg = [&](int64_t k) -> eh_status {
        const int64_t off = k * seg * B, cnt = std::min<int64_t>(n, (k + 1) * seg * B) - off;
        CK(cudaMemcpyAsync(c->d_idx64 + off, perm1 + off, (size_t)cnt * sizeof(int64_t), cudaMemcpyHostToDevice, cs));
        k_idx_convert<<<(unsigned)((cnt + 255) / 256), 256, 0, cs>>>(c->d_idx64 + off, c->d_idx + off, cnt, sp.N, c->d_err);
        CK(cudaGetLastError());
        if (staged) {   // the segment's records in batch order (out-of-range indices were clamped to record 0 above)
            eh_status ss = stage_range(c, n, off, cnt, cs);
            if (ss != EH_OK) return ss;
        }
        CK(cudaEventRecord(c->seg_ev[k], cs));
        return EH_OK;
    };
    s = copy_seg(0);
    if (s != EH_OK) return s;
    const unsigned tag0 = c->epoch_tag, dp0 = c->dp_steps;
    for (int64_t k = 0; k < nseg; k++) {
        if (k + 1 < nseg) {
            s = copy_seg(k + 1);
            if (s != EH_OK) return s;
        }
        const int64_t s0 = k * seg, s1 = std::min<int64_t>(nb, s0 + seg);
        CK(cudaStreamWaitEvent(c->stream, c->seg_ev[k], 0));
        s = prepare_batch_rows_range(c, n, B, s0, s1);
        if (s != EH_OK) return s;
        bool u = false;
        s = enqueue_persistent(c, staged ? c->d_stage : sp.rec, staged ? nullptr : c->d_idx, c->d_bscal, c->d_loss + s0, n, B, s0,
                               s1 - s0, &u, nullptr);
        if (s != EH_OK) return s;
        if (!u) {
            if (k == 0) {  // nothing has trained yet: hand over to the plain path
                CK(cudaStreamSynchronize(cs));
                CK(cudaStreamSynchronize(c->stream));
                return EH_OK;
            }
            return fail(c, EH_ECUDA, "persistent launch refused mid-epoch: %s", c->err.c_str());
        }
    }
    CK(cudaEventRecord(c->ev3, c->stream));
    CK(cudaMemcpyAsync(c->h_loss, c->d_loss, (size_t)nb * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    unsigned herr = 0;
    int ierr = 0;
    CK(cudaMemcpyAsync(&herr, c->d_dperr, sizeof(unsigned), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(&ierr, c->d_err, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    if (herr || ierr) {
        CK(cudaMemcpy(c->d_theta, snap, ((size_t)c->nflat + PARAM_TAIL) * sizeof(float), cudaMemcpyDeviceToDevice));
        CK(cudaMemcpy(c->d_m, snap + c->nflat + PARAM_TAIL, (size_t)c->nflat * sizeof(float), cudaMemcpyDeviceToDevice));
        CK(cudaMemcpy(c->d_v, snap + 2 * c->nflat + PARAM_TAIL, (size_t)c->nflat * sizeof(float), cudaMemcpyDeviceToDevice));
        CK(cudaMemcpy(c->d_ost, snap + 3 * c->nflat + PARAM_TAIL, sizeof(OptState), cudaMemcpyDeviceToDevice));
        c->bn_mean = bn_mean0; c->bn_var = bn_var0;
        c->perm_n = 0; c->perm_B = 0;
        (void)tag0; (void)dp0;  // tags only ever grow: a rolled-back epoch simply leaves a gap
        if (herr) {
            cudaMemset(c->d_dperr, 0, sizeof(unsigned));
            return fail(c, EH_ENCCL, "persistent kernel gave up waiting (a CTA or a data-parallel peer never arrived)");
        }
        return fail(c, EH_EINVAL, "index out of range 1..%lld in batch / permutation", (long long)sp.N);
    }
    CK(cudaEventElapsedTime(&c->last_ms, c->ev2, c->ev3));
    c->last_launches = nseg;
    c->last_step_ms = c->last_ms;
    c->perm_n = n; c->perm_B = B;
    if (staged) c->stage_gen = c->idx_gen;
    if (losses) memcpy(losses, c->h_loss, (size_t)nb * sizeof(float));
    *used = true;
    if (c->use_bn) return update_bn_running(c, n, B, 0, nb);
    return EH_OK;
}

eh_status reset_opt_state(eh_ctx* c)
{
    OptState os;
    os.b1t = c->beta1; os.b2t = c->beta2; os.t = 0; os.skipped = 0;
    // the ctx streams are non-blocking: steps still in flight (eh_step_host_async) must retire before the state they
    // use is overwritten from the legacy stream
    if (c->stream) CK(cudaStreamSynchronize(c->stream));
    CK(cudaMemcpy(c->d_ost, &os, sizeof os, cudaMemcpyHostToDevice));
    CK(cudaMemset(c->d_m, 0, (size_t)c->nflat * sizeof(float)));
    CK(cudaMemset(c->d_v, 0, (size_t)c->nflat * sizeof(float)));
    return EH_OK;
}

eh_status ensure_host_stage(eh_ctx* c, HostStage& h, int64_t B)
{
    if (B <= h.cap) return EH_OK;
    if (h.d_X) cudaFree(h.d_X);
    if (h.d_planes) cudaFree(h.d_planes);
    if (h.d_rec) cudaFree(h.d_rec);
    h.cap = 0;
    int64_t cap = std::max<int64_t>(B, 4096);
    CK(dalloc(&h.d_X, (size_t)cap * c->n_pred_raw));
    CK(dalloc(&h.d_planes, (size_t)cap * (c->n_forc_raw + c->n_targ)));
    CK(dalloc(&h.d_rec, (size_t)cap * c->var->R4));
    if (!h.d_cnt) {
        CK(dalloc(&h.d_cnt, (size_t)MAXT + 1));
        // counters + ticket start at zero; every packer re-arms them after use.  Both streams may launch the
        // first packer of this slot, so the clear is waited for once
        CK(cudaMemsetAsync(h.d_cnt, 0, (MAXT + 1) * sizeof(int), c->stream));
        CK(cudaStreamSynchronize(c->stream));
    }
    if (!h.d_bscal) CK(dalloc(&h.d_bscal, (size_t)BS_STRIDE));
    if (!h.d_loss) CK(dalloc(&h.d_loss, (size_t)1));
    if (!h.ready) CK(cudaEventCreateWithFlags(&h.ready, cudaEventDisableTiming));
    if (!h.freed) CK(cudaEventCreateWithFlags(&h.freed, cudaEventDisableTiming));
    h.cap = cap;
    return EH_OK;
}

eh_status enqueue_host_step_compute(eh_ctx* c, HostStage& h, int64_t B, float* loss_dst, bool heavy, int reserve_sms);

// enqueue one host batch: H2D copies on the copy stream (they overlap the steps of earlier batches still running on
// the compute stream; EH_HOST_SLOTS staging slots), then pack, per-batch scalars, K1, K2 on the compute stream.
// loss_dst: where K2 stores the step's loss -- device memory, or page-locked host memory (written over PCIe by the
// kernel itself, so no separate D2H copy is enqueued).
eh_status enqueue_host_step(eh_ctx* c, HostStage& h, int64_t B, const float* X, const float* const* forc,
                            const float* const* targ, float* loss_dst, float* bn_dst)
{
    const Variant* v = c->var;
    // staging slots alternate between two copy streams: the ramp-up / drain of one batch's transfer overlaps the
    // next batch's (a single stream serialises them and leaves the PCIe link idle in between)
    cudaStream_t cs = c->pack_stream[(&h - c->hs) % EH_NPACK];
    bool heavy = c->use_bn || c->stat_loss;
    for (int t = 0; t < c->n_targ; t++) heavy |= (c->loss_kind[t] == LOSS_NSELOSS);
    // page-locked inputs are read in place by the packer (zero copy); anything else goes through the copy engine
    bool zero_copy = c->host_zero_copy && c->n_forc_raw + c->n_targ <= EH_PACK_MAXPLANES;
    PackHostArgs z;
    if (zero_copy) {
        memset(&z, 0, sizeof z);
        z.X = c->n_pred_raw > 0 ? mapped_host_ptr(X) : nullptr;
        zero_copy = c->n_pred_raw == 0 || z.X != nullptr;
        for (int f = 0; zero_copy && f < c->n_forc_raw; f++) zero_copy = (z.plane[f] = mapped_host_ptr(forc[f])) != nullptr;
        for (int t = 0; zero_copy && t < c->n_targ; t++)
            zero_copy = (z.plane[c->n_forc_raw + t] = mapped_host_ptr(targ[t])) != nullptr;
    }
    if (h.used) CK(cudaStreamWaitEvent(cs, h.freed, 0));  // the step that last read this slot must have retired
    if (zero_copy) {
        z.N = B; z.P_raw = c->n_pred_raw; z.ncols = c->ncols; z.R4 = v->R4;
        for (int i = 0; i < c->ncols; i++) { z.src_kind[i] = c->src_kind[i]; z.src_idx[i] = c->src_idx[i]; }
        z.x_pair = c->n_pred_raw == 2 && c->ncols >= 2 && c->src_kind[0] == 0 && c->src_idx[0] == 0 && c->src_kind[1] == 0 &&
                   c->src_idx[1] == 1 && ((uintptr_t)z.X & 7) == 0;
        z.rec = h.d_rec; z.T = c->n_targ; z.ycol0 = v->P + v->F; z.agg_mean = c->agg_mean;
        z.cnt = h.d_cnt; z.bscal = heavy ? nullptr : h.d_bscal;
        const int ctas = (int)std::min<int64_t>(EH_PACK_HOST_CTAS / EH_NPACK, (B + 1023) / 1024);   // EH_NPACK packers may be in flight
        k_pack_host<<<ctas, 1024, 0, cs>>>(z);
        CK(cudaGetLastError());
        CK(cudaEventRecord(h.ready, cs));
        CK(cudaStreamWaitEvent(c->stream, h.ready, 0));
        h.used = true;
        if (heavy) {
            StatArgs a;
            memset(&a, 0, sizeof a);
            a.rec = h.d_rec; a.R4 = v->R4; a.idx = nullptr; a.rec_base = 0; a.n = B; a.Bfull = (int)B;
            a.P = v->P; a.F = v->F; a.T = c->n_targ;
            const Split& sp = c->split[EH_SPLIT_TRAIN];
            for (int t = 0; t < MAXT; t++) { a.shift_y[t] = sp.shift_y[t]; a.loss_kind[t] = c->loss_kind[t]; }
            for (int k = 0; k < MAXP; k++) a.shift_x[k] = sp.shift_x[k];
            a.agg_mean = c->agg_mean; a.use_bn = c->use_bn; a.bscal = h.d_bscal; a.bn_batch = c->use_bn ? bn_dst : nullptr;
            k_batch_stats<<<1, 256, 0, c->stream>>>(a);
            CK(cudaGetLastError());
        }
        return enqueue_host_step_compute(c, h, B, loss_dst, heavy, EH_PACK_HOST_CTAS);
    }
    CK(cudaMemcpyAsync(h.d_X, X, (size_t)B * c->n_pred_raw * sizeof(float), cudaMemcpyHostToDevice, cs));
    for (int f = 0; f < c->n_forc_raw; f++)
        CK(cudaMemcpyAsync(h.d_planes + (size_t)f * B, forc[f], (size_t)B * sizeof(float), cudaMemcpyHostToDevice, cs));
    for (int t = 0; t < c->n_targ; t++)
        CK(cudaMemcpyAsync(h.d_planes + (size_t)(c->n_forc_raw + t) * B, targ[t], (size_t)B * sizeof(float),
                           cudaMemcpyHostToDevice, cs));
    CK(cudaEventRecord(h.ready, cs));
    CK(cudaStreamWaitEvent(c->stream, h.ready, 0));
    h.used = true;
    PackArgs p;
    memset(&p, 0, sizeof p);
    p.X = h.d_X; p.planes = h.d_planes; p.N = B; p.P_raw = c->n_pred_raw; p.ncols = c->ncols; p.R4 = v->R4;
    for (int i = 0; i < c->ncols; i++) { p.src_kind[i] = c->src_kind[i]; p.src_idx[i] = c->src_idx[i]; }
    p.rec = h.d_rec; p.rec_base = 0;
    if (!heavy) {
        k_pack_count<<<(unsigned)((B + 255) / 256), 256, 0, c->stream>>>(p, c->n_targ, v->P + v->F, h.d_cnt);
        CK(cudaGetLastError());
        k_bscal_from_counts<<<1, 32, 0, c->stream>>>(h.d_bscal, h.d_cnt, c->n_targ, c->agg_mean);
        CK(cudaGetLastError());
    } else {
        k_pack<<<(unsigned)((B + 255) / 256), 256, 0, c->stream>>>(p);
        CK(cudaGetLastError());
        StatArgs a;
        memset(&a, 0, sizeof a);
        a.rec = h.d_rec; a.R4 = v->R4; a.idx = nullptr; a.rec_base = 0; a.n = B; a.Bfull = (int)B;
        a.P = v->P; a.F = v->F; a.T = c->n_targ;
        const Split& sp = c->split[EH_SPLIT_TRAIN];
        for (int t = 0; t < MAXT; t++) { a.shift_y[t] = sp.shift_y[t]; a.loss_kind[t] = c->loss_kind[t]; }
        for (int k = 0; k < MAXP; k++) a.shift_x[k] = sp.shift_x[k];
        a.agg_mean = c->agg_mean; a.use_bn = c->use_bn; a.bscal = h.d_bscal; a.bn_batch = c->use_bn ? bn_dst : nullptr;
        k_batch_stats<<<1, 256, 0, c->stream>>>(a);
        CK(cudaGetLastError());
    }
    return enqueue_host_step_compute(c, h, B, loss_dst, heavy, 0);
}

// second half of a host-batch step: the records of slot `h` are ready on the compute stream
eh_status enqueue_host_step_compute(eh_ctx* c, HostStage& h, int64_t B, float* loss_dst, bool heavy, int reserve_sms)
{
    if (c->wide) {
        if (c->world > 1) return fail(c, EH_EUNSUPPORTED, "host-batch steps of the tensor-core path are single-GPU: use eh_run_steps in data-parallel mode");
        cudaError_t we = c->wide->step(h.d_rec, nullptr, 0, (int)B, h.d_bscal, c->d_theta, c->d_m, c->d_v, c->d_ost, c->d_grad, loss_dst, 1,
                                       c->stream, nullptr, c->split[EH_SPLIT_TRAIN].shift_y);
        if (we != cudaSuccess) return fail(c, EH_ECUDA, "wide path: %s", c->wide->error());
        CK(refresh_tail(c));
        CK(cudaEventRecord(h.freed, c->stream));
        return EH_OK;
    }
    if (c->world > 1) {
        // data parallel: one persistent launch of a single step (the exchange lives in that kernel)
        if (heavy) return fail(c, EH_EUNSUPPORTED, "data-parallel mode needs NaN-free targets, no nseLoss and no input BatchNorm");
        k_fill_bscal<<<1, 32, 0, c->stream>>>(h.d_bscal, 1, B, (int)B, c->n_targ, c->agg_mean, c->world);
        CK(cudaGetLastError());
        if (c->stats_cap < 1) { CK(dalloc(&c->d_stats, (size_t)64 * MAXT)); c->stats_cap = 64; }
        bool used = false;
        eh_status s = enqueue_persistent(c, h.d_rec, nullptr, h.d_bscal, loss_dst, B, B, 0, 1, &used, nullptr);
        if (s != EH_OK) return s;
        if (!used) return fail(c, EH_EUNSUPPORTED, "persistent kernel unavailable for this shape: %s", c->err.c_str());
        CK(cudaEventRecord(h.freed, c->stream));
        return EH_OK;
    }
    if (c->stat_loss) {
        eh_status ps = enqueue_stat_prepass(c, h.d_rec, nullptr, B, h.d_bscal);
        if (ps != EH_OK) return ps;
    }
    StepArgs a;
    fill_step_args(c, a);
    a.rec = reinterpret_cast<const float4*>(h.d_rec);
    a.idx = nullptr; a.rec_base = 0; a.B = (int)B; a.bscal = h.d_bscal;
    Geom g = step_geometry(c, B, reserve_sms);
    const bool pdl = false;  // the step follows memcpy/pack work here, nothing to overlap with
    CK(vlaunch_step(c, pick_variant(c, B), a, g.grid, g.nwarps, g.smem, c->stream, pdl));
    UpdateArgs u;
    fill_update_args(c, u);
    u.G = g.grid; u.bscal = h.d_bscal; u.loss_out = loss_dst;
    CK(launch_update(u, c->stream, pdl));
    CK(cudaEventRecord(h.freed, c->stream));
    return EH_OK;
}

// ---- grouped host batches (HostRing) ----
eh_status ensure_ring(eh_ctx* c, int64_t B)
{
    HostRing& r = c->ring;
    if (B <= r.cap) return EH_OK;
    // growing frees the buffers: nothing may still be reading or writing them (the open group is empty here)
    CK(cudaStreamSynchronize(c->stream));
    for (int i = 0; i < EH_NPACK; i++) CK(cudaStreamSynchronize(c->pack_stream[i]));
    if (r.d_rec) cudaFree(r.d_rec);
    r.d_rec = nullptr; r.cap = 0;
    const int64_t cap = std::max<int64_t>(B, 4096);
    const int nslots = EH_RING_NGRP * EH_RING_GROUP;
    CK(dalloc(&r.d_rec, (size_t)nslots * cap * c->var->R4));
    if (!r.d_bscal) {
        CK(dalloc(&r.d_bscal, (size_t)nslots * BS_STRIDE));
        CK(dalloc(&r.d_cnt, (size_t)nslots * (MAXT + 1)));
        CK(cudaMemsetAsync(r.d_cnt, 0, (size_t)nslots * (MAXT + 1) * sizeof(int), c->stream));
        CK(cudaStreamSynchronize(c->stream));
        for (int i = 0; i < EH_NPACK; i++) CK(cudaEventCreateWithFlags(&r.packed[i], cudaEventDisableTiming));
        for (int i = 0; i < EH_RING_NGRP; i++) CK(cudaEventCreateWithFlags(&r.freed[i], cudaEventDisableTiming));
    }
    for (int i = 0; i < EH_RING_NGRP; i++) r.used[i] = false;
    r.cap = cap;
    return EH_OK;
}

// launch the open group: one persistent kernel for its k batches (or, if that launch is refused, k step / update pairs)
eh_status flush_host_group(eh_ctx* c)
{
    HostRing& r = c->ring;
    if (r.k == 0) return EH_OK;
    const Variant* v = c->var;
    const int k = r.k, g = r.g;
    const int64_t B = r.B;
    r.k = 0;
    r.g = (g + 1) % EH_RING_NGRP;
    for (int i = 0; i < EH_NPACK; i++) {   // (packers rotate over the pack streams across groups: wait for all of them)
        CK(cudaEventRecord(r.packed[i], c->pack_stream[i]));
        CK(cudaStreamWaitEvent(c->stream, r.packed[i], 0));
    }
    const float* rec = r.d_rec + (size_t)g * EH_RING_GROUP * r.cap * v->R4;
    const float* bscal = r.d_bscal + (size_t)g * EH_RING_GROUP * BS_STRIDE;
    bool used = false;
    eh_status s = enqueue_persistent(c, rec, nullptr, bscal, r.loss0, (int64_t)k * B, B, 0, k, &used, nullptr, EH_PACK_HOST_CTAS);
    if (s != EH_OK) return s;
    if (!used && c->world > 1)
        return fail(c, EH_EUNSUPPORTED, "persistent kernel unavailable for this shape (data-parallel host batches need it): %s", c->err.c_str());
    if (!used) {
        for (int i = 0; i < k; i++) {
            StepArgs a;
            fill_step_args(c, a);
            a.rec = reinterpret_cast<const float4*>(rec + (size_t)i * B * v->R4);
            a.idx = nullptr; a.rec_base = 0; a.B = (int)B; a.bscal = bscal + (size_t)i * BS_STRIDE;
            Geom geo = step_geometry(c, B, EH_PACK_HOST_CTAS);
            CK(vlaunch_step(c, pick_variant(c, B), a, geo.grid, geo.nwarps, geo.smem, c->stream, false));
            UpdateArgs u;
            fill_update_args(c, u);
            u.G = geo.grid; u.bscal = a.bscal; u.loss_out = r.loss0 + i;
            CK(launch_update(u, c->stream, false));
        }
    }
    CK(cudaEventRecord(r.freed[g], c->stream));
    r.used[g] = true;
    return EH_OK;
}

// close the running burst of the consumer mode: tell the kernel how many steps there are, wait for it
eh_status end_host_stream(eh_ctx* c)
{
    HostStream& hs = c->hstream;
    if (!hs.active) return EH_OK;
    *reinterpret_cast<volatile int*>(hs.h_total) = hs.count;
    hs.active = false;
    unsigned herr = 0;
    CK(cudaMemcpyAsync(&herr, c->d_dperr, sizeof(unsigned), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    for (int i = 0; i < EH_NPACK; i++) CK(cudaStreamSynchronize(c->pack_stream[i]));
    if (herr) {
        cudaMemset(c->d_dperr, 0, sizeof(unsigned));
        return fail(c, EH_ENCCL, "persistent kernel gave up waiting (a CTA never arrived)");
    }
    return EH_OK;
}

// consumer mode: pack one page-locked batch into its ring slot; the first batch of a burst also launches the persistent
// kernel that trains on the slots as they are published.  *taken = false: not eligible, the caller takes another path.
eh_status stream_enqueue(eh_ctx* c, int64_t B, const PackHostArgs& z0, float* pin, bool* taken)
{
    *taken = false;
    HostStream& hs = c->hstream;
    HostRing& r = c->ring;
    const Variant* v = c->var;
    if (hs.off || c->world > 1 || getenv("EH_NO_COOP")) return EH_OK;
    if (hs.active && (B != hs.B || hs.count >= EH_STREAM_MAX_STEPS)) {
        eh_status s = end_host_stream(c);
        if (s != EH_OK) return s;
    }
    if (B > r.cap) {
        eh_status s = end_host_stream(c);
        if (s != EH_OK) return s;
        s = ensure_ring(c, B);
        if (s != EH_OK) return s;
    }
    const int nslots = EH_RING_NGRP * EH_RING_GROUP;
    if (!hs.h_total) {
        CK(cudaMallocHost((void**)&hs.h_total, 64));
        *hs.h_total = 0;
        CK(dalloc(&hs.d_ready, (size_t)nslots));
        CK(dalloc(&hs.d_done, (size_t)4));
        CK(cudaMemset(hs.d_ready, 0, nslots * sizeof(unsigned)));
        CK(cudaMemset(hs.d_done, 0, 4 * sizeof(unsigned)));
    }
    const unsigned g = hs.global;
    const int slot = (int)(g % (unsigned)nslots);
    if (!hs.active) {
        // open a burst: the consumer kernel first (it waits for slot `slot`), on the compute stream
        *reinterpret_cast<volatile int*>(hs.h_total) = 0;
        if ((size_t)EH_STREAM_MAX_STEPS > c->stats_cap) {
            if (c->d_stats) cudaFree(c->d_stats);
            c->d_stats = nullptr; c->stats_cap = 0;
            CK(dalloc(&c->d_stats, (size_t)EH_STREAM_MAX_STEPS * MAXT));
            c->stats_cap = EH_STREAM_MAX_STEPS;
        }
        StreamLaunch sl{hs.d_ready, g, hs.d_done, hs.h_total, pin, (long long)r.cap};
        bool used = false;
        eh_status s = enqueue_persistent(c, r.d_rec, nullptr, r.d_bscal, nullptr, (int64_t)nslots * B, B, slot, EH_STREAM_MAX_STEPS, &used,
                                         nullptr, EH_PACK_HOST_CTAS, &sl);
        if (s != EH_OK) return s;
        if (!used) { hs.off = true; return EH_OK; }   // (no persistent kernel for this shape: grouped / per-step path)
        hs.active = true; hs.B = B; hs.count = 0;
    }
    PackHostArgs z = z0;
    z.rec = r.d_rec + (size_t)slot * r.cap * v->R4;
    z.cnt = r.d_cnt + (size_t)slot * (MAXT + 1);
    z.bscal = r.d_bscal + (size_t)slot * BS_STRIDE;
    z.wait_done = g >= (unsigned)nslots ? hs.d_done : nullptr;
    z.wait_min = g - (unsigned)nslots + 1u;
    z.ready = hs.d_ready + slot;
    z.ready_val = g + 1u;
    const int ctas = (int)std::min<int64_t>(EH_PACK_HOST_CTAS / EH_NPACK, (B + 1023) / 1024);
    k_pack_host<<<ctas, 1024, 0, c->pack_stream[(r.rr++) % EH_NPACK]>>>(z);
    CK(cudaGetLastError());
    hs.global = g + 1u;
    hs.count++;
    *taken = true;
    return EH_OK;
}

// pack one page-locked batch into the open group; *taken = false when the batch has to go the per-step way
// size of the next group of a burst.  Default ramp 1, 2, 4, 8, 16, 16, ...; EH_RING_RAMP="a,b,c,..." overrides it (the last
// entry repeats), for experiments
int next_group_size(HostRing& r)
{
    static std::vector<int> ramp = [] {
        std::vector<int> v;
        if (const char* e = getenv("EH_RING_RAMP")) {
            for (const char* p = e; *p;) {
                int x = atoi(p);
                if (x >= 1) v.push_back(std::min(x, EH_RING_GROUP));
                while (*p && *p != ',') p++;
                if (*p == ',') p++;
            }
        }
        return v;
    }();
    r.launches++;
    if (ramp.empty()) return std::min(EH_RING_GROUP, 2 * r.limit);
    return ramp[std::min<size_t>((size_t)r.launches, ramp.size() - 1)];
}

eh_status ring_enqueue(eh_ctx* c, int64_t B, const float* X, const float* const* forc, const float* const* targ, float* pin,
                       bool* taken)
{
    *taken = false;
    HostRing& r = c->ring;
    const Variant* v = c->var;
    bool heavy = c->use_bn || c->stat_loss;
    for (int t = 0; t < c->n_targ; t++) heavy |= (c->loss_kind[t] == LOSS_NSELOSS);
    // (large batches amortise their launches anyway; the ring would only cost memory: 48 slots)
    if (B > EH_RING_MAX_BATCH) return EH_OK;
    if (r.off || !c->host_zero_copy || c->wide || heavy || !c->persist_ok || c->profiling ||
        (c->flags & EH_FLAG_NO_PERSIST) || c->n_forc_raw + c->n_targ > EH_PACK_MAXPLANES)
        return EH_OK;
    PackHostArgs z;
    memset(&z, 0, sizeof z);
    if (c->n_pred_raw > 0 && !(z.X = mapped_host_ptr(X))) return EH_OK;
    for (int f = 0; f < c->n_forc_raw; f++)
        if (!(z.plane[f] = mapped_host_ptr(forc[f]))) return EH_OK;
    for (int t = 0; t < c->n_targ; t++)
        if (!(z.plane[c->n_forc_raw + t] = mapped_host_ptr(targ[t]))) return EH_OK;
    z.N = B; z.P_raw = c->n_pred_raw; z.ncols = c->ncols; z.R4 = v->R4;
    for (int i = 0; i < c->ncols; i++) { z.src_kind[i] = c->src_kind[i]; z.src_idx[i] = c->src_idx[i]; }
    z.x_pair = c->n_pred_raw == 2 && c->ncols >= 2 && c->src_kind[0] == 0 && c->src_idx[0] == 0 && c->src_kind[1] == 0 &&
               c->src_idx[1] == 1 && ((uintptr_t)z.X & 7) == 0;
    z.T = c->n_targ; z.ycol0 = v->P + v->F; z.agg_mean = c->agg_mean; z.world = c->world;
    if (r.k == 0) {
        // consumer mode first: one persistent launch per burst, batches picked up as their packers publish them
        bool st = false;
        eh_status s = stream_enqueue(c, B, z, pin, &st);
        if (s != EH_OK) return s;
        if (st) { *taken = true; return EH_OK; }
    }
    if (r.k > 0 && B != r.B) {
        eh_status s = flush_host_group(c);
        if (s != EH_OK) return s;
    }
    if (B > r.cap) {
        eh_status s = ensure_ring(c, B);
        if (s != EH_OK) return s;
    }
    const int g = r.g, k = r.k;
    if (k == 0) {
        r.B = B;
        r.loss0 = pin;
        if (r.used[g]) {   // the launch that last trained on this group's slots must have retired
            for (int i = 0; i < EH_NPACK; i++) CK(cudaStreamWaitEvent(c->pack_stream[i], r.freed[g], 0));
        }
    }
    const int slot = g * EH_RING_GROUP + k;
    z.rec = r.d_rec + ((size_t)g * EH_RING_GROUP * r.cap + (size_t)k * B) * v->R4;
    z.cnt = r.d_cnt + (size_t)slot * (MAXT + 1);
    z.bscal = r.d_bscal + (size_t)slot * BS_STRIDE;
    // EH_NPACK packers may be in flight (one per pack stream): they share the reserved SMs
    const int ctas = (int)std::min<int64_t>(EH_PACK_HOST_CTAS / EH_NPACK, (B + 1023) / 1024);
    k_pack_host<<<ctas, 1024, 0, c->pack_stream[(r.rr++) % EH_NPACK]>>>(z);
    CK(cudaGetLastError());
    r.k = k + 1;
    *taken = true;
    if (r.k >= r.limit) {
        // group sizes within a burst: 1, 2, 4, 8, 16, 16, ... (the first steps start while later batches still cross PCIe;
        // measured at 20 x 65 536-sample batches: 1.84e9 -> 2.27e9 samples/s; constant small groups lose more to the
        // ~50 us every launch costs than they win)
        r.limit = next_group_size(r);
        return flush_host_group(c);
    }
    return EH_OK;
}

}  // namespace

// every entry point that looks at or changes the training state first launches what eh_step_host_async still holds back
#define EH_ENTER(c)                                             \
    do {                                                        \
        CK(cudaSetDevice((c)->device));                         \
        if ((c)->hstream.active) {                              \
            eh_status fs__ = end_host_stream(c);                \
            if (fs__ != EH_OK) return fs__;                     \
        }                                                       \
        if ((c)->ring.k) {                                      \
            eh_status fs__ = flush_host_group(c);               \
            if (fs__ != EH_OK) return fs__;                     \
        }                                                       \
    } while (0)

// =============================== C ABI ===============================
extern "C" {

eh_status eh_create(eh_ctx** out, const eh_model_desc* desc)
{
    if (!out || !desc) return fail(nullptr, EH_EINVAL, "null argument");
    *out = nullptr;
    eh_ctx* c = new (std::nothrow) eh_ctx();
    if (!c) return fail(nullptr, EH_ENOMEM, "out of host memory");
    auto bail = [&](eh_status s) {
        g_create_error = c->err;
        eh_destroy(c);
        return s;
    };
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        fail(c, EH_ECUDA, "no CUDA device available (%s); this library has no CPU fallback", cudaGetErrorString(e));
        return bail(EH_ECUDA);
    }
    c->device = desc->device;
    if (c->device < 0 || c->device >= ndev) { fail(c, EH_EINVAL, "device %d out of range 0..%d", c->device, ndev - 1); return bail(EH_EINVAL); }
    cudaDeviceProp prop;
    if ((e = cudaSetDevice(c->device)) != cudaSuccess || (e = cudaGetDeviceProperties(&prop, c->device)) != cudaSuccess) {
        fail(c, EH_ECUDA, "cudaSetDevice/GetDeviceProperties: %s", cudaGetErrorString(e));
        return bail(EH_ECUDA);
    }
    if (prop.major != 10) {
        fail(c, EH_ECUDA, "device %d is sm_%d%d; this library contains sm_100a code only", c->device, prop.major, prop.minor);
        return bail(EH_ECUDA);
    }
    c->nsm = prop.multiProcessorCount;
    c->smem_optin = prop.sharedMemPerBlockOptin;
    eh_status s = build_plan(c, desc);
    if (s != EH_OK) return bail(s);
    const Variant* v = c->var;
    auto cuda_setup = [&]() -> eh_status {
        CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
        c->pack_stream[0] = c->copy_stream;
        for (int i = 1; i < EH_NPACK; i++) CK(cudaStreamCreateWithFlags(&c->pack_stream[i], cudaStreamNonBlocking));
        if (const char* e = getenv("EH_HOST_NO_ZEROCOPY")) c->host_zero_copy = !(e[0] && e[0] != '0');
        if (const char* e = getenv("EH_HOST_NO_GROUPS")) c->ring.off = e[0] && e[0] != '0';
        if (const char* e = getenv("EH_NO_STAGE")) c->stage_on = !(e[0] && e[0] != '0');
        if (const char* e = getenv("EH_NO_PGRAPH")) c->pg_off = e[0] && e[0] != '0';
        // consumer mode of eh_step_host_async (one persistent launch per burst that waits for the packers): OPT-IN with
        // EH_HOST_STREAM=1.  While a burst is open the kernel spins on host progress, so ANY device-synchronising call of
        // the process (cudaFree / cudaMallocHost / cudaHostRegister, another library's allocator, a finaliser) deadlocks
        // against it; measured it is no faster than the ramped grouped launches (DESIGN.md section 5.6).
        c->hstream.off = true;
        if (const char* e = getenv("EH_HOST_STREAM")) c->hstream.off = !(e[0] && e[0] != '0');
        CK(cudaEventCreate(&c->ev0));
        CK(cudaEventCreate(&c->ev1));
        CK(cudaEventCreate(&c->ev2));
        CK(cudaEventCreate(&c->ev3));
        size_t fixed = (size_t)(rup4(v->NW) + SS_FLOATS) * 4;
        size_t stage = (size_t)std::max(v->stage_floats, v->NPART) * 4;
        int wmax = (int)std::min<size_t>((size_t)v->max_warps, (c->smem_optin - fixed - 8192) / stage);
        if (wmax < 1) return fail(c, EH_EUNSUPPORTED, "variant %s needs %zu B of shared memory per warp", v->name, stage);
        if (c->jit_on) {
            std::string jerr;
            if (!jit_load(c->jit_cubin, c->jit_names, &c->jit, &jerr)) return fail(c, EH_ECUDA, "run-time compiled kernels: %s", jerr.c_str());
            c->jit_var.epoch_func = c->jit.k_epoch;
            std::string().swap(c->jit_cubin);
            CK(jit_prepare(c->jit, c->smem_optin - 256, fixed));
        }
        if (v->prepare) CK(v->prepare(c->smem_optin - 256, fixed));  // kernels carry a few bytes of static shared memory
        if (c->var2) CK(c->var2->prepare(c->smem_optin - 256, fixed));
        if (c->var_tc) CK(c->var_tc->prepare(c->smem_optin - 256, fixed));
        CK(dalloc(&c->d_wsrc, c->h_wsrc.size()));
        CK(dalloc(&c->d_pmap, c->h_pmap.size()));
        CK(dalloc(&c->d_pspan, c->h_pspan.size()));
        if (c->l2_on) {
            CK(dalloc(&c->d_l2coef, c->h_l2coef.size()));
            CK(cudaMemcpy(c->d_l2coef, c->h_l2coef.data(), c->h_l2coef.size() * sizeof(float), cudaMemcpyHostToDevice));
        }
        CK(cudaMemcpy(c->d_wsrc, c->h_wsrc.data(), c->h_wsrc.size() * sizeof(int), cudaMemcpyHostToDevice));
        CK(cudaMemcpy(c->d_pmap, c->h_pmap.data(), c->h_pmap.size() * sizeof(int), cudaMemcpyHostToDevice));
        CK(cudaMemcpy(c->d_pspan, c->h_pspan.data(), c->h_pspan.size() * sizeof(float), cudaMemcpyHostToDevice));
        CK(dalloc(&c->d_theta, (size_t)c->nflat + PARAM_TAIL));
        CK(dalloc(&c->d_cells, c->h_cells.size()));
        CK(dalloc(&c->d_slot_of_flat, c->h_slot_of_flat.size()));
        CK(dalloc(&c->d_losskind, (size_t)MAXT));
        CK(cudaMemcpy(c->d_cells, c->h_cells.data(), c->h_cells.size() * sizeof(int), cudaMemcpyHostToDevice));
        CK(cudaMemcpy(c->d_slot_of_flat, c->h_slot_of_flat.data(), c->h_slot_of_flat.size() * sizeof(int), cudaMemcpyHostToDevice));
        CK(cudaMemcpy(c->d_losskind, c->loss_kind, MAXT * sizeof(int), cudaMemcpyHostToDevice));
        CK(dalloc(&c->d_pbuf, (size_t)4 * (c->nsm + EH_PBUF_EXTRA_ROWS) * rup4(v->NPART)));  // [2][rows][npartp] {value, tag}: CTA partials + totals, by step parity
        CK(cudaMemset(c->d_pbuf, 0, (size_t)4 * (c->nsm + EH_PBUF_EXTRA_ROWS) * rup4(v->NPART) * sizeof(float)));
        CK(dalloc(&c->d_dperr, (size_t)1));
        CK(cudaMemset(c->d_dperr, 0, sizeof(unsigned)));
        CK(dalloc(&c->d_m, (size_t)c->nflat));
        CK(dalloc(&c->d_v, (size_t)c->nflat));
        CK(dalloc(&c->d_grad, (size_t)c->nflat));
        CK(dalloc(&c->d_ost, (size_t)1));
        CK(dalloc(&c->d_partial, (size_t)(c->nsm + 8) * v->NPART));
        CK(dalloc(&c->d_gvec, (size_t)v->NPART));
        CK(dalloc(&c->d_err, (size_t)1));
        CK(dalloc(&c->d_evalpart, (size_t)c->nsm * 4 * MAXT * EVAL_NSTAT));
        CK(dalloc(&c->d_bn_test, (size_t)BS_STRIDE));
        if (c->small_prog) {
            CK(cudaMalloc((void**)&c->d_prog, sizeof(PmProgData)));
            CK(cudaMemcpy(c->d_prog, &c->h_prog, sizeof(PmProgData), cudaMemcpyHostToDevice));
        }
        CK(cudaMemset(c->d_theta, 0, ((size_t)c->nflat + PARAM_TAIL) * sizeof(float)));
        CK(refresh_tail(c));
        if (v->engine == 3) {
            c->wide_model.d_slot_of_flat = c->d_slot_of_flat;
            c->wide_model.d_l2coef = c->l2_on ? c->d_l2coef : nullptr;
            char werr[256] = {0};
            c->wide = eh::wide::WideNet::create(c->wide_model, werr, sizeof werr);
            if (!c->wide) return fail(c, EH_ECUDA, "%s", werr);
            eh_status rs = reset_opt_state(c);
            if (rs != EH_OK) return rs;
            cudaError_t we = c->wide->refresh_images(c->d_theta, c->d_m, c->d_v, c->d_ost, c->stream);
            if (we != cudaSuccess) return fail(c, EH_ECUDA, "wide path: %s", c->wide->error());
            return EH_OK;
        }
        return reset_opt_state(c);
    };
    s = cuda_setup();
    if (s != EH_OK) return bail(s);
    *out = c;
    return EH_OK;
}

void eh_destroy(eh_ctx* c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->hstream.active) end_host_stream(c);   // a consumer kernel still waiting for batches: close its burst first
    if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
    for (int i = 1; i < EH_NPACK; i++)
        if (c->pack_stream[i]) cudaStreamSynchronize(c->pack_stream[i]);
    if (c->stream) cudaStreamSynchronize(c->stream);
    delete c->wide;
    c->wide = nullptr;
    if (c->gexec) cudaGraphExecDestroy(c->gexec);
    if (c->pg_exec) cudaGraphExecDestroy(c->pg_exec);
    jit_unload(&c->jit);
    if (c->pg_graph) cudaGraphDestroy(c->pg_graph);
    for (int r = 0; r < c->world && c->world > 1; r++)
        if (r != c->rank && c->dp_peer[r]) cudaIpcCloseMemHandle(c->dp_peer[r]);
    if (c->dp_block) cudaFree(c->dp_block);
    void* ptrs[] = {c->d_wsrc, c->d_pmap, c->d_pspan, c->d_theta, c->d_m, c->d_v, c->d_grad, c->d_ost, c->d_partial,
                    c->d_gvec, c->d_dperr, c->d_cells, c->d_slot_of_flat, c->d_losskind, c->d_pbuf, c->d_stats, c->d_bscal, c->d_bn_batch, c->d_idx, c->d_idx64, c->d_err, c->d_loss, c->d_evalpart, c->d_statpart, c->d_l2coef,
                    c->d_bn_test, c->d_prog, c->d_stage, c->split[0].rec, c->split[1].rec};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    {
        HostRing& r = c->ring;
        void* rp[] = {r.d_rec, r.d_bscal, r.d_cnt};
        for (void* p : rp)
            if (p) cudaFree(p);
        for (cudaEvent_t e : r.packed)
            if (e) cudaEventDestroy(e);
        for (cudaEvent_t e : r.freed)
            if (e) cudaEventDestroy(e);
    }
    for (HostStage& h : c->hs) {
        void* hp[] = {h.d_X, h.d_planes, h.d_rec, h.d_cnt, h.d_bscal, h.d_loss};
        for (void* p : hp)
            if (p) cudaFree(p);
        if (h.ready) cudaEventDestroy(h.ready);
        if (h.freed) cudaEventDestroy(h.freed);
    }
    if (c->h_loss) cudaFreeHost(c->h_loss);
    if (c->hstream.h_total) cudaFreeHost(c->hstream.h_total);
    if (c->hstream.d_ready) cudaFree(c->hstream.d_ready);
    if (c->hstream.d_done) cudaFree(c->hstream.d_done);
    if (c->h_async_loss) cudaFreeHost(c->h_async_loss);
    if (c->h_async_bn) cudaFreeHost(c->h_async_bn);
    if (c->h_bn0) cudaFreeHost(c->h_bn0);
    for (cudaEvent_t e : c->prof_ev) cudaEventDestroy(e);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->ev2) cudaEventDestroy(c->ev2);
    if (c->ev3) cudaEventDestroy(c->ev3);
    for (cudaEvent_t e : c->seg_ev) cudaEventDestroy(e);
    if (c->d_snap) cudaFree(c->d_snap);
    if (c->stream) cudaStreamDestroy(c->stream);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    for (int i = 1; i < EH_NPACK; i++)
        if (c->pack_stream[i]) cudaStreamDestroy(c->pack_stream[i]);
    delete c;
}

const char* eh_last_error(const eh_ctx* c) { return c ? c->err.c_str() : g_create_error.c_str(); }

int64_t eh_num_params(const eh_ctx* c) { return c ? c->nflat : -1; }

eh_status eh_upload(eh_ctx* c, int32_t split, int64_t N, const float* X, const float* const* forc,
                    const float* const* targ)
{
    if (!c) return EH_EINVAL;
    if (split < 0 || split > 1 || N < 0 || (N > 0 && (!X || !targ))) return fail(c, EH_EINVAL, "bad eh_upload arguments");
    if (N > 0x7fffffffLL) return fail(c, EH_EUNSUPPORTED, "split larger than 2^31-1 samples");
    EH_ENTER(c);
    Split& sp = c->split[split];
    if (sp.rec) { cudaFree(sp.rec); sp.rec = nullptr; }
    sp.N = N;
    sp.has_nan = false;
    if (split == EH_SPLIT_TRAIN) { c->perm_n = 0; c->perm_B = 0; c->idx_gen++; }
    if (N == 0) return EH_OK;
    const Variant* v = c->var;
    // numerically convenient shifts + NaN census on the host (one pass over the targets)
    for (int t = 0; t < c->n_targ; t++) {
        double s = 0; int64_t n = 0;
        for (int64_t i = 0; i < N; i++) { float y = targ[t][i]; if (y == y) { s += y; n++; } else sp.has_nan = true; }
        sp.shift_y[t] = n ? (float)(s / (double)n) : 0.f;
    }
    if (c->use_bn) {
        for (int k = 0; k < c->real_in; k++) {
            double s = 0;
            int col = c->src_idx[k];
            for (int64_t i = 0; i < N; i++) s += X[(size_t)i * c->n_pred_raw + col];
            sp.shift_x[k] = (float)(s / (double)N);
        }
    }
    float *dX = nullptr, *dP = nullptr;
    size_t nplanes = (size_t)(c->n_forc_raw + c->n_targ);
    CK(dalloc(&sp.rec, (size_t)N * v->R4));
    CK(dalloc(&dX, (size_t)N * c->n_pred_raw));
    CK(dalloc(&dP, (size_t)N * nplanes));
    CK(cudaMemcpyAsync(dX, X, (size_t)N * c->n_pred_raw * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    for (int f = 0; f < c->n_forc_raw; f++)
        CK(cudaMemcpyAsync(dP + (size_t)f * N, forc[f], (size_t)N * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    for (int t = 0; t < c->n_targ; t++)
        CK(cudaMemcpyAsync(dP + (size_t)(c->n_forc_raw + t) * N, targ[t], (size_t)N * sizeof(float), cudaMemcpyHostToDevice,
                           c->stream));
    PackArgs p;
    memset(&p, 0, sizeof p);
    p.X = dX; p.planes = dP; p.N = N; p.P_raw = c->n_pred_raw; p.ncols = c->ncols; p.R4 = v->R4;
    for (int i = 0; i < c->ncols; i++) { p.src_kind[i] = c->src_kind[i]; p.src_idx[i] = c->src_idx[i]; }
    p.rec = sp.rec; p.rec_base = 0;
    k_pack<<<(unsigned)((N + 255) / 256), 256, 0, c->stream>>>(p);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(c->stream));
    cudaFree(dX);
    cudaFree(dP);
    return EH_OK;
}

eh_status eh_set_params(eh_ctx* c, const float* flat, int64_t n)
{
    if (!c) return EH_EINVAL;
    if (!flat || n != c->nflat) return fail(c, EH_EINVAL, "eh_set_params: expected %d entries, got %lld", c->nflat, (long long)n);
    EH_ENTER(c);
    CK(cudaMemcpyAsync(c->d_theta, flat, (size_t)n * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    CK(refresh_tail(c));
    if (c->wide && c->wide->refresh_images(c->d_theta, c->d_m, c->d_v, c->d_ost, c->stream) != cudaSuccess)
        return fail(c, EH_ECUDA, "wide path: %s", c->wide->error());
    CK(cudaStreamSynchronize(c->stream));
    return EH_OK;
}

eh_status eh_get_params(eh_ctx* c, float* flat, int64_t n)
{
    if (!c) return EH_EINVAL;
    if (!flat || n != c->nflat) return fail(c, EH_EINVAL, "eh_get_params: expected %d entries, got %lld", c->nflat, (long long)n);
    EH_ENTER(c);
    CK(cudaMemcpyAsync(flat, c->d_theta, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return EH_OK;
}

eh_status eh_set_opt_state(eh_ctx* c, const float* m, const float* v, int64_t n, int64_t t)
{
    if (!c) return EH_EINVAL;
    if (n != c->nflat || t < 0) return fail(c, EH_EINVAL, "eh_set_opt_state: bad size or step count");
    EH_ENTER(c);
    eh_status s = reset_opt_state(c);
    if (s != EH_OK) return s;
    if (m) CK(cudaMemcpy(c->d_m, m, (size_t)n * sizeof(float), cudaMemcpyHostToDevice));
    if (v) CK(cudaMemcpy(c->d_v, v, (size_t)n * sizeof(float), cudaMemcpyHostToDevice));
    OptState os;
    os.b1t = c->beta1; os.b2t = c->beta2; os.t = t; os.skipped = 0;
    for (int64_t i = 0; i < t; i++) { os.b1t *= c->beta1; os.b2t *= c->beta2; }
    CK(cudaMemcpy(c->d_ost, &os, sizeof os, cudaMemcpyHostToDevice));
    return EH_OK;
}

eh_status eh_get_opt_state(eh_ctx* c, float* m, float* v, int64_t n, int64_t* t)
{
    if (!c) return EH_EINVAL;
    if (n != c->nflat) return fail(c, EH_EINVAL, "eh_get_opt_state: bad size");
    EH_ENTER(c);
    CK(cudaStreamSynchronize(c->stream));
    if (m) CK(cudaMemcpy(m, c->d_m, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost));
    if (v) CK(cudaMemcpy(v, c->d_v, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost));
    if (t) {
        OptState os;
        CK(cudaMemcpy(&os, c->d_ost, sizeof os, cudaMemcpyDeviceToHost));
        *t = os.t;
    }
    return EH_OK;
}

eh_status eh_set_bn_state(eh_ctx* c, int32_t chain, const float* mean, const float* var, int32_t n)
{
    if (!c) return EH_EINVAL;
    if (chain < 0 || chain >= c->n_chains || n != c->chain_nin[chain] || !mean || !var)
        return fail(c, EH_EINVAL, "eh_set_bn_state: chain %d has %d inputs (got n=%d)", chain, chain >= 0 && chain < c->n_chains ? c->chain_nin[chain] : -1, n);
    EH_ENTER(c);
    CK(cudaStreamSynchronize(c->stream));   // steps in flight may still fold their batch moments in (eh_sync does that)
    const int o = c->chain_in0[chain];
    for (int i = 0; i < n; i++) { c->bn_mean[o + i] = mean[i]; c->bn_var[o + i] = var[i]; }
    return EH_OK;
}

eh_status eh_get_bn_state(eh_ctx* c, int32_t chain, float* mean, float* var, int32_t n)
{
    if (!c) return EH_EINVAL;
    if (chain < 0 || chain >= c->n_chains || n != c->chain_nin[chain] || !mean || !var)
        return fail(c, EH_EINVAL, "eh_get_bn_state: chain %d has %d inputs (got n=%d)", chain, chain >= 0 && chain < c->n_chains ? c->chain_nin[chain] : -1, n);
    if (!c->pending_bn.empty()) {   // host batches still in flight: their moments belong to the state that is asked for
        eh_status s = eh_sync(c);
        if (s != EH_OK) return s;
    }
    const int o = c->chain_in0[chain];
    for (int i = 0; i < n; i++) { mean[i] = c->bn_mean[o + i]; var[i] = c->bn_var[o + i]; }
    return EH_OK;
}

static eh_status step_on_indices(eh_ctx* c, const int64_t* idx1, int64_t B, float* loss_out, float* grad_out, int apply)
{
    if (!c) return EH_EINVAL;
    if (!idx1 || B <= 0) return fail(c, EH_EINVAL, "empty batch");
    EH_ENTER(c);
    const Split& sp = c->split[EH_SPLIT_TRAIN];
    if (!sp.rec) return fail(c, EH_EINVAL, "train split not uploaded");
    eh_status s = upload_indices(c, idx1, B, sp.N);
    if (s != EH_OK) return s;
    c->perm_n = 0; c->perm_B = 0;  // the resident index stream was overwritten
    s = prepare_batch_rows(c, B, B);
    if (s != EH_OK) return s;
    float L = 0.f;
    s = run_steps(c, B, B, 0, 1, &L, apply, grad_out);
    if (s != EH_OK) return s;
    if (loss_out) *loss_out = L;
    return EH_OK;
}

eh_status eh_loss_grad(eh_ctx* c, const int64_t* idx1, int64_t B, float* loss_out, float* grad_out)
{
    return step_on_indices(c, idx1, B, loss_out, grad_out, 0);
}

eh_status eh_step(eh_ctx* c, const int64_t* idx1, int64_t B, float* loss_out, float* grad_out)
{
    return step_on_indices(c, idx1, B, loss_out, grad_out, 1);
}

eh_status eh_set_perm(eh_ctx* c, const int64_t* perm1, int64_t n)
{
    if (!c) return EH_EINVAL;
    if (!perm1 || n <= 0) return fail(c, EH_EINVAL, "empty permutation");
    EH_ENTER(c);
    const Split& sp = c->split[EH_SPLIT_TRAIN];
    if (!sp.rec) return fail(c, EH_EINVAL, "train split not uploaded");
    eh_status s = upload_indices(c, perm1, n, sp.N);
    if (s != EH_OK) return s;
    c->perm_n = n;
    c->perm_B = 0;
    return EH_OK;
}

eh_status eh_run_steps(eh_ctx* c, int64_t B, int64_t first_step, int64_t n_steps, float* losses)
{
    if (!c) return EH_EINVAL;
    if (c->perm_n <= 0) return fail(c, EH_EINVAL, "no resident permutation (call eh_set_perm)");
    if (B <= 0) return fail(c, EH_EINVAL, "batch size must be positive");
    EH_ENTER(c);
    if (c->perm_B != B) {
        eh_status s = prepare_batch_rows(c, c->perm_n, B);
        if (s != EH_OK) return s;
        c->perm_B = B;
    }
    return run_steps(c, c->perm_n, B, first_step, n_steps, losses, 1, nullptr);
}

eh_status eh_epoch(eh_ctx* c, const int64_t* perm1, int64_t n, int64_t B, float* losses)
{
    if (!c) return EH_EINVAL;
    if (!perm1 || n <= 0) return fail(c, EH_EINVAL, "empty permutation");
    if (B <= 0) return fail(c, EH_EINVAL, "batch size must be positive");
    EH_ENTER(c);
    bool piped = false;
    eh_status ps = epoch_pipelined(c, perm1, n, B, losses, &piped);
    if (ps != EH_OK || piped) return ps;
    eh_status s = eh_set_perm(c, perm1, n);
    if (s != EH_OK) return s;
    if (B <= 0) return fail(c, EH_EINVAL, "batch size must be positive");
    return eh_run_steps(c, B, 0, (n + B - 1) / B, losses);
}

eh_status eh_step_host(eh_ctx* c, int64_t B, const float* X, const float* const* forc, const float* const* targ,
                       float* loss_out)
{
    if (!c) return EH_EINVAL;
    if (B <= 0 || !X || !targ) return fail(c, EH_EINVAL, "bad eh_step_host arguments");
    EH_ENTER(c);
    HostStage& h = c->hs[0];
    eh_status s = ensure_host_stage(c, h, B);
    if (s != EH_OK) return s;
    if (c->use_bn && !c->h_bn0) CK(cudaMallocHost((void**)&c->h_bn0, 2 * MAXP * sizeof(float)));
    s = enqueue_host_step(c, h, B, X, forc, targ, h.d_loss, c->h_bn0);
    if (s != EH_OK) return s;
    float L = 0.f;
    CK(cudaMemcpyAsync(&L, h.d_loss, sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    if (loss_out) *loss_out = L;
    // Lux updates the running statistics of the input BatchNorm on every training step (momentum 0.1)
    if (c->use_bn && !c->wide) fold_bn_host_batch(c, c->h_bn0, B, L);
    return EH_OK;
}

eh_status eh_step_host_async(eh_ctx* c, int64_t B, const float* X, const float* const* forc, const float* const* targ,
                             float* loss_slot)
{
    if (!c) return EH_EINVAL;
    if (B <= 0 || !X || !targ) return fail(c, EH_EINVAL, "bad eh_step_host_async arguments");
    CK(cudaSetDevice(c->device));   // (no flush: this call adds to the open group)
    if (c->async_used == c->async_cap) {
        if (c->async_used) {
            eh_status s = eh_sync(c);
            if (s != EH_OK) return s;
        }
        if (!c->h_async_loss) {
            c->async_cap = 4096;
            CK(cudaMallocHost((void**)&c->h_async_loss, c->async_cap * sizeof(float)));
            if (c->use_bn) CK(cudaMallocHost((void**)&c->h_async_bn, c->async_cap * 2 * MAXP * sizeof(float)));
        }
    }
    {
        // grouped form: the batch is packed now, its step runs with the group's persistent launch
        bool taken = false;
        eh_status rs = ring_enqueue(c, B, X, forc, targ, c->h_async_loss + c->async_used, &taken);
        if (rs != EH_OK) return rs;
        if (taken) {
            c->pending_loss.emplace_back(c->h_async_loss + c->async_used, loss_slot);
            c->async_used++;
            return EH_OK;
        }
        rs = flush_host_group(c);   // keep the order of the steps
        if (rs != EH_OK) return rs;
    }
    HostStage& h = c->hs[c->hs_next];
    c->hs_next = (c->hs_next + 1) % EH_HOST_SLOTS;
    if (B > h.cap && h.used) {
        // growing a slot frees its buffers: nothing may still be reading them
        CK(cudaStreamSynchronize(c->stream));
        for (int i = 0; i < EH_NPACK; i++) CK(cudaStreamSynchronize(c->pack_stream[i]));
    }
    eh_status s = ensure_host_stage(c, h, B);
    if (s != EH_OK) return s;
    // the update kernel stores the loss straight into the page-locked ring (device-visible under UVA):
    // the device->host read of the step's result costs no extra enqueue
    float* bnp = c->h_async_bn ? c->h_async_bn + c->async_used * 2 * MAXP : nullptr;
    float* pin = c->h_async_loss + c->async_used++;
    s = enqueue_host_step(c, h, B, X, forc, targ, pin, bnp);
    if (s != EH_OK) return s;
    c->pending_loss.emplace_back(pin, loss_slot);
    if (c->use_bn && !c->wide && bnp) c->pending_bn.push_back({pin, bnp, B});
    return EH_OK;
}

eh_status eh_sync(eh_ctx* c)
{
    if (!c) return EH_EINVAL;
    EH_ENTER(c);
    unsigned herr = 0;
    CK(cudaMemcpyAsync(&herr, c->d_dperr, sizeof(unsigned), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    if (herr) {
        cudaMemset(c->d_dperr, 0, sizeof(unsigned));
        return fail(c, EH_ENCCL, "persistent kernel gave up waiting (a CTA or a data-parallel peer never arrived)");
    }
    for (auto& pr : c->pending_loss)
        if (pr.second) *pr.second = *pr.first;
    c->pending_loss.clear();
    c->ring.limit = 1;   // the next burst ramps its group sizes up again
    c->ring.launches = 0;
    if (const char* e = getenv("EH_RING_RAMP")) c->ring.limit = std::max(1, std::min(atoi(e), EH_RING_GROUP));
    // the retired host batches' BatchNorm moments, in step order (Lux: running statistics move on every training step)
    for (auto& pb : c->pending_bn) fold_bn_host_batch(c, pb.mom, pb.B, *pb.loss);
    c->pending_bn.clear();
    c->async_used = 0;
    return EH_OK;
}

eh_status eh_eval(eh_ctx* c, int32_t split, float* yhat, double* stats, float* nn_out)
{
    if (!c) return EH_EINVAL;
    if (split < 0 || split > 1) return fail(c, EH_EINVAL, "bad split");
    EH_ENTER(c);
    const Split& sp = c->split[split];
    if (!sp.rec) return fail(c, EH_EINVAL, "split %d not uploaded", split);
    const Variant* v = c->var;
    const int64_t N = sp.N;
    // temporaries are released on every exit path (the CK macro returns early)
    struct Scoped {
        void* p = nullptr;
        ~Scoped() { if (p) cudaFree(p); }
    } g_yhat, g_par, g_acc;
    float *d_yhat = nullptr, *d_par = nullptr;
    if (yhat) CK(dalloc(&d_yhat, (size_t)N * v->T));
    g_yhat.p = d_yhat;
    if (nn_out) CK(dalloc(&d_par, (size_t)N * v->NPS));
    g_par.p = d_par;
    EvalArgs a;
    memset(&a, 0, sizeof a);
    a.rec = reinterpret_cast<const float4*>(sp.rec);
    a.rec_base = 0; a.N = N; a.pblock = c->d_theta; a.nflat = c->nflat; a.wsrc = c->d_wsrc;
    a.use_bn = c->use_bn; a.prog = c->d_prog; a.scale_rt = c->scale_rt;
    for (int l = 0; l < 3; l++) a.pass_mask[l] = c->pass_mask[l];
    if (c->use_bn) {
        // test mode: running statistics (LuxCore.testmode(st), compute_loss.jl:37)
        float row[BS_STRIDE];
        memset(row, 0, sizeof row);
        for (int k = 0; k < c->real_in; k++) {
            row[BS_BN + 2 * k] = c->bn_mean[k];
            row[BS_BN + 2 * k + 1] = 1.0f / std::sqrt(c->bn_var[k] + 1e-5f);
        }
        CK(cudaMemcpyAsync(c->d_bn_test, row, sizeof row, cudaMemcpyHostToDevice, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        a.bscal = c->d_bn_test;
    }
    for (int s = 0; s < MAXPS; s++) a.slot[s] = c->slots[s];
    for (int i = 0; i < 4; i++) a.pmc[i] = c->pmc[i];
    for (int t = 0; t < MAXT; t++) a.shift_y[t] = sp.shift_y[t];
    a.yhat = d_yhat; a.parout = d_par; a.partial = c->d_evalpart;
    if (c->wide) {
        // wide chains: forward GEMMs over chunks of rows, statistics accumulated on the device
        double* d_acc = nullptr;
        CK(dalloc(&d_acc, (size_t)MAXT * EVAL_NSTAT));
        g_acc.p = d_acc;
        CK(cudaMemsetAsync(d_acc, 0, MAXT * EVAL_NSTAT * sizeof(double), c->stream));
        CK(cudaEventRecord(c->ev0, c->stream));
        const int64_t chunk = c->wide->eval_chunk();
        for (int64_t r0 = 0; r0 < N; r0 += chunk) {
            const int bc = (int)std::min<int64_t>(chunk, N - r0);
            if (c->wide->eval_rows(sp.rec, N, r0, bc, a.bscal, c->d_theta, d_yhat, d_par, N, d_acc, sp.shift_y, c->stream) != cudaSuccess) {
                return fail(c, EH_ECUDA, "wide path: %s", c->wide->error());
            }
        }
        CK(cudaEventRecord(c->ev1, c->stream));
        double acc[MAXT * EVAL_NSTAT];
        CK(cudaMemcpyAsync(acc, d_acc, sizeof acc, cudaMemcpyDeviceToHost, c->stream));
        if (yhat) CK(cudaMemcpyAsync(yhat, d_yhat, (size_t)N * v->T * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        CK(cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1));
        if (nn_out) {
            for (int pi = 0; pi < c->nparam_desc; pi++) {
                int s = c->slot_of_param[pi];
                if (s < 0 || c->slots[s].role != ROLE_NEURAL) continue;
                CK(cudaMemcpy(nn_out + (size_t)pi * N, d_par + (size_t)s * N, (size_t)N * sizeof(float), cudaMemcpyDeviceToHost));
            }
        }
        if (stats)
            for (int t = 0; t < v->T; t++) {
                for (int q = 0; q < EVAL_NSTAT; q++) stats[(size_t)t * EH_EVAL_STATS + q] = acc[t * EVAL_NSTAT + q];
                stats[(size_t)t * EH_EVAL_STATS + 8] = sp.shift_y[t];
            }
        return EH_OK;
    }
    const int nwarps = 8;
    int64_t nchunks = (N + CHUNK - 1) / CHUNK;
    int grid = (int)std::min<int64_t>((nchunks + nwarps - 1) / nwarps, (int64_t)c->nsm * 4);
    if (grid < 1) grid = 1;
    size_t smem = (size_t)(rup4(v->NW) + SS_FLOATS) * 4;
    CK(cudaEventRecord(c->ev0, c->stream));
    CK(vlaunch_eval(c, v, a, grid, nwarps, smem, c->stream));
    CK(cudaEventRecord(c->ev1, c->stream));
    std::vector<double> part((size_t)grid * v->T * EVAL_NSTAT);
    CK(cudaMemcpyAsync(part.data(), c->d_evalpart, part.size() * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    if (yhat) CK(cudaMemcpyAsync(yhat, d_yhat, (size_t)N * c->n_targ * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaEventElapsedTime(&c->last_ms, c->ev0, c->ev1));
    c->last_launches = 1;
    if (nn_out) {
        // rows of nn_out are indexed by the descriptor's parameter order
        for (int pi = 0; pi < c->nparam_desc; pi++) {
            int s = c->slot_of_param[pi];
            if (s < 0 || c->slots[s].role != ROLE_NEURAL) continue;
            CK(cudaMemcpy(nn_out + (size_t)pi * N, d_par + (size_t)s * N, (size_t)N * sizeof(float), cudaMemcpyDeviceToHost));
        }
    }
    if (stats) {
        for (int t = 0; t < c->n_targ; t++) {   // (the generic variants carry unused, always-masked target columns)
            for (int q = 0; q < EVAL_NSTAT; q++) {
                double s = 0;
                for (int g = 0; g < grid; g++) s += part[(size_t)g * v->T * EVAL_NSTAT + t * EVAL_NSTAT + q];
                stats[(size_t)t * EH_EVAL_STATS + q] = s;
            }
            stats[(size_t)t * EH_EVAL_STATS + 8] = sp.shift_y[t];
        }
    }
    return EH_OK;
}

eh_status eh_comm_id(eh_ctx* c, void* id_out)
{
    if (!c) return EH_EINVAL;
    if (!id_out) return fail(c, EH_EINVAL, "null id_out");
    EH_ENTER(c);
    if (!c->dp_block) {
        const size_t bytes = c->wide ? c->wide->dp_block_bytes()                                            // [2][xlen] floats + flags
                                     : (size_t)2 * EH_MAX_WORLD * rup4(c->var->NPART) * sizeof(uint2);  // {value, tag} slots
        CK(cudaMalloc(&c->dp_block, bytes));
        CK(cudaMemset(c->dp_block, 0, bytes));
    }
    static_assert(sizeof(cudaIpcMemHandle_t) <= EH_COMM_ID_BYTES, "IPC handle does not fit the id blob");
    cudaIpcMemHandle_t h;
    CK(cudaIpcGetMemHandle(&h, c->dp_block));
    memset(id_out, 0, EH_COMM_ID_BYTES);
    memcpy(id_out, &h, sizeof h);
    return EH_OK;
}

eh_status eh_comm_init(eh_ctx* c, int32_t rank, int32_t world, const void* ids)
{
    if (!c) return EH_EINVAL;
    if (world < 1 || world > EH_MAX_WORLD || rank < 0 || rank >= world || !ids)
        return fail(c, EH_EINVAL, "eh_comm_init: world must be 1..%d and 0 <= rank < world", EH_MAX_WORLD);
    if (!c->dp_block) return fail(c, EH_EINVAL, "eh_comm_init: call eh_comm_id on this ctx first");
    if (!c->persist_ok && !c->wide) return fail(c, EH_EUNSUPPORTED, "data-parallel mode needs the persistent kernel, unavailable for this model");
    // (the seeds of these losses need statistics of the GLOBAL batch's predictions, which the ranks do not exchange)
    if (c->wide && (c->stat_loss || c->l2_on))
        return fail(c, EH_EUNSUPPORTED, "data-parallel mode on the tensor-core path: rmse over several targets, pearsonLoss, kgeLoss, "
                                        "pbkgeLoss and weight_l2 train on one GPU only");
    EH_ENTER(c);
    for (int r = 0; r < world; r++) {
        if (r == rank) { c->dp_peer[r] = c->dp_block; continue; }
        cudaIpcMemHandle_t h;
        memcpy(&h, reinterpret_cast<const char*>(ids) + (size_t)r * EH_COMM_ID_BYTES, sizeof h);
        cudaError_t e = cudaIpcOpenMemHandle(&c->dp_peer[r], h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess)
            return fail(c, EH_ENCCL, "cudaIpcOpenMemHandle for rank %d failed: %s (peer access over NVLink required)", r,
                        cudaGetErrorString(e));
    }
    c->rank = rank;
    c->world = world;
    c->dp_steps = 0;
    c->perm_B = 0;  // per-batch scalars depend on the world size
    return EH_OK;
}

// ---- data parallel: per-batch data statistics are statistics of the GLOBAL batch ----
static void fill_stat_args(const eh_ctx* c, StatArgs& a, int64_t n, int64_t B)
{
    const Split& sp = c->split[EH_SPLIT_TRAIN];
    memset(&a, 0, sizeof a);
    a.rec = sp.rec; a.R4 = c->var->R4; a.idx = c->d_idx; a.n = n; a.Bfull = (int)B;
    a.P = c->var->P; a.F = c->var->F; a.T = c->n_targ;
    for (int t = 0; t < MAXT; t++) { a.shift_y[t] = 0.f; a.loss_kind[t] = c->loss_kind[t]; }  // common shift on every rank
    for (int k = 0; k < MAXP; k++) a.shift_x[k] = 0.f;
    a.agg_mean = c->agg_mean; a.use_bn = 1;  // input sums are always taken: the ranks must agree on the layout
    a.bscal = c->d_bscal; a.bn_batch = c->use_bn ? c->d_bn_batch : nullptr;
}

eh_status eh_dp_batch_moments(eh_ctx* c, int64_t B, double* out)
{
    if (!c) return EH_EINVAL;
    if (!out || B <= 0) return fail(c, EH_EINVAL, "bad eh_dp_batch_moments arguments");
    if (c->perm_n <= 0) return fail(c, EH_EINVAL, "no resident permutation (call eh_set_perm)");
    EH_ENTER(c);
    const int64_t n = c->perm_n, nb = (n + B - 1) / B;
    eh_status s = ensure_bscal_cap(c, (size_t)nb);
    if (s != EH_OK) return s;
    double* d_mom = nullptr;
    CK(dalloc(&d_mom, (size_t)nb * DP_MOMENTS));
    StatArgs a;
    fill_stat_args(c, a, n, B);
    a.moments = d_mom;
    k_batch_stats<<<(unsigned)nb, 256, 0, c->stream>>>(a);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, d_mom, (size_t)nb * DP_MOMENTS * sizeof(double), cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    cudaFree(d_mom);
    if (e != cudaSuccess) return fail(c, EH_ECUDA, "eh_dp_batch_moments: %s", cudaGetErrorString(e));
    return EH_OK;
}

eh_status eh_dp_set_batch_moments(eh_ctx* c, int64_t B, const double* global)
{
    if (!c) return EH_EINVAL;
    if (!global || B <= 0) return fail(c, EH_EINVAL, "bad eh_dp_set_batch_moments arguments");
    if (c->perm_n <= 0) return fail(c, EH_EINVAL, "no resident permutation (call eh_set_perm)");
    EH_ENTER(c);
    const int64_t n = c->perm_n, nb = (n + B - 1) / B;
    eh_status s = ensure_bscal_cap(c, (size_t)nb);
    if (s != EH_OK) return s;
    double* d_mom = nullptr;
    CK(dalloc(&d_mom, (size_t)nb * DP_MOMENTS));
    StatArgs a;
    fill_stat_args(c, a, n, B);
    a.use_bn = c->use_bn;
    cudaError_t e = cudaMemcpyAsync(d_mom, global, (size_t)nb * DP_MOMENTS * sizeof(double), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) {
        k_bscal_from_moments<<<(unsigned)((nb + 127) / 128), 128, 0, c->stream>>>(a, d_mom, (int)nb);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    cudaFree(d_mom);
    if (e != cudaSuccess) return fail(c, EH_ECUDA, "eh_dp_set_batch_moments: %s", cudaGetErrorString(e));
    c->perm_B = B;  // the rows of this permutation / batch size are in place
    return EH_OK;
}

const char* eh_kernel_variant(const eh_ctx* c)
{
    return (c && c->var && c->var->name) ? c->var->name : "";
}

eh_status eh_jit_check(const eh_model_desc* desc, char* info, size_t info_bytes)
{
    if (!desc) return fail(nullptr, EH_EINVAL, "null argument");
    eh_ctx* c = new (std::nothrow) eh_ctx();
    if (!c) return fail(nullptr, EH_ENOMEM, "out of host memory");
    c->nsm = 148; c->smem_optin = 232448;   // B200; the plan does not depend on a device being present
    eh_model_desc d = *desc;
    d.flags |= EH_FLAG_JIT;
    eh_status s = build_plan(c, &d);
    if (s == EH_OK && !c->jit_on) s = fail(c, EH_EUNSUPPORTED, "the planner did not choose a generic exact-fp32 variant for this model (variant %s)", c->var ? c->var->name : "?");
    if (s != EH_OK) g_create_error = c->err;
    if (s == EH_OK && info && info_bytes)
        snprintf(info, info_bytes, "%s cubin=%zu cached=%d seconds=%.2f", c->jit.name.c_str(), c->jit_cubin.size(), c->jit.from_cache ? 1 : 0, c->jit.compile_seconds);
    delete c;
    return s;
}

const char* eh_epoch_variant(const eh_ctx* c, int64_t batch)
{
    if (!c || !c->var) return "";
    const Variant* v = c->wide ? c->var : pick_epoch_variant(c, batch);
    return (v && v->name) ? v->name : "";
}

eh_status eh_host_alloc(void** out, size_t bytes)
{
    if (!out) return EH_EINVAL;
    cudaError_t e = cudaMallocHost(out, bytes ? bytes : 1);
    if (e != cudaSuccess) {
        g_create_error = std::string("cudaMallocHost: ") + cudaGetErrorString(e);
        return e == cudaErrorMemoryAllocation ? EH_ENOMEM : EH_ECUDA;
    }
    return EH_OK;
}

eh_status eh_host_free(void* p)
{
    if (p && cudaFreeHost(p) != cudaSuccess) return EH_ECUDA;
    return EH_OK;
}

eh_status eh_last_timing(eh_ctx* c, float* total_ms, int64_t* launches, float* step_kernel_ms)
{
    if (!c) return EH_EINVAL;
    if (total_ms) *total_ms = c->last_ms;
    if (launches) *launches = c->last_launches;
    if (step_kernel_ms) *step_kernel_ms = c->last_step_ms;
    return EH_OK;
}

eh_status eh_set_profiling(eh_ctx* c, int32_t on)
{
    if (!c) return EH_EINVAL;
    c->profiling = on ? 1 : 0;
    return EH_OK;
}

}  // extern "C"
