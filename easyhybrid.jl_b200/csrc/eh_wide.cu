// eh_wide.cu -- host side of the wide-hidden-layer path: TMA descriptors, GEMM launches, self-test entry.
#include <cuda_runtime.h>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/easyhybrid_cuda.h"
#include "eh_stat_seeds.cuh"
#include "eh_wide.h"
#include "eh_wide_gemm.cuh"
#include "eh_wide_kernels.cuh"

namespace eh {
namespace wide {

namespace {
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn()
{
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}
}  // namespace

// 2-D bf16 tensor map: `inner` contiguous elements per row, `rows` rows of `pitch_elems`; box = 64 x box_rows,
// 128-byte swizzle (the shared-memory layout tcgen05 descriptors expect)
bool make_map_bf16(CUtensorMap* map, const void* ptr, uint64_t inner, uint64_t rows, uint64_t pitch_elems, uint32_t box_rows)
{
    EncodeTiledFn fn = encode_fn();
    if (!fn) return false;
    cuuint64_t dims[2] = {inner, rows};
    cuuint64_t strides[1] = {pitch_elems * 2};
    cuuint32_t box[2] = {64, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}

cudaError_t gemm_prepare()
{
    static bool done = false;
    if (done) return cudaSuccess;
    cudaError_t e;
    if ((e = cudaFuncSetAttribute(k_wide_gemm<GEMM_FWD>, cudaFuncAttributeMaxDynamicSharedMemorySize, gemm_smem(GEMM_FWD))) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_wide_gemm<GEMM_BWD>, cudaFuncAttributeMaxDynamicSharedMemorySize, gemm_smem(GEMM_BWD))) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_wide_gemm<GEMM_WGRAD>, cudaFuncAttributeMaxDynamicSharedMemorySize, gemm_smem(GEMM_WGRAD))) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_wide_gemm_p<GEMM_FWD, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, PG_SMEM)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_wide_gemm_p<GEMM_BWD, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, PG_SMEM)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_wide_gemm_p<GEMM_FWD, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, PG_SMEM)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_wide_gemm_p<GEMM_BWD, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, PG_SMEM)) != cudaSuccess) return e;
    done = true;
    return cudaSuccess;
}

// out = act(A W^T + bias): A [M x K] bf16, W [N x K] bf16 (K contiguous in both)
cudaError_t gemm_fwd(const CUtensorMap& tmA, const CUtensorMap& tmW, int M, int N, int K, const float* bias, int act,
                     __nv_bfloat16* out, cudaStream_t st)
{
    GemmArgs g{};
    g.M = M; g.N = N; g.K = K; g.ksplits = 1; g.act = act; g.bias = bias; g.out16 = out;
    k_wide_gemm<GEMM_FWD><<<dim3(M / BM, N / gemm_bn(GEMM_FWD), 1), GEMM_THREADS, gemm_smem(GEMM_FWD), st>>>(tmA, tmW, g);
    return cudaGetLastError();
}
// out = (D Wt^T) .* act'(aux): D [M x K] bf16, Wt [N x K] bf16, aux [M x N] bf16
cudaError_t gemm_bwd(const CUtensorMap& tmD, const CUtensorMap& tmWt, int M, int N, int K, const __nv_bfloat16* aux, int act,
                     __nv_bfloat16* out, cudaStream_t st, float* colsum, const float* xb, const float* bscal, int R4, int P1,
                     int use_bn)
{
    GemmArgs g{};
    g.M = M; g.N = N; g.K = K; g.ksplits = 1; g.act = act; g.aux = aux; g.out16 = out;
    g.colsum = colsum; g.xb = xb; g.bscal = bscal; g.R4 = R4; g.P1 = P1; g.use_bn = use_bn;
    k_wide_gemm<GEMM_BWD><<<dim3(M / BM, N / gemm_bn(GEMM_BWD), 1), GEMM_THREADS, gemm_smem(GEMM_BWD), st>>>(tmD, tmWt, g);
    return cudaGetLastError();
}
// persistent forms (one CTA per SM, 128 x 256 tiles, double-buffered accumulator); tmW / tmWt must be built with
// box rows = pg_box_rows().  With an even number of row tiles the CTAs run
// can run as clusters of two that share the weight tile by multicast (EH_WIDE_CLUSTER=1; measured 4 us SLOWER per GEMM than
// single CTAs: the kernels are bound by shared-memory bandwidth -- TMA writes plus MMA operand reads -- not by L2 reads).
static bool pg_cluster() { static const bool on = getenv("EH_WIDE_CLUSTER") != nullptr; return on; }
int pg_box_rows() { return pg_cluster() ? PG_BN / 2 : PG_BN; }
template <int MODE>
static cudaError_t launch_gemm_p(const CUtensorMap& tmA, const CUtensorMap& tmB, const GemmArgs& g, cudaStream_t st)
{
    static int nsm = 0, max_clusters = -1;
    if (!nsm) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
    }
    const int mt = g.M / BM, nn = g.N / PG_BN;
    cudaLaunchConfig_t cfg{};
    cfg.blockDim = dim3(PG_THREADS);
    cfg.dynamicSmemBytes = PG_SMEM;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    if (pg_cluster()) {
        if (mt % 2) return cudaErrorInvalidValue;   // (the opt-in cluster form needs an even number of row tiles)
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        if (max_clusters < 0) {
            cfg.gridDim = dim3((unsigned)(nsm & ~1));
            int mc = 0;
            if (cudaOccupancyMaxActiveClusters(&mc, k_wide_gemm_p<MODE, 2>, &cfg) != cudaSuccess || mc < 1) { cudaGetLastError(); mc = 0; }
            max_clusters = mc;
        }
        if (max_clusters > 0) {
            const int units = (mt / 2) * nn;
            const int ncl = std::min(std::min(max_clusters, nsm / 2), units);
            cfg.gridDim = dim3((unsigned)(2 * ncl));
            return cudaLaunchKernelEx(&cfg, k_wide_gemm_p<MODE, 2>, tmA, tmB, g);
        }
        cfg.attrs = nullptr;
        cfg.numAttrs = 0;
    }
    cfg.gridDim = dim3((unsigned)std::min(mt * nn, nsm));
    return cudaLaunchKernelEx(&cfg, k_wide_gemm_p<MODE, 1>, tmA, tmB, g);
}
int persistent_grid(int M, int N)
{
    static int nsm = 0;
    if (!nsm) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
    }
    const int tiles = (M / BM) * (N / PG_BN);
    return tiles < nsm ? tiles : nsm;
}
cudaError_t gemm_fwd_p(const CUtensorMap& tmA, const CUtensorMap& tmW, int M, int N, int K, const float* bias, int act,
                       __nv_bfloat16* out, cudaStream_t st)
{
    GemmArgs g{};
    g.M = M; g.N = N; g.K = K; g.ksplits = 1; g.act = act; g.bias = bias; g.out16 = out;
    return launch_gemm_p<GEMM_FWD>(tmA, tmW, g, st);
}
cudaError_t gemm_bwd_p(const CUtensorMap& tmD, const CUtensorMap& tmWt, int M, int N, int K, const __nv_bfloat16* aux, int act,
                       __nv_bfloat16* out, cudaStream_t st, float* colsum, const float* xb, const float* bscal, int R4, int P1,
                       int use_bn)
{
    GemmArgs g{};
    g.M = M; g.N = N; g.K = K; g.ksplits = 1; g.act = act; g.aux = aux; g.out16 = out;
    g.colsum = colsum; g.xb = xb; g.bscal = bscal; g.R4 = R4; g.P1 = P1; g.use_bn = use_bn;
    return launch_gemm_p<GEMM_BWD>(tmD, tmWt, g, st);
}

// partial[z] = D[rows z]^T A[rows z]: D [Kall x M] bf16, A [Kall x N] bf16 (batch rows), ksplits slices of Kall
cudaError_t gemm_wgrad(const CUtensorMap& tmD, const CUtensorMap& tmA, int M, int N, int Kall, int ksplits, float* partial,
                       cudaStream_t st)
{
    GemmArgs g{};
    g.M = M; g.N = N; g.K = Kall / ksplits; g.ksplits = ksplits; g.out32 = partial;
    k_wide_gemm<GEMM_WGRAD><<<dim3(M / BM, N / gemm_bn(GEMM_WGRAD), ksplits), GEMM_THREADS, gemm_smem(GEMM_WGRAD), st>>>(tmD, tmA, g);
    return cudaGetLastError();
}


// ------------------------------------------------------------------------------------------------
// WideNet
// ------------------------------------------------------------------------------------------------
namespace {

typedef void (*HeadKernel)(const HeadArgs);
struct HeadEntry { int pm, nout, scale, hch, aff; HeadKernel fn; };
#define EH_HEAD(PMF, NOUT, SCALE, HCH, AFF) {PMF::ID, NOUT, SCALE, HCH, AFF, k_wide_head<HeadCfg<PMF, NOUT, (SCALE != 0), (AFF != 0)>, HCH>},
#define EH_HEAD_PMA(PMF, AFF) EH_HEAD(PMF, 1, 0, 1, AFF) EH_HEAD(PMF, 1, 1, 1, AFF) EH_HEAD(PMF, 2, 0, 1, AFF) EH_HEAD(PMF, 2, 1, 1, AFF) \
                              EH_HEAD(PMF, 1, 0, 2, AFF) EH_HEAD(PMF, 1, 1, 2, AFF) EH_HEAD(PMF, 2, 0, 2, AFF) EH_HEAD(PMF, 2, 1, 2, AFF)
#define EH_HEAD_PM(PMF) EH_HEAD_PMA(PMF, 0) EH_HEAD_PMA(PMF, 1)
const HeadEntry g_heads[] = {EH_HEAD_PM(PmRbQ10) EH_HEAD_PM(PmExpo) EH_HEAD_PM(PmLinear) EH_HEAD_PM(PmLinear2) EH_HEAD_PM(PmExpo2)
                             EH_HEAD_PM(PmProgram)};

// aff: the training head of a model with LOSS_AFFINE targets (the statistics and evaluation modes take aff = 0)
HeadKernel find_head(int pm, int nout, int scale, int hch, bool aff = false)
{
    for (const HeadEntry& e : g_heads)
        if (e.pm == pm && e.nout == nout && e.scale == (scale ? 1 : 0) && e.hch == hch && e.aff == (aff ? 1 : 0)) return e.fn;
    return nullptr;
}

// CTAs of k_wide_gradpost: a function of the shape only, so that its sums of theta^2 have one fixed order
int gradpost_grid(const WideModel& m) { return std::max(1, std::min((m.nflat + 255) / 256, 2 * m.nsm)); }

WideDims dims_of(const WideModel& m)
{
    WideDims d{};
    d.P = m.P; d.H = m.H; d.NH = m.NH; d.NOUT = m.NOUT; d.R4 = m.R4; d.nflat = m.nflat; d.ntheta = m.ntheta;
    return d;
}
}  // namespace

#define WN(call)                                                                                       \
    do {                                                                                               \
        cudaError_t e__ = (call);                                                                      \
        if (e__ != cudaSuccess) {                                                                      \
            snprintf(err_, sizeof err_, "%s: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return e__;                                                                                \
        }                                                                                              \
    } while (0)

bool WideNet::supported(int P, int hmax, int NH, int NOUT, int act, int pm)
{
    if (P < 1 || P > WIDE_MAXP || NH < 2 || NH > 6 || NOUT < 1 || NOUT > 2) return false;
    if (hmax < 1 || hmax > 512) return false;
    if (act != ACT_TANH && act != ACT_SIGMOID && act != ACT_RELU && act != ACT_IDENTITY) return false;
    return find_head(pm, NOUT, 0, padded_width(hmax) / 256) != nullptr;
}

WideNet* WideNet::create(const WideModel& m, char* err, size_t errlen)
{
    WideNet* w = new WideNet();
    w->m_ = m;
    w->persist_ = getenv("EH_WIDE_NO_PERSIST") == nullptr;   // persistent forward / backward-data GEMMs (default)
    auto bail = [&](const char* what, cudaError_t e) -> WideNet* {
        snprintf(err, errlen, "wide path: %s: %s", what, cudaGetErrorString(e));
        delete w;
        return nullptr;
    };
    cudaError_t e = gemm_prepare();
    if (e != cudaSuccess) return bail("gemm_prepare", e);
    for (int t = 0; t < m.T && t < 4; t++) w->affine_ |= m.loss_kind[t] == LOSS_AFFINE;
    for (int aff = 0; aff <= (w->affine_ ? 1 : 0); aff++) {
        HeadKernel hk = find_head(m.pm, m.NOUT, m.scale, m.H / 256, aff != 0);
        if (!hk) { snprintf(err, errlen, "wide path: no head kernel for this process model / shape"); delete w; return nullptr; }
        const int head_smem = (8 * (m.NOUT + 1) + m.NOUT) * m.H * (int)sizeof(float);   // warps' scratch / row rings + the output-layer weights
        e = cudaFuncSetAttribute((const void*)hk, cudaFuncAttributeMaxDynamicSharedMemorySize, head_smem);
        if (e != cudaSuccess) return bail("head smem", e);
    }
    const size_t HH = (size_t)m.H * m.H;
    const int bn = w->persist_ ? pg_box_rows() : gemm_bn(GEMM_FWD);
    // images of the embedded chain: everything outside the real entries (padding, other chains' units) stays zero
    for (int l = 1; l <= m.NH; l++) {
        if ((e = cudaMalloc(&w->Bp_[l - 1], (size_t)m.H * 4)) != cudaSuccess) return bail("cudaMalloc", e);
        cudaMemset(w->Bp_[l - 1], 0, (size_t)m.H * 4);
        if (l == 1) continue;
        if ((e = cudaMalloc(&w->Wf_[l - 1], HH * 2)) != cudaSuccess) return bail("cudaMalloc", e);
        if ((e = cudaMalloc(&w->Wb_[l - 1], HH * 2)) != cudaSuccess) return bail("cudaMalloc", e);
        cudaMemset(w->Wf_[l - 1], 0, HH * 2);
        cudaMemset(w->Wb_[l - 1], 0, HH * 2);
        if (!make_map_bf16(&w->tmWf_[l - 1], w->Wf_[l - 1], m.H, m.H, m.H, bn) ||
            !make_map_bf16(&w->tmWb_[l - 1], w->Wb_[l - 1], m.H, m.H, m.H, bn)) {
            snprintf(err, errlen, "wide path: cuTensorMapEncodeTiled failed for a weight image");
            delete w;
            return nullptr;
        }
    }
    if ((e = cudaMalloc(&w->W1img_, (size_t)WIDE_MAXP * m.H * 4)) != cudaSuccess) return bail("cudaMalloc", e);
    if ((e = cudaMalloc(&w->WOimg_, (size_t)4 * m.H * 4)) != cudaSuccess) return bail("cudaMalloc", e);
    if ((e = cudaMalloc(&w->BOimg_, 16)) != cudaSuccess) return bail("cudaMalloc", e);
    cudaMemset(w->W1img_, 0, (size_t)WIDE_MAXP * m.H * 4);
    cudaMemset(w->WOimg_, 0, (size_t)4 * m.H * 4);
    cudaMemset(w->BOimg_, 0, 16);
    {
        static_assert(sizeof(ParamMap) == 16, "ParamMap is four ints");
        if ((e = cudaMalloc(&w->d_map_, (size_t)m.nflat * sizeof(ParamMap))) != cudaSuccess) return bail("cudaMalloc", e);
        if ((e = cudaMemcpy(w->d_map_, m.h_map, (size_t)m.nflat * sizeof(ParamMap), cudaMemcpyHostToDevice)) != cudaSuccess) return bail("cudaMemcpy", e);
        std::vector<int> small;
        for (int p = 0; p < m.nflat; p++)
            if (m.h_map[4 * p] != WK_WH) small.push_back(p);
        w->n_small_ = (int)small.size();
        if ((e = cudaMalloc(&w->d_small_, small.size() * sizeof(int) + 4)) != cudaSuccess) return bail("cudaMalloc", e);
        if ((e = cudaMemcpy(w->d_small_, small.data(), small.size() * sizeof(int), cudaMemcpyHostToDevice)) != cudaSuccess) return bail("cudaMemcpy", e);
        w->m_.h_map = nullptr;   // the caller's table is not retained
    }
    if (m.pm == PM_PROGRAM) {
        static_assert(PM_MAXLEN == 48, "WideModel program arrays");
        PmProgData pd;
        memset(&pd, 0, sizeof pd);
        pd.len = m.prog_len; pd.nt = m.T; pd.nf = m.F; pd.np = m.NPS;
        for (int t = 0; t < 4; t++) pd.out[t] = m.prog_out[t];
        for (int i = 0; i < m.prog_len; i++) { pd.op[i] = m.prog_op[i]; pd.a[i] = m.prog_a[i]; pd.b[i] = m.prog_b[i]; pd.imm[i] = m.prog_imm[i]; }
        if ((e = cudaMalloc(&w->d_prog_, sizeof pd)) != cudaSuccess) return bail("cudaMalloc", e);
        if ((e = cudaMemcpy(w->d_prog_, &pd, sizeof pd, cudaMemcpyHostToDevice)) != cudaSuccess) return bail("cudaMemcpy", e);
    }
    w->n_head_ = 3 * m.nsm;   // three CTAs of the head kernel are resident per SM (80 registers)
    if (cudaStreamCreateWithFlags(&w->side_, cudaStreamNonBlocking) != cudaSuccess || cudaEventCreateWithFlags(&w->ev_wgrad_, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&w->ev_wred_, cudaEventDisableTiming) != cudaSuccess) {
        cudaGetLastError();
        if (w->side_) cudaStreamDestroy(w->side_);
        w->side_ = nullptr;   // no side stream: the reductions stay on the main stream
    }
    if ((e = cudaMalloc(&w->head_partial_, (size_t)w->n_head_ * head_npart(m.H, m.NOUT) * 4)) != cudaSuccess) return bail("cudaMalloc", e);
    if ((e = cudaMalloc(&w->stats_, 16 * 4)) != cudaSuccess) return bail("cudaMalloc", e);
    if ((e = cudaMalloc(&w->skip_, 4)) != cudaSuccess) return bail("cudaMalloc", e);
    if ((e = cudaMalloc(&w->evalpart_, (size_t)w->n_head_ * 4 * 8 * sizeof(double))) != cudaSuccess) return bail("cudaMalloc", e);
    cudaMemset(w->skip_, 0, 4);
    for (int t = 0; t < m.T && t < 4; t++) w->post_ |= m.loss_kind[t] == LOSS_RMSE;
    if (m.d_l2coef) {
        w->post_ = true;
        if ((e = cudaMalloc(&w->l2part_, (size_t)gradpost_grid(m) * 4)) != cudaSuccess) return bail("cudaMalloc", e);
        if ((e = cudaMalloc(&w->ticket_, 4)) != cudaSuccess) return bail("cudaMalloc", e);
        cudaMemset(w->ticket_, 0, 4);
    }
    return w;
}

WideNet::~WideNet()
{
    if (side_) { cudaStreamSynchronize(side_); cudaStreamDestroy(side_); }
    if (ev_wgrad_) cudaEventDestroy(ev_wgrad_);
    if (ev_wred_) cudaEventDestroy(ev_wred_);
    for (int i = 0; i < 8; i++) {
        if (A_[i]) cudaFree(A_[i]);
        if (Wf_[i]) cudaFree(Wf_[i]);
        if (Wb_[i]) cudaFree(Wb_[i]);
        if (Bp_[i]) cudaFree(Bp_[i]);
        if (colsum_[i]) cudaFree(colsum_[i]);
    }
    void* ps[] = {xb_, D_[0], D_[1], partial_, head_partial_, stats_, skip_, evalpart_, l2part_, ticket_, d_prog_, W1img_, WOimg_, BOimg_,
                  d_map_, d_small_};
    for (void* p : ps)
        if (p) cudaFree(p);
}

// activation / delta buffers and their tensor maps for batches of B rows
cudaError_t WideNet::ensure(int B)
{
    const int H = m_.H;
    if (B > cap_) {
        for (int i = 0; i < 8; i++) { if (A_[i]) cudaFree(A_[i]); A_[i] = nullptr; if (colsum_[i]) cudaFree(colsum_[i]); colsum_[i] = nullptr; }
        for (int i = 0; i < 2; i++) { if (D_[i]) cudaFree(D_[i]); D_[i] = nullptr; }
        if (xb_) cudaFree(xb_);
        if (partial_) cudaFree(partial_);
        xb_ = nullptr; partial_ = nullptr; cap_ = 0; mapB_ = 0;
        WN(cudaMalloc(&xb_, (size_t)B * m_.R4 * 4));
        for (int l = 1; l <= m_.NH; l++) WN(cudaMalloc(&A_[l - 1], (size_t)B * H * 2));
        for (int i = 0; i < 2; i++) WN(cudaMalloc(&D_[i], (size_t)B * H * 2));
        WN(cudaMalloc(&partial_, (size_t)16 * H * H * 4));
        const int slabs = (B + 127) / 128;
        for (int l = 1; l < m_.NH; l++) WN(cudaMalloc(&colsum_[l - 1], (size_t)slabs * (1 + (l == 1 ? m_.P : 0)) * H * 4));
        cap_ = B;
    }
    if (B != mapB_) {
        bool ok = true;
        for (int l = 1; l <= m_.NH; l++) {
            ok &= make_map_bf16(&tmA_k_[l - 1], A_[l - 1], H, B, H, BM);
            ok &= make_map_bf16(&tmA_mn_[l - 1], A_[l - 1], H, B, H, BK);
        }
        for (int i = 0; i < 2; i++) {
            ok &= make_map_bf16(&tmD_k_[i], D_[i], H, B, H, BM);
            ok &= make_map_bf16(&tmD_mn_[i], D_[i], H, B, H, BK);
        }
        if (!ok) { snprintf(err_, sizeof err_, "cuTensorMapEncodeTiled failed"); return cudaErrorUnknown; }
        mapB_ = B;
        n_slab_ = (B + 127) / 128;
        ksplit_ = 1;
        for (int s : {16, 8, 4, 2})
            if (B % (s * BK) == 0) { ksplit_ = s; break; }
    }
    return cudaSuccess;
}

cudaError_t WideNet::refresh_images(float* pblock, float* m, float* v, void* ost, cudaStream_t st)
{
    WUpdArgs u{};
    u.d = dims_of(m_);
    u.theta = pblock; u.m = m; u.v = v; u.ost = reinterpret_cast<OptState*>(ost);
    u.skip = skip_;
    u.map = reinterpret_cast<const ParamMap*>(d_map_);
    u.W1img = W1img_; u.WOimg = WOimg_; u.BOimg = BOimg_;
    for (int l = 1; l <= m_.NH; l++) { u.Wf[l - 1] = Wf_[l - 1]; u.Wb[l - 1] = Wb_[l - 1]; u.Bp[l - 1] = Bp_[l - 1]; }
    u.apply = 0;
    k_wide_update<<<(m_.nflat + 255) / 256, 256, 0, st>>>(u);
    WN(cudaGetLastError());
    return cudaSuccess;
}

cudaError_t WideNet::forward(const float* rec, const int* idx, long long rec_base, long long nrec, int B, int Bvalid,
                             const float* bscal, const float* pblock, cudaStream_t st)
{
    const int H = m_.H;
    const WideDims d = dims_of(m_);
    k_wide_gather<<<(B + 255) / 256, 256, 0, st>>>(reinterpret_cast<const float4*>(rec), idx, rec_base, nrec, B, Bvalid, m_.R4 / 4,
                                                   reinterpret_cast<float4*>(xb_));
    WN(cudaGetLastError());
    const int rows_per_cta = (256 / (H / 8)) * FIRST_ROWS;
    {
        const unsigned g1 = (unsigned)((B + rows_per_cta - 1) / rows_per_cta);
        if (d.P <= 2) k_wide_first<2><<<g1, 256, 0, st>>>(xb_, W1img_, Bp_[0], bscal, m_.use_bn, d, B, m_.act, A_[0]);
        else if (d.P <= 4) k_wide_first<4><<<g1, 256, 0, st>>>(xb_, W1img_, Bp_[0], bscal, m_.use_bn, d, B, m_.act, A_[0]);
        else k_wide_first<8><<<g1, 256, 0, st>>>(xb_, W1img_, Bp_[0], bscal, m_.use_bn, d, B, m_.act, A_[0]);
    }
    WN(cudaGetLastError());
    for (int l = 2; l <= m_.NH; l++) {
        if (persist_) WN(gemm_fwd_p(tmA_k_[l - 2], tmWf_[l - 1], B, H, H, Bp_[l - 1], m_.act, A_[l - 1], st));
        else WN(gemm_fwd(tmA_k_[l - 2], tmWf_[l - 1], B, H, H, Bp_[l - 1], m_.act, A_[l - 1], st));
    }
    return cudaSuccess;
}

cudaError_t WideNet::step(const float* rec, const int* idx, long long rec_base, int Bvalid, float* bscal, float* pblock,
                          float* m, float* v, void* ost, float* grad_final, float* loss_out, int apply, cudaStream_t st,
                          const WideDp* dp, const float* shift_y)
{
    const int H = m_.H, NH = m_.NH;
    const int B = (Bvalid + 127) / 128 * 128;   // GEMM tiles are 128 rows: padded rows are masked in the head kernel
    const bool isdp = dp && dp->world > 1;
    const int par = isdp ? (int)(dp->tag & 1u) : 0;
    // data parallel: this rank's gradient goes into its exchange block, the all-reduce leaves the sum in grad_final
    float* grad = isdp ? dp->peer[dp->rank] + (size_t)par * dp_xlen() : grad_final;
    WN(ensure(B));
    WN(forward(rec, idx, rec_base, 1ll << 62, B, Bvalid, bscal, pblock, st));
    const WideDims d = dims_of(m_);
    HeadKernel hk = find_head(m_.pm, m_.NOUT, m_.scale, H / 256, affine_);
    HeadArgs ha{};
    ha.A = A_[NH - 1]; ha.xb = xb_; ha.pblock = pblock; ha.WOimg = WOimg_; ha.BOimg = BOimg_; ha.bscal = bscal; ha.D = D_[NH & 1];
    ha.partial = head_partial_;
    ha.d = d; ha.B = B; ha.Bvalid = Bvalid; ha.act = m_.act; ha.train = 1;
    ha.prog = reinterpret_cast<const PmProgData*>(d_prog_); ha.nf = m_.F; ha.nt = m_.T;
    for (int t = 0; t < 4; t++) ha.loss_kind[t] = m_.loss_kind[t];
    for (int s = 0; s < 8; s++) { ha.slot[s].role = m_.slot[s].role; ha.slot[s].idx = m_.slot[s].idx; ha.slot[s].lo = m_.slot[s].lo; ha.slot[s].span = m_.slot[s].span; ha.slot[s].fixedv = m_.slot[s].fixedv; }
    for (int i = 0; i < 4; i++) ha.pmc[i] = m_.pmc[i];
    const int head_smem = (8 * (m_.NOUT + 1) + m_.NOUT) * H * (int)sizeof(float);
    if (affine_) {
        // prediction-statistics losses: the head kernel's statistics mode over the training forward (train-mode
        // BatchNorm is in A_NH already) leaves per-CTA sufficient statistics of the batch; k_stat_seeds turns them into
        // the seed coefficients and the loss value in the batch's scalar row, which the training head reads next
        if (!shift_y) { snprintf(err_, sizeof err_, "step: prediction-statistics losses need the train split's shift_y"); return cudaErrorInvalidValue; }
        HeadArgs hs = ha;
        hs.train = 0; hs.D = nullptr; hs.partial = nullptr; hs.yhat = nullptr; hs.parout = nullptr; hs.ldy = 0; hs.row0 = 0;
        hs.evalstat = evalpart_;
        for (int t = 0; t < 4; t++) hs.shift_y[t] = shift_y[t];
        find_head(m_.pm, m_.NOUT, m_.scale, H / 256)<<<n_head_, 256, head_smem, st>>>(hs);
        WN(cudaGetLastError());
        StatSeedArgs z{};
        z.partial = evalpart_; z.nparts = n_head_; z.Tk = m_.T; z.T = m_.T; z.agg_mean = m_.agg_mean; z.bscal = bscal;
        for (int t = 0; t < 4; t++) { z.kind[t] = m_.loss_kind[t] == LOSS_AFFINE ? m_.loss_kind_abi[t] : -1; z.shift_y[t] = shift_y[t]; }
        k_stat_seeds<<<1, 32, 0, st>>>(z);
        WN(cudaGetLastError());
    }
    hk<<<n_head_, 256, head_smem, st>>>(ha);
    WN(cudaGetLastError());
    const bool fork = side_ != nullptr && !getenv("EH_WIDE_NO_SIDE_STREAM");
    bool pending = false;   // a split-K reduction is in flight on the side stream (it reads partial_, it writes grad)
    for (int l = NH; l >= 2; l--) {
        const int cur = l & 1, nxt = (l - 1) & 1;
        if (pending) { WN(cudaStreamWaitEvent(st, ev_wred_, 0)); pending = false; }   // partial_ is free again
        WN(gemm_wgrad(tmD_mn_[cur], tmA_mn_[l - 2], H, H, B, ksplit_, partial_, st));
        cudaStream_t rs = st;
        if (fork) {
            WN(cudaEventRecord(ev_wgrad_, st));
            WN(cudaStreamWaitEvent(side_, ev_wgrad_, 0));
            rs = side_;
        }
        for (int bi = 0; bi < m_.n_blocks; bi++) {
            const auto& bk = m_.blocks[bi];
            if (bk.l != l) continue;
            k_wide_wreduce<<<dim3((bk.hin + 31) / 32, (bk.hout + 31) / 32), 256, 0, rs>>>(partial_, ksplit_, H, bk.hout, bk.hin, bk.o_off,
                                                                                     bk.i_off, grad + bk.flat_off);
            WN(cudaGetLastError());
        }
        if (fork) { WN(cudaEventRecord(ev_wred_, side_)); pending = true; }
        // backward data; its epilogue also leaves the 32-row column sums of D_{l-1} (bias gradient of layer l-1 and,
        // for layer 1, the x-weighted sums = its weight gradient)
        if (persist_)
            WN(gemm_bwd_p(tmD_k_[cur], tmWb_[l - 1], B, H, H, A_[l - 2], m_.act, D_[nxt], st, colsum_[l - 2], xb_, bscal, m_.R4,
                          (l - 1 == 1) ? m_.P : 0, m_.use_bn));
        else
            WN(gemm_bwd(tmD_k_[cur], tmWb_[l - 1], B, H, H, A_[l - 2], m_.act, D_[nxt], st, colsum_[l - 2], xb_, bscal, m_.R4,
                        (l - 1 == 1) ? m_.P : 0, m_.use_bn));
    }
    if (pending) WN(cudaStreamWaitEvent(st, ev_wred_, 0));   // the flat gradient is complete from here on
    FinArgs fa{};
    fa.d = d; fa.head_partial = head_partial_; fa.n_head = n_head_; fa.n_slab = n_slab_;
    fa.map = reinterpret_cast<const ParamMap*>(d_map_); fa.small = d_small_; fa.n_small = n_small_;
    for (int l = 1; l < NH; l++) fa.colsum[l - 1] = colsum_[l - 1];
    fa.bscal = bscal; fa.theta = pblock; fa.grad = grad; fa.stats = stats_; fa.loss_out = m_.d_l2coef ? nullptr : loss_out;
    fa.T = m_.T; fa.agg_mean = m_.agg_mean;
    for (int t = 0; t < 4; t++) fa.loss_kind[t] = m_.loss_kind[t];
    for (int s = 0; s < 8; s++) fa.slot[s] = ha.slot[s];
    fa.slot_of_flat = m_.d_slot_of_flat; fa.skip_out = skip_; fa.dp = isdp ? 1 : 0;
    k_wide_gradfin<<<(n_small_ + 31) / 32, 256, 0, st>>>(fa);
    WN(cudaGetLastError());
    if (post_) {   // (single GPU only: data-parallel mode refuses rmse and weight_l2)
        PostArgs pa{};
        pa.map = reinterpret_cast<const ParamMap*>(d_map_); pa.nflat = m_.nflat; pa.theta = pblock; pa.grad = grad;
        pa.stats = stats_; pa.bscal = bscal; pa.T = m_.T;
        for (int t = 0; t < 4; t++) pa.loss_kind[t] = m_.loss_kind[t];
        pa.l2coef = m_.d_l2coef; pa.l2_aggw = m_.l2_aggw; pa.l2_loss_coef = m_.l2_loss_coef;
        pa.l2part = l2part_; pa.ticket = ticket_; pa.loss_out = loss_out;
        k_wide_gradpost<<<gradpost_grid(m_), 256, 0, st>>>(pa);
        WN(cudaGetLastError());
    }
    if (isdp) {
        AllredArgs ar{};
        for (int r = 0; r < dp->world; r++) ar.peer[r] = dp->peer[r];
        ar.world = dp->world; ar.rank = dp->rank; ar.par = par; ar.xlen = dp_xlen(); ar.nflat = m_.nflat; ar.tag = dp->tag;
        ar.grad_out = grad_final; ar.stats = stats_; ar.loss_out = loss_out; ar.skip_out = skip_; ar.bscal = bscal;
        ar.T = m_.T; ar.agg_mean = m_.agg_mean;
        for (int t = 0; t < 4; t++) ar.loss_kind[t] = m_.loss_kind[t];
        ar.err = dp->err;
        k_wide_allreduce<<<2 * m_.nsm, 256, 0, st>>>(ar);
        WN(cudaGetLastError());
        grad = grad_final;
    }
    if (apply) {
        WUpdArgs u{};
        u.d = d; u.theta = pblock; u.m = m; u.v = v; u.ost = reinterpret_cast<OptState*>(ost); u.grad = grad; u.skip = skip_;
        u.map = reinterpret_cast<const ParamMap*>(d_map_);
        u.W1img = W1img_; u.WOimg = WOimg_; u.BOimg = BOimg_;
        u.opt_kind = m_.opt_kind; u.adamw_coupled = m_.adamw_coupled;
        u.eta = m_.eta; u.beta1 = m_.beta1; u.beta2 = m_.beta2; u.eps = m_.eps; u.lambda = m_.lambda;
        for (int l = 1; l <= NH; l++) { u.Wf[l - 1] = Wf_[l - 1]; u.Wb[l - 1] = Wb_[l - 1]; u.Bp[l - 1] = Bp_[l - 1]; }
        u.apply = 1;
        k_wide_update<<<(m_.nflat + 255) / 256, 256, 0, st>>>(u);
        WN(cudaGetLastError());
        k_wide_advance<<<1, 1, 0, st>>>(reinterpret_cast<OptState*>(ost), skip_, m_.beta1, m_.beta2, 1);
        WN(cudaGetLastError());
    }
    return cudaSuccess;
}

__global__ void k_wide_evalsum(const double* part, int n, int cnt, double* acc)
{
    const int q = threadIdx.x;
    if (q >= cnt) return;
    double s = 0.0;
    for (int g = 0; g < n; g++) s += part[(size_t)g * cnt + q];
    acc[q] += s;
}

cudaError_t WideNet::eval_rows(const float* rec, long long nrec, long long row0, int Bvalid, const float* bscal, const float* pblock,
                               float* yhat, float* parout, long long ldy, double* evalstat_dev, const float* shift_y,
                               cudaStream_t st)
{
    const int H = m_.H, NH = m_.NH;
    const int B = (Bvalid + 127) / 128 * 128;
    WN(ensure(B));
    WN(forward(rec, nullptr, row0, nrec, B, B, bscal, pblock, st));
    HeadKernel hk = find_head(m_.pm, m_.NOUT, m_.scale, H / 256);
    HeadArgs ha{};
    ha.A = A_[NH - 1]; ha.xb = xb_; ha.pblock = pblock; ha.WOimg = WOimg_; ha.BOimg = BOimg_; ha.bscal = bscal; ha.D = nullptr;
    ha.partial = nullptr;
    ha.yhat = yhat; ha.parout = parout; ha.ldy = ldy; ha.row0 = row0; ha.evalstat = evalstat_dev ? evalpart_ : nullptr;
    for (int t = 0; t < 4; t++) { ha.shift_y[t] = shift_y[t]; ha.loss_kind[t] = m_.loss_kind[t]; }
    ha.d = dims_of(m_); ha.B = B; ha.Bvalid = Bvalid; ha.act = m_.act; ha.train = 0;
    ha.prog = reinterpret_cast<const PmProgData*>(d_prog_); ha.nf = m_.F; ha.nt = m_.T;
    for (int s = 0; s < 8; s++) { ha.slot[s].role = m_.slot[s].role; ha.slot[s].idx = m_.slot[s].idx; ha.slot[s].lo = m_.slot[s].lo; ha.slot[s].span = m_.slot[s].span; ha.slot[s].fixedv = m_.slot[s].fixedv; }
    for (int i = 0; i < 4; i++) ha.pmc[i] = m_.pmc[i];
    const int head_smem = (8 * (m_.NOUT + 1) + m_.NOUT) * H * (int)sizeof(float);
    hk<<<n_head_, 256, head_smem, st>>>(ha);
    WN(cudaGetLastError());
    if (evalstat_dev) {
        k_wide_evalsum<<<1, 64, 0, st>>>(evalpart_, n_head_, m_.T * 8, evalstat_dev);
        WN(cudaGetLastError());
    }
    return cudaSuccess;
}

}  // namespace wide
}  // namespace eh

using namespace eh::wide;

#define WCK(call)                                                                             \
    do {                                                                                      \
        cudaError_t e__ = (call);                                                             \
        if (e__ != cudaSuccess) {                                                             \
            fprintf(stderr, "eh_wide: %s failed: %s\n", #call, cudaGetErrorString(e__));      \
            return EH_ECUDA;                                                                  \
        }                                                                                     \
    } while (0)

extern "C" eh_status eh_selftest_wide_gemm(int32_t mode, int32_t M, int32_t N, int32_t K, int32_t ksplits, int32_t act,
                                           const uint16_t* A, const uint16_t* B, const float* bias, const uint16_t* aux,
                                           void* out, int32_t device, float* ms_out)
{
    if (!A || !B || !out || mode < 0 || mode > 4) return EH_EINVAL;
    const bool pers = mode >= 3;   // 3 / 4: the persistent forms of 0 / 1
    if (pers) mode -= 3;
    if (M % BM || N % (pers ? PG_BN : gemm_bn(mode)) || ksplits < 1) return EH_EINVAL;
    WCK(cudaSetDevice(device));
    cudaDeviceProp prop;
    WCK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return EH_ECUDA;
    WCK(gemm_prepare());
    const bool wg = mode == GEMM_WGRAD;
    if (wg ? (K % (ksplits * BK) != 0) : (K % BK != 0)) return EH_EINVAL;
    // FWD/BWD: A [M x K], B [N x K].  WGRAD: A = deltas [K x M], B = activations [K x N].
    const size_t nA = (size_t)M * K, nB = (size_t)N * K;
    __nv_bfloat16 *dA = nullptr, *dB = nullptr, *dAux = nullptr, *dO16 = nullptr;
    float *dBias = nullptr, *dO32 = nullptr;
    WCK(cudaMalloc(&dA, nA * 2));
    WCK(cudaMalloc(&dB, nB * 2));
    WCK(cudaMemcpy(dA, A, nA * 2, cudaMemcpyHostToDevice));
    WCK(cudaMemcpy(dB, B, nB * 2, cudaMemcpyHostToDevice));
    if (mode == GEMM_FWD) {
        WCK(cudaMalloc(&dBias, (size_t)N * 4));
        WCK(cudaMemcpy(dBias, bias, (size_t)N * 4, cudaMemcpyHostToDevice));
    }
    if (mode == GEMM_BWD) {
        WCK(cudaMalloc(&dAux, (size_t)M * N * 2));
        WCK(cudaMemcpy(dAux, aux, (size_t)M * N * 2, cudaMemcpyHostToDevice));
    }
    if (wg) WCK(cudaMalloc(&dO32, (size_t)ksplits * M * N * 4));
    else WCK(cudaMalloc(&dO16, (size_t)M * N * 2));
    CUtensorMap tmA, tmB;
    bool ok;
    if (!wg) ok = make_map_bf16(&tmA, dA, K, M, K, BM) && make_map_bf16(&tmB, dB, K, N, K, pers ? pg_box_rows() : gemm_bn(mode));
    else ok = make_map_bf16(&tmA, dA, M, K, M, BK) && make_map_bf16(&tmB, dB, N, K, N, BK);
    if (!ok) return EH_ECUDA;
    cudaEvent_t e0, e1;
    WCK(cudaEventCreate(&e0));
    WCK(cudaEventCreate(&e1));
    const int reps = ms_out ? 5 : 1;
    for (int r = 0; r < reps; r++) {
        if (r == reps - 1) WCK(cudaEventRecord(e0));
        if (mode == GEMM_FWD && pers) WCK(gemm_fwd_p(tmA, tmB, M, N, K, dBias, act, dO16, 0));
        else if (mode == GEMM_BWD && pers) WCK(gemm_bwd_p(tmA, tmB, M, N, K, dAux, act, dO16, 0, nullptr, nullptr, nullptr, 0, 0, 0));
        else if (mode == GEMM_FWD) WCK(gemm_fwd(tmA, tmB, M, N, K, dBias, act, dO16, 0));
        else if (mode == GEMM_BWD) WCK(gemm_bwd(tmA, tmB, M, N, K, dAux, act, dO16, 0, nullptr, nullptr, nullptr, 0, 0, 0));
        else WCK(gemm_wgrad(tmA, tmB, M, N, K, ksplits, dO32, 0));
        if (r == reps - 1) WCK(cudaEventRecord(e1));
    }
    WCK(cudaDeviceSynchronize());
    if (ms_out) WCK(cudaEventElapsedTime(ms_out, e0, e1));
    if (wg) WCK(cudaMemcpy(out, dO32, (size_t)ksplits * M * N * 4, cudaMemcpyDeviceToHost));
    else WCK(cudaMemcpy(out, dO16, (size_t)M * N * 2, cudaMemcpyDeviceToHost));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(dA); cudaFree(dB); cudaFree(dAux); cudaFree(dO16); cudaFree(dBias); cudaFree(dO32);
    return EH_OK;
}
