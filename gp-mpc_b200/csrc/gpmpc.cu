// libgpmpc.so -- host side of the C ABI declared in include/gpmpc.h.
// One handle = one GPU = one CUDA stream.  No CPU fallback exists in this library.
#include "../../include/gpmpc.h"

#include <dlfcn.h>
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <vector>

#include <nvtx3/nvToolsExt.h>

#include "common.cuh"
#include "gemm_dmma.cuh"
#include "predict_streamk.cuh"
#include "kernels.cuh"

#define GPMPC_VERSION 100
#define HB 64                 // test points per predict pass (rows of the KS^T operand)
#define NX_MAX 32
#define PSK_MAX_CTAS 2048
#define MAX_DEPTH 12           // recursion depth bound: 128 * 2^12 rows

// ------------------------------------------------------------------------------------
// minimal NCCL surface, bound at run time with dlopen (no link-time dependency)
// ------------------------------------------------------------------------------------
typedef struct { char internal[128]; } nccl_uid_t;
typedef void* nccl_comm_t;
struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(nccl_uid_t*) = nullptr;
    int (*CommInitRank)(nccl_comm_t*, int, nccl_uid_t, int) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, nccl_comm_t, cudaStream_t) = nullptr;
    int (*CommDestroy)(nccl_comm_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
static NcclApi g_nccl;
static char g_create_err[512] = "";

static bool nccl_load(char* err, size_t errn)
{
    if (g_nccl.lib) return true;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
        g_nccl.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (g_nccl.lib) break;
    }
    if (!g_nccl.lib) { snprintf(err, errn, "dlopen(libnccl.so.2) failed: %s", dlerror()); return false; }
    g_nccl.GetUniqueId = (int (*)(nccl_uid_t*))dlsym(g_nccl.lib, "ncclGetUniqueId");
    g_nccl.CommInitRank = (int (*)(nccl_comm_t*, int, nccl_uid_t, int))dlsym(g_nccl.lib, "ncclCommInitRank");
    g_nccl.AllGather = (int (*)(const void*, void*, size_t, int, nccl_comm_t, cudaStream_t))dlsym(g_nccl.lib, "ncclAllGather");
    g_nccl.CommDestroy = (int (*)(nccl_comm_t))dlsym(g_nccl.lib, "ncclCommDestroy");
    g_nccl.GetErrorString = (const char* (*)(int))dlsym(g_nccl.lib, "ncclGetErrorString");
    if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllGather || !g_nccl.CommDestroy) {
        snprintf(err, errn, "libnccl is missing required symbols");
        g_nccl.lib = nullptr;
        return false;
    }
    return true;
}

// ------------------------------------------------------------------------------------
struct gpmpc_handle_s {
    int N = 0, Nx = 0, Ny = 0, a0 = 0, nloc = 0, Npad = 0, device = 0;
    int nloc_max = 0;                 // ceil(Ny / world): slots per rank in the gather buffer
    cudaStream_t st = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // factorisation overlap: step 5a of every recursion depth runs on its own side stream
    cudaStream_t sideSt[MAX_DEPTH] = {nullptr}; cudaEvent_t evA[MAX_DEPTH] = {nullptr}, evB[MAX_DEPTH] = {nullptr}, evT[MAX_DEPTH] = {nullptr}, evS[MAX_DEPTH] = {nullptr};
    long long w2off[MAX_DEPTH + 1] = {0}; int opt_overlap = 1, opt_lookahead = 1, opt_lookahead_min = 1024;
    // model
    double *dXT = nullptr, *dMu = nullptr, *dY = nullptr, *dHyp = nullptr, *dJit = nullptr, *dHypTmp = nullptr;
    double *dL = nullptr, *dLi = nullptr, *dW1 = nullptr, *dW2 = nullptr;
    double *dAlpha = nullptr, *dTmp = nullptr, *dRes = nullptr;
    int* dInfo = nullptr;
    // predict
    double *dKST = nullptr, *dPart = nullptr, *dPMJ = nullptr, *dSQ = nullptr, *dV = nullptr, *dR = nullptr, *dR2 = nullptr;
    unsigned int* dCnt = nullptr;     // stream-K counters: [nloc*nt tile | nloc output | 1 done], self-cleaning
    int psk_ctas = 0, opt_predict_ctas = 0, partCtas = 0;   // persistent grid of the predict product (2 CTAs per SM)
    double *dCovV = nullptr, *dCovOut = nullptr; long long covVcap = 0, covOutcap = 0;   // GP.covar scratch pool
    // predict_grad: U = Linv^T per output (lazy), beta rows, partial sums, per-batch derivative slabs
    double *dUall = nullptr, *dBeta = nullptr, *dPDV = nullptr, *dPH = nullptr, *dGradOut = nullptr; bool u_valid = false; int gradHcap = 0;
    // predict_hess: pair-sum partials / sums, Gram of W = L^-1 dks, Sigma Hm scratch, per-batch second-derivative slab
    double *dHP = nullptr, *dHS = nullptr, *dGram = nullptr, *dSH = nullptr, *dHessOut = nullptr; int hessHcap = 0;
    double *dG = nullptr, *dZ = nullptr, *dSigma = nullptr, *dMean = nullptr, *dVar = nullptr, *dJ = nullptr, *dCov = nullptr;
    double* dRoll = nullptr; size_t rollCap = 0;   // gpmpc_rollout: [Z | Sigma | U | scale | means | vars | cov]
    double *dIn = nullptr, *dOut = nullptr;   // [Z | Sigma] and [mean | var | J | cov] slabs: one H2D + one D2H per host call
    int Hcap = 0;
    double* hPinned = nullptr; double* dPinnedAlias = nullptr; size_t hPinnedBytes = 0; int opt_zero_copy = 1;
    // nlml scratch
    double *dU = nullptr, *dKinv = nullptr, *dGradPart = nullptr, *dGrad = nullptr;
    bool has_data = false, has_hyper = false, factorized = false;
    // EM scratch
    double *dEmTr = nullptr, *dEMP = nullptr, *dEmE = nullptr, *dEmF = nullptr, *dEmW = nullptr, *dEmIJ = nullptr;
    double *dEmMeanPart = nullptr, *dEmPart = nullptr, *dEmLQ = nullptr, *dEmVec = nullptr, *dEmE2 = nullptr, *dEmF2 = nullptr;
    int emHcap = 0;
    std::vector<double> hyper;        // (nloc, Nx+2)
    std::vector<double> logdet, yalpha;
    std::vector<int> jitter_used;
    // FITC sparse model (gpmpc_fitc): L holds Luu, Li holds R (R^T R = K~^-1), alpha holds alpha_s
    bool sparse = false; int opt_fitc_panel = 4096;
    double fitc_ms[5] = {0, 0, 0, 0, 0};   // last build: Kuf, V product, column pass + b, SYRK, M-sized factorisations
    int opt_refine = 0, opt_gemm_variant = 3, opt_leaf_variant = 3, opt_small_tiles = 592;   // 128x64-tile count below which 64x32 tiles are used
    // comm
    nccl_comm_t comm = nullptr; int rank = 0, world = 1;
    // peer (CUDA IPC) exchange: [flags: 2*MAXW u64][gather buffer parity 0][parity 1]
    double* dPeerBlock = nullptr; long long peerGsz = 0; int peerHcap = 0; bool peer_ready = false;
    double* peerBase[GPMPC_MAXW] = {nullptr}; bool peerOpened[GPMPC_MAXW] = {false};
    int* dPeerStatus = nullptr; int* hPeerStatus = nullptr;
    unsigned long long peer_step = 0; int opt_peer = 1; double opt_peer_timeout_s = 60.0; int clock_khz = 1965000;
    char err[512] = "";
};

static void set_error(gpmpc_handle_t h, const char* fmt, ...)
{
    va_list ap; va_start(ap, fmt);
    vsnprintf(h ? h->err : g_create_err, 512, fmt, ap);
    va_end(ap);
}

// NVTX range per phase (header-only nvtx3: a no-op unless a profiler injects the library)
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

static inline long long slab(gpmpc_handle_t h) { return (long long)h->Npad * h->Npad; }
static inline long long wslab(gpmpc_handle_t h) { return (long long)h->Npad * h->Npad / 4 + 128; }
static inline long long w2slab(gpmpc_handle_t h) { return h->w2off[MAX_DEPTH]; }   // all depths, one batch entry

// ------------------------------------------------------------------------------------
// GEMM helpers (all operands live in slabs with leading dimension ld)
// ------------------------------------------------------------------------------------
static cudaError_t gemm128_on(gpmpc_handle_t h, cudaStream_t st, bool bt, const GemmParams& p, int batch);

// callers describe the problem in 128x128 tiles (mt, nt); variant 1 re-tiles N by 64
static cudaError_t gemm128(gpmpc_handle_t h, bool bt, const GemmParams& p, int batch)
{
    return gemm128_on(h, h->st, bt, p, batch);
}

static cudaError_t gemm128_on(gpmpc_handle_t h, cudaStream_t st, bool bt, const GemmParams& p, int batch)
{
    if (h->opt_gemm_variant == 3) {
        // tile-granular TMA (tensor maps, 128B swizzle) for the NT products that fill the GPU for at
        // least two waves; everything else (NN products, small launches) takes the cp.async variant
        const long long tiles = (long long)batch * (p.lower ? (long long)p.mt * (p.mt + 1) : 2LL * p.mt * p.nt);
        GemmParams q = p;
        if (tiles < h->opt_small_tiles) {
            // deep recursion levels: a handful of 128x64 tiles cannot occupy 148 SMs; 64x32 tiles
            // (8x more CTAs, 4 CTAs/SM) cut the latency of these critical-path launches
            q.mt = p.mt * 2; q.nt = p.nt * 4;
            return bt ? gemm_launch<64, 32, 2, 2, true, 3, 4>(q, batch, 1, st)
                      : gemm_launch<64, 32, 2, 2, false, 3, 4>(q, batch, 1, st);
        }
        q.nt = p.nt * 2;
        if (bt && tiles >= 592) return gemm_tmap_launch<128, 64, 2, 2, 4, 2>(q, batch, 1, st);
        return bt ? gemm_launch<128, 64, 2, 2, true, 3, 2>(q, batch, 1, st)
                  : gemm_launch<128, 64, 2, 2, false, 3, 2>(q, batch, 1, st);
    }
    if (h->opt_gemm_variant == 2) {       // variant 1 with the TMA (cp.async.bulk + mbarrier) feed
        GemmParams q = p;
        q.nt = p.nt * 2;
        return bt ? gemm_launch<128, 64, 2, 2, true, 3, 2, true>(q, batch, 1, st)
                  : gemm_launch<128, 64, 2, 2, false, 3, 2, true>(q, batch, 1, st);
    }
    if (h->opt_gemm_variant == 1) {       // 128x64 tiles, 4 warps, 3 stages, 2 CTAs/SM
        GemmParams q = p;
        q.nt = p.nt * 2;
        return bt ? gemm_launch<128, 64, 2, 2, true, 3, 2>(q, batch, 1, st)
                  : gemm_launch<128, 64, 2, 2, false, 3, 2>(q, batch, 1, st);
    }
    return bt ? gemm_launch<128, 128, 2, 4, true, 4, 1>(p, batch, 1, st)
              : gemm_launch<128, 128, 2, 4, false, 4, 1>(p, batch, 1, st);
}

// Recursive blocked Cholesky + triangular inverse on the diagonal block
// [off, off+n) of every slab in the batch:  A -> L (in place, lower), Li -> L^-1.
//   1. (L11, Li11) = rec(A11)
//   2. L21 = A21 Li11^T                 (explicit-inverse panel solve, DMMA GEMM NT)
//   3. A22 -= L21 L21^T                 (trailing SYRK update, DMMA GEMM NT, lower tiles)
//   4. (L22, Li22) = rec(A22)
//   5. Li21 = -Li22 (L21 Li11)          (two DMMA GEMMs NN)
// All flops except the 128x128 leaves run on the fp64 tensor pipe.
static int potrf_inv_rec(gpmpc_handle_t h, double* A, double* Li, long long sA, long long sLi,
                         int* dInfo, int off, int n, int batch, int depth = 0, cudaEvent_t pend = nullptr)
{
    const int ld = h->Npad;
    if (n <= LEAF_N) {
        if (pend) CUDA_TRY(cudaStreamWaitEvent(h->st, pend, 0));
        static std::atomic<bool> conf[GPMPC_MAX_DEVICES];
        if (!conf[h->device % GPMPC_MAX_DEVICES].load(std::memory_order_acquire)) {
            CUDA_TRY(cudaFuncSetAttribute(leaf_potrf_trtri_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, LEAF_N * LEAF_LD * 8));
            CUDA_TRY(cudaFuncSetAttribute(leaf_potrf_trtri_v2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, LF_SMEM_DOUBLES * 8));
            CUDA_TRY(cudaFuncSetAttribute(leaf_potrf_trtri_v3_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, LF3_SMEM_DOUBLES * 8));
            CUDA_TRY(cudaFuncSetAttribute(leaf_potrf_trtri_v3_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, LF3_SMEM_DOUBLES * 8));
            conf[h->device % GPMPC_MAX_DEVICES].store(true, std::memory_order_release);
        }
        if (h->opt_leaf_variant == 0)
            leaf_potrf_trtri_kernel<<<batch, 256, LEAF_N * LEAF_LD * 8, h->st>>>(A + (long long)off * ld + off, ld, sA,
                                                                              Li + (long long)off * ld + off, ld, sLi, dInfo, off);
        else if (h->opt_leaf_variant == 1)
            leaf_potrf_trtri_v2_kernel<<<batch, 256, LF_SMEM_DOUBLES * 8, h->st>>>(A + (long long)off * ld + off, ld, sA,
                                                                                Li + (long long)off * ld + off, ld, sLi, dInfo, off);
        else if (h->opt_leaf_variant == 2)
            leaf_potrf_trtri_v3_kernel<false><<<batch, 256, LF3_SMEM_DOUBLES * 8, h->st>>>(A + (long long)off * ld + off, ld, sA,
                                                                                        Li + (long long)off * ld + off, ld, sLi, dInfo, off);
        else       // 3: v3 with two pivots per step
            leaf_potrf_trtri_v3_kernel<true><<<batch, 256, LF3_SMEM_DOUBLES * 8, h->st>>>(A + (long long)off * ld + off, ld, sA,
                                                                                       Li + (long long)off * ld + off, ld, sLi, dInfo, off);
        CUDA_TRY(cudaGetLastError());
        return GPMPC_OK;
    }
    const int nb = n / GPMPC_TILE;
    const int n1 = (nb / 2) * GPMPC_TILE, n2 = n - n1;
    int rc = potrf_inv_rec(h, A, Li, sA, sLi, dInfo, off, n1, batch, depth + 1, nullptr);
    if (rc) return rc;
    // the caller deferred part of its trailing update to its side stream (look-ahead, see below): everything outside this
    // sub-problem's leading n1 x n1 block is only valid once that work has finished
    if (pend) CUDA_TRY(cudaStreamWaitEvent(h->st, pend, 0));
    double* A21 = A + (long long)(off + n1) * ld + off;
    double* A22 = A + (long long)(off + n1) * ld + off + n1;
    double* Li11 = Li + (long long)off * ld + off;
    double* Li21 = Li + (long long)(off + n1) * ld + off;
    double* Li22 = Li + (long long)(off + n1) * ld + off + n1;
    double* W1 = h->dW1 + h->w2off[depth];                 // one region per depth (deferred work of different depths is in flight together)
    double* W2 = h->dW2 + h->w2off[depth];
    const long long sW = w2slab(h), sW2 = w2slab(h);
    const bool ovl = h->opt_overlap && depth < MAX_DEPTH;
    cudaStream_t side = ovl ? h->sideSt[depth] : h->st;
    // LOOK-AHEAD.  rec(A22) starts with the leading h2 x h2 block of A22 (its own first half) and does not touch the rest
    // before its panel step.  So only the top h2 rows of the panel and the (1,1) block of the trailing update stay on the
    // critical stream; the bottom panel rows, the (2,1) and (2,2) blocks of the update and W2 run on this depth's
    // low-priority side stream beside the latency-bound recursion into A22_11 (leaves, small products) and are joined by
    // the child right before its panel step (`pend`).  On-chain share of a level's flops: 0.44 instead of 0.75.
    const int h2 = ((n2 / GPMPC_TILE) / 2) * GPMPC_TILE;
    const bool split = ovl && h->opt_lookahead && h2 >= GPMPC_TILE && n >= h->opt_lookahead_min;
    GemmParams p;
    auto panel = [&](cudaStream_t st, int r0, int rows) -> cudaError_t {     // W1[r0:r0+rows] = A21[r0:..] Li11^T ; L21 rows <- W1 rows
        GemmParams q;
        memset(&q, 0, sizeof(q));
        q.A = A21 + (long long)r0 * ld; q.lda = ld; q.sA = sA;
        q.B = Li11; q.ldb = ld; q.sB = sLi;                                   // B[j][k] = Li11[j][k] != 0 only for k <= j
        q.C = W1 + (long long)r0 * n1; q.ldc = n1; q.sC = sW;
        q.mt = rows / 128; q.nt = n1 / 128; q.K = n1; q.alpha = 1.0; q.beta = 0.0; q.kflags = GEMM_KJ_LE;
        cudaError_t e = gemm128_on(h, st, true, q, batch);
        if (e != cudaSuccess) return e;
        dim3 g(std::max(1, std::min(64, n1 / 2 / 128)), std::min(rows, 4096), batch);
        copy2d_kernel<<<g, 128, 0, st>>>(W1 + (long long)r0 * n1, n1, sW, A21 + (long long)r0 * ld, ld, sA, rows, n1);
        return cudaGetLastError();
    };
    auto update = [&](cudaStream_t st, int r0, int rows, int c0, int cols, int lower) -> cudaError_t {   // A22[r0.., c0..] -= W1[r0..] W1[c0..]^T
        GemmParams q;
        memset(&q, 0, sizeof(q));
        q.A = W1 + (long long)r0 * n1; q.lda = n1; q.sA = sW;
        q.B = W1 + (long long)c0 * n1; q.ldb = n1; q.sB = sW;
        q.C = A22 + (long long)r0 * ld + c0; q.ldc = ld; q.sC = sA; q.Cin = q.C; q.ldcin = ld; q.sCin = sA;
        q.mt = rows / 128; q.nt = cols / 128; q.K = n1; q.alpha = -1.0; q.beta = 1.0; q.lower = lower;
        return gemm128_on(h, st, true, q, batch);
    };
    if (ovl) {
        CUDA_TRY(cudaEventRecord(h->evA[depth], h->st));
        CUDA_TRY(cudaStreamWaitEvent(side, h->evA[depth], 0));
    }
    if (split) {
        CUDA_TRY(panel(h->st, 0, h2));                                        // 2. top rows (critical)
        CUDA_TRY(cudaEventRecord(h->evT[depth], h->st));
        CUDA_TRY(update(h->st, 0, h2, 0, h2, 1));                             // 3. (1,1) block (critical)
        CUDA_TRY(panel(side, h2, n2 - h2));                                   // 2. bottom rows (side)
        CUDA_TRY(cudaStreamWaitEvent(side, h->evT[depth], 0));                //    needs W1's top rows
        CUDA_TRY(update(side, h2, n2 - h2, 0, h2, 0));                        // 3. (2,1) block
        CUDA_TRY(update(side, h2, n2 - h2, h2, n2 - h2, 1));                  // 3. (2,2) block
        CUDA_TRY(cudaEventRecord(h->evS[depth], side));
    } else {
        CUDA_TRY(panel(h->st, 0, n2));                                        // 2. W1 = A21 Li11^T, L21 <- W1
        CUDA_TRY(update(h->st, 0, n2, 0, n2, 1));                             // 3. A22 -= W1 W1^T (lower tiles)
        if (ovl) {       // the side stream must not start 5a before L21 is in place
            CUDA_TRY(cudaEventRecord(h->evT[depth], h->st));
            CUDA_TRY(cudaStreamWaitEvent(side, h->evT[depth], 0));
        }
    }
    // 5a. W2 = L21 * Li11     Bop[k][j] = Li11[k][j] != 0 only for k >= j.  Independent of step 4: on the side stream it
    //     fills the SMs the recursion into A22 leaves idle.  L21 is read from the matrix; W2 has one region per depth.
    memset(&p, 0, sizeof(p));
    p.A = A21; p.lda = ld; p.sA = sA;
    p.B = Li11; p.ldb = ld; p.sB = sLi;
    p.C = W2; p.ldc = n1; p.sC = sW2;
    p.mt = n2 / 128; p.nt = n1 / 128; p.K = n1; p.alpha = 1.0; p.beta = 0.0; p.kflags = GEMM_KJ_GE;
    if (ovl) {
        CUDA_TRY(gemm128_on(h, side, false, p, batch));
        CUDA_TRY(cudaEventRecord(h->evB[depth], side));
    }
    // 4.
    rc = potrf_inv_rec(h, A, Li, sA, sLi, dInfo, off + n1, n2, batch, depth + 1, split ? h->evS[depth] : nullptr);
    if (rc) return rc;
    if (ovl) CUDA_TRY(cudaStreamWaitEvent(h->st, h->evB[depth], 0));
    else CUDA_TRY(gemm128(h, false, p, batch));
    // 5b. Li21 = -Li22 * W2   A[i][k] = Li22[i][k] != 0 only for k <= i
    memset(&p, 0, sizeof(p));
    p.A = Li22; p.lda = ld; p.sA = sLi;
    p.B = W2; p.ldb = n1; p.sB = sW2;
    p.C = Li21; p.ldc = ld; p.sC = sLi;
    p.mt = n2 / 128; p.nt = n1 / 128; p.K = n2; p.alpha = -1.0; p.beta = 0.0; p.kflags = GEMM_KI_LE;
    CUDA_TRY(gemm128(h, false, p, batch));
    return GPMPC_OK;
}

// K(theta) for `batch` consecutive outputs: hyper rows at dHyp (stride Nx+2), jitter at dJit,
// output slabs at K (stride slab).  full = 1 writes the whole square, 0 the lower triangle.
static int launch_kbuild(gpmpc_handle_t h, const double* dHyp, const double* dJit, double* K, int batch, int full)
{
    static std::atomic<bool> conf[GPMPC_MAX_DEVICES];
    const int KD = (h->Nx + 3) & ~3, S = ((KD >> 2) & 1) ? KD : KD + 4;
    const int smem = (2 * KB2_TILE * S + 2 * KB2_TILE + 256) * 8;
    if (!conf[h->device % GPMPC_MAX_DEVICES].load(std::memory_order_acquire)) {
        CUDA_TRY(cudaFuncSetAttribute(kbuild_dmma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (2 * KB2_TILE * 36 + 2 * KB2_TILE + 256) * 8));
        CUDA_TRY(cudaFuncSetAttribute(kbuild_dmma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (2 * KB2_TILE * 36 + 2 * KB2_TILE + 256) * 8));
        conf[h->device % GPMPC_MAX_DEVICES].store(true, std::memory_order_release);
    }
    const int T = h->Npad / KB2_TILE;
    dim3 grid(T * (T + 1) / 2, 1, batch);
    if (full)
        kbuild_dmma_kernel<true><<<grid, 256, smem, h->st>>>(h->dXT, h->Npad, h->N, h->Nx, h->dMu, dHyp, h->Nx + 2, dJit, K, h->Npad, slab(h));
    else
        kbuild_dmma_kernel<false><<<grid, 256, smem, h->st>>>(h->dXT, h->Npad, h->N, h->Nx, h->dMu, dHyp, h->Nx + 2, dJit, K, h->Npad, slab(h));
    CUDA_TRY(cudaGetLastError());
    return GPMPC_OK;
}

// alpha = Li^T (Li y) for `batch` consecutive local outputs starting at local index a
static int launch_alpha(gpmpc_handle_t h, int a, int batch)
{
    const int n = h->Npad;
    const double* Li = h->dLi + (long long)a * slab(h);
    dim3 g1((n + 7) / 8, 1, batch);
    trmv_lower_kernel<<<g1, 256, 0, h->st>>>(Li, n, slab(h), h->dY + (long long)a * n, n,
                                              h->dTmp + (long long)a * n, n, n);
    CUDA_TRY(cudaGetLastError());
    // alpha = Li^T tmp in row chunks (partials in the W1 workspace, free outside the recursion), then
    // one pass that sums the partials, takes log det and y . alpha
    const int nch = (n + TRT_ROWS - 1) / TRT_ROWS;
    double* P = h->dW1 + (long long)a * w2slab(h);
    dim3 g2(n / 32, nch, batch);
    trmv_lower_T_part_kernel<<<g2, 256, 0, h->st>>>(Li, n, slab(h), h->dTmp + (long long)a * n, n, P, w2slab(h), n);
    CUDA_TRY(cudaGetLastError());
    alpha_logdet_kernel<<<batch, 1024, 0, h->st>>>(P, w2slab(h), nch, h->dL + (long long)a * slab(h), n, slab(h),
                                                   h->dY + (long long)a * n, n, h->dAlpha + (long long)a * n, n, n, h->dRes + 2 * a);
    CUDA_TRY(cudaGetLastError());
    return GPMPC_OK;
}

// K(theta) -> L, Li for local output a with the reference's single jitter retry.
// used: 0 ok, 1 jitter used, >1: 1 + failing pivot.  dHyp = device hyper row of that output.
static int factor_one(gpmpc_handle_t h, int a, const double* dHyp, double jitter, int* used)
{
    double* L = h->dL + (long long)a * slab(h);
    double* Li = h->dLi + (long long)a * slab(h);
    *used = 0;
    for (int attempt = 0; attempt < 2; ++attempt) {
        const double jit = attempt ? jitter : 0.0;
        CUDA_TRY(cudaMemcpyAsync(h->dJit + a, &jit, sizeof(double), cudaMemcpyHostToDevice, h->st));
        CUDA_TRY(cudaMemsetAsync(h->dInfo + a, 0, sizeof(int), h->st));
        {   // kbuild indexes hyper/jitter by blockIdx.z (== 0 here): pass row pointers
            int rck = launch_kbuild(h, dHyp, h->dJit + a, L, 1, 0);
            if (rck) return rck;
        }
        int rc = potrf_inv_rec(h, L, Li, slab(h), slab(h), h->dInfo + a, 0, h->Npad, 1);
        if (rc) return rc;
        int info = 0;
        CUDA_TRY(cudaMemcpyAsync(&info, h->dInfo + a, sizeof(int), cudaMemcpyDeviceToHost, h->st));
        CUDA_TRY(cudaStreamSynchronize(h->st));
        if (info == 0) { *used = attempt; return GPMPC_OK; }
        *used = 1 + info;
    }
    return GPMPC_ERR_NOTPD;
}

// ------------------------------------------------------------------------------------
extern "C" int gpmpc_version(void) { return GPMPC_VERSION; }

extern "C" const char* gpmpc_last_error(gpmpc_handle_t h) { return h ? h->err : g_create_err; }

#define ALLOC(ptr, count)                                                               \
    do {                                                                                \
        cudaError_t _e = cudaMalloc((void**)&(ptr), (size_t)(count) * sizeof(*(ptr)));  \
        if (_e != cudaSuccess) {                                                        \
            set_error(h, "cudaMalloc(%s, %zu bytes) failed: %s", #ptr,                  \
                      (size_t)(count) * sizeof(*(ptr)), cudaGetErrorString(_e));        \
            return GPMPC_ERR_CUDA;                                                      \
        }                                                                               \
        cudaMemsetAsync((ptr), 0, (size_t)(count) * sizeof(*(ptr)), h->st);             \
    } while (0)

extern "C" int gpmpc_destroy(gpmpc_handle_t h);

static int create_fill(gpmpc_handle_t h, int N, int Nx, int Ny, int out_begin, int out_count, int device)
{
    h->N = N; h->Nx = Nx; h->Ny = Ny; h->a0 = out_begin; h->nloc = out_count; h->device = device;
    h->nloc_max = out_count; h->world = 1; h->rank = 0;
    h->Npad = (N + GPMPC_TILE - 1) / GPMPC_TILE * GPMPC_TILE;
    CUDA_TRY(cudaSetDevice(device));
    {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        CUDA_TRY(cudaStreamCreateWithPriority(&h->st, cudaStreamNonBlocking, hi));   // critical path first
    }
    CUDA_TRY(cudaEventCreate(&h->ev0));
    CUDA_TRY(cudaEventCreate(&h->ev1));
    const long long np = h->Npad;
    ALLOC(h->dXT, (long long)Nx * np);
    ALLOC(h->dMu, NX_MAX);
    ALLOC(h->dY, (long long)out_count * np);
    ALLOC(h->dHyp, (long long)out_count * (Nx + 2));
    ALLOC(h->dHypTmp, Nx + 2);
    ALLOC(h->dJit, out_count);
    ALLOC(h->dL, out_count * slab(h));
    ALLOC(h->dLi, out_count * slab(h));
    {   // W2 workspace: one region per recursion depth (n_d = ceil(nb / 2^d) * 128 rows at depth d)
        const int nb = h->Npad / 128;
        long long off = 0;
        for (int d = 0; d < MAX_DEPTH; ++d) {
            h->w2off[d] = off;
            const long long nd = (long long)((nb + (1 << d) - 1) >> d) * 128;
            off += nd * nd / 4 + 128;
        }
        h->w2off[MAX_DEPTH] = off;
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        for (int d = 0; d < MAX_DEPTH; ++d) {
            CUDA_TRY(cudaStreamCreateWithPriority(&h->sideSt[d], cudaStreamNonBlocking, lo));
            CUDA_TRY(cudaEventCreateWithFlags(&h->evA[d], cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&h->evB[d], cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&h->evT[d], cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&h->evS[d], cudaEventDisableTiming));
        }
    }
    ALLOC(h->dW1, out_count * w2slab(h));      // same per-depth layout as W2
    ALLOC(h->dW2, out_count * w2slab(h));
    ALLOC(h->dAlpha, (long long)out_count * np);
    ALLOC(h->dTmp, (long long)out_count * np);
    ALLOC(h->dRes, 2 * out_count);
    ALLOC(h->dInfo, out_count);
    ALLOC(h->dGrad, Nx + 2);
    h->hyper.assign((size_t)out_count * (Nx + 2), 0.0);
    h->logdet.assign(out_count, 0.0); h->yalpha.assign(out_count, 0.0); h->jitter_used.assign(out_count, 0);
    CUDA_TRY(cudaStreamSynchronize(h->st));
    return GPMPC_OK;
}


extern "C" int gpmpc_create(int N, int Nx, int Ny, int out_begin, int out_count, int device, gpmpc_handle_t* out)
{
    gpmpc_handle_t h = nullptr;
    if (!out) return GPMPC_ERR_ARG;
    *out = nullptr;
    if (N < 1 || Nx < 1 || Nx > NX_MAX || Ny < 1 || out_begin < 0 || out_count < 1 || out_begin + out_count > Ny) {
        set_error(nullptr, "gpmpc_create: bad sizes N=%d Nx=%d (max %d) Ny=%d outputs [%d,%d)", N, Nx, NX_MAX, Ny,
                  out_begin, out_begin + out_count);
        return GPMPC_ERR_ARG;
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev < 1 || device < 0 || device >= ndev) {
        set_error(nullptr, "gpmpc_create: no usable CUDA device %d (count %d, %s) -- this engine has no CPU path",
                  device, ndev, cudaGetErrorString(e));
        return GPMPC_ERR_CUDA;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major < 10) {
        set_error(nullptr, "gpmpc_create: device %d is sm_%d%d; this library is built for sm_100a only", device,
                  prop.major, prop.minor);
        return GPMPC_ERR_CUDA;
    }
    h = new gpmpc_handle_s();
    const int rc = create_fill(h, N, Nx, Ny, out_begin, out_count, device);
    if (rc != GPMPC_OK) {            // no partially built handle survives: message to the create slot, everything freed
        snprintf(g_create_err, sizeof(g_create_err), "gpmpc_create: %s", h->err);
        gpmpc_destroy(h);
        return rc;
    }
    *out = h;
    return GPMPC_OK;
}

extern "C" int gpmpc_destroy(gpmpc_handle_t h)
{
    if (!h) return GPMPC_OK;
    cudaSetDevice(h->device);
    if (h->st) cudaStreamSynchronize(h->st);
    if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
    for (int r = 0; r < GPMPC_MAXW; ++r) if (h->peerOpened[r]) cudaIpcCloseMemHandle(h->peerBase[r]);
    if (h->dPeerBlock) cudaFree(h->dPeerBlock);
    if (h->dCnt) cudaFree(h->dCnt);
    if (h->hPeerStatus) cudaFreeHost(h->hPeerStatus);
    double* bufs[] = {h->dXT, h->dMu, h->dY, h->dHyp, h->dHypTmp, h->dJit, h->dL, h->dLi, h->dW1, h->dW2, h->dAlpha, h->dTmp,
                      h->dRes, h->dKST, h->dPart, h->dPMJ, h->dSQ, h->dV, h->dR, h->dR2, h->dCovV, h->dCovOut, h->dUall, h->dBeta, h->dPDV, h->dPH, h->dGradOut, h->dHP, h->dHS, h->dGram, h->dSH, h->dHessOut, h->dG, h->dRoll, h->dIn, h->dOut, h->dU, h->dKinv, h->dGradPart, h->dGrad,
                      h->dEmTr, h->dEmLQ, h->dEmVec, h->dEmE2, h->dEmF2, h->dEMP, h->dEmE, h->dEmF, h->dEmW, h->dEmIJ, h->dEmMeanPart, h->dEmPart};
    for (double* b : bufs) if (b) cudaFree(b);
    if (h->dInfo) cudaFree(h->dInfo);
    if (h->hPinned) cudaFreeHost(h->hPinned);
    for (int d = 0; d < MAX_DEPTH; ++d) {
        if (h->sideSt[d]) { cudaStreamSynchronize(h->sideSt[d]); cudaStreamDestroy(h->sideSt[d]); }
        if (h->evA[d]) cudaEventDestroy(h->evA[d]);
        if (h->evB[d]) cudaEventDestroy(h->evB[d]);
        if (h->evT[d]) cudaEventDestroy(h->evT[d]);
        if (h->evS[d]) cudaEventDestroy(h->evS[d]);
    }
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->st) cudaStreamDestroy(h->st);
    delete h;
    return GPMPC_OK;
}

static int ensure_pinned(gpmpc_handle_t h, size_t bytes)
{
    if (h->hPinnedBytes >= bytes) return GPMPC_OK;
    if (h->hPinned) cudaFreeHost(h->hPinned);
    h->hPinned = nullptr; h->hPinnedBytes = 0;
    // mapped: small batches are read / written by the kernels directly (zero copy), see gpmpc_predict
    CUDA_TRY(cudaHostAlloc((void**)&h->hPinned, bytes, cudaHostAllocMapped));
    CUDA_TRY(cudaHostGetDevicePointer((void**)&h->dPinnedAlias, h->hPinned, 0));
    h->hPinnedBytes = bytes;
    return GPMPC_OK;
}

extern "C" int gpmpc_set_data(gpmpc_handle_t h, const double* X, const double* Y)
{
    if (!h || !X || !Y) return GPMPC_ERR_ARG;
    CUDA_TRY(cudaSetDevice(h->device));
    const int N = h->N, Nx = h->Nx, np = h->Npad;
    std::vector<double> xt((size_t)Nx * np, 0.0), yl((size_t)h->nloc * np, 0.0);
    for (int i = 0; i < N; ++i)
        for (int d = 0; d < Nx; ++d) xt[(size_t)d * np + i] = X[(size_t)i * Nx + d];
    for (int a = 0; a < h->nloc; ++a)
        for (int i = 0; i < N; ++i) yl[(size_t)a * np + i] = Y[(size_t)i * h->Ny + h->a0 + a];
    double mu[NX_MAX] = {0.0};              // column means: the K build centres its inputs (translation invariant)
    for (int d = 0; d < Nx; ++d) {
        double sacc = 0.0;
        for (int i = 0; i < N; ++i) sacc += X[(size_t)i * Nx + d];
        mu[d] = sacc / N;
    }
    CUDA_TRY(cudaMemcpyAsync(h->dMu, mu, NX_MAX * 8, cudaMemcpyHostToDevice, h->st));
    CUDA_TRY(cudaMemcpyAsync(h->dXT, xt.data(), xt.size() * 8, cudaMemcpyHostToDevice, h->st));
    CUDA_TRY(cudaMemcpyAsync(h->dY, yl.data(), yl.size() * 8, cudaMemcpyHostToDevice, h->st));
    CUDA_TRY(cudaStreamSynchronize(h->st));
    h->has_data = true; h->factorized = false;
    return GPMPC_OK;
}

static int local_index(gpmpc_handle_t h, int a);

// Replace the target vector of global output a (N doubles): GP passes the residual y - m(X) when a
// prior mean function is in use (alpha = K^-1 (y - m(X)), optimize.py:492-494).
extern "C" int gpmpc_set_y(gpmpc_handle_t h, int a, const double* y)
{
    if (!h || !y) return GPMPC_ERR_ARG;
    if (!h->has_data) { set_error(h, "gpmpc_set_y: set_data first"); return GPMPC_ERR_STATE; }
    CUDA_TRY(cudaSetDevice(h->device));
    const int al = local_index(h, a);
    if (al < 0) return GPMPC_ERR_ARG;
    CUDA_TRY(cudaMemcpyAsync(h->dY + (long long)al * h->Npad, y, (size_t)h->N * 8, cudaMemcpyHostToDevice, h->st));
    CUDA_TRY(cudaStreamSynchronize(h->st));
    h->factorized = false;
    return GPMPC_OK;
}

extern "C" int gpmpc_set_hyper(gpmpc_handle_t h, const double* hyper, int ld)
{
    if (!h || !hyper || ld < h->Nx + 2) { if (h) set_error(h, "gpmpc_set_hyper: ld < Nx+2"); return GPMPC_ERR_ARG; }
    CUDA_TRY(cudaSetDevice(h->device));
    const int m = h->Nx + 2;
    for (int a = 0; a < h->nloc; ++a)
        for (int q = 0; q < m; ++q) {
            const double v = hyper[(size_t)(h->a0 + a) * ld + q];
            if (q < h->Nx && v == 0.0) { set_error(h, "gpmpc_set_hyper: zero length scale"); return GPMPC_ERR_ARG; }
            h->hyper[(size_t)a * m + q] = v;
        }
    CUDA_TRY(cudaMemcpyAsync(h->dHyp, h->hyper.data(), h->hyper.size() * 8, cudaMemcpyHostToDevice, h->st));
    CUDA_TRY(cudaStreamSynchronize(h->st));
    h->has_hyper = true; h->factorized = false;
    return GPMPC_OK;
}

static int local_index(gpmpc_handle_t h, int a)
{
    if (a < h->a0 || a >= h->a0 + h->nloc) { set_error(h, "output %d is not owned by this handle [%d,%d)", a, h->a0, h->a0 + h->nloc); return -1; }
    return a - h->a0;
}

static int ensure_nlml_scratch(gpmpc_handle_t h)
{
    if (!h->dU) { ALLOC(h->dU, slab(h)); }
    if (!h->dKinv) { ALLOC(h->dKinv, slab(h)); }
    if (!h->dGradPart) {
        const int T = h->Npad / KB_TILE;
        ALLOC(h->dGradPart, (long long)T * (T + 1) / 2 * (h->Nx + 2));
    }
    return GPMPC_OK;
}

static int extract_to_host(gpmpc_handle_t h, const double* src, double* dst, int mode)
{
    const int N = h->N;
    if (!h->dKinv) { int rc = ensure_nlml_scratch(h); if (rc) return rc; }
    // stage through dU (N*N fits: Npad >= N)
    dim3 g((N + 127) / 128, N);
    extract_kernel<<<g, 128, 0, h->st>>>(src, h->Npad, h->dU, N, mode);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(dst, h->dU, (size_t)N * N * 8, cudaMemcpyDeviceToHost, h->st));
    CUDA_TRY(cudaStreamSynchronize(h->st));
    return GPMPC_OK;
}

extern "C" int gpmpc_build_K(gpmpc_handle_t h, int a, double* K_out)
{
    if (!h) return GPMPC_ERR_ARG;
    if (!h->has_data || !h->has_hyper) { set_error(h, "gpmpc_build_K: set_data and set_hyper first"); return GPMPC_ERR_STATE; }
    CUDA_TRY(cudaSetDevice(h->device));
    const int al = local_index(h, a);
    if (al < 0) return GPMPC_ERR_ARG;
    int rc = ensure_nlml_scratch(h);
    if (rc) return rc;
    const double zero = 0.0;
    CUDA_TRY(cudaMemcpyAsync(h->dJit + al, &zero, 8, cudaMemcpyHostToDevice, h->st));
    rc = launch_kbuild(h, h->dHyp + (long long)al * (h->Nx + 2), h->dJit + al, h->dKinv, 1, 1);
    if (rc) return rc;
    if (K_out) return extract_to_host(h, h->dKinv, K_out, 0);
    CUDA_TRY(cudaStreamSynchronize(h->st));
    return GPMPC_OK;
}

extern "C" int gpmpc_factorize(gpmpc_handle_t h, double jitter, int* info)
{
    if (!h) return GPMPC_ERR_ARG;
    if (!h->has_data || !h->has_hyper) { set_error(h, "gpmpc_factorize: set_data and set_hyper first"); return GPMPC_ERR_STATE; }
    CUDA_TRY(cudaSetDevice(h->device));
    NvtxRange nvtx_r("gpmpc.factorize");
    const int nl = h->nloc;
    CUDA_TRY(cudaMemsetAsync(h->dJit, 0, nl * sizeof(double), h->st));
    CUDA_TRY(cudaMemsetAsync(h->dInfo, 0, nl * sizeof(int), h->st));
    int rc = launch_kbuild(h, h->dHyp, h->dJit, h->dL, nl, 0);
    if (rc) return rc;
    rc = potrf_inv_rec(h, h->dL, h->dLi, slab(h), slab(h), h->dInfo, 0, h->Npad, nl);
    if (rc) return rc;
    std::vector<int> inf(nl, 0);
    CUDA_TRY(cudaMemcpyAsync(inf.data(), h->dInfo, nl * sizeof(int), cudaMemcpyDeviceToHost, h->st));
    CUDA_TRY(cudaStreamSynchronize(h->st));
    int worst = GPMPC_OK;
    for (int a = 0; a < nl; ++a) {
        h->jitter_used[a] = 0;
        if (inf[a] != 0) {      // optimize.py:483-488: add jitter once, retry, else propagate
            int used = 0;
            rc = factor_one(h, a, h->dHyp + (long long)a * (h->Nx + 2), jitter, &used);
            h->jitter_used[a] = used;
            if (rc == GPMPC_ERR_NOTPD) { worst = rc; set_error(h, "output %d: K not positive definite even with jitter %g (pivot %d)", h->a0 + a, jitter, used - 1); }
            else if (rc) return rc;
        }
        if (info) info[a] = h->jitter_used[a];
    }
    if (worst) return worst;
    rc = launch_alpha(h, 0, nl);
    if (rc) return rc;
    std::vector<double> res(2 * nl);
    CUDA_TRY(cudaMemcpyAsync(res.data(), h->dRes, 2 * nl * 8, cudaMemcpyDeviceToHost, h->st));
    CUDA_TRY(cudaStreamSynchronize(h->st));
    for (int a = 0; a < nl; ++a) { h->logdet[a] = res[2 * a]; h->yalpha[a] = res[2 * a + 1]; }
    h->factorized = true; h->u_valid = false; h->sparse = false;
    return GPMPC_OK;
}

// K^-1 (lower) of local output al into dKinv:  U = Li^T,  K^-1 = U U^T
static int compute_kinv(gpmpc_handle_t h, int al)
{
    int rc = ensure_nlml_scratch(h);
    if (rc) return rc;
    const int np = h->Npad;
    dim3 g(np / 32, np / 32), b(32, 8);
    transpose_lower_kernel<<<g, b, 0, h->st>>>(h->dLi + (long long)al * slab(h), h->dU, np, np / 32);
    CUDA_TRY(cudaGetLastError());
    GemmParams p;
    memset(&p, 0, sizeof(p));
    p.A = h->dU; p.lda = np; p.B = h->dU; p.ldb = np; p.C = h->dKinv; p.ldc = np;
    p.mt = np / 128; p.nt = np / 128; p.K = np; p.alpha = 1.0; p.beta = 0.0;
    p.kflags = GEMM_KI_GE | GEMM_KJ_GE; p.lower = 1;
    CUDA_TRY(gemm128(h, true, p, 1));
    return GPMPC_OK;
}

// ------------------------------------------------------------------------------------
// FITC sparse model (the reference's GP.sparse, gp_class.py:682-689).  The handle's own M points are the inducing points;
// the N training points stream through the GPU in column panels of opt_fitc_panel points:
//   Luu = chol(Kuu + jitter sf2 I),  V = Luu^-1 Kuf,  Lambda = diag(Kff - V^T V) + sn2 I,  A = I + V Lambda^-1 V^T = LA LA^T
//   B = I - A^-1 = Luu^T K~^-1 Luu,  S^T S = B (reverse Cholesky),  R = S Luu^-1,  alpha_s = Luu^-T LA^-T LA^-1 V Lambda^-1 y
// R goes to the L^-1 slab and alpha_s to alpha, so every predict kernel evaluates the FITC predictive distribution.
// ------------------------------------------------------------------------------------
#define FITC_N_MAX (1 << 30)          // panel column indices and the padded column count stay in int
#define FITC_B_SHIFT 1e-10            // retry shift of B: moves the variance by at most FITC_B_SHIFT * Qss <= 1e-10 sf2

// build buffers: allocated per call, freed on every return path (only L, L^-1 and alpha outlive the build)
struct FitcBufs {
    gpmpc_handle_t h;
    double *X = nullptr, *Y = nullptr, *Kuf = nullptr, *V = nullptr, *P[4] = {nullptr, nullptr, nullptr, nullptr};
    double *b = nullptr, *t = nullptr, *w = nullptr, *part = nullptr, *res = nullptr, *hyp = nullptr;
    std::vector<cudaEvent_t> ev;        // phase boundaries: [Kuu start, Kuu end, 4 per panel..., panels end, build end]
    explicit FitcBufs(gpmpc_handle_t hh) : h(hh) {}
    ~FitcBufs()
    {
        cudaStreamSynchronize(h->st);
        for (cudaEvent_t e : ev) cudaEventDestroy(e);
        double* bufs[] = {X, Y, Kuf, V, P[0], P[1], P[2], P[3], b, t, w, part, res, hyp};
        for (double* q : bufs) if (q) cudaFree(q);
    }
};

static int fitc_check_info(gpmpc_handle_t h, const char* what, std::vector<int>& inf)
{
    CUDA_TRY(cudaMemcpyAsync(inf.data(), h->dInfo, inf.size() * sizeof(int), cudaMemcpyDeviceToHost, h->st));
    CUDA_TRY(cudaStreamSynchronize(h->st));
    for (size_t a = 0; a < inf.size(); ++a)
        if (inf[a]) {
            set_error(h, "gpmpc_fitc: output %d: %s is not positive definite (pivot %d)", h->a0 + (int)a, what, inf[a] - 1);
            return GPMPC_ERR_NOTPD;
        }
    return GPMPC_OK;
}

extern "C" int gpmpc_fitc(gpmpc_handle_t h, int N, const double* X, const double* Y, double jitter, int* info, double* nll)
{
    if (!h) return GPMPC_ERR_ARG;
    if (!X || !Y || N < 1 || N > FITC_N_MAX || !(jitter >= 0.0)) {
        set_error(h, "gpmpc_fitc: need X, Y, 1 <= N <= %d (got %d) and jitter >= 0", FITC_N_MAX, N);
        return GPMPC_ERR_ARG;
    }
    if (!h->has_data || !h->has_hyper) { set_error(h, "gpmpc_fitc: set_data (the inducing points) and set_hyper first"); return GPMPC_ERR_STATE; }
    if (h->opt_refine) { set_error(h, "gpmpc_fitc: option refine needs the dense factor; switch it off first"); return GPMPC_ERR_STATE; }
    const int nl = h->nloc, Nx = h->Nx, M = h->N, mp = h->Npad, m = Nx + 2;
    for (int a = 0; a < nl; ++a)
        if (!(h->hyper[(size_t)a * m + Nx + 1] != 0.0)) { set_error(h, "gpmpc_fitc: output %d has sn = 0 (FITC needs noise)", h->a0 + a); return GPMPC_ERR_ARG; }
    CUDA_TRY(cudaSetDevice(h->device));
    NvtxRange nvtx_r("gpmpc.fitc");
    h->factorized = false; h->sparse = false; h->u_valid = false;
    const int nb = h->opt_fitc_panel, npan = (int)(((long long)N + nb - 1) / nb), cpp = nb / 32;
    const long long Nq = (long long)npan * nb, sK = (long long)mp * nb, sP = slab(h), nparts = (long long)npan * cpp;
    FitcBufs f(h);
    ALLOC(f.X, (long long)Nx * Nq); ALLOC(f.Y, (long long)nl * Nq);
    ALLOC(f.Kuf, nl * sK); ALLOC(f.V, nl * sK);
    for (int k = 0; k < 4; ++k) ALLOC(f.P[k], nl * sP);
    ALLOC(f.b, (long long)nl * mp); ALLOC(f.t, 2LL * nl * mp); ALLOC(f.w, (long long)nl * nb);
    ALLOC(f.part, 2 * nl * nparts); ALLOC(f.res, nl); ALLOC(f.hyp, (long long)nl * m);
    {   // training set, transposed (X^T: Nx x Nq) and per owned output (Y: nl x Nq), zero padded to whole panels
        std::vector<double> xt((size_t)Nx * Nq, 0.0), yl((size_t)nl * Nq, 0.0);
        for (long long i = 0; i < N; ++i)
            for (int d = 0; d < Nx; ++d) xt[(size_t)d * Nq + i] = X[(size_t)i * Nx + d];
        for (int a = 0; a < nl; ++a)
            for (long long i = 0; i < N; ++i) yl[(size_t)a * Nq + i] = Y[(size_t)i * h->Ny + h->a0 + a];
        CUDA_TRY(cudaMemcpyAsync(f.X, xt.data(), xt.size() * 8, cudaMemcpyHostToDevice, h->st));
        CUDA_TRY(cudaMemcpyAsync(f.Y, yl.data(), yl.size() * 8, cudaMemcpyHostToDevice, h->st));
        CUDA_TRY(cudaStreamSynchronize(h->st));
    }
    f.ev.assign(4 * npan + 4, nullptr);
    for (auto& e : f.ev) CUDA_TRY(cudaEventCreate(&e));
    std::vector<int> inf(nl, 0);
    // 1. Kuu + jitter sf2 I (the K build with sn = 0) -> Luu (L slab), Luu^-1 (P0)
    {
        std::vector<double> hk(h->hyper), jit(nl);
        for (int a = 0; a < nl; ++a) {
            const double sf = hk[(size_t)a * m + Nx];
            hk[(size_t)a * m + Nx + 1] = 0.0;
            jit[a] = jitter * sf * sf;
        }
        CUDA_TRY(cudaMemcpyAsync(f.hyp, hk.data(), hk.size() * 8, cudaMemcpyHostToDevice, h->st));
        CUDA_TRY(cudaMemcpyAsync(h->dJit, jit.data(), nl * 8, cudaMemcpyHostToDevice, h->st));
        CUDA_TRY(cudaStreamSynchronize(h->st));
    }
    CUDA_TRY(cudaMemsetAsync(h->dInfo, 0, nl * sizeof(int), h->st));
    CUDA_TRY(cudaEventRecord(f.ev[0], h->st));
    int rc = launch_kbuild(h, f.hyp, h->dJit, h->dL, nl, 0);
    if (rc) return rc;
    rc = potrf_inv_rec(h, h->dL, f.P[0], sP, sP, h->dInfo, 0, mp, nl);
    if (rc) return rc;
    CUDA_TRY(cudaEventRecord(f.ev[1], h->st));
    rc = fitc_check_info(h, "Kuu + jitter sf2 I", inf);
    if (rc) return rc;
    // 2. panels: Kuf -> V = Luu^-1 Kuf -> column pass -> b += Vs w, Phi += Vs Vs^T (Phi in P1)
    {
        const int KD = (Nx + 3) & ~3, S = ((KD >> 2) & 1) ? KD : KD + 4;
        const int smem = (2 * KB2_TILE * S + 2 * KB2_TILE + 256) * 8;
        CUDA_TRY(cudaFuncSetAttribute(kcross_dmma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        for (int p = 0; p < npan; ++p) {
            const long long c0 = (long long)p * nb;
            const int ncols = (int)std::min<long long>(nb, N - c0);
            CUDA_TRY(cudaEventRecord(f.ev[2 + 4 * p], h->st));
            dim3 gk((mp / KB2_TILE) * (nb / KB2_TILE), 1, nl);
            kcross_dmma_kernel<<<gk, 256, smem, h->st>>>(h->dXT, mp, M, f.X + c0, Nq, ncols, Nx, h->dMu, h->dHyp, m,
                                                          f.Kuf, nb, sK, nb / KB2_TILE);
            CUDA_TRY(cudaGetLastError());
            GemmParams q;
            memset(&q, 0, sizeof(q));
            q.A = f.P[0]; q.lda = mp; q.sA = sP;                        // Luu^-1: lower
            q.B = f.Kuf; q.ldb = nb; q.sB = sK;
            q.C = f.V; q.ldc = nb; q.sC = sK;
            q.mt = mp / 128; q.nt = nb / 128; q.K = mp; q.alpha = 1.0; q.beta = 0.0; q.kflags = GEMM_KI_LE;
            CUDA_TRY(cudaEventRecord(f.ev[3 + 4 * p], h->st));
            CUDA_TRY(gemm128(h, false, q, nl));
            CUDA_TRY(cudaEventRecord(f.ev[4 + 4 * p], h->st));
            fitc_column_kernel<<<dim3(cpp, nl), 256, 0, h->st>>>(f.V, nb, sK, mp, ncols, h->dHyp, m, Nx, f.Y + c0, Nq,
                                                                 f.w, nb, f.part + 2LL * p * cpp, 2 * nparts);
            CUDA_TRY(cudaGetLastError());
            fitc_bvec_kernel<<<dim3(mp / 8, nl), 256, 0, h->st>>>(f.V, nb, sK, nb, f.w, nb, f.b, mp);
            CUDA_TRY(cudaGetLastError());
            CUDA_TRY(cudaEventRecord(f.ev[5 + 4 * p], h->st));
            memset(&q, 0, sizeof(q));
            q.A = f.V; q.lda = nb; q.sA = sK;
            q.B = f.V; q.ldb = nb; q.sB = sK;
            q.C = f.P[1]; q.ldc = mp; q.sC = sP; q.Cin = f.P[1]; q.ldcin = mp; q.sCin = sP;
            q.mt = mp / 128; q.nt = mp / 128; q.K = nb; q.alpha = 1.0; q.beta = 1.0; q.lower = 1;
            CUDA_TRY(gemm128(h, true, q, nl));
        }
    }
    CUDA_TRY(cudaEventRecord(f.ev[2 + 4 * npan], h->st));
    // 3. A = I + Phi -> LA (P1), LA^-1 (P2)
    fitc_add_identity_kernel<<<dim3((mp + 255) / 256, nl), 256, 0, h->st>>>(f.P[1], mp, sP, mp);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemsetAsync(h->dInfo, 0, nl * sizeof(int), h->st));
    rc = potrf_inv_rec(h, f.P[1], f.P[2], sP, sP, h->dInfo, 0, mp, nl);
    if (rc) return rc;
    rc = fitc_check_info(h, "A = I + V Lambda^-1 V^T", inf);
    if (rc) return rc;
    // 6./7. t = LA^-1 b, NLML, alpha_s = Luu^-T (LA^-T t)   (enqueued before P1 / P2 are reused below)
    double* t1 = f.t;
    double* t2 = f.t + (long long)nl * mp;
    trmv_lower_kernel<<<dim3((mp + 7) / 8, 1, nl), 256, 0, h->st>>>(f.P[2], mp, sP, f.b, mp, t1, mp, mp);
    CUDA_TRY(cudaGetLastError());
    fitc_nll_kernel<<<nl, 256, 0, h->st>>>(f.part, 2 * nparts, (int)nparts, f.P[1], mp, sP, t1, mp, mp, f.res);
    CUDA_TRY(cudaGetLastError());
    trmv_lower_T_kernel<<<dim3(mp / 32, 1, nl), 256, 0, h->st>>>(f.P[2], mp, sP, t1, mp, t2, mp, mp);
    CUDA_TRY(cudaGetLastError());
    trmv_lower_T_kernel<<<dim3(mp / 32, 1, nl), 256, 0, h->st>>>(f.P[0], mp, sP, t2, mp, h->dAlpha, mp, mp);
    CUDA_TRY(cudaGetLastError());
    // 4. X = LA^-T LA^-1 (lower, P1) through U = (LA^-1)^T (P3), the product compute_kinv uses; B' = J (I - X) J (P3)
    for (int a = 0; a < nl; ++a) {
        transpose_lower_kernel<<<dim3(mp / 32, mp / 32), dim3(32, 8), 0, h->st>>>(f.P[2] + a * sP, f.P[3] + a * sP, mp, mp / 32);
        CUDA_TRY(cudaGetLastError());
    }
    {
        GemmParams q;
        memset(&q, 0, sizeof(q));
        q.A = f.P[3]; q.lda = mp; q.sA = sP; q.B = f.P[3]; q.ldb = mp; q.sB = sP; q.C = f.P[1]; q.ldc = mp; q.sC = sP;
        q.mt = mp / 128; q.nt = mp / 128; q.K = mp; q.alpha = 1.0; q.beta = 0.0;
        q.kflags = GEMM_KI_GE | GEMM_KJ_GE; q.lower = 1;
        CUDA_TRY(gemm128(h, true, q, nl));
    }
    const dim3 gf(mp / 32, mp / 32, nl), bf(32, 8);
    fitc_flip_kernel<<<gf, bf, 0, h->st>>>(f.P[1], f.P[3], mp, sP, M, -1.0, 1.0);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemsetAsync(h->dInfo, 0, nl * sizeof(int), h->st));
    rc = potrf_inv_rec(h, f.P[3], f.P[2], sP, sP, h->dInfo, 0, mp, nl);       // G (P3); G^-1 (P2) is not used
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(inf.data(), h->dInfo, nl * sizeof(int), cudaMemcpyDeviceToHost, h->st));
    CUDA_TRY(cudaStreamSynchronize(h->st));
    std::vector<int> shifted(nl, 0);
    for (int a = 0; a < nl; ++a) {
        if (!inf[a]) continue;
        // a non-positive pivot (B is only semi-definite, e.g. duplicate inducing points give phi = 0): one retry with B + eps I
        shifted[a] = 1;
        fitc_flip_kernel<<<dim3(mp / 32, mp / 32, 1), bf, 0, h->st>>>(f.P[1] + a * sP, f.P[3] + a * sP, mp, sP, M, -1.0, 1.0 + FITC_B_SHIFT);
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaMemsetAsync(h->dInfo + a, 0, sizeof(int), h->st));
        rc = potrf_inv_rec(h, f.P[3] + a * sP, f.P[2] + a * sP, sP, sP, h->dInfo + a, 0, mp, 1);
        if (rc) return rc;
        int i2 = 0;
        CUDA_TRY(cudaMemcpyAsync(&i2, h->dInfo + a, sizeof(int), cudaMemcpyDeviceToHost, h->st));
        CUDA_TRY(cudaStreamSynchronize(h->st));
        if (i2) {
            set_error(h, "gpmpc_fitc: output %d: B = I - A^-1 is not positive definite even with the shift %g (pivot %d)",
                      h->a0 + a, FITC_B_SHIFT, i2 - 1);
            return GPMPC_ERR_NOTPD;
        }
    }
    // 5. S = J G^T J (P1);  R = S Luu^-1 into the L^-1 slab: lower, exact zeros above the diagonal, identity tail
    fitc_flip_kernel<<<gf, bf, 0, h->st>>>(f.P[3], f.P[1], mp, sP, M, 1.0, 0.0);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemsetAsync(h->dLi, 0, (size_t)nl * sP * 8, h->st));
    {
        GemmParams q;
        memset(&q, 0, sizeof(q));
        q.A = f.P[1]; q.lda = mp; q.sA = sP;                            // S: lower
        q.B = f.P[0]; q.ldb = mp; q.sB = sP;                            // Luu^-1: lower -> Bop[k][j] = 0 for k < j
        q.C = h->dLi; q.ldc = mp; q.sC = sP;
        q.mt = mp / 128; q.nt = mp / 128; q.K = mp; q.alpha = 1.0; q.beta = 0.0;
        q.kflags = GEMM_KI_LE | GEMM_KJ_GE; q.lower = 1;
        CUDA_TRY(gemm128(h, false, q, nl));
    }
    CUDA_TRY(cudaEventRecord(f.ev[3 + 4 * npan], h->st));
    std::vector<double> res(nl);
    CUDA_TRY(cudaMemcpyAsync(res.data(), f.res, nl * 8, cudaMemcpyDeviceToHost, h->st));
    CUDA_TRY(cudaStreamSynchronize(h->st));
    {
        auto el = [&](int i, int j) { float ms = 0.f; cudaEventElapsedTime(&ms, f.ev[i], f.ev[j]); return (double)ms; };
        double t[5] = {0, 0, 0, 0, 0};
        for (int p = 0; p < npan; ++p) {
            const int e = 2 + 4 * p;
            t[0] += el(e, e + 1); t[1] += el(e + 1, e + 2); t[2] += el(e + 2, e + 3); t[3] += el(e + 3, e + 4);
        }
        t[4] = el(0, 1) + el(2 + 4 * npan, 3 + 4 * npan);
        for (int k = 0; k < 5; ++k) h->fitc_ms[k] = t[k];
    }
    for (int a = 0; a < nl; ++a) {
        if (info) info[a] = shifted[a];
        if (nll) nll[a] = res[a];
        h->jitter_used[a] = 0;
    }
    h->factorized = true; h->sparse = true; h->u_valid = false;
    return GPMPC_OK;
}

template <int NXP>
static cudaError_t launch_grad(gpmpc_handle_t h, int al, const double* dHyp)
{
    const int T = h->Npad / KB_TILE;
    const int smem = 2 * h->Nx * KB_TILE * 8;
    nlml_grad_kernel<NXP><<<T * (T + 1) / 2, 256, smem, h->st>>>(h->dXT, h->Npad, h->N, h->Nx, dHyp, h->dKinv, h->Npad,
                                                                 h->dAlpha + (long long)al * h->Npad, h->dGradPart);
    return cudaGetLastError();
}

extern "C" int gpmpc_nlml(gpmpc_handle_t h, int a, const double* theta, double* nll, double* grad)
{
    if (!h || !theta || !nll) return GPMPC_ERR_ARG;
    if (!h->has_data) { set_error(h, "gpmpc_nlml: set_data first"); return GPMPC_ERR_STATE; }
    CUDA_TRY(cudaSetDevice(h->device));
    const int al = local_index(h, a);
    if (al < 0) return GPMPC_ERR_ARG;
    const int m = h->Nx + 2;
    for (int d = 0; d < h->Nx; ++d) if (theta[d] == 0.0) { set_error(h, "gpmpc_nlml: zero length scale"); return GPMPC_ERR_ARG; }
    h->factorized = false;
    NvtxRange nvtx_r("gpmpc.nlml");
    CUDA_TRY(cudaMemcpyAsync(h->dHypTmp, theta, m * 8, cudaMemcpyHostToDevice, h->st));
    int used = 0;
    int rc = factor_one(h, al, h->dHypTmp, 1e-8, &used);     // optimize.py:345-350
    if (rc) { if (rc == GPMPC_ERR_NOTPD) set_error(h, "gpmpc_nlml: K not positive definite even with jitter"); return rc; }
    rc = launch_alpha(h, al, 1);
    if (rc) return rc;
    double res[2];
    CUDA_TRY(cudaMemcpyAsync(res, h->dRes + 2 * al, 16, cudaMemcpyDeviceToHost, h->st));
    if (grad) {
        rc = compute_kinv(h, al);
        if (rc) return rc;
        cudaError_t e = (h->Nx <= 8) ? launch_grad<8>(h, al, h->dHypTmp)
                      : (h->Nx <= 16) ? launch_grad<16>(h, al, h->dHypTmp) : launch_grad<32>(h, al, h->dHypTmp);
        CUDA_TRY(e);
        const int T = h->Npad / KB_TILE;
        nlml_grad_final_kernel<<<m, 256, 0, h->st>>>(h->dGradPart, T * (T + 1) / 2, h->Nx, h->dHypTmp, h->dGrad);
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaMemcpyAsync(grad, h->dGrad, m * 8, cudaMemcpyDeviceToHost, h->st));
    }
    CUDA_TRY(cudaStreamSynchronize(h->st));
    *nll = 0.5 * res[1] + 0.5 * res[0];                      // optimize.py:355
    return GPMPC_OK;
}

extern "C" int gpmpc_fitc_timings(gpmpc_handle_t h, double* ms5)
{
    if (!h || !ms5) return GPMPC_ERR_ARG;
    if (!h->sparse) { set_error(h, "gpmpc_fitc_timings: no FITC build on this handle"); return GPMPC_ERR_STATE; }
    for (int k = 0; k < 5; ++k) ms5[k] = h->fitc_ms[k];
    return GPMPC_OK;
}

extern "C" int gpmpc_get(gpmpc_handle_t h, int what, int a, double* dst)
{
    if (!h || !dst) return GPMPC_ERR_ARG;
    CUDA_TRY(cudaSetDevice(h->device));
    const int al = local_index(h, a);
    if (al < 0) return GPMPC_ERR_ARG;
    if (h->sparse && h->factorized && (what == GPMPC_GET_CHOL || what == GPMPC_GET_K || what == GPMPC_GET_INVK || what == GPMPC_GET_LOGDET)) {
        set_error(h, "gpmpc_get: selector %d has no FITC counterpart (the handle holds a sparse model: GET_ALPHA / GET_LINV)", what);
        return GPMPC_ERR_STATE;
    }
    if (what == GPMPC_GET_K) return gpmpc_build_K(h, a, dst);
    if (what == GPMPC_GET_ALPHA_NLML) {       // alpha of the last gpmpc_nlml(a, theta) evaluation
        CUDA_TRY(cudaMemcpyAsync(dst, h->dAlpha + (long long)al * h->Npad, h->N * 8, cudaMemcpyDeviceToHost, h->st));
        CUDA_TRY(cudaStreamSynchronize(h->st));
        return GPMPC_OK;
    }
    if (!h->factorized) { set_error(h, "gpmpc_get: call gpmpc_factorize first"); return GPMPC_ERR_STATE; }
    switch (what) {
    case GPMPC_GET_CHOL: return extract_to_host(h, h->dL + (long long)al * slab(h), dst, 1);
    case GPMPC_GET_LINV: return extract_to_host(h, h->dLi + (long long)al * slab(h), dst, 1);
    case GPMPC_GET_ALPHA:
        CUDA_TRY(cudaMemcpyAsync(dst, h->dAlpha + (long long)al * h->Npad, h->N * 8, cudaMemcpyDeviceToHost, h->st));
        CUDA_TRY(cudaStreamSynchronize(h->st));
        return GPMPC_OK;
    case GPMPC_GET_LOGDET: dst[0] = h->logdet[al]; return GPMPC_OK;
    case GPMPC_GET_INVK: {
        int rc = compute_kinv(h, al);
        if (rc) return rc;
        // dKinv -> host through dU is not possible (dU is an input of compute_kinv but free now)
        return extract_to_host(h, h->dKinv, dst, 2);
    }
    default: set_error(h, "gpmpc_get: unknown selector %d", what); return GPMPC_ERR_ARG;
    }
}

extern "C" int gpmpc_set_option(gpmpc_handle_t h, const char* name, double value)
{
    if (!h || !name) return GPMPC_ERR_ARG;
    if (!strcmp(name, "refine")) {
        if (h->sparse) { set_error(h, "refine: a FITC model keeps Luu, not the factor of R, in the L slab"); return GPMPC_ERR_STATE; }
        h->opt_refine = value != 0.0; return GPMPC_OK;
    }
    if (!strcmp(name, "fitc_panel")) {       // training points per FITC panel (multiple of 128)
        const int v = (int)value;
        if (v < 128 || v % 128 || v > 65536) { set_error(h, "fitc_panel must be a multiple of 128 in [128, 65536]"); return GPMPC_ERR_ARG; }
        h->opt_fitc_panel = v; return GPMPC_OK;
    }
    if (!strcmp(name, "predict_ctas")) {       // persistent grid of the predict product (0 = 2 per SM)
        const int v = (int)value;
        if (v < 0 || v > PSK_MAX_CTAS) { set_error(h, "predict_ctas must be in [0, %d]", PSK_MAX_CTAS); return GPMPC_ERR_ARG; }
        h->opt_predict_ctas = v; return GPMPC_OK;
    }
    if (!strcmp(name, "zero_copy")) { h->opt_zero_copy = value != 0.0; return GPMPC_OK; }
    if (!strcmp(name, "peer_timeout_s")) { h->opt_peer_timeout_s = value > 0.0 ? value : 60.0; return GPMPC_OK; }
    if (!strcmp(name, "gemm_variant")) { h->opt_gemm_variant = (int)value; return GPMPC_OK; }
    if (!strcmp(name, "small_tiles")) { h->opt_small_tiles = (int)value; return GPMPC_OK; }
    if (!strcmp(name, "overlap")) { h->opt_overlap = value != 0.0; return GPMPC_OK; }
    if (!strcmp(name, "lookahead")) { h->opt_lookahead = value != 0.0; return GPMPC_OK; }
    if (!strcmp(name, "lookahead_min")) { h->opt_lookahead_min = (int)value; return GPMPC_OK; }
    if (!strcmp(name, "peer")) { h->opt_peer = value != 0.0; return GPMPC_OK; }
    if (!strcmp(name, "leaf_variant")) { h->opt_leaf_variant = (int)value; return GPMPC_OK; }
    set_error(h, "unknown option %s", name);
    return GPMPC_ERR_ARG;
}

// ------------------------------------------------------------------------------------
// predict
// ------------------------------------------------------------------------------------
static inline int ks_chunk(gpmpc_handle_t h);

static int ensure_predict_bufs(gpmpc_handle_t h, int H)
{
    const long long np = h->Npad;
    if (!h->dKST) {
        int sms = 148;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
        cudaDeviceGetAttribute(&h->clock_khz, cudaDevAttrClockRate, h->device);
        h->psk_ctas = 2 * sms;
        const long long nt = np / 128;
        ALLOC(h->dKST, (long long)h->nloc * HB * np);
        ALLOC(h->dPMJ, (long long)h->nloc * HB * ((np + ks_chunk(h) - 1) / ks_chunk(h)) * (h->Nx + 1));
        ALLOC(h->dSQ, (long long)h->nloc * HB * nt);
        ALLOC(h->dCnt, (long long)h->nloc * nt + h->nloc + 1);
    }
    {   // parked stream-K partials: two BM x 128 slots per persistent CTA
        const int want = std::max(h->psk_ctas, h->opt_predict_ctas);
        if (want > h->partCtas) {
            CUDA_TRY(cudaStreamSynchronize(h->st));
            if (h->dPart) cudaFree(h->dPart);
            h->dPart = nullptr; h->partCtas = 0;
            ALLOC(h->dPart, (long long)want * 2 * HB * PSK_BN);
            h->partCtas = want;
        }
    }
    if (h->opt_refine && !h->dR2) {
        if (!h->dV) { ALLOC(h->dV, (long long)h->nloc * HB * np); ALLOC(h->dR, (long long)h->nloc * HB * np); }
        ALLOC(h->dR2, (long long)h->nloc * HB * np);
    }
    if (H > h->Hcap) {
        CUDA_TRY(cudaStreamSynchronize(h->st));
        double* bufs[] = {h->dG, h->dIn, h->dOut};
        for (double* b : bufs) if (b) cudaFree(b);
        h->dG = h->dIn = h->dOut = nullptr;
        const long long cap = std::max(H, HB);
        const int nyp = h->nloc_max * h->world;
        const long long Nx = h->Nx, Ny = h->Ny;
        ALLOC(h->dG, (long long)nyp * cap * (Nx + 2));
        ALLOC(h->dIn, cap * Nx + cap * Nx * Nx);
        ALLOC(h->dOut, cap * (2 * Ny + Ny * Nx + Ny * Ny));
        // defined contents for the profiling selectors when every call so far went through the zero-copy path
        CUDA_TRY(cudaMemsetAsync(h->dIn, 0, (size_t)(cap * Nx + cap * Nx * Nx) * 8, h->st));
        h->dZ = h->dIn; h->dSigma = h->dIn + cap * Nx;
        h->dMean = h->dOut; h->dVar = h->dOut + cap * Ny; h->dJ = h->dOut + 2 * cap * Ny;
        h->dCov = h->dOut + 2 * cap * Ny + cap * Ny * Nx;
        h->Hcap = (int)cap;
    }
    return GPMPC_OK;
}

// Persistent stream-K launch of the fused predict product (predict_streamk.cuh)
template <int BM>
static cudaError_t psk_launch_bm(const PredictParams& p, const double* A, long long sA, const double* B, long long sB,
                                 int np, int grid, cudaStream_t st)
{
    auto kern = predict_streamk_kernel<BM>;
    constexpr int BYTES = PSK_STAGES * (BM + PSK_BN) * GEMM_BK * 8 + 2 * PSK_STAGES * 8 + 1024;
    static std::atomic<bool> configured[GPMPC_MAX_DEVICES];
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < GPMPC_MAX_DEVICES && !configured[dev].load(std::memory_order_acquire)) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, BYTES);
        if (e != cudaSuccess) return e;
        configured[dev].store(true, std::memory_order_release);
    }
    CUtensorMap tmA, tmB;
    if (!tmap_make(&tmA, A, np, BM, np, sA, p.nloc, BM)) return cudaErrorInvalidValue;
    if (!tmap_make(&tmB, B, np, np, np, sB, p.nloc, PSK_BN)) return cudaErrorInvalidValue;
    // programmatic dependent launch after the ks kernel (the kernel's griddepcontrol.wait guards its inputs)
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(PSK_THREADS); cfg.dynamicSmemBytes = BYTES; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, p, tmA, tmB);
}

static cudaError_t psk_launch(int bm, const PredictParams& p, const double* A, long long sA, const double* B, long long sB,
                              int np, int grid, cudaStream_t st)
{
    switch (bm) {
    case 8: return psk_launch_bm<8>(p, A, sA, B, sB, np, grid, st);
    case 16: return psk_launch_bm<16>(p, A, sA, B, sB, np, grid, st);
    case 24: return psk_launch_bm<24>(p, A, sA, B, sB, np, grid, st);
    case 32: return psk_launch_bm<32>(p, A, sA, B, sB, np, grid, st);
    case 40: return psk_launch_bm<40>(p, A, sA, B, sB, np, grid, st);
    case 48: return psk_launch_bm<48>(p, A, sA, B, sB, np, grid, st);
    case 56: return psk_launch_bm<56>(p, A, sA, B, sB, np, grid, st);
    default: return psk_launch_bm<64>(p, A, sA, B, sB, np, grid, st);
    }
}

// persistent grid: 2 CTAs per SM, but never fewer than 4 k-steps per CTA (measured at N=1000, 6 outputs: 296 CTAs of
// 6 steps beat 144 of 12 -- the fixed cost per CTA overlaps across SMs, the steps do not)
static int psk_grid(gpmpc_handle_t h, long long G)
{
    int ctas = h->opt_predict_ctas > 0 ? h->opt_predict_ctas : h->psk_ctas;
    ctas = std::min(ctas, PSK_MAX_CTAS);
    const long long by_work = std::max(1LL, G / 4);
    return (int)std::min<long long>(ctas, h->opt_predict_ctas > 0 ? G : by_work);
}

static void psk_base(gpmpc_handle_t h, PredictParams& p, int Hc)
{
    memset(&p, 0, sizeof(p));
    const long long nt = h->Npad / 128;
    p.nloc = h->nloc; p.nt = (int)nt; p.Hc = Hc;
    p.T = 4 * nt * (nt + 1); p.G = p.T * h->nloc;
    p.part = h->dPart;
    p.tile_cnt = h->dCnt; p.out_cnt = h->dCnt + (long long)h->nloc * nt; p.done_cnt = p.out_cnt + h->nloc;
    p.SQ = h->dSQ;
    p.hyp = h->dHyp; p.hyp_ld = h->Nx + 2; p.Nx = h->Nx;
}

// training points per CTA of the ks kernel (ks_tile_kernel): 128-point chunks below N = 8192 so small problems still fill
// the machine; 512 at large N (few partial blocks for the record sums); 1024 when a rank also holds several outputs --
// the per-CTA prologue / epilogue (~2 us of a ~5 us CTA at 512) is then amortised over twice the evaluations, and the
// 16 chunks x 7 row groups x outputs still cover the SMs.  (Nx <= 12: the chunk of X^T must leave room for 2 CTAs per SM.)
static inline int ks_chunk(gpmpc_handle_t h)
{
    if (h->Npad < 8192) return 128;
    return (h->nloc >= 2 && h->Nx <= 12) ? 1024 : 512;
}

template <int NXP, int CH>
static cudaError_t launch_ks(gpmpc_handle_t h, const double* dZc, int Hc, int bm, int nblk)
{
    auto kern = ks_tile_kernel<NXP, CH, 2>;
    const int smem = (NXP + 1) * CH * 8;
    static std::atomic<bool> conf[GPMPC_MAX_DEVICES];
    if (!conf[h->device % GPMPC_MAX_DEVICES].load(std::memory_order_acquire)) {      // static + dynamic may pass 48 KB
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
        conf[h->device % GPMPC_MAX_DEVICES].store(true, std::memory_order_release);
    }
    dim3 g(nblk, bm / 8, h->nloc);
    kern<<<g, 256, smem, h->st>>>(h->dXT, h->Npad, h->N, h->Nx, h->dHyp, h->Nx + 2, h->dAlpha, h->Npad,
                                  dZc, Hc, h->dKST, h->Npad, (long long)HB * h->Npad, h->dPMJ, nblk);
    return cudaGetLastError();
}

template <int CH>
static cudaError_t launch_ks_nx(gpmpc_handle_t h, const double* dZc, int Hc, int bm, int nblk)
{
    const int Nx = h->Nx;       // register-array extent NXP: the next even count up to 12, then 16 / 24 / 32
    if (Nx <= 4) return launch_ks<4, CH>(h, dZc, Hc, bm, nblk);
    if (Nx <= 6) return launch_ks<6, CH>(h, dZc, Hc, bm, nblk);
    if (Nx <= 8) return launch_ks<8, CH>(h, dZc, Hc, bm, nblk);
    if (Nx <= 10) return launch_ks<10, CH>(h, dZc, Hc, bm, nblk);
    if (Nx <= 12) return launch_ks<12, CH>(h, dZc, Hc, bm, nblk);
    if (CH <= 512) {
        if (Nx <= 16) return launch_ks<16, (CH <= 512 ? CH : 512)>(h, dZc, Hc, bm, nblk);
        if (Nx <= 24) return launch_ks<24, (CH <= 512 ? CH : 512)>(h, dZc, Hc, bm, nblk);
        return launch_ks<32, (CH <= 512 ? CH : 512)>(h, dZc, Hc, bm, nblk);
    }
    return cudaErrorInvalidValue;                              // ks_chunk never picks 1024 above Nx = 12
}

// bm = the chunk's row count rounded up to 8 (the rows of the product's A operand)
static cudaError_t launch_ks_any(gpmpc_handle_t h, const double* dZc, int Hc, int bm, int nblk)
{
    switch (ks_chunk(h)) {
    case 1024: return launch_ks_nx<1024>(h, dZc, Hc, bm, nblk);
    case 512: return launch_ks_nx<512>(h, dZc, Hc, bm, nblk);
    default: return launch_ks_nx<128>(h, dZc, Hc, bm, nblk);
    }
}

// rows of Amat (h-major, stride HB*np per output) times T^T with T = Li or L (lower triangular):
// the solved rows go to Vout (may be null), their per-tile squared norms to dSQ
static int tri_product(gpmpc_handle_t h, const double* Amat, const double* T, int bm, int Hc, double* Vout)
{
    const int np = h->Npad;
    PredictParams p;
    psk_base(h, p, Hc);
    p.Vout = Vout; p.sV = (long long)HB * np; p.ldv = np;
    CUDA_TRY(psk_launch(bm, p, Amat, (long long)HB * np, T, slab(h), np, psk_grid(h, p.G), h->st));
    return GPMPC_OK;
}

// r = ks - L v   (elementwise epilogue of the refinement residual) and v += dv
__global__ void axpby_rows_kernel(const double* __restrict__ x, const double* __restrict__ y, double a, double b,
                                  double* __restrict__ out, long long rowlen, long long srow, int rows)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int r = blockIdx.y, bz = blockIdx.z;
    if (i >= rowlen || r >= rows) return;
    const long long o = (long long)bz * srow + (long long)r * rowlen + i;
    out[o] = a * x[o] + b * y[o];
}

static int predict_core(gpmpc_handle_t h, int method, int H, const double* dZ, const double* dSigma, int spp,
                        double* d_mean, double* d_var, double* d_cov, double* d_jac)
{
    const int np = h->Npad, Nx = h->Nx;
    const int nblk_mj = (np + ks_chunk(h) - 1) / ks_chunk(h);
    NvtxRange nvtx_r("gpmpc.predict");
    // fused epilogue + all-gather over peer memory when the exchange block is attached
    const int use_peers = (h->world > 1 && h->peer_ready && h->opt_peer && H <= h->peerHcap) ? 1 : 0;
    const int nccl_gather = (h->world > 1 && !use_peers) ? 1 : 0;
    const long long timeout_clocks = (long long)(h->opt_peer_timeout_s * 1e3 * (double)h->clock_khz);
    PeerArgs pa;
    memset(&pa, 0, sizeof(pa));
    if (use_peers) {
        h->peer_step += 1;
        for (int r = 0; r < h->world; ++r) pa.base[r] = h->peerBase[r];
        pa.world = h->world; pa.rank = h->rank;
        pa.goff = 2 * GPMPC_MAXW + (long long)(h->peer_step & 1) * h->peerGsz;
        pa.flag_idx = (int)(h->peer_step & 1) * GPMPC_MAXW + h->rank;
        pa.step = h->peer_step;
        pa.timeout_clocks = timeout_clocks;
    }
    AssembleArgs as;
    memset(&as, 0, sizeof(as));
    as.G = use_peers ? h->dPeerBlock + pa.goff : h->dG;
    as.Ny = h->Ny; as.Nx = Nx; as.H = H; as.method_ta = (method == GPMPC_METHOD_TA);
    as.Sigma = dSigma; as.sigma_per_point = spp;
    as.mean = d_mean; as.var = d_var; as.J = d_jac; as.cov = d_cov;
    as.flags = use_peers ? reinterpret_cast<const unsigned long long*>(h->dPeerBlock) + (h->peer_step & 1) * GPMPC_MAXW : nullptr;
    as.world = h->world; as.step = h->peer_step; as.status = h->dPeerStatus; as.timeout_clocks = timeout_clocks;
    // one chunk and no NCCL call in between: the product kernel's last CTA assembles too (2 launches per step)
    // (it keeps J Sigma for all H points in the pipeline's shared memory: H Ny Nx doubles, >= 68 KB available)
    const bool fused_assemble = (H <= HB) && !nccl_gather && ((long long)H * h->Ny * Nx * 8 <= 64 * 1024);
    {   // gather records next to J Sigma in the product kernel's stage buffers (PSK_STAGES (bm + 128) 16 doubles)
        const long long bm1 = (std::min(H, HB) + 7) / 8 * 8;
        as.stage_g = (assemble_rows_doubles(H, h->Ny, Nx) <= (long long)PSK_STAGES * (bm1 + PSK_BN) * GEMM_BK) ? 1 : 0;
    }
    for (int h0 = 0; h0 < H; h0 += HB) {
        const int Hc = std::min(HB, H - h0);
        const int bm = (Hc + 7) / 8 * 8;
        const bool last_chunk = (h0 + HB >= H);
        const double* dZc = dZ + (long long)h0 * Nx;
        CUDA_TRY(launch_ks_any(h, dZc, Hc, bm, nblk_mj));
        PredictParams p;
        psk_base(h, p, Hc);
        p.finalize = 1;
        p.PMJ = h->dPMJ; p.nblk_mj = nblk_mj;
        p.Gloc = h->dG; p.slot0 = h->a0; p.Htot = H; p.h0 = h0;
        p.pa = pa; p.use_peers = use_peers; p.publish = last_chunk ? 1 : 0;
        p.as = as; p.do_assemble = (fused_assemble && !h->opt_refine) ? 1 : 0;
        if (!h->opt_refine) {
            CUDA_TRY(psk_launch(bm, p, h->dKST, (long long)HB * np, h->dLi, slab(h), np, psk_grid(h, p.G), h->st));
        } else {
            // v1 = Li ks ; r = ks - L v1 ; v = v1 + Li r   (one step of iterative refinement)
            int rc = tri_product(h, h->dKST, h->dLi, bm, Hc, h->dV);
            if (rc) return rc;
            rc = tri_product(h, h->dV, h->dL, bm, Hc, h->dR);                  // dR = L v1
            if (rc) return rc;
            dim3 g((np + 255) / 256, bm, h->nloc);
            axpby_rows_kernel<<<g, 256, 0, h->st>>>(h->dKST, h->dR, 1.0, -1.0, h->dR, np, (long long)HB * np, bm);
            CUDA_TRY(cudaGetLastError());
            rc = tri_product(h, h->dR, h->dLi, bm, Hc, h->dR2);                // dR2 = Li r
            if (rc) return rc;
            axpby_rows_kernel<<<g, 256, 0, h->st>>>(h->dV, h->dR2, 1.0, 1.0, h->dV, np, (long long)HB * np, bm);
            CUDA_TRY(cudaGetLastError());
            sq_rows_kernel<<<dim3(np / 128, Hc, h->nloc), 128, 0, h->st>>>(h->dV, np, (long long)HB * np, h->dSQ, np / 128);
            CUDA_TRY(cudaGetLastError());
            finalize_kernel<<<h->nloc, PSK_THREADS, 0, h->st>>>(p);
            CUDA_TRY(cudaGetLastError());
        }
    }
    if (nccl_gather) {
        const size_t cnt = (size_t)h->nloc_max * H * (Nx + 2);
        int r = g_nccl.AllGather(h->dG + (size_t)h->rank * cnt, h->dG, cnt, 8 /* ncclFloat64 */, h->comm, h->st);
        if (r) { set_error(h, "ncclAllGather failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?"); return GPMPC_ERR_NCCL; }
    }
    if (!fused_assemble || h->opt_refine) {
        const int smem = (2 * h->Ny * Nx + h->Ny) * 8;
        assemble_kernel<<<std::min(H, 2048), 128, smem, h->st>>>(as);
        CUDA_TRY(cudaGetLastError());
    }
    return GPMPC_OK;
}

// ------------------------------------------------------------------------------------
// 'EM' exact moment matching (gp_functions.py:344-418): small dense helpers on the host
// (Nx <= 32), everything O(N), O(N^2) on the GPU
// ------------------------------------------------------------------------------------
static bool lu_factor(int n, double* A, int* piv, double* det)
{
    double d = 1.0;
    for (int k = 0; k < n; ++k) {
        int p = k; double mx = fabs(A[k * n + k]);
        for (int i = k + 1; i < n; ++i) if (fabs(A[i * n + k]) > mx) { mx = fabs(A[i * n + k]); p = i; }
        piv[k] = p;
        if (mx == 0.0) { *det = 0.0; return false; }
        if (p != k) { for (int j = 0; j < n; ++j) std::swap(A[k * n + j], A[p * n + j]); d = -d; }
        d *= A[k * n + k];
        for (int i = k + 1; i < n; ++i) {
            const double f = A[i * n + k] / A[k * n + k];
            A[i * n + k] = f;
            for (int j = k + 1; j < n; ++j) A[i * n + j] -= f * A[k * n + j];
        }
    }
    *det = d;
    return true;
}

static void lu_solve(int n, const double* LU, const int* piv, double* B, int m)
{
    for (int k = 0; k < n; ++k) if (piv[k] != k) for (int j = 0; j < m; ++j) std::swap(B[k * m + j], B[piv[k] * m + j]);
    for (int k = 0; k < n; ++k)
        for (int i = k + 1; i < n; ++i) { const double f = LU[i * n + k]; for (int j = 0; j < m; ++j) B[i * m + j] -= f * B[k * m + j]; }
    for (int k = n - 1; k >= 0; --k) {
        for (int j = 0; j < m; ++j) B[k * m + j] /= LU[k * n + k];
        for (int i = 0; i < k; ++i) { const double f = LU[i * n + k]; for (int j = 0; j < m; ++j) B[i * m + j] -= f * B[k * m + j]; }
    }
}

// pack the per-output / per-pair Nx x Nx quantities of one test point (layout: kernels.cuh)
static int em_prepare_point(gpmpc_handle_t h, const double* S, double* out)
{
    const int Nx = h->Nx, Ny = h->Ny, nn = Nx * Nx, m = Nx + 2;
    std::vector<double> R(nn), B(nn), lc(Ny);
    std::vector<int> piv(Nx);
    double det = 0.0;
    for (int a = 0; a < Ny; ++a) {
        const double* hp = &h->hyper[(size_t)a * m];
        for (int i = 0; i < Nx; ++i) for (int j = 0; j < Nx; ++j) R[i * Nx + j] = S[i * Nx + j] + (i == j ? hp[i] * hp[i] : 0.0);
        if (!lu_factor(Nx, R.data(), piv.data(), &det) || !(det > 0.0)) { set_error(h, "EM: Sigma + Lambda is not positive definite"); return GPMPC_ERR_ARG; }
        for (int i = 0; i < nn; ++i) B[i] = 0.0;
        for (int i = 0; i < Nx; ++i) B[i * Nx + i] = 1.0;
        lu_solve(Nx, R.data(), piv.data(), B.data(), Nx);                 // iR = (Sigma + Lambda)^-1   (:383-385)
        double* o = out + (size_t)a * (2 * nn + 2);
        memcpy(o, B.data(), nn * 8);
        double pe = 1.0;
        for (int d = 0; d < Nx; ++d) pe *= hp[d];
        o[nn] = hp[Nx] * hp[Nx] / sqrt(det) * pe;                         // c (:386-387)
        // G_a = Lambda^-1 Sigma (Sigma + Lambda)^-1  (= Lambda^-1 - (Sigma+Lambda)^-1, formed without the subtraction)
        for (int i = 0; i < Nx; ++i)
            for (int j = 0; j < Nx; ++j) {
                double sacc = 0.0;
                for (int k = 0; k < Nx; ++k) sacc += S[i * Nx + k] * B[k * Nx + j];
                o[nn + 1 + i * Nx + j] = sacc / (hp[i] * hp[i]);
            }
        // lc_a = log sf2_a - log c_a = 1/2 log det(I + Sigma Lambda^-1): determinant of I + small, not a difference of logs
        for (int i = 0; i < Nx; ++i) for (int j = 0; j < Nx; ++j) R[i * Nx + j] = S[i * Nx + j] / (hp[j] * hp[j]) + (i == j ? 1.0 : 0.0);
        if (!lu_factor(Nx, R.data(), piv.data(), &det) || !(det > 0.0)) { set_error(h, "EM: det(I + Sigma Lambda^-1) <= 0"); return GPMPC_ERR_ARG; }
        lc[a] = 0.5 * log(det);
        o[2 * nn + 1] = lc[a];
    }
    int p = 0;
    for (int a = 0; a < Ny; ++a)
        for (int b = 0; b <= a; ++b, ++p) {
            const double* ha = &h->hyper[(size_t)a * m];
            const double* hb = &h->hyper[(size_t)b * m];
            for (int i = 0; i < Nx; ++i)
                for (int j = 0; j < Nx; ++j)
                    R[i * Nx + j] = S[i * Nx + j] * (1.0 / (ha[j] * ha[j]) + 1.0 / (hb[j] * hb[j])) + (i == j ? 1.0 : 0.0);   // :396-397
            if (!lu_factor(Nx, R.data(), piv.data(), &det) || !(det > 0.0)) { set_error(h, "EM: det(R_ab) <= 0"); return GPMPC_ERR_ARG; }
            for (int i = 0; i < nn; ++i) B[i] = 0.5 * S[i];
            lu_solve(Nx, R.data(), piv.data(), B.data(), Nx);             // solve(R, Sigma/2)  (:402)
            double* o = out + (size_t)Ny * (2 * nn + 2) + (size_t)p * (nn + 4);
            memcpy(o, B.data(), nn * 8);
            o[nn] = 1.0 / sqrt(det); o[nn + 1] = a; o[nn + 2] = b;        // t (:398)
            o[nn + 3] = -0.5 * log(det) + lc[a] + lc[b];                  // log t + (log sf2_a - log c_a) + (log sf2_b - log c_b)
        }
    return GPMPC_OK;
}

template <int NXP>
static cudaError_t launch_em_prep(gpmpc_handle_t h, int npairs, const double* dz, const double* dEMP, int nblk)
{
    dim3 g(nblk, h->Ny + npairs);
    em_prep_kernel<NXP><<<g, 256, 0, h->st>>>(h->dXT, h->Npad, h->N, h->Nx, h->Ny, npairs, h->dHyp, h->Nx + 2, h->dAlpha, h->Npad,
                                              dz, dEMP, h->dEmMeanPart, nblk, h->dEmE, h->dEmF, h->dEmW, h->dEmIJ, h->Npad, h->dEmLQ, h->dEmE2, h->dEmF2);
    return cudaGetLastError();
}

static int predict_em(gpmpc_handle_t h, int H, const double* Z, const double* Sigma, int spp,
                      double* mean, double* var, double* cov)
{
    const int Nx = h->Nx, Ny = h->Ny, nn = Nx * Nx, np = h->Npad;
    NvtxRange nvtx_r("gpmpc.predict_em");
    if (h->nloc != Ny) { set_error(h, "EM needs all outputs on one handle (replicate the model, shard the points)"); return GPMPC_ERR_STATE; }
    if (!Sigma) { set_error(h, "EM needs an input covariance"); return GPMPC_ERR_ARG; }
    const int npairs = Ny * (Ny + 1) / 2;
    if (npairs > 1024) { set_error(h, "EM supports Ny <= 44"); return GPMPC_ERR_ARG; }
    const size_t per = (size_t)Ny * (2 * nn + 2) + (size_t)npairs * (nn + 4);
    const int nblk = (np + 255) / 256, T = (h->N + 63) / 64, Tq = np / 64, ntr = Tq * (Tq + 1) / 2;
    if (!h->dEmTr) {
        ALLOC(h->dEmTr, (long long)Ny * ntr);
        ALLOC(h->dEmLQ, (long long)Ny * np);
        ALLOC(h->dEmVec, 2LL * np + Ny);
        ALLOC(h->dEmE, (long long)npairs * np); ALLOC(h->dEmF, (long long)npairs * np);
        ALLOC(h->dEmE2, (long long)npairs * np); ALLOC(h->dEmF2, (long long)npairs * np);
        ALLOC(h->dEmW, (long long)npairs * Nx * np); ALLOC(h->dEmIJ, (long long)npairs * Nx * np);
        ALLOC(h->dEmMeanPart, (long long)Ny * nblk); ALLOC(h->dEmPart, (long long)npairs * T * T);
    }
    { int rcs = ensure_nlml_scratch(h); if (rcs) return rcs; }      // dKinv <- Q_aa, dU <- L^-1 Q_aa (one slab each)
    if (H > h->emHcap) {
        CUDA_TRY(cudaStreamSynchronize(h->st));
        if (h->dEMP) cudaFree(h->dEMP);
        h->dEMP = nullptr;
        ALLOC(h->dEMP, (long long)H * per);
        h->emHcap = H;
    }
    std::vector<double> emp((size_t)H * per);
    for (int p = 0; p < H; ++p) {
        int rc = em_prepare_point(h, Sigma + (spp ? (size_t)p * nn : 0), emp.data() + (size_t)p * per);
        if (rc) return rc;
    }
    CUDA_TRY(cudaMemcpyAsync(h->dEMP, emp.data(), emp.size() * 8, cudaMemcpyHostToDevice, h->st));
    CUDA_TRY(cudaMemcpyAsync(h->dZ, Z, (size_t)H * Nx * 8, cudaMemcpyHostToDevice, h->st));
    for (int p = 0; p < H; ++p) {
        const double* dz = h->dZ + (size_t)p * Nx;
        const double* dP = h->dEMP + (size_t)p * per;
        cudaError_t e = (Nx <= 8) ? launch_em_prep<8>(h, npairs, dz, dP, nblk)
                      : (Nx <= 16) ? launch_em_prep<16>(h, npairs, dz, dP, nblk) : launch_em_prep<32>(h, npairs, dz, dP, nblk);
        CUDA_TRY(e);
        em_pair_kernel<<<dim3(T, T, npairs), 256, 2 * Nx * 64 * 8, h->st>>>(h->N, Nx, Ny, dP, h->dAlpha, np,
                                                                          h->dEmE, h->dEmF, h->dEmW, h->dEmIJ, np, h->dEmLQ, h->dEmE2, h->dEmF2, h->dEmPart, 0, 0, nullptr, 0);
        CUDA_TRY(cudaGetLastError());
        // E[var] term of the diagonal pairs, Cholesky-based: t tr(K^-1 Q_aa) = t tr(L^-1 Q_aa L^-T)
        for (int a = 0; a < Ny; ++a) {
            const int paa = a * (a + 1) / 2 + a;
            em_pair_kernel<<<dim3(Tq, Tq, 1), 256, 2 * Nx * 64 * 8, h->st>>>(h->N, Nx, Ny, dP, h->dAlpha, np,
                                                                          h->dEmE, h->dEmF, h->dEmW, h->dEmIJ, np, h->dEmLQ, h->dEmE2, h->dEmF2, nullptr, 1, paa, h->dKinv, np);
            CUDA_TRY(cudaGetLastError());
            // rank-one backbone: |L^-1 e^E|^2 (same kernels as alpha's first half)
            em_qvec_kernel<<<(np + 255) / 256, 256, 0, h->st>>>(h->dEmE + (long long)paa * np, h->N, np, h->dEmVec);
            CUDA_TRY(cudaGetLastError());
            trmv_lower_kernel<<<dim3((np + 7) / 8, 1, 1), 256, 0, h->st>>>(h->dLi + (long long)a * slab(h), np, 0, h->dEmVec, 0, h->dEmVec + np, 0, np);
            CUDA_TRY(cudaGetLastError());
            sumsq_kernel<<<1, 256, 0, h->st>>>(h->dEmVec + np, np, h->dEmVec + 2LL * np + a);
            CUDA_TRY(cudaGetLastError());
            GemmParams gp;
            memset(&gp, 0, sizeof(gp));
            gp.A = h->dLi + (long long)a * slab(h); gp.lda = np;
            gp.B = h->dKinv; gp.ldb = np;                 // Q symmetric: row-major (j,k) storage is the NT operand
            gp.C = h->dU; gp.ldc = np;
            gp.mt = np / 128; gp.nt = np / 128; gp.K = np; gp.alpha = 1.0; gp.beta = 0.0;
            gp.kflags = GEMM_KI_LE; gp.lower = 1;
            CUDA_TRY(gemm128(h, true, gp, 1));
            em_trdot_kernel<<<ntr, 256, 0, h->st>>>(h->dU, h->dLi + (long long)a * slab(h), np, h->dEmTr + (long long)a * ntr);
            CUDA_TRY(cudaGetLastError());
        }
        em_finalize_kernel<<<1, 1024, 0, h->st>>>(Nx, Ny, npairs, dP, h->dHyp, Nx + 2, h->dEmMeanPart, nblk, h->dEmPart, T * T,
                                                   h->dEmTr, ntr, h->dEmVec + 2LL * np,
                                                   h->dMean + (size_t)p * Ny, h->dVar + (size_t)p * Ny, h->dCov + (size_t)p * Ny * Ny);
        CUDA_TRY(cudaGetLastError());
    }
    if (mean) CUDA_TRY(cudaMemcpyAsync(mean, h->dMean, (size_t)H * Ny * 8, cudaMemcpyDeviceToHost, h->st));
    if (var) CUDA_TRY(cudaMemcpyAsync(var, h->dVar, (size_t)H * Ny * 8, cudaMemcpyDeviceToHost, h->st));
    if (cov) CUDA_TRY(cudaMemcpyAsync(cov, h->dCov, (size_t)H * Ny * Ny * 8, cudaMemcpyDeviceToHost, h->st));
    CUDA_TRY(cudaStreamSynchronize(h->st));
    return GPMPC_OK;
}

// after a stream sync: did a consumer give up waiting for a peer's flag?
static int peer_status_check(gpmpc_handle_t h)
{
    if (!h->peer_ready) return GPMPC_OK;
    const int st = h->hPeerStatus ? *(volatile int*)h->hPeerStatus : 0;
    if (st) {
        set_error(h, "peer exchange timed out waiting for rank %d (step %llu)", st - 1, h->peer_step);
        *h->hPeerStatus = 0;
        return GPMPC_ERR_NCCL;
    }
    return GPMPC_OK;
}

static int predict_check(gpmpc_handle_t h, int method, int H)
{
    if (!h) return GPMPC_ERR_ARG;
    if (!h->factorized) { set_error(h, "gpmpc_predict: call gpmpc_factorize first"); return GPMPC_ERR_STATE; }
    if (H < 1) { set_error(h, "gpmpc_predict: H < 1"); return GPMPC_ERR_ARG; }
    if (method != GPMPC_METHOD_ME && method != GPMPC_METHOD_TA && method != GPMPC_METHOD_EM) { set_error(h, "gpmpc_predict: unknown method %d", method); return GPMPC_ERR_ARG; }
    return GPMPC_OK;
}

extern "C" int gpmpc_predict_device(gpmpc_handle_t h, int method, int H, const double* dZ, const double* dSigma,
                                    int spp, double* d_mean, double* d_var, double* d_cov, double* d_jac, int sync)
{
    int rc = predict_check(h, method, H);
    if (rc) return rc;
    if (method == GPMPC_METHOD_EM) { set_error(h, "gpmpc_predict_device: EM needs host inputs (use gpmpc_predict)"); return GPMPC_ERR_ARG; }
    if (!dZ || (method == GPMPC_METHOD_TA && d_cov && !dSigma)) { set_error(h, "gpmpc_predict_device: null Z / Sigma"); return GPMPC_ERR_ARG; }
    CUDA_TRY(cudaSetDevice(h->device));
    rc = ensure_predict_bufs(h, H);
    if (rc) return rc;
    rc = predict_core(h, method, H, dZ, dSigma, spp, d_mean, d_var, d_cov, d_jac);
    if (rc) return rc;
    if (sync) CUDA_TRY(cudaStreamSynchronize(h->st));
    return GPMPC_OK;
}

// ------------------------------------------------------------------------------------
// Open-loop multi-step prediction with the state kept on the device (GP.rollout = the numeric loop of
// predict_compare, gp_class.py:746-804).  The host loop pays a call (launches + sync + copies + Python) per step
// although a step's device work at MPC sizes is tens of microseconds; here all Nt steps are enqueued back to back:
//   z_t = [ (mean_{t-1} sY + mY - mX) / sX , u_{t-1} ],  Sigma_t = [cov_{t-1} 0; 0 Sigma_uu]  ->  (mean_t, cov_t)
// with the reference's operation order (gp_class.py:629-638), so the trajectory is the host loop's bit for bit.
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
rollout_feedback_kernel(const double* __restrict__ mean_t, const double* __restrict__ cov_t, const double* __restrict__ u_t,
                        const double* __restrict__ scale, int Ny, int Nu, double* __restrict__ Z, double* __restrict__ Sigma)
{
    const int Nx = Ny + Nu, tid = threadIdx.x;
    for (int j = tid; j < Nx; j += 256) {
        if (j < Ny) {
            double z = mean_t[j];
            if (scale) {                                     // [sY | mY | mX | sX]; no fused multiply-add: numpy does not fuse
                const double x = __dadd_rn(__dmul_rn(z, scale[j]), scale[Ny + j]);
                z = __ddiv_rn(__dsub_rn(x, scale[2 * Ny + j]), scale[3 * Ny + j]);
            }
            Z[j] = z;
        } else {
            Z[j] = u_t[j - Ny];
        }
    }
    for (int idx = tid; idx < Ny * Ny; idx += 256) {
        const int r = idx / Ny, c = idx - r * Ny;
        Sigma[r * Nx + c] = cov_t[idx];
    }
}

extern "C" int gpmpc_rollout(gpmpc_handle_t h, int method, int Nt, const double* z0, const double* U, const double* Sigma0,
                             const double* scale, double* means, double* vars, double* cov_last)
{
    int rc = predict_check(h, method, 1);
    if (rc) return rc;
    const int Nx = h->Nx, Ny = h->Ny, Nu = Nx - Ny;
    if (method == GPMPC_METHOD_EM) { set_error(h, "gpmpc_rollout: methods ME and TA (EM prepares every point on the host)"); return GPMPC_ERR_ARG; }
    if (Nt < 1 || !z0 || !Sigma0 || !means || !vars || (Nu > 0 && !U)) { set_error(h, "gpmpc_rollout: null argument / Nt < 1"); return GPMPC_ERR_ARG; }
    if (Nu < 0) { set_error(h, "gpmpc_rollout: needs Nx = Ny + Nu with Nu >= 0 (Nx=%d, Ny=%d)", Nx, Ny); return GPMPC_ERR_ARG; }
    if (h->world != 1 || h->nloc != Ny) { set_error(h, "gpmpc_rollout: all outputs must live on this handle"); return GPMPC_ERR_STATE; }
    CUDA_TRY(cudaSetDevice(h->device));
    rc = ensure_predict_bufs(h, 1);
    if (rc) return rc;
    NvtxRange nvtx_r("gpmpc.rollout");
    // device slab: [Z | Sigma | U | scale | means | vars | cov], host mirror in the pinned buffer
    const size_t o_sig = Nx, o_u = o_sig + (size_t)Nx * Nx, o_sc = o_u + (size_t)Nt * Nu, o_m = o_sc + 4 * (size_t)Ny;
    const size_t o_v = o_m + (size_t)Nt * Ny, o_c = o_v + (size_t)Nt * Ny, tot = o_c + (size_t)Nt * Ny * Ny;   // one cov per step
    if (tot > h->rollCap) {
        CUDA_TRY(cudaStreamSynchronize(h->st));
        if (h->dRoll) cudaFree(h->dRoll);
        h->dRoll = nullptr; h->rollCap = 0;
        ALLOC(h->dRoll, tot);
        h->rollCap = tot;
    }
    rc = ensure_pinned(h, tot * 8);
    if (rc) return rc;
    double* pin = h->hPinned;
    memcpy(pin, z0, (size_t)Nx * 8);
    memcpy(pin + o_sig, Sigma0, (size_t)Nx * Nx * 8);
    if (Nu > 0) memcpy(pin + o_u, U, (size_t)Nt * Nu * 8);
    if (scale) memcpy(pin + o_sc, scale, 4 * (size_t)Ny * 8);
    CUDA_TRY(cudaMemcpyAsync(h->dRoll, pin, o_m * 8, cudaMemcpyHostToDevice, h->st));
    double* d = h->dRoll;
    for (int t = 0; t < Nt; ++t) {
        double* cov_t = d + o_c + (size_t)t * Ny * Ny;
        rc = predict_core(h, method, 1, d, d + o_sig, 0, d + o_m + (size_t)t * Ny, d + o_v + (size_t)t * Ny, cov_t, nullptr);
        if (rc) return rc;
        if (t + 1 < Nt) {
            rollout_feedback_kernel<<<1, 256, 0, h->st>>>(d + o_m + (size_t)t * Ny, cov_t, d + o_u + (size_t)(t + 1) * Nu,
                                                          scale ? d + o_sc : nullptr, Ny, Nu, d, d + o_sig);
            CUDA_TRY(cudaGetLastError());
        }
    }
    CUDA_TRY(cudaMemcpyAsync(pin + o_m, d + o_m, (tot - o_m) * 8, cudaMemcpyDeviceToHost, h->st));
    CUDA_TRY(cudaStreamSynchronize(h->st));
    memcpy(means, pin + o_m, (size_t)Nt * Ny * 8);
    // the reference records diag(covar_x) of every step (gp_class.py:793): the propagated variance, JSigmaJ^T included
    for (int t = 0; t < Nt; ++t)
        for (int a = 0; a < Ny; ++a) vars[(size_t)t * Ny + a] = pin[o_c + (size_t)t * Ny * Ny + (size_t)a * Ny + a];
    if (cov_last) memcpy(cov_last, pin + o_c + (size_t)(Nt - 1) * Ny * Ny, (size_t)Ny * Ny * 8);
    return GPMPC_OK;
}

extern "C" int gpmpc_predict(gpmpc_handle_t h, int method, int H, const double* Z, const double* Sigma,
                             int spp, double* mean, double* var, double* cov, double* jac)
{
    int rc = predict_check(h, method, H);
    if (rc) return rc;
    if (!Z || (method == GPMPC_METHOD_TA && cov && !Sigma)) { set_error(h, "gpmpc_predict: null Z / Sigma"); return GPMPC_ERR_ARG; }
    CUDA_TRY(cudaSetDevice(h->device));
    rc = ensure_predict_bufs(h, H);
    if (rc) return rc;
    if (method == GPMPC_METHOD_EM) {
        if (jac) { set_error(h, "gpmpc_predict: EM does not return a Jacobian"); return GPMPC_ERR_ARG; }
        return predict_em(h, H, Z, Sigma, spp, mean, var, cov);
    }
    const int Nx = h->Nx, Ny = h->Ny;
    const size_t nz = (size_t)H * Nx, ns = (method == GPMPC_METHOD_TA && Sigma) ? (size_t)(spp ? H : 1) * Nx * Nx : 0;
    const size_t nm = (size_t)H * Ny, nj = (size_t)H * Ny * Nx, nc = (size_t)H * Ny * Ny;
    // device slabs: [Z | Sigma] and [mean | var | J | cov] at capacity-based offsets -> one copy each way
    const size_t cap = (size_t)h->Hcap;
    const size_t in_span = ns ? cap * Nx + ns : nz;
    const size_t off_var = cap * Ny, off_j = 2 * cap * Ny, off_c = 2 * cap * Ny + cap * Ny * Nx;
    size_t lo = (size_t)-1, hi = 0;
    if (mean) { lo = std::min(lo, (size_t)0); hi = std::max(hi, nm); }
    if (var) { lo = std::min(lo, off_var); hi = std::max(hi, off_var + nm); }
    if (jac) { lo = std::min(lo, off_j); hi = std::max(hi, off_j + nj); }
    if (cov) { lo = std::min(lo, off_c); hi = std::max(hi, off_c + nc); }
    const size_t out_span = (hi > lo) ? hi - lo : 0;
    rc = ensure_pinned(h, (in_span + out_span) * 8);
    if (rc) return rc;
    double* pin = h->hPinned;
    memcpy(pin, Z, nz * 8);
    if (ns) memcpy(pin + cap * Nx, Sigma, ns * 8);
    // Small batches skip both copy operations: the ks kernel reads Z / Sigma from the mapped pinned buffer
    // (each of its CTAs reads HG x Nx doubles once: only worthwhile while that re-read volume is small) and the
    // assembling CTA writes mean / var / J / cov straight into it (posted writes, visible after the stream sync).
    const int np_ = h->Npad;
    const long long ks_ctas = (long long)((np_ + ks_chunk(h) - 1) / ks_chunk(h)) * ((std::min(H, HB) + 7) / 8 * 8) * h->nloc;
    const bool zc_in = h->opt_zero_copy && H <= HB && ks_ctas * Nx * 8 <= 256 * 1024 && in_span * 8 <= 64 * 1024;
    const bool zc_out = h->opt_zero_copy && out_span * 8 <= 1024 * 1024;
    double* po = pin + in_span;
    const double* dZ_ = h->dZ; const double* dS_ = h->dSigma;
    if (zc_in) { dZ_ = h->dPinnedAlias; dS_ = h->dPinnedAlias + cap * Nx; }
    else CUDA_TRY(cudaMemcpyAsync(h->dIn, pin, in_span * 8, cudaMemcpyHostToDevice, h->st));
    auto fld = [&](size_t off) { return zc_out ? h->dPinnedAlias + in_span + (off - lo) : h->dOut + off; };
    rc = predict_core(h, method, H, dZ_, dS_, spp, mean ? fld(0) : nullptr, var ? fld(off_var) : nullptr,
                      cov ? fld(off_c) : nullptr, jac ? fld(off_j) : nullptr);
    if (rc) return rc;
    if (out_span && !zc_out) CUDA_TRY(cudaMemcpyAsync(po, h->dOut + lo, out_span * 8, cudaMemcpyDeviceToHost, h->st));
    CUDA_TRY(cudaStreamSynchronize(h->st));
    { int prc = peer_status_check(h); if (prc) return prc; }
    if (mean) memcpy(mean, po + (0 - lo), nm * 8);
    if (var) memcpy(var, po + (off_var - lo), nm * 8);
    if (jac) memcpy(jac, po + (off_j - lo), nj * 8);
    if (cov) memcpy(cov, po + (off_c - lo), nc * 8);
    return GPMPC_OK;
}

// ------------------------------------------------------------------------------------
// predict + first derivatives w.r.t. the test inputs (SURVEY 8f row 1: the GPU half of the
// CasADi adapter).  Same outputs as gpmpc_predict plus
//   dvar_dz (H,Ny,Nx), dcov_dz (H,Ny,Ny,Nx), hess (H,Ny,Nx,Nx) = d^2 mean / dz^2   (each optional)
// (d mean / dz is `jac`.)  Needs all outputs on this handle.
// ------------------------------------------------------------------------------------
template <int NXP>
static cudaError_t launch_grad_reduce(gpmpc_handle_t h, const double* dZc, int Hc, int nblk)
{
    dim3 g(nblk, Hc, h->nloc);
    const int smem = (h->Nx * 257 + 256) * 8;
    static std::atomic<bool> conf[GPMPC_MAX_DEVICES];
    if (!conf[h->device % GPMPC_MAX_DEVICES].load(std::memory_order_acquire)) {      // static + dynamic may pass 48 KB
        cudaError_t e = cudaFuncSetAttribute(grad_reduce_kernel<NXP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (NX_MAX * 257 + 256) * 8);
        if (e != cudaSuccess) return e;
        conf[h->device % GPMPC_MAX_DEVICES].store(true, std::memory_order_release);
    }
    grad_reduce_kernel<NXP><<<g, 256, smem, h->st>>>(h->dXT, h->Npad, h->N, h->Nx, h->dHyp, h->Nx + 2, h->dAlpha, h->Npad, dZc,
                                                      h->dKST, h->dBeta, h->Npad, (long long)HB * h->Npad, h->dPDV, h->dPH, nblk, Hc);
    return cudaGetLastError();
}

template <int NXP>
static cudaError_t launch_hess_reduce(gpmpc_handle_t h, const double* dZc, int Hc, int nblk)
{
    dim3 g(nblk, Hc, h->nloc);
    const int smem = (h->Nx * 257 + 512) * 8;
    static std::atomic<bool> conf[GPMPC_MAX_DEVICES];
    if (!conf[h->device % GPMPC_MAX_DEVICES].load(std::memory_order_acquire)) {      // dynamic shared memory may pass 48 KB
        cudaError_t e = cudaFuncSetAttribute(hess_reduce_kernel<NXP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (NX_MAX * 257 + 512) * 8);
        if (e != cudaSuccess) return e;
        conf[h->device % GPMPC_MAX_DEVICES].store(true, std::memory_order_release);
    }
    hess_reduce_kernel<NXP><<<g, 256, smem, h->st>>>(h->dXT, h->Npad, h->N, h->Nx, h->dHyp, h->Nx + 2, h->dAlpha, h->Npad, dZc,
                                                      h->dKST, h->dBeta, h->Npad, (long long)HB * h->Npad, h->dHP, nblk, Hc);
    return cudaGetLastError();
}

// Second-order work of one chunk of Hc points (after its first-order kernels): W = L^-1 dks on the stream-K product in
// passes of whole points (floor(HB / Nx) points = up to 64 rows of the A operand, staged in dR; the solved rows land in
// dV, free once beta is formed), the Gram of each pass, the beta / third-order pair sums, d2var and d2cov.
static int hess_chunk(gpmpc_handle_t h, int method, int H, int h0, int Hc, const double* dZc, int spp,
                      const double* d_hess, double* d_d2var, double* d_d2cov)
{
    const int np = h->Npad, Nx = h->Nx, Ny = h->Ny;
    const int nblk_g = (np + GR_CHUNK - 1) / GR_CHUNK;
    const int ppp = HB / Nx;                                  // points per W pass (NX_MAX = 32 <= HB: at least 2)
    for (int p0 = 0; p0 < Hc; p0 += ppp) {
        const int npts = std::min(ppp, Hc - p0), nrows = npts * Nx, bm = (nrows + 7) / 8 * 8;
        hess_wrows_kernel<<<dim3(np / 128, bm, h->nloc), 128, 0, h->st>>>(h->dXT, np, h->N, Nx, h->dHyp, Nx + 2, dZc,
                                                                           h->dKST, np, (long long)HB * np, p0, nrows,
                                                                           h->dR, (long long)HB * np);
        CUDA_TRY(cudaGetLastError());
        int rc = tri_product(h, h->dR, h->dLi, bm, nrows, h->dV);
        if (rc) return rc;
        hess_gram_kernel<<<dim3(npts, h->nloc), 256, Nx * 129 * 8, h->st>>>(h->dV, np, (long long)HB * np, np, Nx, p0, Hc, h->dGram);
        CUDA_TRY(cudaGetLastError());
    }
    cudaError_t e = (Nx <= 8) ? launch_hess_reduce<8>(h, dZc, Hc, nblk_g)
                  : (Nx <= 16) ? launch_hess_reduce<16>(h, dZc, Hc, nblk_g) : launch_hess_reduce<32>(h, dZc, Hc, nblk_g);
    CUDA_TRY(e);
    hess_finalize_kernel<<<dim3(Hc, h->nloc), 128, 0, h->st>>>(h->dHP, nblk_g, Hc, h->dGram, h->dHyp, Nx + 2, Nx, Ny,
                                                               h->dG, H, h0, h->dHS, d_d2var);
    CUDA_TRY(cudaGetLastError());
    hess_cov_kernel<<<Hc, 256, 3 * Ny * Nx * 8, h->st>>>(Ny, Nx, method == GPMPC_METHOD_TA, h->dSigma, spp, h->dG, H, h0,
                                                         h->dHyp, Nx + 2, h->dHS, Hc, d_hess, d_d2var, h->dSH, d_d2cov);
    CUDA_TRY(cudaGetLastError());
    return GPMPC_OK;
}

// predict_grad and predict_hess: the first-order outputs of both come from this one sequence of kernels
static int predict_deriv(gpmpc_handle_t h, const char* fn, int method, int H, const double* Z, const double* Sigma, int spp,
                         double* mean, double* var, double* cov, double* jac, double* dvar_dz, double* dcov_dz, double* hess,
                         bool second, double* d2var_dz2, double* d2cov_dz2)
{
    int rc = predict_check(h, method, H);
    if (rc) return rc;
    if (method == GPMPC_METHOD_EM) { set_error(h, "%s: derivatives are available for ME and TA", fn); return GPMPC_ERR_ARG; }
    if (!Z || (method == GPMPC_METHOD_TA && !Sigma)) { set_error(h, "%s: null Z / Sigma", fn); return GPMPC_ERR_ARG; }
    if (h->nloc != h->Ny || h->world != 1) { set_error(h, "%s needs all outputs on one handle (replicate the model, shard the points)", fn); return GPMPC_ERR_STATE; }
    CUDA_TRY(cudaSetDevice(h->device));
    rc = ensure_predict_bufs(h, H);
    if (rc) return rc;
    NvtxRange nvtx_r(second ? "gpmpc.predict_hess" : "gpmpc.predict_grad");
    const int np = h->Npad, Nx = h->Nx, Ny = h->Ny, npairs = Nx * (Nx + 1) / 2;
    const int nblk_g = (np + GR_CHUNK - 1) / GR_CHUNK, nblk_mj = (np + ks_chunk(h) - 1) / ks_chunk(h);
    if (!h->dUall) {
        ALLOC(h->dUall, (long long)h->nloc * slab(h));
        ALLOC(h->dBeta, (long long)h->nloc * HB * np);
        ALLOC(h->dPDV, (long long)h->nloc * HB * nblk_g * Nx);
        ALLOC(h->dPH, (long long)h->nloc * HB * nblk_g * npairs);
        if (!h->dV) { ALLOC(h->dV, (long long)h->nloc * HB * np); ALLOC(h->dR, (long long)h->nloc * HB * np); }
    }
    if (second && !h->dHP) {
        ALLOC(h->dHP, (long long)h->nloc * HB * nblk_g * npairs * (Nx + 1));
        ALLOC(h->dHS, (long long)h->nloc * HB * npairs * (Nx + 1));
        ALLOC(h->dGram, (long long)h->nloc * HB * npairs);
        ALLOC(h->dSH, (long long)HB * Ny * Nx * Nx);
    }
    if (!h->u_valid) {                 // U = Linv^T (upper): the K-contiguous operand of beta = Linv^T v
        dim3 g(np / 32, np / 32), b(32, 8);
        for (int a = 0; a < h->nloc; ++a) {
            transpose_lower_kernel<<<g, b, 0, h->st>>>(h->dLi + (long long)a * slab(h), h->dUall + (long long)a * slab(h), np, np / 32);
            CUDA_TRY(cudaGetLastError());
        }
        h->u_valid = true;
    }
    const long long per = (long long)Ny * Nx + (long long)Ny * Ny * Nx + (long long)Ny * Nx * Nx;   // dvar | dcov | hess per point
    if (H > h->gradHcap) {
        CUDA_TRY(cudaStreamSynchronize(h->st));
        if (h->dGradOut) cudaFree(h->dGradOut);
        h->dGradOut = nullptr; h->gradHcap = 0;
        ALLOC(h->dGradOut, (long long)std::max(H, HB) * per);
        h->gradHcap = std::max(H, HB);
    }
    const long long per2 = (long long)Ny * Nx * Nx + (long long)Ny * Ny * Nx * Nx;                  // d2var | d2cov per point
    if (second && H > h->hessHcap) {
        CUDA_TRY(cudaStreamSynchronize(h->st));
        if (h->dHessOut) cudaFree(h->dHessOut);
        h->dHessOut = nullptr; h->hessHcap = 0;
        ALLOC(h->dHessOut, (long long)std::max(H, HB) * per2);
        h->hessHcap = std::max(H, HB);
    }
    double* d_dvar = h->dGradOut;
    double* d_dcov = d_dvar + (long long)H * Ny * Nx;
    double* d_hess = d_dcov + (long long)H * Ny * Ny * Nx;
    double* d_d2var = second ? h->dHessOut : nullptr;
    double* d_d2cov = second ? h->dHessOut + (long long)H * Ny * Nx * Nx : nullptr;
    const size_t nz = (size_t)H * Nx, ns = (method == GPMPC_METHOD_TA) ? (size_t)(spp ? H : 1) * Nx * Nx : 0;
    CUDA_TRY(cudaMemcpyAsync(h->dZ, Z, nz * 8, cudaMemcpyHostToDevice, h->st));
    if (ns) CUDA_TRY(cudaMemcpyAsync(h->dSigma, Sigma, ns * 8, cudaMemcpyHostToDevice, h->st));
    AssembleArgs as;
    memset(&as, 0, sizeof(as));
    as.G = h->dG; as.Ny = Ny; as.Nx = Nx; as.H = H; as.method_ta = (method == GPMPC_METHOD_TA);
    as.Sigma = h->dSigma; as.sigma_per_point = spp;
    as.mean = h->dMean; as.var = h->dVar; as.J = h->dJ; as.cov = h->dCov;
    as.world = 1;
    for (int h0 = 0; h0 < H; h0 += HB) {
        const int Hc = std::min(HB, H - h0), bm = (Hc + 7) / 8 * 8;
        const double* dZc = h->dZ + (long long)h0 * Nx;
        CUDA_TRY(launch_ks_any(h, dZc, Hc, bm, nblk_mj));
        PredictParams p;
        psk_base(h, p, Hc);                                   // v = Linv ks: records + the rows themselves
        p.finalize = 1; p.PMJ = h->dPMJ; p.nblk_mj = nblk_mj;
        p.Gloc = h->dG; p.slot0 = h->a0; p.Htot = H; p.h0 = h0;
        p.Vout = h->dV; p.sV = (long long)HB * np; p.ldv = np;
        CUDA_TRY(psk_launch(bm, p, h->dKST, (long long)HB * np, h->dLi, slab(h), np, psk_grid(h, p.G), h->st));
        psk_base(h, p, Hc);                                   // beta = Linv^T v = K^-1 ks  (rows of V times U^T)
        p.upper = 1; p.Vout = h->dBeta; p.sV = (long long)HB * np; p.ldv = np;
        CUDA_TRY(psk_launch(bm, p, h->dV, (long long)HB * np, h->dUall, slab(h), np, psk_grid(h, p.G), h->st));
        cudaError_t e = (Nx <= 8) ? launch_grad_reduce<8>(h, dZc, Hc, nblk_g)
                      : (Nx <= 16) ? launch_grad_reduce<16>(h, dZc, Hc, nblk_g) : launch_grad_reduce<32>(h, dZc, Hc, nblk_g);
        CUDA_TRY(e);
        grad_finalize_kernel<<<dim3(Hc, h->nloc), 128, 0, h->st>>>(h->dPDV, h->dPH, nblk_g, Hc, h->dHyp, Nx + 2, Nx, Ny,
                                                                   h->dG, H, h0, d_dvar, d_hess);
        CUDA_TRY(cudaGetLastError());
        if (second) {
            rc = hess_chunk(h, method, H, h0, Hc, dZc, spp, d_hess, d_d2var, d_d2cov);
            if (rc) return rc;
        }
    }
    {
        const int smem = (2 * Ny * Nx + Ny) * 8;
        assemble_kernel<<<std::min(H, 2048), 128, smem, h->st>>>(as);
        CUDA_TRY(cudaGetLastError());
        grad_cov_kernel<<<H, 128, 2 * Ny * Nx * 8, h->st>>>(Ny, Nx, method == GPMPC_METHOD_TA, h->dSigma, spp, h->dJ, d_dvar, d_hess, d_dcov);
        CUDA_TRY(cudaGetLastError());
    }
    if (mean) CUDA_TRY(cudaMemcpyAsync(mean, h->dMean, (size_t)H * Ny * 8, cudaMemcpyDeviceToHost, h->st));
    if (var) CUDA_TRY(cudaMemcpyAsync(var, h->dVar, (size_t)H * Ny * 8, cudaMemcpyDeviceToHost, h->st));
    if (cov) CUDA_TRY(cudaMemcpyAsync(cov, h->dCov, (size_t)H * Ny * Ny * 8, cudaMemcpyDeviceToHost, h->st));
    if (jac) CUDA_TRY(cudaMemcpyAsync(jac, h->dJ, (size_t)H * Ny * Nx * 8, cudaMemcpyDeviceToHost, h->st));
    if (dvar_dz) CUDA_TRY(cudaMemcpyAsync(dvar_dz, d_dvar, (size_t)H * Ny * Nx * 8, cudaMemcpyDeviceToHost, h->st));
    if (dcov_dz) CUDA_TRY(cudaMemcpyAsync(dcov_dz, d_dcov, (size_t)H * Ny * Ny * Nx * 8, cudaMemcpyDeviceToHost, h->st));
    if (hess) CUDA_TRY(cudaMemcpyAsync(hess, d_hess, (size_t)H * Ny * Nx * Nx * 8, cudaMemcpyDeviceToHost, h->st));
    if (d2var_dz2) CUDA_TRY(cudaMemcpyAsync(d2var_dz2, d_d2var, (size_t)H * Ny * Nx * Nx * 8, cudaMemcpyDeviceToHost, h->st));
    if (d2cov_dz2) CUDA_TRY(cudaMemcpyAsync(d2cov_dz2, d_d2cov, (size_t)H * Ny * Ny * Nx * Nx * 8, cudaMemcpyDeviceToHost, h->st));
    CUDA_TRY(cudaStreamSynchronize(h->st));
    return GPMPC_OK;
}

extern "C" int gpmpc_predict_grad(gpmpc_handle_t h, int method, int H, const double* Z, const double* Sigma, int spp,
                                  double* mean, double* var, double* cov, double* jac,
                                  double* dvar_dz, double* dcov_dz, double* hess)
{
    return predict_deriv(h, "gpmpc_predict_grad", method, H, Z, Sigma, spp, mean, var, cov, jac, dvar_dz, dcov_dz, hess,
                         false, nullptr, nullptr);
}

// ------------------------------------------------------------------------------------
// predict + first and second derivatives w.r.t. the test inputs: everything gpmpc_predict_grad returns plus
//   d2var_dz2 (H,Ny,Nx,Nx), d2cov_dz2 (H,Ny,Ny,Nx,Nx)   (each optional; formulas above hess_wrows_kernel)
// ------------------------------------------------------------------------------------
extern "C" int gpmpc_predict_hess(gpmpc_handle_t h, int method, int H, const double* Z, const double* Sigma, int spp,
                                  double* mean, double* var, double* cov, double* jac,
                                  double* dvar_dz, double* dcov_dz, double* hess,
                                  double* d2var_dz2, double* d2cov_dz2)
{
    return predict_deriv(h, "gpmpc_predict_hess", method, H, Z, Sigma, spp, mean, var, cov, jac, dvar_dz, dcov_dz, hess,
                         true, d2var_dz2, d2cov_dz2);
}

extern "C" int gpmpc_append(gpmpc_handle_t h, const double* x_new, const double* y_new)
{
    if (!h || !x_new || !y_new) return GPMPC_ERR_ARG;
    if (!h->factorized) { set_error(h, "gpmpc_append: call gpmpc_factorize first"); return GPMPC_ERR_STATE; }
    if (h->sparse) { set_error(h, "gpmpc_append: the handle holds a FITC model (rebuild it with gpmpc_fitc)"); return GPMPC_ERR_STATE; }
    if (h->N >= h->Npad) { set_error(h, "gpmpc_append: capacity %d reached, refit on a new handle", h->Npad); return GPMPC_ERR_STATE; }
    CUDA_TRY(cudaSetDevice(h->device));
    int rc = ensure_predict_bufs(h, 1);
    if (rc) return rc;
    const int N = h->N, Nx = h->Nx, np = h->Npad, nl = h->nloc;
    // k(X, x_new) for every owned output through the predict ks kernel (H = 1): row 0 of KS^T
    CUDA_TRY(cudaMemcpyAsync(h->dZ, x_new, Nx * 8, cudaMemcpyHostToDevice, h->st));
    CUDA_TRY(launch_ks_any(h, h->dZ, 1, 8, (np + ks_chunk(h) - 1) / ks_chunk(h)));
    // l = Li k (rows < N), r = Li^T l
    if (!h->dV) { ALLOC(h->dV, (long long)nl * HB * np); ALLOC(h->dR, (long long)nl * HB * np); }
    dim3 g1((np + 7) / 8, 1, nl);
    trmv_lower_kernel<<<g1, 256, 0, h->st>>>(h->dLi, np, slab(h), h->dKST, (long long)HB * np, h->dV, (long long)HB * np, N);
    CUDA_TRY(cudaGetLastError());
    // rows >= N of l must be zero for the transposed product over the padded matrix
    for (int a = 0; a < nl; ++a)
        CUDA_TRY(cudaMemsetAsync(h->dV + (long long)a * HB * np + N, 0, (size_t)(np - N) * 8, h->st));
    dim3 g2(np / 32, 1, nl);
    trmv_lower_T_kernel<<<g2, 256, 0, h->st>>>(h->dLi, np, slab(h), h->dV, (long long)HB * np, h->dR, (long long)HB * np, np);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemsetAsync(h->dInfo, 0, nl * sizeof(int), h->st));
    append_row_kernel<<<nl, 256, 0, h->st>>>(h->dL, h->dLi, np, slab(h), h->dV, h->dR, (long long)HB * np, h->dHyp, Nx + 2, Nx, N, h->dInfo);
    CUDA_TRY(cudaGetLastError());
    std::vector<int> inf(nl, 0);
    CUDA_TRY(cudaMemcpyAsync(inf.data(), h->dInfo, nl * sizeof(int), cudaMemcpyDeviceToHost, h->st));
    // the new point joins X^T (column N) and Y
    for (int d = 0; d < Nx; ++d) CUDA_TRY(cudaMemcpyAsync(h->dXT + (long long)d * np + N, x_new + d, 8, cudaMemcpyHostToDevice, h->st));
    for (int a = 0; a < nl; ++a) CUDA_TRY(cudaMemcpyAsync(h->dY + (long long)a * np + N, y_new + h->a0 + a, 8, cudaMemcpyHostToDevice, h->st));
    CUDA_TRY(cudaStreamSynchronize(h->st));
    for (int a = 0; a < nl; ++a)
        if (inf[a]) {
            h->factorized = false;       // row N of that output is unusable: the caller must refactorise
            set_error(h, "gpmpc_append: output %d lost positive definiteness (refactorise, jitter applies there)", h->a0 + a);
            h->N = N + 1;
            return GPMPC_ERR_NOTPD;
        }
    h->N = N + 1;
    h->u_valid = false;
    rc = launch_alpha(h, 0, nl);
    if (rc) return rc;
    std::vector<double> res(2 * nl);
    CUDA_TRY(cudaMemcpyAsync(res.data(), h->dRes, 2 * nl * 8, cudaMemcpyDeviceToHost, h->st));
    CUDA_TRY(cudaStreamSynchronize(h->st));
    for (int a = 0; a < nl; ++a) { h->logdet[a] = res[2 * a]; h->yalpha[a] = res[2 * a + 1]; }
    return GPMPC_OK;
}

extern "C" int gpmpc_posterior_cov(gpmpc_handle_t h, int H, const double* Z, double* out)
{
    if (!h || !Z || !out || H < 1) return GPMPC_ERR_ARG;
    if (!h->factorized) { set_error(h, "gpmpc_posterior_cov: call gpmpc_factorize first"); return GPMPC_ERR_STATE; }
    CUDA_TRY(cudaSetDevice(h->device));
    int rc = ensure_predict_bufs(h, H);
    if (rc) return rc;
    const int np = h->Npad, Nx = h->Nx, nl = h->nloc;
    const long long sVall = (long long)H * np;            // all H solved rows of one output
    // scratch is pooled on the handle (grown on demand), not allocated per call
    if ((long long)nl * sVall > h->covVcap) {
        CUDA_TRY(cudaStreamSynchronize(h->st));
        if (h->dCovV) cudaFree(h->dCovV);
        h->dCovV = nullptr; h->covVcap = 0;
        ALLOC(h->dCovV, (long long)nl * sVall);
        h->covVcap = (long long)nl * sVall;
    }
    if ((long long)nl * H * H > h->covOutcap) {
        CUDA_TRY(cudaStreamSynchronize(h->st));
        if (h->dCovOut) cudaFree(h->dCovOut);
        h->dCovOut = nullptr; h->covOutcap = 0;
        ALLOC(h->dCovOut, (long long)nl * H * H);
        h->covOutcap = (long long)nl * H * H;
    }
    double *dVall = h->dCovV, *dOut = h->dCovOut;
    if (!h->dV) { ALLOC(h->dV, (long long)nl * HB * np); ALLOC(h->dR, (long long)nl * HB * np); }
    CUDA_TRY(cudaMemcpyAsync(h->dZ, Z, (size_t)H * Nx * 8, cudaMemcpyHostToDevice, h->st));
    const int nblk_mj = (np + ks_chunk(h) - 1) / ks_chunk(h);
    for (int h0 = 0; h0 < H && rc == GPMPC_OK; h0 += HB) {
        const int Hc = std::min(HB, H - h0), bm = (Hc + 7) / 8 * 8;
        const double* dZc = h->dZ + (long long)h0 * Nx;
        cudaError_t e = launch_ks_any(h, dZc, Hc, bm, nblk_mj);
        if (e != cudaSuccess) { set_error(h, "posterior_cov ks: %s", cudaGetErrorString(e)); rc = GPMPC_ERR_CUDA; break; }
        rc = tri_product(h, h->dKST, h->dLi, bm, Hc, h->dV);
        if (rc) break;
        dim3 g(1, Hc, nl);
        copy2d_kernel<<<dim3(16, std::min(Hc, 64), nl), 128, 0, h->st>>>(h->dV, np, (long long)HB * np,
                                                                     dVall + (long long)h0 * np, np, sVall, Hc, np);
        if (cudaGetLastError() != cudaSuccess) { rc = GPMPC_ERR_CUDA; break; }
    }
    if (rc == GPMPC_OK) {
        gram_cov_kernel<<<dim3(H, H, nl), 256, 0, h->st>>>(dVall, np, sVall, np, h->dHyp, Nx + 2, Nx, H, dOut);
        if (cudaGetLastError() != cudaSuccess) rc = GPMPC_ERR_CUDA;
    }
    if (rc == GPMPC_OK && cudaMemcpyAsync(out, dOut, (size_t)nl * H * H * 8, cudaMemcpyDeviceToHost, h->st) != cudaSuccess) rc = GPMPC_ERR_CUDA;
    cudaStreamSynchronize(h->st);
    if (rc == GPMPC_ERR_CUDA) set_error(h, "gpmpc_posterior_cov: CUDA failure %s", cudaGetErrorString(cudaGetLastError()));
    return rc;
}

// ------------------------------------------------------------------------------------
// multi-GPU
// ------------------------------------------------------------------------------------
extern "C" int gpmpc_comm_unique_id(void* id128)
{
    if (!id128) return GPMPC_ERR_ARG;
    if (!nccl_load(g_create_err, sizeof(g_create_err))) return GPMPC_ERR_NCCL;
    nccl_uid_t id;
    int r = g_nccl.GetUniqueId(&id);
    if (r) { snprintf(g_create_err, sizeof(g_create_err), "ncclGetUniqueId failed (%d)", r); return GPMPC_ERR_NCCL; }
    memcpy(id128, &id, 128);
    return GPMPC_OK;
}

extern "C" int gpmpc_comm_init(gpmpc_handle_t h, const void* id128, int rank, int world)
{
    if (!h || !id128 || world < 1 || rank < 0 || rank >= world) return GPMPC_ERR_ARG;
    CUDA_TRY(cudaSetDevice(h->device));
    const int nlm = (h->Ny + world - 1) / world;
    if (h->a0 != std::min(h->Ny, rank * nlm) || h->nloc > nlm) {
        set_error(h, "gpmpc_comm_init: rank %d of %d must own outputs starting at %d (at most %d); handle owns [%d,%d)",
                  rank, world, rank * nlm, nlm, h->a0, h->a0 + h->nloc);
        return GPMPC_ERR_ARG;
    }
    if (world > 1) {
        if (!nccl_load(h->err, sizeof(h->err))) return GPMPC_ERR_NCCL;
        nccl_uid_t id;
        memcpy(&id, id128, 128);
        int r = g_nccl.CommInitRank(&h->comm, world, id, rank);
        if (r) { set_error(h, "ncclCommInitRank failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?"); return GPMPC_ERR_NCCL; }
    }
    h->rank = rank; h->world = world; h->nloc_max = nlm;
    h->Hcap = 0;      // gather buffer must be re-sized for the padded output count
    return GPMPC_OK;
}

extern "C" int gpmpc_peer_export(gpmpc_handle_t h, int Hcap, void* handle64)
{
    if (!h || !handle64 || Hcap < 1) return GPMPC_ERR_ARG;
    CUDA_TRY(cudaSetDevice(h->device));
    if (h->world > GPMPC_MAXW) { set_error(h, "peer exchange supports at most %d ranks", GPMPC_MAXW); return GPMPC_ERR_ARG; }
    if (h->dPeerBlock) { set_error(h, "gpmpc_peer_export: already exported"); return GPMPC_ERR_STATE; }
    const int nyp = h->nloc_max * h->world;
    h->peerGsz = (long long)nyp * Hcap * (h->Nx + 2);
    h->peerHcap = Hcap;
    ALLOC(h->dPeerBlock, 2 * GPMPC_MAXW + 2 * h->peerGsz);
    if (!h->dPeerStatus) {     // status word in mapped pinned host memory: the host reads it without a copy
        CUDA_TRY(cudaHostAlloc((void**)&h->hPeerStatus, sizeof(int), cudaHostAllocMapped));
        *h->hPeerStatus = 0;
        CUDA_TRY(cudaHostGetDevicePointer((void**)&h->dPeerStatus, h->hPeerStatus, 0));
    }
    CUDA_TRY(cudaStreamSynchronize(h->st));
    cudaIpcMemHandle_t mh;
    CUDA_TRY(cudaIpcGetMemHandle(&mh, h->dPeerBlock));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    memcpy(handle64, &mh, 64);
    return GPMPC_OK;
}

extern "C" int gpmpc_peer_attach(gpmpc_handle_t h, const void* handles)
{
    if (!h || !handles) return GPMPC_ERR_ARG;
    if (!h->dPeerBlock) { set_error(h, "gpmpc_peer_attach: call gpmpc_peer_export first"); return GPMPC_ERR_STATE; }
    CUDA_TRY(cudaSetDevice(h->device));
    for (int r = 0; r < h->world; ++r) {
        if (r == h->rank) { h->peerBase[r] = h->dPeerBlock; continue; }
        cudaIpcMemHandle_t mh;
        memcpy(&mh, (const char*)handles + 64 * r, 64);
        void* ptr = nullptr;
        CUDA_TRY(cudaIpcOpenMemHandle(&ptr, mh, cudaIpcMemLazyEnablePeerAccess));
        h->peerBase[r] = (double*)ptr; h->peerOpened[r] = true;
    }
    h->peer_ready = true; h->peer_step = 0;
    return GPMPC_OK;
}

extern "C" int gpmpc_get_size(gpmpc_handle_t h, int* N, int* Nx, int* Ny)
{
    if (!h) return GPMPC_ERR_ARG;
    if (N) *N = h->N;
    if (Nx) *Nx = h->Nx;
    if (Ny) *Ny = h->Ny;
    return GPMPC_OK;
}

extern "C" void* gpmpc_stream(gpmpc_handle_t h) { return h ? (void*)h->st : nullptr; }

extern "C" int gpmpc_synchronize(gpmpc_handle_t h)
{
    if (!h) return GPMPC_ERR_ARG;
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(cudaStreamSynchronize(h->st));
    return peer_status_check(h);
}

// load balance of the persistent predict product: per-CTA busy time (globaltimer at CTA start / end)
//   out = {shortest CTA, longest CTA, mean CTA, first start -> last end} in microseconds
extern "C" int gpmpc_profile_balance(gpmpc_handle_t h, int H, double* out4)
{
    if (!h || !out4 || H < 1 || H > HB) return GPMPC_ERR_ARG;
    if (!h->factorized) { set_error(h, "gpmpc_profile_balance: call gpmpc_factorize first"); return GPMPC_ERR_STATE; }
    CUDA_TRY(cudaSetDevice(h->device));
    int rc = ensure_predict_bufs(h, HB);
    if (rc) return rc;
    PredictParams p;
    psk_base(h, p, H);
    const int grid = psk_grid(h, p.G);
    unsigned long long* dbg = nullptr;
    CUDA_TRY(cudaMalloc((void**)&dbg, (size_t)grid * 16));
    p.dbg = dbg;
    const int np = h->Npad, bm = (H + 7) / 8 * 8;
    for (int rep = 0; rep < 2; ++rep) {
        cudaError_t e = psk_launch(bm, p, h->dKST, (long long)HB * np, h->dLi, slab(h), np, grid, h->st);
        if (e != cudaSuccess) { cudaFree(dbg); set_error(h, "profile_balance: %s", cudaGetErrorString(e)); return GPMPC_ERR_CUDA; }
    }
    std::vector<unsigned long long> t((size_t)grid * 2);
    cudaMemcpyAsync(t.data(), dbg, t.size() * 8, cudaMemcpyDeviceToHost, h->st);
    cudaStreamSynchronize(h->st);
    cudaFree(dbg);
    unsigned long long lo = ~0ull, hi = 0; double mn = 1e300, mx = 0.0, sum = 0.0;
    for (int c = 0; c < grid; ++c) {
        const double d = (double)(t[2 * c + 1] - t[2 * c]) * 1e-3;
        mn = std::min(mn, d); mx = std::max(mx, d); sum += d;
        lo = std::min(lo, t[2 * c]); hi = std::max(hi, t[2 * c + 1]);
    }
    out4[0] = mn; out4[1] = mx; out4[2] = sum / grid; out4[3] = (double)(hi - lo) * 1e-3;
    return GPMPC_OK;
}

// phase stamps of the fused kernel's serial tail (the CTA that completes the step): out8 = microseconds, relative to the
// latest end of every OTHER CTA, of {last output complete, records built, step counter passed, records staged,
// J Sigma done, outputs written}, then the kernel's span and the tail CTA's own span.  Needs a predict call before it.
extern "C" int gpmpc_profile_tail(gpmpc_handle_t h, int H, double* out8)
{
    if (!h || !out8 || H < 1 || H > HB) return GPMPC_ERR_ARG;
    if (!h->factorized) { set_error(h, "gpmpc_profile_tail: call gpmpc_factorize first"); return GPMPC_ERR_STATE; }
    if (h->world != 1 || h->nloc != h->Ny) { set_error(h, "gpmpc_profile_tail: single-rank handles only"); return GPMPC_ERR_STATE; }
    CUDA_TRY(cudaSetDevice(h->device));
    int rc = ensure_predict_bufs(h, HB);
    if (rc) return rc;
    const int np = h->Npad, bm = (H + 7) / 8 * 8;
    PredictParams p;
    psk_base(h, p, H);
    const int grid = psk_grid(h, p.G);
    unsigned long long* dbg = nullptr;
    CUDA_TRY(cudaMalloc((void**)&dbg, (size_t)(grid * 2 + 8) * 8));
    CUDA_TRY(cudaMemset(dbg, 0, (size_t)(grid * 2 + 8) * 8));
    p.dbg = dbg;
    p.finalize = 1; p.PMJ = h->dPMJ; p.nblk_mj = (np + ks_chunk(h) - 1) / ks_chunk(h);
    p.Gloc = h->dG; p.slot0 = h->a0; p.Htot = H; p.h0 = 0;
    AssembleArgs as;
    memset(&as, 0, sizeof(as));
    as.G = h->dG; as.Ny = h->Ny; as.Nx = h->Nx; as.H = H; as.method_ta = 1; as.Sigma = h->dSigma;
    as.mean = h->dMean; as.var = h->dVar; as.J = h->dJ; as.cov = h->dCov; as.world = 1;
    as.stage_g = (assemble_rows_doubles(H, h->Ny, h->Nx) <= (long long)PSK_STAGES * (bm + PSK_BN) * GEMM_BK) ? 1 : 0;
    as.dbg = dbg + 2 * grid;
    p.as = as; p.do_assemble = 1;
    for (int rep = 0; rep < 2; ++rep) {
        cudaError_t e = psk_launch(bm, p, h->dKST, (long long)HB * np, h->dLi, slab(h), np, grid, h->st);
        if (e != cudaSuccess) { cudaFree(dbg); set_error(h, "profile_tail: %s", cudaGetErrorString(e)); return GPMPC_ERR_CUDA; }
    }
    std::vector<unsigned long long> t((size_t)grid * 2 + 8);
    cudaMemcpyAsync(t.data(), dbg, t.size() * 8, cudaMemcpyDeviceToHost, h->st);
    cudaStreamSynchronize(h->st);
    cudaFree(dbg);
    unsigned long long lo = ~0ull, hi = 0, hi2 = 0; int cmax = 0;
    for (int c = 0; c < grid; ++c) {
        lo = std::min(lo, t[2 * c]);
        if (t[2 * c + 1] > hi) { hi2 = hi; hi = t[2 * c + 1]; cmax = c; } else hi2 = std::max(hi2, t[2 * c + 1]);
    }
    for (int k = 0; k < 6; ++k) out8[k] = ((double)t[2 * grid + k] - (double)hi2) * 1e-3;
    out8[6] = (double)(hi - lo) * 1e-3;
    out8[7] = (double)(t[2 * cmax + 1] - t[2 * cmax]) * 1e-3;
    return GPMPC_OK;
}

// phase clock stamps of one 128x128 leaf (potrf + trtri): out15 = clock64 at
// {start, loaded, first panel, after block steps 1..7, L stored, inverse levels 16/32/64, Linv stored}
extern "C" int gpmpc_profile_leaf(gpmpc_handle_t h, double* out15)
{
    if (!h || !out15) return GPMPC_ERR_ARG;
    if (!h->has_data || !h->has_hyper) { set_error(h, "gpmpc_profile_leaf: set_data and set_hyper first"); return GPMPC_ERR_STATE; }
    CUDA_TRY(cudaSetDevice(h->device));
    long long* d = nullptr;
    CUDA_TRY(cudaMalloc((void**)&d, 16 * sizeof(long long)));
    CUDA_TRY(cudaMemset(d, 0, 16 * sizeof(long long)));
    CUDA_TRY(cudaMemcpyToSymbol(d_leaf_prof, &d, sizeof(d)));
    int rc = GPMPC_OK;
    for (int rep = 0; rep < 2 && rc == GPMPC_OK; ++rep) {           // second run: warm instruction cache
        rc = launch_kbuild(h, h->dHyp, h->dJit, h->dL, 1, 0);
        if (rc == GPMPC_OK) rc = potrf_inv_rec(h, h->dL, h->dLi, slab(h), slab(h), h->dInfo, 0, 128, 1);
    }
    cudaStreamSynchronize(h->st);
    long long hst[16];
    cudaMemcpy(hst, d, sizeof(hst), cudaMemcpyDeviceToHost);
    long long* nul = nullptr;
    cudaMemcpyToSymbol(d_leaf_prof, &nul, sizeof(nul));
    cudaFree(d);
    for (int k = 0; k < 15; ++k) out15[k] = (double)(hst[k] - hst[0]);
    h->factorized = false;
    return rc;
}

// ------------------------------------------------------------------------------------
// kernel-level timing for the roofline report (CUDA events on the handle's stream)
// ------------------------------------------------------------------------------------
extern "C" int gpmpc_profile(gpmpc_handle_t h, int what, int n, int reps, double* ms_out)
{
    if (!h || !ms_out || reps < 1) return GPMPC_ERR_ARG;
    if (!h->has_data || !h->has_hyper) { set_error(h, "gpmpc_profile: set_data and set_hyper first"); return GPMPC_ERR_STATE; }
    CUDA_TRY(cudaSetDevice(h->device));
    const int np = h->Npad;
    float ms = 0.f;
    int rc = GPMPC_OK;
    auto run = [&](int rep) -> int {
        switch (what) {
        case GPMPC_PROF_KBUILD_FULL: return launch_kbuild(h, h->dHyp, h->dJit, h->dL, 1, 1);
        case GPMPC_PROF_KBUILD_LOWER: return launch_kbuild(h, h->dHyp, h->dJit, h->dL, 1, 0);
        case GPMPC_PROF_SYRK: {
            // trailing update shape of the top recursion level: C(n2 x n2, lower) -= P P^T, K = n1
            const int nn = (n > 0 && n <= np) ? n / 128 * 128 : np;
            const int n1 = (nn / 128 / 2) * 128, n2 = nn - n1;
            if (n1 < 128) { set_error(h, "gpmpc_profile: SYRK needs N >= 256"); return GPMPC_ERR_ARG; }
            GemmParams p;
            memset(&p, 0, sizeof(p));
            p.A = h->dW1; p.lda = n1; p.B = h->dW1; p.ldb = n1;
            p.C = h->dLi; p.ldc = np; p.Cin = h->dLi; p.ldcin = np;
            p.mt = n2 / 128; p.nt = n2 / 128; p.K = n1; p.alpha = -1e-30; p.beta = 1.0; p.lower = 1;
            cudaError_t e = gemm128(h, true, p, 1);
            if (e != cudaSuccess) { set_error(h, "profile syrk: %s", cudaGetErrorString(e)); return GPMPC_ERR_CUDA; }
            return GPMPC_OK;
        }
        case GPMPC_PROF_FACTORIZE: {
            int r = launch_kbuild(h, h->dHyp, h->dJit, h->dL, 1, 0);
            if (r) return r;
            return potrf_inv_rec(h, h->dL, h->dLi, slab(h), slab(h), h->dInfo, 0, np, 1);
        }
        case GPMPC_PROF_TRIGEMM: {
            const int Hc = (n > 0 && n <= HB) ? n : 56;
            return tri_product(h, h->dKST, h->dLi, (Hc + 7) / 8 * 8, Hc, nullptr);
        }
        case GPMPC_PROF_KS: {             // the ks / mean / Jacobian partial kernel alone (Z = the last batch's inputs)
            const int Hc = (n > 0 && n <= HB) ? n : 56;
            cudaError_t e = launch_ks_any(h, h->dZ, Hc, (Hc + 7) / 8 * 8, (np + ks_chunk(h) - 1) / ks_chunk(h));
            if (e != cudaSuccess) { set_error(h, "profile ks: %s", cudaGetErrorString(e)); return GPMPC_ERR_CUDA; }
            return GPMPC_OK;
        }
        case GPMPC_PROF_PREDICT_TAIL: {   // the fused kernel WITH finalize + assembly, without the ks kernel in front
            const int Hc = (n > 0 && n <= HB) ? n : 56;
            PredictParams p;
            psk_base(h, p, Hc);
            p.finalize = 1; p.PMJ = h->dPMJ; p.nblk_mj = (np + ks_chunk(h) - 1) / ks_chunk(h);
            p.Gloc = h->dG; p.slot0 = h->a0; p.Htot = Hc; p.h0 = 0;
            AssembleArgs as;
            memset(&as, 0, sizeof(as));
            as.G = h->dG; as.Ny = h->Ny; as.Nx = h->Nx; as.H = Hc; as.method_ta = 1; as.Sigma = h->dSigma;
            as.mean = h->dMean; as.var = h->dVar; as.J = h->dJ; as.cov = h->dCov; as.world = 1;
            as.stage_g = (assemble_rows_doubles(Hc, h->Ny, h->Nx) <= (long long)PSK_STAGES * ((Hc + 7) / 8 * 8 + PSK_BN) * GEMM_BK) ? 1 : 0;
            p.as = as; p.do_assemble = (h->world == 1 && h->nloc == h->Ny) ? 1 : 0;
            cudaError_t e = psk_launch((Hc + 7) / 8 * 8, p, h->dKST, (long long)HB * np, h->dLi, slab(h), np, psk_grid(h, p.G), h->st);
            if (e != cudaSuccess) { set_error(h, "profile predict tail: %s", cudaGetErrorString(e)); return GPMPC_ERR_CUDA; }
            return GPMPC_OK;
        }
        default: set_error(h, "gpmpc_profile: unknown selector %d", what); return GPMPC_ERR_ARG;
        }
    };
    if (what == GPMPC_PROF_TRIGEMM || what == GPMPC_PROF_KS || what == GPMPC_PROF_PREDICT_TAIL) { rc = ensure_predict_bufs(h, HB); if (rc) return rc; }
    CUDA_TRY(cudaMemsetAsync(h->dJit, 0, h->nloc * sizeof(double), h->st));
    rc = run(-1);
    if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(h->st));
    CUDA_TRY(cudaEventRecord(h->ev0, h->st));
    for (int r = 0; r < reps; ++r) { rc = run(r); if (rc) return rc; }
    CUDA_TRY(cudaEventRecord(h->ev1, h->st));
    CUDA_TRY(cudaEventSynchronize(h->ev1));
    CUDA_TRY(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    ms_out[0] = (double)ms / reps;
    if (what != GPMPC_PROF_TRIGEMM && what != GPMPC_PROF_KS && what != GPMPC_PROF_PREDICT_TAIL) h->factorized = false;   // slabs were used as scratch
    return GPMPC_OK;
}
