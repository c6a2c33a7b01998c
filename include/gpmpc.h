/* gpmpc.h -- C ABI of the B200-native GP regression engine (libgpmpc.so).
 *
 * This is the drop-in boundary for the dense Gaussian-process hot path of
 * helgeanl/GP-MPC.  The reference has no FFI layer of its own (it is pure Python on
 * numpy/CasADi); the entry points below are what a ctypes binding inside the
 * reference's gp_mpc/gp_class.py would call instead of numpy/CasADi.  Each entry
 * point cites the reference code it replaces (file:line relative to the reference
 * checkout).  See INTEGRATION.md for the binding a maintainer would add.
 *
 * Conventions
 *   - all matrices are fp64, row-major, caller-owned;  "host" pointers are ordinary
 *     CPU memory, "device" pointers are CUDA device memory on the handle's GPU
 *   - hyper rows are [ell_1..ell_Nx, sf, sn] with sf, sn STANDARD DEVIATIONS
 *     (gp_class.py:139-142);  prior mean is zero (the only mean the reference's
 *     prediction graph ever uses, gp_class.py:69-71)
 *   - return value: 0 ok, <0 error (gpmpc_last_error(h) has the text),
 *     GPMPC_ERR_NOTPD when the Cholesky failed even after the jitter retry
 *   - a handle owns one CUDA stream and is not thread-safe; calls are synchronous
 *     unless stated otherwise
 *   - the library has NO CPU fallback: without a CUDA device gpmpc_create fails
 */
#ifndef GPMPC_H
#define GPMPC_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gpmpc_handle_s* gpmpc_handle_t;

enum {
    GPMPC_OK = 0,
    GPMPC_ERR_ARG = -1,
    GPMPC_ERR_CUDA = -2,
    GPMPC_ERR_STATE = -3,
    GPMPC_ERR_NCCL = -4,
    GPMPC_ERR_NOTPD = -5
};

/* propagation method of GP.set_method / GP.predict (gp_class.py:193-237) */
enum { GPMPC_METHOD_ME = 0, GPMPC_METHOD_TA = 1, GPMPC_METHOD_EM = 2 /* gp_exact_moment, gp_functions.py:344-418; host API only */ };

/* selector of gpmpc_get */
enum {
    GPMPC_GET_CHOL = 0,    /* (N,N) lower factor, exact zeros above the diagonal (optimize.py:491) */
    GPMPC_GET_ALPHA = 1,   /* (N,)  K^-1 y                                      (optimize.py:494) */
    GPMPC_GET_INVK = 2,    /* (N,N) K^-1, symmetric                             (optimize.py:489-490) */
    GPMPC_GET_K = 3,       /* (N,N) K + sn2 I                                   (optimize.py:480-482) */
    GPMPC_GET_LOGDET = 4,  /* (1,)  2 sum log L_ii                              (optimize.py:352) */
    GPMPC_GET_LINV = 5,    /* (N,N) L^-1 lower                                  (optimize.py:489 invL) */
    GPMPC_GET_ALPHA_NLML = 6 /* (N,) alpha of the last gpmpc_nlml evaluation for that output (mean-parameter gradient) */
};

/* selector of gpmpc_profile */
enum {
    GPMPC_PROF_KBUILD_FULL = 0,   /* covSEard K build, full square                     */
    GPMPC_PROF_KBUILD_LOWER = 1,  /* covSEard K build, lower triangle only            */
    GPMPC_PROF_SYRK = 2,          /* Cholesky trailing update C -= P P^T (DMMA GEMM)  */
    GPMPC_PROF_FACTORIZE = 3,     /* potrf + trtri of one output (K prebuilt each rep) */
    GPMPC_PROF_TRIGEMM = 4,       /* predict v = Linv ks product, all local outputs    */
    GPMPC_PROF_KS = 5,            /* ks / partial mean / partial Jacobian kernel alone (after a predict call) */
    GPMPC_PROF_PREDICT_TAIL = 6   /* product + finalize + assembly in one launch, no ks kernel in front (after a predict call) */
};

int gpmpc_version(void);

/* Create an engine for N training points, Nx inputs, Ny outputs of which this handle
 * owns the contiguous block [out_begin, out_begin+out_count) (one block per GPU rank;
 * independent per-output GPs, optimize.py:433 / gp_functions.py:128).  device = CUDA
 * ordinal.  Replaces the array allocations of train_gp_numpy, optimize.py:424-427. */
int gpmpc_create(int N, int Nx, int Ny, int out_begin, int out_count, int device, gpmpc_handle_t* out);
int gpmpc_destroy(gpmpc_handle_t h);
const char* gpmpc_last_error(gpmpc_handle_t h);   /* h may be NULL: last create error */

/* Training data already in the GP's input space (standardised by the caller when
 * normalize=True, gp_class.py:101-117).  X:(N,Nx) Y:(N,Ny) host. */
int gpmpc_set_data(gpmpc_handle_t h, const double* X, const double* Y);

/* hyper:(Ny,ld) host, ld >= Nx+2; only the owned rows are used (gp_class.py:134-142). */
int gpmpc_set_hyper(gpmpc_handle_t h, const double* hyper, int ld);

/* Replace the target vector of global output a with y (N doubles, host): the GP class passes the
 * residual y - m(X) of a prior mean function (alpha = K^-1 (y - m(X)), optimize.py:492-494;
 * get_mean_function, gp_functions.py:25-69).  Invalidates the factorisation. */
int gpmpc_set_y(gpmpc_handle_t h, int a, const double* y);

/* K = covSEard(X,X) + sn2 I for global output a into K_out:(N,N) host (may be NULL:
 * build only).  Replaces calc_cov_matrix + noise + symmetrise, optimize.py:303-319,
 * :480-482 and GP.covSEard gp_class.py:314-350. */
int gpmpc_build_K(gpmpc_handle_t h, int a, double* K_out);

/* Post-fit block for every owned output: K -> L (blocked Cholesky on fp64 tensor
 * cores) -> L^-1 -> alpha, logdet.  On a non-positive pivot adds `jitter` (reference:
 * 1e-8) to that output's diagonal ONCE and retries; a second failure returns
 * GPMPC_ERR_NOTPD.  info:(out_count,) host, may be NULL: 0 ok, 1 = ok after jitter,
 * >1 = 1 + failing pivot index.  Replaces optimize.py:479-494 (= :267-285,
 * gp_class.py:516-537). */
int gpmpc_factorize(gpmpc_handle_t h, double jitter, int* info);

/* FITC sparse model (the reference's GP.sparse, gp_class.py:682-689): the handle's own points (gpmpc_set_data, M rows)
 * are the inducing points U; X:(N,Nx), Y:(N,Ny) host are the training set in the GP's input space, streamed through the
 * GPU in column panels (option "fitc_panel", default 4096 points), so device memory is O(M^2 + M * panel + N (Nx+Ny)).
 * With Kuu = k(U,U) + jitter * sf2 I (jitter e.g. 1e-6), Lambda = diag(Kff - Kfu Kuu^-1 Kuf) + sn2 I:
 *   mean(z) = k(U,z)^T alpha_s,  var(z) = sf2 - k(U,z)^T K~^-1 k(U,z),  K~^-1 = Kuu^-1 - (Kuu + Kuf Lambda^-1 Kfu)^-1
 * After the call the handle is factorised and sparse: the L^-1 slab holds R (lower, R^T R = K~^-1) and alpha holds
 * alpha_s, so every predict entry point (and gp_b200_bind) evaluates the FITC prediction with the dense kernels.
 * gpmpc_get returns alpha_s for GET_ALPHA and R for GET_LINV, GPMPC_ERR_STATE for CHOL, K, INVK and LOGDET;
 * gpmpc_append and option "refine" return GPMPC_ERR_STATE; gpmpc_factorize turns the handle back into a dense GP on
 * its own points.  info:(out_count,) may be NULL: 0 ok, 1 = B = I - A^-1 needed the retry shift 1e-10 I (the variance
 * then moves by at most 1e-10 sf2).  nll:(out_count,) may be NULL: FITC negative log marginal likelihood per owned output
 * (no N/2 log 2 pi term, as gpmpc_nlml).  GPMPC_ERR_ARG for N < 1, N > 2^30 (panel indexing is int), a zero noise
 * level or a negative jitter; GPMPC_ERR_NOTPD (the text names the output and Kuu, A or B) when a factor fails. */
int gpmpc_fitc(gpmpc_handle_t h, int N, const double* X, const double* Y, double jitter, int* info, double* nll);

/* CUDA-event phase times (ms) of the handle's last gpmpc_fitc, summed over panels and outputs: ms5 = {Kuf build,
 * V = Luu^-1 Kuf product, column pass + b, SYRK, M-sized factorisations and products (Kuu, A, B, R, alpha_s)}. */
int gpmpc_fitc_timings(gpmpc_handle_t h, double* ms5);

/* Negative log marginal likelihood of global output a at theta:(Nx+2,) host and
 * (grad != NULL) its analytic gradient:  NLL = 1/2 y^T alpha + 1/2 logdet K (no
 * N/2 log 2pi term), with the same jitter retry.  Replaces calc_NLL_numpy,
 * optimize.py:322-356; the gradient replaces SLSQP's finite differences
 * (optimize.py:466-467).  Invalidates the factorisation of output a. */
int gpmpc_nlml(gpmpc_handle_t h, int a, const double* theta, double* nll, double* grad);

/* Batched prediction at H test points (host buffers; copies are part of the call).
 * Z:(H,Nx) in the GP's input space; Sigma:(Nx,Nx) or (H,Nx,Nx) when sigma_per_point
 * (ignored for ME, may be NULL); outputs (any may be NULL): mean:(H,Ny) var:(H,Ny)
 * cov:(H,Ny,Ny) jac:(H,Ny,Nx).  With a communicator attached every rank passes the
 * same Z/Sigma and receives all Ny outputs (one all-gather of H*(2+Nx) doubles per
 * output).  Replaces build_gp / build_TA_cov evaluation gp_functions.py:111-147,
 * :167-171 and GP.covar gp_class.py:353-381. */
int gpmpc_predict(gpmpc_handle_t h, int method, int H, const double* Z, const double* Sigma,
                  int sigma_per_point, double* mean, double* var, double* cov, double* jac);

/* Append ONE training point (x_new:(Nx,), y_new:(Ny,) host, GP input space) to a factorised
 * model in O(N^2): new rows of L and L^-1, alpha refreshed.  Capacity is the padded size
 * ceil(N/128)*128 (GPMPC_ERR_STATE beyond it: refit on a new handle).  GPMPC_ERR_NOTPD if the
 * Schur complement is not positive: refactorise (the jitter policy applies there).  The correct
 * counterpart of the reference's broken GP.update_data (gp_class.py:384-471). */
int gpmpc_append(gpmpc_handle_t h, const double* x_new, const double* y_new);

/* Full posterior covariance between H test points for every OWNED output:
 * out:(out_count,H,H) host, out[a] = sf2_a - V_a^T V_a with V_a = L_a \ k(X, Z)  (the scalar
 * kss = sf2 is broadcast over the whole matrix exactly as the reference does).  Replaces
 * GP.covar, gp_class.py:353-381. */
int gpmpc_posterior_cov(gpmpc_handle_t h, int H, const double* Z, double* out);

/* Prediction plus its first derivatives w.r.t. the test inputs -- what CasADi's AD extracts from
 * the symbolic build_gp / build_TA_cov graphs (gp_functions.py:111-173) when nlpsol differentiates
 * the MPC's NLP (mpc_class.py:390-412, :496-513).  Same arguments and outputs as gpmpc_predict
 * (methods ME and TA; jac = d mean / d z), plus, each optional (NULL to skip):
 *   dvar_dz (H,Ny,Nx)     d var_a / d z_e    = -2 (K^-1 ks)^T d ks/d z_e   (one extra L^-T product)
 *   dcov_dz (H,Ny,Ny,Nx)  d cov[a][b] / d z_e of diag(var) + J Sigma J^T  (needs the mean Hessian)
 *   hess    (H,Ny,Nx,Nx)  d^2 mean_a / d z_d d z_e
 * d cov[a][b] / d Sigma[d][e] = J_a[d] J_b[e] ('TA') is formed by the caller from jac.
 * The handle must own all outputs (single process, or a replicated handle). */
int gpmpc_predict_grad(gpmpc_handle_t h, int method, int H, const double* Z, const double* Sigma,
                       int sigma_per_point, double* mean, double* var, double* cov, double* jac,
                       double* dvar_dz, double* dcov_dz, double* hess);

/* Prediction plus its first AND second derivatives w.r.t. the test inputs -- what IPOPT's default exact Hessian
 * needs from the GP when nlpsol builds the MPC's NLP with 'expand': True and no hessian_approximation
 * (mpc_class.py:496-513; CasADi differentiates the symbolic build_gp / build_TA_cov graphs of gp_functions.py:111-173
 * twice).  Same arguments and outputs as gpmpc_predict_grad (equal to them bit for bit), plus, each optional:
 *   d2var_dz2 (H,Ny,Nx,Nx)     d^2 var_a / d z_d d z_e          (one extra L^-1 product with H*Nx rows per output)
 *   d2cov_dz2 (H,Ny,Ny,Nx,Nx)  d^2 cov[a][b] / d z_d d z_e of diag(var) ('ME') or diag(var) + J Sigma J^T ('TA')
 * Both are exactly symmetric in (d, e).  The mixed block d^2 cov[a][b] / d z_d d Sigma[f][g] =
 * hess_a[f][d] J_b[g] + J_a[f] hess_b[g][d] is formed by the caller from jac and hess; the Sigma-Sigma block is 0.
 * Methods ME and TA; the handle must own all outputs (GPMPC_ERR_STATE otherwise). */
int gpmpc_predict_hess(gpmpc_handle_t h, int method, int H, const double* Z, const double* Sigma,
                       int sigma_per_point, double* mean, double* var, double* cov, double* jac,
                       double* dvar_dz, double* dcov_dz, double* hess, double* d2var_dz2, double* d2cov_dz2);

/* Open-loop multi-step prediction with the state kept on the device: the numeric loop of GP.predict_compare
 * (gp_class.py:746-804, :779-792: mean_t, covar_x = predict(mean_t, u_t, covar); covar[:Ny,:Ny] = covar_x) for a
 * model whose inputs are z = [x, u] (Nx = Ny + Nu).  All Nt steps are enqueued back to back, one synchronisation.
 *   z0      (Nx)        first input [x_0, u_0], already in the GP's input units (standardised when the GP normalises)
 *   U       (Nt, Nu)    inputs u_0 .. u_{Nt-1}, GP input units (row 0 repeats z0's tail); may be NULL when Nu = 0
 *   Sigma0  (Nx, Nx)    covariance of z0; afterwards only its top-left Ny x Ny block is replaced by cov_t
 *   scale   (4, Ny)     [stdY | meanY | meanX | stdX] or NULL: next x = ((mean * stdY + meanY) - meanX) / stdX, the
 *                       inverse_mean / standardize pair of gp_class.py:629-638 in the same operation order
 *   means, vars (Nt, Ny) predicted means / diag(cov_t) (the propagated variance the reference records, gp_class.py:793)
 *                       in the GP's output units, cov_last (Ny, Ny) or NULL
 * method GPMPC_METHOD_ME or _TA; the handle must own all outputs. */
int gpmpc_rollout(gpmpc_handle_t h, int method, int Nt, const double* z0, const double* U, const double* Sigma0,
                  const double* scale, double* means, double* vars, double* cov_last);

/* Problem sizes of a handle (GP.get_size, gp_class.py:266-274: N, and Nx, Ny). */
int gpmpc_get_size(gpmpc_handle_t h, int* N, int* Nx, int* Ny);

/* Same with DEVICE pointers, enqueued on the handle's stream; returns without
 * synchronising unless sync != 0. */
int gpmpc_predict_device(gpmpc_handle_t h, int method, int H, const double* dZ, const double* dSigma,
                         int sigma_per_point, double* d_mean, double* d_var, double* d_cov,
                         double* d_jac, int sync);

/* Copy a result of the last factorisation for global output a into dst (host). */
int gpmpc_get(gpmpc_handle_t h, int what, int a, double* dst);

/* Engine options: "refine" (0/1: one step of iterative refinement of v = L\ks through
 * the stored factor), "predict_ctas" (persistent grid of the stream-K predict product,
 * 0 = two CTAs per SM), "peer" (0/1), "peer_timeout_s" (consumer wait for a peer's flag),
 * "overlap", "gemm_variant", "leaf_variant", "small_tiles" (factorisation A/B switches). */
int gpmpc_set_option(gpmpc_handle_t h, const char* name, double value);

/* Multi-GPU: one process per GPU.  Rank 0 calls gpmpc_comm_unique_id and ships the
 * 128 bytes to the other ranks (any transport); every rank then calls
 * gpmpc_comm_init.  NCCL is loaded with dlopen("libnccl.so.2"). */
int gpmpc_comm_unique_id(void* id128);
int gpmpc_comm_init(gpmpc_handle_t h, const void* id128, int rank, int world);

/* Fused epilogue + all-gather over NVLink peer memory (optional, after gpmpc_comm_init):
 * every rank exports one exchange block (gpmpc_peer_export -> 64-byte CUDA IPC handle, room
 * for Hcap test points), the handles of ALL ranks (world x 64 bytes, rank order) are passed
 * to gpmpc_peer_attach.  gpmpc_predict* then stores each rank's results directly into every
 * peer's buffer from the predict epilogue and synchronises with flags; ncclAllGather remains
 * the fallback (H > Hcap, option "peer" = 0, or no attach). */
int gpmpc_peer_export(gpmpc_handle_t h, int Hcap, void* handle64);
int gpmpc_peer_attach(gpmpc_handle_t h, const void* handles);

/* The handle's CUDA stream (cudaStream_t) so a caller can record events on it. */
void* gpmpc_stream(gpmpc_handle_t h);
int gpmpc_synchronize(gpmpc_handle_t h);

/* Time one kernel of the path with CUDA events on the handle's stream: `reps` launches
 * after one warm-up, average milliseconds in ms_out[0]; n = problem size override
 * (0 = the handle's N).  flops/bytes are derived by the caller (DESIGN.md). */
int gpmpc_profile(gpmpc_handle_t h, int what, int n, int reps, double* ms_out);

/* Load balance of the persistent predict product for an H-point batch: per-CTA busy time
 * out4 = {shortest, longest, mean, first start -> last end} in microseconds (%globaltimer). */
int gpmpc_profile_balance(gpmpc_handle_t h, int H, double* out4);

/* Serial tail of the fused predict kernel (the CTA that completes the step), H-point batch, after a predict call:
 * out8 = microseconds relative to the latest end of every other CTA of {last output complete, records built,
 * step counter passed, records staged, J Sigma done, outputs written}, kernel span, tail CTA span. */
int gpmpc_profile_tail(gpmpc_handle_t h, int H, double* out8);

/* Phase clock stamps (SM cycles since kernel start) of one 128x128 potrf+trtri leaf: out15 =
 * {start, block loaded, first panel, block steps 1..7, L stored, inverse levels 16/32/64, L^-1 stored}. */
int gpmpc_profile_leaf(gpmpc_handle_t h, double* out15);

#ifdef __cplusplus
}
#endif
#endif /* GPMPC_H */
