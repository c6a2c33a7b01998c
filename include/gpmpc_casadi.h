/* CasADi `external` entry points of libgpmpc.so -- the C side of the adapter that lets
 * mpc_class.py keep its CasADi/IPOPT NLP while the GP inside it runs on the GPU
 * (SURVEY.md 8f row 1; reference call sites mpc_class.py:361-423, :496-513,
 * gp_class.py:207-263).  Usage from Python, once CasADi is installed:
 *
 *     lib.gp_b200_bind(engine_handle, GPMPC_METHOD_TA, Nt)
 *     F = casadi.external('gp_b200', '.../libgpmpc.so')    # F(z, sigma) -> (mean, cov)
 *
 * CasADi resolves `gp_b200`, `gp_b200_n_in/_n_out/_name_in/_name_out/_sparsity_in/_sparsity_out/
 * _work/_incref/_decref` and, for derivatives, the Jacobian function `jac_gp_b200` with the same
 * family of helpers.  Conventions: casadi_int = long long, casadi_real = double, dense blocks are
 * column-major, sparsity patterns are compressed-column {nrow, ncol, colind[ncol+1], row[nnz]}
 * ({nrow, ncol, 1} = dense).  Shapes for Nt shooting nodes (all in the GP's standardised space;
 * the scaling of gp_class.py:253-262 is two elementwise CasADi expressions around F):
 *   z (Nx x Nt), sigma (Nx x Nx*Nt)  ->  mean (Ny x Nt), cov (Ny x Ny*Nt)
 *   jac_gp_b200(z, sigma, mean, cov) -> jac_mean_z, jac_mean_sigma (empty), jac_cov_z, jac_cov_sigma
 *   (block-diagonal: node t only depends on node t's inputs).
 * For IPOPT's exact Hessian the next level, jac_jac_gp_b200 (around gpmpc_predict_hess), takes jac's four inputs
 * and its four nominal outputs (z, sigma, out_mean, out_cov, out_jac_mean_z, out_jac_mean_sigma, out_jac_cov_z,
 * out_jac_cov_sigma) and returns the 16 blocks jac_<o>_<i> of jac's outputs o w.r.t. its inputs i, o-major
 * (jac_jac_mean_z_z, jac_jac_mean_z_sigma, ...).  Block (o, i) is numel(o) x numel(i): its rows follow the
 * column-major vectorisation of o's FULL dimensions, not o's nonzeros.  That row convention is the one
 * assumption here not verified against CasADi.  Non-empty blocks (block-diagonal over nodes):
 *   jac_jac_mean_z_z      d^2 mean_a / dz_d dz_e                           (the mean Hessian)
 *   jac_jac_cov_z_z       d^2 cov[a][b] / dz_d dz_e                        (d2cov_dz2)
 *   jac_jac_cov_z_sigma   d^2 cov[a][b] / dz_d dSigma[f][g] = Hm_a[f][d] J_b[g] + J_a[f] Hm_b[g][d]   ('TA')
 *   jac_jac_cov_sigma_z   the same mixed block seen from jac_cov_sigma                             ('TA')
 */
#ifndef GPMPC_CASADI_H
#define GPMPC_CASADI_H
#include "gpmpc.h"
#ifdef __cplusplus
extern "C" {
#endif

int gp_b200_bind(gpmpc_handle_t h, int method, int Nt);
void gp_b200_unbind(void);

long long gp_b200_n_in(void);
long long gp_b200_n_out(void);
const char* gp_b200_name_in(long long i);
const char* gp_b200_name_out(long long i);
const long long* gp_b200_sparsity_in(long long i);
const long long* gp_b200_sparsity_out(long long i);
int gp_b200_work(long long* sz_arg, long long* sz_res, long long* sz_iw, long long* sz_w);
void gp_b200_incref(void);
void gp_b200_decref(void);
int gp_b200(const double** arg, double** res, long long* iw, double* w, int mem);

long long jac_gp_b200_n_in(void);
long long jac_gp_b200_n_out(void);
const char* jac_gp_b200_name_in(long long i);
const char* jac_gp_b200_name_out(long long i);
const long long* jac_gp_b200_sparsity_in(long long i);
const long long* jac_gp_b200_sparsity_out(long long i);
int jac_gp_b200_work(long long* sz_arg, long long* sz_res, long long* sz_iw, long long* sz_w);
int jac_gp_b200(const double** arg, double** res, long long* iw, double* w, int mem);

long long jac_jac_gp_b200_n_in(void);
long long jac_jac_gp_b200_n_out(void);
const char* jac_jac_gp_b200_name_in(long long i);
const char* jac_jac_gp_b200_name_out(long long i);
const long long* jac_jac_gp_b200_sparsity_in(long long i);
const long long* jac_jac_gp_b200_sparsity_out(long long i);
int jac_jac_gp_b200_work(long long* sz_arg, long long* sz_res, long long* sz_iw, long long* sz_w);
int jac_jac_gp_b200(const double** arg, double** res, long long* iw, double* w, int mem);

#ifdef __cplusplus
}
#endif
#endif /* GPMPC_CASADI_H */
