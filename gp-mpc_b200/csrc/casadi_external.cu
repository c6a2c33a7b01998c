// CasADi `external`-shaped entry points around gpmpc_predict_grad (SURVEY 8f row 1).
//
// mpc_class.py:361-423 calls gp.predict(mean_t, u_t, covar_t) once per shooting node with MX
// symbols and nlpsol (:496-513) differentiates the resulting graph.  With
//     F = casadi.external('gp_b200', 'libgpmpc.so')
// the GP becomes ONE opaque call for all Nt nodes per NLP iterate, evaluated on the GPU, with the
// analytic Jacobian function `jac_gp_b200` CasADi looks up by name.  The signatures follow
// CasADi's C API for external functions (casadi_int = long long, casadi_real = double; dense
// matrices are column-major, sparsity patterns are compressed-column: {nrow, ncol, colind[ncol+1],
// row[nnz]}, with the 3-entry form {nrow, ncol, 1} meaning dense).  Nothing here needs CasADi to
// compile or to be tested: tests drive these entry points through ctypes.
//
//   inputs : i0 = Z     (Nx  x Nt)     test inputs of all shooting nodes, standardised space
//            i1 = Sigma (Nx  x Nx*Nt)  input covariance of every node (Nt blocks side by side)
//   outputs: o0 = mean  (Ny  x Nt)
//            o1 = cov   (Ny  x Ny*Nt)  'TA' / 'ME' covariance blocks
//   jac_gp_b200: inputs (i0, i1, o0, o1), outputs block-diagonal sparse
//            jac_o0_i0 (Ny*Nt x Nx*Nt), jac_o0_i1 (empty), jac_o1_i0 (Ny*Ny*Nt x Nx*Nt),
//            jac_o1_i1 (Ny*Ny*Nt x Nx*Nx*Nt;  d cov[a][b] / d Sigma[d][e] = J_a[d] J_b[e] for 'TA')
//   jac_jac_gp_b200 (around gpmpc_predict_hess): inputs jac's four inputs and its four nominal outputs, outputs the
//            16 blocks jac_<o>_<i> (o-major), numel(o) x numel(i) each: rows follow the column-major vectorisation of
//            o's full dimensions (not its nonzeros).  Non-empty: jac_mean_z / z (the mean Hessian), jac_cov_z / z
//            (d2cov), jac_cov_z / sigma and jac_cov_sigma / z (the mixed z-Sigma block, 'TA' only).  This row
//            convention is the one assumption of this file that has not been checked against CasADi itself.
#include "../../include/gpmpc.h"

#include <mutex>
#include <string>
#include <vector>

typedef long long casadi_int;
typedef double casadi_real;

namespace {
struct Bound {
    gpmpc_handle_t h = nullptr;
    int method = GPMPC_METHOD_TA, Nt = 0, Nx = 0, Ny = 0;
    std::vector<casadi_int> sp_in[2], sp_out[2], sp_jac[4], sp_hess[16];
    std::vector<double> sig, mean, var, cov, jac, dvar, dcov, hess, d2cov;
    int refs = 0;
};
Bound g_b;
std::mutex g_mtx;

std::vector<casadi_int> dense_sp(casadi_int r, casadi_int c) { return {r, c, 1}; }

// block-diagonal CCS pattern: Nt dense blocks of R rows x Cc columns
std::vector<casadi_int> blockdiag_sp(casadi_int R, casadi_int Cc, casadi_int Nt)
{
    std::vector<casadi_int> sp;
    sp.reserve(2 + Cc * Nt + 1 + R * Cc * Nt);
    sp.push_back(R * Nt); sp.push_back(Cc * Nt);
    for (casadi_int c = 0; c <= Cc * Nt; ++c) sp.push_back(c * R);
    for (casadi_int t = 0; t < Nt; ++t)
        for (casadi_int c = 0; c < Cc; ++c)
            for (casadi_int r = 0; r < R; ++r) sp.push_back(t * R + r);
    return sp;
}
std::vector<casadi_int> empty_sp(casadi_int r, casadi_int c)
{
    std::vector<casadi_int> sp(2 + c + 1, 0);
    sp[0] = r; sp[1] = c;
    return sp;
}

// second-level block pattern: numel(o) rows x (cpn*Nt) columns; every column of node t holds the rows row(t, k),
// k = 0 .. rpn-1 (ascending in k)
template <class RowFn>
std::vector<casadi_int> node_sp(casadi_int nrow, casadi_int cpn, casadi_int rpn, casadi_int Nt, RowFn row)
{
    std::vector<casadi_int> sp;
    sp.reserve(2 + cpn * Nt + 1 + rpn * cpn * Nt);
    sp.push_back(nrow); sp.push_back(cpn * Nt);
    for (casadi_int c = 0; c <= cpn * Nt; ++c) sp.push_back(c * rpn);
    for (casadi_int t = 0; t < Nt; ++t)
        for (casadi_int c = 0; c < cpn; ++c)
            for (casadi_int k = 0; k < rpn; ++k) sp.push_back(row(t, k));
    return sp;
}

// evaluate mean/cov (+ derivatives when grad) for the bound handle; Sigma blocks are transposed to
// the engine's row-major convention (a symmetric Sigma is unchanged)
int eval(const casadi_real* Z, const casadi_real* Sigma, bool grad)
{
    Bound& b = g_b;
    if (!b.h || !Z) return 1;
    const int Nt = b.Nt, Nx = b.Nx;
    const bool ta = b.method == GPMPC_METHOD_TA;
    if (ta) {
        if (!Sigma) return 1;
        for (int t = 0; t < Nt; ++t)
            for (int d = 0; d < Nx; ++d)
                for (int e = 0; e < Nx; ++e)
                    b.sig[((size_t)t * Nx + d) * Nx + e] = Sigma[((size_t)t * Nx + e) * Nx + d];
    }
    if (!grad)
        return gpmpc_predict(b.h, b.method, Nt, Z, ta ? b.sig.data() : nullptr, 1, b.mean.data(), b.var.data(),
                             b.cov.data(), b.jac.data()) == GPMPC_OK ? 0 : 1;
    return gpmpc_predict_grad(b.h, b.method, Nt, Z, ta ? b.sig.data() : nullptr, 1, b.mean.data(), b.var.data(),
                              b.cov.data(), b.jac.data(), b.dvar.data(), b.dcov.data(), nullptr) == GPMPC_OK ? 0 : 1;
}

// the second derivatives of jac_jac_gp_b200: jac, the mean Hessian and d2cov for the bound handle
int eval_hess(const casadi_real* Z, const casadi_real* Sigma)
{
    Bound& b = g_b;
    if (!b.h || !Z) return 1;
    const int Nt = b.Nt, Nx = b.Nx;
    const bool ta = b.method == GPMPC_METHOD_TA;
    if (ta) {
        if (!Sigma) return 1;
        for (int t = 0; t < Nt; ++t)
            for (int d = 0; d < Nx; ++d)
                for (int e = 0; e < Nx; ++e)
                    b.sig[((size_t)t * Nx + d) * Nx + e] = Sigma[((size_t)t * Nx + e) * Nx + d];
    }
    return gpmpc_predict_hess(b.h, b.method, Nt, Z, ta ? b.sig.data() : nullptr, 1, nullptr, nullptr, nullptr, b.jac.data(),
                              nullptr, nullptr, b.hess.data(), nullptr, b.d2cov.data()) == GPMPC_OK ? 0 : 1;
}
}  // namespace

// Bind the (process-global) external to a factorised engine handle: method GPMPC_METHOD_ME / _TA,
// Nt shooting nodes per call.  Call again to re-bind (e.g. after a refit or another horizon).
extern "C" int gp_b200_bind(gpmpc_handle_t h, int method, int Nt)
{
    std::lock_guard<std::mutex> lock(g_mtx);
    int N = 0, Nx = 0, Ny = 0;
    if (!h || Nt < 1 || (method != GPMPC_METHOD_ME && method != GPMPC_METHOD_TA)) return GPMPC_ERR_ARG;
    if (gpmpc_get_size(h, &N, &Nx, &Ny) != GPMPC_OK) return GPMPC_ERR_ARG;
    Bound& b = g_b;
    b.h = h; b.method = method; b.Nt = Nt; b.Nx = Nx; b.Ny = Ny;
    b.sp_in[0] = dense_sp(Nx, Nt); b.sp_in[1] = dense_sp(Nx, (casadi_int)Nx * Nt);
    b.sp_out[0] = dense_sp(Ny, Nt); b.sp_out[1] = dense_sp(Ny, (casadi_int)Ny * Nt);
    b.sp_jac[0] = blockdiag_sp(Ny, Nx, Nt);
    b.sp_jac[1] = empty_sp((casadi_int)Ny * Nt, (casadi_int)Nx * Nx * Nt);
    b.sp_jac[2] = blockdiag_sp((casadi_int)Ny * Ny, Nx, Nt);
    b.sp_jac[3] = (method == GPMPC_METHOD_TA) ? blockdiag_sp((casadi_int)Ny * Ny, (casadi_int)Nx * Nx, Nt)
                                              : empty_sp((casadi_int)Ny * Ny * Nt, (casadi_int)Nx * Nx * Nt);
    b.sig.assign((size_t)Nt * Nx * Nx, 0.0);
    b.mean.assign((size_t)Nt * Ny, 0.0); b.var.assign((size_t)Nt * Ny, 0.0);
    b.cov.assign((size_t)Nt * Ny * Ny, 0.0); b.jac.assign((size_t)Nt * Ny * Nx, 0.0);
    b.dvar.assign((size_t)Nt * Ny * Nx, 0.0); b.dcov.assign((size_t)Nt * Ny * Ny * Nx, 0.0);
    // jac_jac_gp_b200: block k = 4 o + i of jac output o (numel no[o]) w.r.t. jac input i (numel ni[i])
    const casadi_int T = Nt, X = Nx, Y = Ny;
    const casadi_int no[4] = {Y * T * X * T, Y * T * X * X * T, Y * Y * T * X * T, Y * Y * T * X * X * T};
    const casadi_int ni[4] = {X * T, X * X * T, Y * T, Y * Y * T};
    for (int k = 0; k < 16; ++k) b.sp_hess[k] = empty_sp(no[k / 4], ni[k % 4]);
    // jac_mean_z (Ny*Nt x Nx*Nt) entry (t Ny + a, t Nx + d) / z[e][t]: column e of node t, rows k = d Ny + a
    b.sp_hess[0] = node_sp(no[0], X, Y * X, T, [=](casadi_int t, casadi_int k) {
        const casadi_int d = k / Y, a = k % Y;
        return (t * Y + a) + Y * T * (t * X + d); });
    // jac_cov_z (Ny*Ny*Nt x Nx*Nt) entry (t Ny^2 + a + Ny b, t Nx + d): rows k = (d Ny + b) Ny + a
    auto row_cz = [=](casadi_int t, casadi_int k) {
        const casadi_int d = k / (Y * Y), bb = (k / Y) % Y, a = k % Y;
        return (t * Y * Y + a + Y * bb) + Y * Y * T * (t * X + d); };
    b.sp_hess[8] = node_sp(no[2], X, Y * Y * X, T, row_cz);
    if (method == GPMPC_METHOD_TA) {
        b.sp_hess[9] = node_sp(no[2], X * X, Y * Y * X, T, row_cz);          // columns f + Nx g of node t's Sigma
        // jac_cov_sigma (Ny*Ny*Nt x Nx*Nx*Nt) entry (t Ny^2 + a + Ny b, t Nx^2 + f + Nx g): rows k = ((g Nx + f) Ny + b) Ny + a
        b.sp_hess[12] = node_sp(no[3], X, Y * Y * X * X, T, [=](casadi_int t, casadi_int k) {
            const casadi_int g = k / (Y * Y * X), f = (k / (Y * Y)) % X, bb = (k / Y) % Y, a = k % Y;
            return (t * Y * Y + a + Y * bb) + Y * Y * T * (t * X * X + f + X * g); });
    }
    b.hess.assign((size_t)Nt * Ny * Nx * Nx, 0.0); b.d2cov.assign((size_t)Nt * Ny * Ny * Nx * Nx, 0.0);
    return GPMPC_OK;
}

extern "C" void gp_b200_unbind(void)
{
    std::lock_guard<std::mutex> lock(g_mtx);
    g_b = Bound();
}

// ---- the function itself
extern "C" casadi_int gp_b200_n_in(void) { return 2; }
extern "C" casadi_int gp_b200_n_out(void) { return 2; }
extern "C" const char* gp_b200_name_in(casadi_int i) { return i == 0 ? "z" : (i == 1 ? "sigma" : nullptr); }
extern "C" const char* gp_b200_name_out(casadi_int i) { return i == 0 ? "mean" : (i == 1 ? "cov" : nullptr); }
extern "C" const casadi_int* gp_b200_sparsity_in(casadi_int i) { return (i >= 0 && i < 2 && g_b.h) ? g_b.sp_in[i].data() : nullptr; }
extern "C" const casadi_int* gp_b200_sparsity_out(casadi_int i) { return (i >= 0 && i < 2 && g_b.h) ? g_b.sp_out[i].data() : nullptr; }
extern "C" int gp_b200_work(casadi_int* sz_arg, casadi_int* sz_res, casadi_int* sz_iw, casadi_int* sz_w)
{
    if (sz_arg) *sz_arg = 2;
    if (sz_res) *sz_res = 2;
    if (sz_iw) *sz_iw = 0;
    if (sz_w) *sz_w = 0;
    return 0;
}
extern "C" void gp_b200_incref(void) { std::lock_guard<std::mutex> lock(g_mtx); ++g_b.refs; }
extern "C" void gp_b200_decref(void) { std::lock_guard<std::mutex> lock(g_mtx); --g_b.refs; }

extern "C" int gp_b200(const casadi_real** arg, casadi_real** res, casadi_int* iw, casadi_real* w, int mem)
{
    (void)iw; (void)w; (void)mem;
    std::lock_guard<std::mutex> lock(g_mtx);
    if (!arg || !res) return 1;
    if (eval(arg[0], arg[1], false)) return 1;
    const Bound& b = g_b;
    // (Nt,Ny) row-major == Ny x Nt column-major; each Ny x Ny block is written column-major
    // (element (a,b) at a + Ny*b) -- the blocks are symmetric only up to rounding
    if (res[0]) std::copy(b.mean.begin(), b.mean.end(), res[0]);
    if (res[1])
        for (int t = 0; t < b.Nt; ++t)
            for (int bb = 0; bb < b.Ny; ++bb)
                for (int a = 0; a < b.Ny; ++a)
                    res[1][((size_t)t * b.Ny + bb) * b.Ny + a] = b.cov[((size_t)t * b.Ny + a) * b.Ny + bb];
    return 0;
}

// ---- its Jacobian: inputs (z, sigma, mean, cov), outputs the four blocks in CCS nonzero order
extern "C" casadi_int jac_gp_b200_n_in(void) { return 4; }
extern "C" casadi_int jac_gp_b200_n_out(void) { return 4; }
extern "C" const char* jac_gp_b200_name_in(casadi_int i)
{
    static const char* n[] = {"z", "sigma", "out_mean", "out_cov"};
    return (i >= 0 && i < 4) ? n[i] : nullptr;
}
extern "C" const char* jac_gp_b200_name_out(casadi_int i)
{
    static const char* n[] = {"jac_mean_z", "jac_mean_sigma", "jac_cov_z", "jac_cov_sigma"};
    return (i >= 0 && i < 4) ? n[i] : nullptr;
}
extern "C" const casadi_int* jac_gp_b200_sparsity_in(casadi_int i)
{
    if (!g_b.h || i < 0 || i > 3) return nullptr;
    return i < 2 ? g_b.sp_in[i].data() : g_b.sp_out[i - 2].data();
}
extern "C" const casadi_int* jac_gp_b200_sparsity_out(casadi_int i) { return (i >= 0 && i < 4 && g_b.h) ? g_b.sp_jac[i].data() : nullptr; }
extern "C" int jac_gp_b200_work(casadi_int* sz_arg, casadi_int* sz_res, casadi_int* sz_iw, casadi_int* sz_w)
{
    if (sz_arg) *sz_arg = 4;
    if (sz_res) *sz_res = 4;
    if (sz_iw) *sz_iw = 0;
    if (sz_w) *sz_w = 0;
    return 0;
}

extern "C" int jac_gp_b200(const casadi_real** arg, casadi_real** res, casadi_int* iw, casadi_real* w, int mem)
{
    (void)iw; (void)w; (void)mem;
    std::lock_guard<std::mutex> lock(g_mtx);
    if (!arg || !res) return 1;
    if (eval(arg[0], arg[1], true)) return 1;
    const Bound& b = g_b;
    const int Nt = b.Nt, Nx = b.Nx, Ny = b.Ny;
    if (res[0])          // block t, column d, row a:  d mean_a / d z_d
        for (int t = 0; t < Nt; ++t)
            for (int d = 0; d < Nx; ++d)
                for (int a = 0; a < Ny; ++a) res[0][((size_t)t * Nx + d) * Ny + a] = b.jac[((size_t)t * Ny + a) * Nx + d];
    if (res[2])          // block t, column e, row a + Ny*b (column-major vec of the Ny x Ny block)
        for (int t = 0; t < Nt; ++t)
            for (int e = 0; e < Nx; ++e)
                for (int bb = 0; bb < Ny; ++bb)
                    for (int a = 0; a < Ny; ++a)
                        res[2][(((size_t)t * Nx + e) * Ny + bb) * Ny + a] = b.dcov[(((size_t)t * Ny + a) * Ny + bb) * Nx + e];
    if (res[3] && b.method == GPMPC_METHOD_TA)   // column d + Nx*e (vec of Sigma), row a + Ny*b:  J_a[d] J_b[e]
        for (int t = 0; t < Nt; ++t)
            for (int e = 0; e < Nx; ++e)
                for (int d = 0; d < Nx; ++d)
                    for (int bb = 0; bb < Ny; ++bb)
                        for (int a = 0; a < Ny; ++a)
                            res[3][((((size_t)t * Nx + e) * Nx + d) * Ny + bb) * Ny + a] =
                                b.jac[((size_t)t * Ny + a) * Nx + d] * b.jac[((size_t)t * Ny + bb) * Nx + e];
    return 0;
}

// ---- the Jacobian of jac_gp_b200: inputs (z, sigma, out_mean, out_cov, and jac's four nominal outputs), 16 blocks
extern "C" casadi_int jac_jac_gp_b200_n_in(void) { return 8; }
extern "C" casadi_int jac_jac_gp_b200_n_out(void) { return 16; }
extern "C" const char* jac_jac_gp_b200_name_in(casadi_int i)
{
    static const char* n[] = {"z", "sigma", "out_mean", "out_cov", "out_jac_mean_z", "out_jac_mean_sigma", "out_jac_cov_z",
                              "out_jac_cov_sigma"};
    return (i >= 0 && i < 8) ? n[i] : nullptr;
}
extern "C" const char* jac_jac_gp_b200_name_out(casadi_int i)
{
    static const std::vector<std::string> n = [] {
        const char* o[] = {"jac_mean_z", "jac_mean_sigma", "jac_cov_z", "jac_cov_sigma"};
        const char* in[] = {"z", "sigma", "out_mean", "out_cov"};
        std::vector<std::string> v;
        for (const char* oo : o)
            for (const char* ii : in) v.push_back(std::string("jac_") + oo + "_" + ii);
        return v;
    }();
    return (i >= 0 && i < 16) ? n[i].c_str() : nullptr;
}
extern "C" const casadi_int* jac_jac_gp_b200_sparsity_in(casadi_int i)
{
    if (!g_b.h || i < 0 || i > 7) return nullptr;
    return i < 2 ? g_b.sp_in[i].data() : (i < 4 ? g_b.sp_out[i - 2].data() : g_b.sp_jac[i - 4].data());
}
extern "C" const casadi_int* jac_jac_gp_b200_sparsity_out(casadi_int i)
{
    return (i >= 0 && i < 16 && g_b.h) ? g_b.sp_hess[i].data() : nullptr;
}
extern "C" int jac_jac_gp_b200_work(casadi_int* sz_arg, casadi_int* sz_res, casadi_int* sz_iw, casadi_int* sz_w)
{
    if (sz_arg) *sz_arg = 8;
    if (sz_res) *sz_res = 16;
    if (sz_iw) *sz_iw = 0;
    if (sz_w) *sz_w = 0;
    return 0;
}

// nonzeros in the CCS order of the patterns built by gp_b200_bind
extern "C" int jac_jac_gp_b200(const casadi_real** arg, casadi_real** res, casadi_int* iw, casadi_real* w, int mem)
{
    (void)iw; (void)w; (void)mem;
    std::lock_guard<std::mutex> lock(g_mtx);
    if (!arg || !res) return 1;
    if (eval_hess(arg[0], arg[1])) return 1;
    const Bound& b = g_b;
    const size_t Nt = b.Nt, Nx = b.Nx, Ny = b.Ny;
    auto J = [&](size_t t, size_t a, size_t d) { return b.jac[(t * Ny + a) * Nx + d]; };
    auto Hm = [&](size_t t, size_t a, size_t f, size_t d) { return b.hess[((t * Ny + a) * Nx + f) * Nx + d]; };
    if (res[0]) {        // column (t, e), rows (d, a): d^2 mean_a / dz_d dz_e
        casadi_real* o = res[0];
        for (size_t t = 0; t < Nt; ++t)
            for (size_t e = 0; e < Nx; ++e)
                for (size_t d = 0; d < Nx; ++d)
                    for (size_t a = 0; a < Ny; ++a) *o++ = Hm(t, a, d, e);
    }
    if (res[8]) {        // column (t, e), rows (d, b, a): d^2 cov[a][b] / dz_d dz_e
        casadi_real* o = res[8];
        for (size_t t = 0; t < Nt; ++t)
            for (size_t e = 0; e < Nx; ++e)
                for (size_t d = 0; d < Nx; ++d)
                    for (size_t bb = 0; bb < Ny; ++bb)
                        for (size_t a = 0; a < Ny; ++a) *o++ = b.d2cov[(((t * Ny + a) * Ny + bb) * Nx + d) * Nx + e];
    }
    if (b.method == GPMPC_METHOD_TA && res[9]) {   // column (t, f + Nx g), rows (d, b, a): Hm_a[f][d] J_b[g] + J_a[f] Hm_b[g][d]
        casadi_real* o = res[9];
        for (size_t t = 0; t < Nt; ++t)
            for (size_t g = 0; g < Nx; ++g)
                for (size_t f = 0; f < Nx; ++f)
                    for (size_t d = 0; d < Nx; ++d)
                        for (size_t bb = 0; bb < Ny; ++bb)
                            for (size_t a = 0; a < Ny; ++a) *o++ = Hm(t, a, f, d) * J(t, bb, g) + J(t, a, f) * Hm(t, bb, g, d);
    }
    if (b.method == GPMPC_METHOD_TA && res[12]) {  // column (t, e), rows (g, f, b, a): Hm_a[f][e] J_b[g] + J_a[f] Hm_b[g][e]
        casadi_real* o = res[12];
        for (size_t t = 0; t < Nt; ++t)
            for (size_t e = 0; e < Nx; ++e)
                for (size_t g = 0; g < Nx; ++g)
                    for (size_t f = 0; f < Nx; ++f)
                        for (size_t bb = 0; bb < Ny; ++bb)
                            for (size_t a = 0; a < Ny; ++a) *o++ = Hm(t, a, f, e) * J(t, bb, g) + J(t, a, f) * Hm(t, bb, g, e);
    }
    return 0;
}
