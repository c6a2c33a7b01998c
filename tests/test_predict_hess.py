"""Second derivatives of the prediction w.r.t. the test input (gpmpc_predict_hess, jac_jac_gp_b200,
GP.predict_batch_hess): what IPOPT's exact Hessian needs from the GP inside the reference's MPC NLP
(mpc_class.py:496-513).

CPU: the closed forms of tests/_hess_oracle.py against central differences (first order against the oracle's
predict_grad_fd, second order against differences of the first-order closed form), the jac_jac_gp_b200 metadata and
the host-side refusals.  GPU: the engine against those closed forms and against differences of its own first
derivatives, bitwise identities, edge shapes, the CasADi entry point through ctypes and the GP-class view."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from oracle import gp_oracle as orc
from tests._hess_oracle import predict_grad_closed, predict_hess_closed
from tests._util import load_fixture, load_golden, relinf

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _problem(case):
    """X, Y, hyper, Z, Sigma (Nx,Nx) of a named case.  The synthetic Sigmas are made non-symmetric on purpose."""
    if case in ('tank', 'car'):
        m = load_fixture(case); X, Y, hyper = m['X'], m['Y'], m['hyper']
        rng = np.random.default_rng(5)
        Z = X[rng.choice(X.shape[0], 6, replace=False)] + 0.05 * rng.standard_normal((6, X.shape[1]))
        A = rng.standard_normal((X.shape[1],) * 2)
        return X, Y, hyper, Z, 1e-3 * np.eye(X.shape[1]) + 1e-4 * A @ A.T
    N, Nx, Ny, H = dict(synA=(90, 3, 2, 4), synB=(160, 5, 3, 4), syn700=(700, 7, 3, 9), syn1500=(1500, 17, 3, 66))[case]
    p = orc.synthetic_problem(N, Nx, Ny, config_id=N, H=H)
    A = np.random.default_rng(2).standard_normal((Nx, Nx))
    return p['X'], p['Y'], p['hyper'], p['Z'], p['Sigma'] + 1e-5 * A


def _fd_of_grad(X, hyper, post, Z, S, method, rel=1e-4):
    """Central differences of predict_grad_closed: d2var, d2cov and the mean Hessian."""
    g0 = predict_grad_closed(X, hyper, post['alpha'], post['chol'], Z, S, method)
    out = dict(d2var=np.zeros(g0['dvar'].shape + (Z.shape[1],)), d2cov=np.zeros(g0['dcov'].shape + (Z.shape[1],)),
               hess=np.zeros_like(g0['hess']))
    for e in range(Z.shape[1]):
        h = rel * np.maximum(1.0, np.abs(Z[:, e]))
        Zp = Z.copy(); Zp[:, e] += h
        Zm = Z.copy(); Zm[:, e] -= h
        gp = predict_grad_closed(X, hyper, post['alpha'], post['chol'], Zp, S, method)
        gm = predict_grad_closed(X, hyper, post['alpha'], post['chol'], Zm, S, method)
        out['d2var'][..., e] = (gp['dvar'] - gm['dvar']) / (2 * h[:, None, None])
        out['d2cov'][..., e] = (gp['dcov'] - gm['dcov']) / (2 * h[:, None, None, None])
        out['hess'][..., e] = (gp['dmean'] - gm['dmean']) / (2 * h[:, None, None])
    return out


# ------------------------------------------------------------------ CPU: the closed forms
@pytest.mark.parametrize('case', ['tank', 'car', 'synA', 'synB'])
def test_closed_form_first_derivatives_vs_central_differences(case):
    """predict_grad_closed against the oracle's predict_grad_fd with the tolerances of the GPU first-derivative test
    (1e-5; car 3e-5: cond(K) ~ 1e10 makes the difference quotient of var noisy)."""
    X, Y, hyper, Z, S = _problem(case)
    post = orc.postfit(X, Y, hyper, lapack_general_solve=False)
    tol = 1e-5 if case != 'car' else 3e-5
    for method in ('TA', 'ME'):
        c = predict_grad_closed(X, hyper, post['alpha'], post['chol'], Z, S, method)
        fd = orc.predict_grad_fd(X, hyper, post['alpha'], post['chol'], Z, S, method)
        for k in ('dmean', 'dvar', 'dcov', 'hess'):
            assert relinf(c[k], fd[k]) < tol, (method, k, relinf(c[k], fd[k]))


@pytest.mark.parametrize('case', ['tank', 'car', 'synA', 'synB'])
def test_closed_form_second_derivatives_vs_central_differences(case):
    """predict_hess_closed's d2var, d2cov ('TA', 'ME') and mean Hessian against central differences of
    predict_grad_closed.  Measured worst: 1.5e-6 (car d2var), 8e-7 (tank), <= 1e-7 (synthetic); bound 1e-5."""
    X, Y, hyper, Z, S = _problem(case)
    post = orc.postfit(X, Y, hyper, lapack_general_solve=False)
    for method in ('TA', 'ME'):
        c = predict_hess_closed(X, hyper, post['alpha'], post['chol'], Z, S, method)
        fd = _fd_of_grad(X, hyper, post, Z, S, method)
        for k in ('d2var', 'd2cov', 'hess'):
            assert relinf(c[k], fd[k]) < 1e-5, (method, k, relinf(c[k], fd[k]))
        g = predict_grad_closed(X, hyper, post['alpha'], post['chol'], Z, S, method)
        for k in g:
            assert np.array_equal(c[k], g[k])


# ------------------------------------------------------------------ CPU: the CasADi entry point's metadata
def _lib():
    import __graft_entry__ as g
    g.build()
    import gp_mpc_b200
    return gp_mpc_b200._lib


JJ_IN = ['z', 'sigma', 'out_mean', 'out_cov', 'out_jac_mean_z', 'out_jac_mean_sigma', 'out_jac_cov_z', 'out_jac_cov_sigma']
JJ_OUT = ['jac_%s_%s' % (o, i) for o in ('jac_mean_z', 'jac_mean_sigma', 'jac_cov_z', 'jac_cov_sigma')
          for i in ('z', 'sigma', 'out_mean', 'out_cov')]


def test_jac_jac_metadata_without_a_gpu():
    """jac_jac_gp_b200's helpers answer without a device; patterns exist only once bound; every jac_jac_gp_b200*
    name of include/gpmpc_casadi.h is exported and bound by _lib.load()."""
    L = _lib()
    lib = L.load()
    hdr = open(os.path.join(ROOT, 'include', 'gpmpc_casadi.h')).read().split('#ifndef GPMPC_CASADI_H')[1]
    declared = set(re.findall(r'\b(jac_jac_gp_b200[A-Za-z_0-9]*)\s*\(', hdr))
    assert len(declared) == 8 and declared == {s[0] for s in L.SYMBOLS_HESS}
    for name in declared:
        assert getattr(lib, name) is not None
    assert lib.jac_jac_gp_b200_n_in() == 8 and lib.jac_jac_gp_b200_n_out() == 16
    assert [lib.jac_jac_gp_b200_name_in(i).decode() for i in range(8)] == JJ_IN
    assert [lib.jac_jac_gp_b200_name_out(i).decode() for i in range(16)] == JJ_OUT
    assert lib.jac_jac_gp_b200_name_in(8) is None and lib.jac_jac_gp_b200_name_out(16) is None
    sz = [C.c_longlong(-1) for _ in range(4)]
    assert lib.jac_jac_gp_b200_work(*[C.byref(x) for x in sz]) == 0 and [x.value for x in sz] == [8, 16, 0, 0]
    assert not any(lib.jac_jac_gp_b200_sparsity_in(i) for i in range(8))         # not bound
    assert not any(lib.jac_jac_gp_b200_sparsity_out(i) for i in range(16))
    assert 'gpmpc_predict_hess' in {s[0] for s in L.SYMBOLS}


def test_gp_view_refuses_em_and_sharded_models():
    """Host-side refusals of GP.predict_batch_hess (same conditions as predict_batch_grad)."""
    import gp_mpc_b200
    from tests._fake_engine import OracleEngine

    class TwoRankComm:                       # rank 0 of two with the outputs sharded across the ranks
        rank, world = 0, 2

        def allgather_object(self, obj):
            return [obj, obj]

        def broadcast_object(self, obj, src=0):
            return obj

        def barrier(self):
            pass

    p = orc.synthetic_problem(40, 4, 3, config_id=5, H=3)
    gp = gp_mpc_b200.GP(p['X'], p['Y'], hyper=dict(hyper=p['hyper']), normalize=False, engine_factory=OracleEngine,
                        comm=TwoRankComm())
    with pytest.raises(NotImplementedError, match='all outputs on one GPU'):
        gp.predict_batch_hess(p['Z'][:, :3], p['Z'][:, 3:], p['Sigma'])
    gp1 = gp_mpc_b200.GP(p['X'], p['Y'], hyper=dict(hyper=p['hyper']), normalize=False, engine_factory=OracleEngine)
    with pytest.raises(NotImplementedError, match="'ME' and 'TA'"):
        gp1.predict_batch_hess(p['Z'][:, :3], p['Z'][:, 3:], p['Sigma'], method='EM')


# ------------------------------------------------------------------ GPU
def _fit(X, Y, hyper):
    import gp_mpc_b200
    eng = gp_mpc_b200.Engine(X.shape[0], X.shape[1], Y.shape[1], device=0)
    eng.set_data(X, Y)
    eng.set_hyper(hyper)
    eng.factorize()
    return eng


def _check_identities(g, g1, method):
    """predict_hess's first-order outputs equal predict_grad's bit for bit; d2var / d2cov are exactly symmetric in
    (d, e); 'ME': d2cov is diag(d2var) exactly."""
    for k in ('mean', 'var', 'cov', 'jac', 'dvar_dz', 'dcov_dz', 'hess'):
        assert np.array_equal(g[k], g1[k]), k
    assert np.array_equal(g['d2var_dz2'], np.swapaxes(g['d2var_dz2'], -1, -2))
    assert np.array_equal(g['d2cov_dz2'], np.swapaxes(g['d2cov_dz2'], -1, -2))
    if method == 'ME':
        Ny = g['var'].shape[1]
        for a in range(Ny):
            assert np.array_equal(g['d2cov_dz2'][:, a, a], g['d2var_dz2'][:, a])
            for b in range(Ny):
                if b != a:
                    assert not g['d2cov_dz2'][:, a, b].any()


# car: cond(K) ~ 1e10.  The engine's beta = K^-1 ks and the L^-1 products carry ~cond(K) eps relative error, and
# the second derivatives of var are sums of terms far larger than their result.  Bound set from the measured error.
HESS_TOL = dict(tank=1e-6, car=1e-4, syn700=1e-6, syn1500=1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize('case', ['tank', 'car', 'syn700', 'syn1500'])
def test_predict_hess_vs_oracle_and_differences(case):
    """gpmpc_predict_hess against predict_hess_closed (batch-inf-norm relative, HESS_TOL) and against central
    differences of the engine's own predict_grad (dvar_dz, dcov_dz; 1e-5, car 1e-3), 'TA' and 'ME'.  syn1500
    (Nx = 17, H = 66) takes the Nx > 16 reduction, two 64-point chunks and W passes of 3 points (51 rows)."""
    L = __import__('gp_mpc_b200')._lib
    X, Y, hyper, Z, S = _problem(case)
    eng = _fit(X, Y, hyper)
    post = orc.postfit(X, Y, hyper, lapack_general_solve=False)
    Sg = np.stack([S * (1 + 0.05 * h) for h in range(Z.shape[0])])
    for method, name, Sx in ((L.METHOD_TA, 'TA', Sg), (L.METHOD_ME, 'ME', None)):
        g = eng.predict_hess(Z, Sx, method)
        g1 = eng.predict_grad(Z, Sx, method, want_hess=True)
        _check_identities(g, g1, name)
        c = predict_hess_closed(X, hyper, post['alpha'], post['chol'], Z, Sg, name)
        e_var, e_cov = relinf(g['d2var_dz2'], c['d2var']), relinf(g['d2cov_dz2'], c['d2cov'])
        print('[hess] %s %s oracle d2var %.2e d2cov %.2e' % (case, name, e_var, e_cov))
        assert e_var < HESS_TOL[case] and e_cov < HESS_TOL[case]
        # the engine's own first derivatives, differenced
        fdv = np.zeros_like(g['d2var_dz2']); fdc = np.zeros_like(g['d2cov_dz2'])
        for e in range(Z.shape[1]):
            h = 1e-4 * np.maximum(1.0, np.abs(Z[:, e]))
            Zp = Z.copy(); Zp[:, e] += h
            Zm = Z.copy(); Zm[:, e] -= h
            gp_, gm_ = eng.predict_grad(Zp, Sx, method), eng.predict_grad(Zm, Sx, method)
            fdv[..., e] = (gp_['dvar_dz'] - gm_['dvar_dz']) / (2 * h[:, None, None])
            fdc[..., e] = (gp_['dcov_dz'] - gm_['dcov_dz']) / (2 * h[:, None, None, None])
        f_var, f_cov = relinf(g['d2var_dz2'], fdv), relinf(g['d2cov_dz2'], fdc)
        print('[hess] %s %s differences d2var %.2e d2cov %.2e' % (case, name, f_var, f_cov))
        tol = 1e-5 if case != 'car' else 1e-3
        assert f_var < tol and f_cov < tol
    eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize('shape', [(1, 1, 1, 1), (300, 12, 3, 5), (130, 32, 2, 3)])
def test_predict_hess_edge_shapes(shape):
    """N=1, Nx=1, Ny=1, H=1; Nx=12 (the 8 < Nx <= 16 reduction); N=130, Nx=NX_MAX=32, Ny=2, H=3 (two points per W
    pass, 528 pairs) vs the oracle."""
    L = __import__('gp_mpc_b200')._lib
    N, Nx, Ny, H = shape
    rng = np.random.default_rng(11)
    X = rng.standard_normal((N, Nx)); Y = rng.standard_normal((N, Ny))
    hyper = np.column_stack([rng.uniform(1.5, 4.0, (Ny, Nx)), np.ones(Ny), 0.1 * np.ones(Ny)])
    Z = X[:1] + 0.3 * rng.standard_normal((H, Nx))
    A = rng.standard_normal((Nx, Nx)); S = 1e-3 * np.eye(Nx) + 1e-4 * A
    eng = _fit(X, Y, hyper)
    post = orc.postfit(X, Y, hyper, lapack_general_solve=False)
    for method, name, Sx in ((L.METHOD_TA, 'TA', S), (L.METHOD_ME, 'ME', None)):
        g = eng.predict_hess(Z, Sx, method)
        _check_identities(g, eng.predict_grad(Z, Sx, method, want_hess=True), name)
        c = predict_hess_closed(X, hyper, post['alpha'], post['chol'], Z, S, name)
        e_var, e_cov = relinf(g['d2var_dz2'], c['d2var']), relinf(g['d2cov_dz2'], c['d2cov'])
        print('[hess] edge %s %s d2var %.2e d2cov %.2e' % (shape, name, e_var, e_cov))
        assert e_var < 1e-6 and e_cov < 1e-6
    eng.close()
    import gp_mpc_b200
    part = gp_mpc_b200.Engine(N, Nx, Ny, out_begin=0, out_count=1, device=0) if Ny > 1 else None
    if part is not None:                       # a handle that owns only part of the outputs refuses
        part.set_data(X, Y); part.set_hyper(hyper); part.factorize()
        with pytest.raises(L.GpmpcError) as ex:
            part.predict_hess(Z, S, L.METHOD_TA)
        assert ex.value.code == L.ERR_STATE
        part.close()


def _ccs(ptr):
    nrow, ncol = ptr[0], ptr[1]
    colind = np.array([ptr[2 + k] for k in range(ncol + 1)])
    rows = np.array([ptr[2 + ncol + 1 + k] for k in range(colind[-1])], dtype=np.int64)
    return nrow, ncol, colind, rows


def _dense(pat, vals):
    nrow, ncol, colind, rows = pat
    D = np.zeros((nrow, ncol))
    for c in range(ncol):
        D[rows[colind[c]:colind[c + 1]], c] = vals[colind[c]:colind[c + 1]]
    return D


@pytest.mark.gpu
@pytest.mark.parametrize('method_name', ['TA', 'ME'])
def test_jac_jac_gp_b200_entry_point(method_name):
    """jac_jac_gp_b200 driven through ctypes: valid CCS patterns of numel(o) x numel(i) with the stated nnz, and the
    densified blocks equal the derivative of the column-major vectorisation of jac_gp_b200's full output matrices,
    built here from predict_hess (hess, d2cov_dz2, jac) -- zero off the node block diagonal."""
    Lb = __import__('gp_mpc_b200')._lib
    lib = Lb.load()
    method = Lb.METHOD_TA if method_name == 'TA' else Lb.METHOD_ME
    m = load_fixture('tank'); X, Y, hyper = m['X'], m['Y'], m['hyper']
    Ny, Nx, Nt = 4, 6, 5
    eng = _fit(X, Y, hyper)
    rng = np.random.default_rng(8)
    Z = X[:Nt] + 0.1 * rng.standard_normal((Nt, Nx))
    Sg = np.stack([1e-3 * np.eye(Nx) + 1e-4 * rng.standard_normal((Nx, Nx)) for _ in range(Nt)])
    assert lib.gp_b200_bind(eng.h, method, Nt) == 0
    jac_pats = [_ccs(lib.jac_gp_b200_sparsity_out(k)) for k in range(4)]
    for k in range(4):                         # inputs 4..7 are jac's outputs
        a, b = _ccs(lib.jac_jac_gp_b200_sparsity_in(4 + k)), jac_pats[k]
        assert a[:2] == b[:2] and np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])
    numel_o = [p[0] * p[1] for p in jac_pats]
    numel_i = [Nx * Nt, Nx * Nx * Nt, Ny * Nt, Ny * Ny * Nt]
    nonempty = {0: Nt * Nx * Ny * Nx, 8: Nt * Nx * Ny * Ny * Nx}
    if method_name == 'TA':
        nonempty.update({9: Nt * Nx * Nx * Ny * Ny * Nx, 12: Nt * Nx * Ny * Ny * Nx * Nx})
    pats = []
    for k in range(16):
        nrow, ncol, colind, rows = p = _ccs(lib.jac_jac_gp_b200_sparsity_out(k))
        assert (nrow, ncol) == (numel_o[k // 4], numel_i[k % 4]), k
        assert colind[0] == 0 and (np.diff(colind) >= 0).all() and colind[-1] == nonempty.get(k, 0), k
        for c in range(ncol):
            r = rows[colind[c]:colind[c + 1]]
            assert (np.diff(r) > 0).all() and (r.size == 0 or (r[0] >= 0 and r[-1] < nrow))
        pats.append(p)
    dp = C.POINTER(C.c_double)
    z_cm = np.ascontiguousarray(Z)
    s_cm = np.ascontiguousarray(np.transpose(Sg, (0, 2, 1)))
    ins = [z_cm, s_cm, np.zeros(Nt * Ny), np.zeros(Nt * Ny * Ny)] + [np.zeros(max(1, p[2][-1])) for p in jac_pats]
    outs = [np.full(max(1, p[2][-1]), np.nan) for p in pats]
    arg = (dp * 8)(*[a.ctypes.data_as(dp) for a in ins])
    res = (dp * 16)(*[o.ctypes.data_as(dp) for o in outs])
    assert lib.jac_jac_gp_b200(arg, res, None, None, 0) == 0
    g = eng.predict_hess(Z, Sg if method_name == 'TA' else None, method)
    J, Hm, d2c = g['jac'], g['hess'], g['d2cov_dz2']
    # expected: column (node t, input entry) = vec_F(d M_o / d input entry) for jac's full output matrices M_o
    exp = {k: np.zeros((numel_o[k // 4], numel_i[k % 4])) for k in nonempty}
    for t in range(Nt):
        for e in range(Nx):
            M0 = np.zeros((Ny * Nt, Nx * Nt)); M0[t * Ny:(t + 1) * Ny, t * Nx:(t + 1) * Nx] = Hm[t][:, :, e]
            exp[0][:, e + Nx * t] = M0.flatten(order='F')
            M2 = np.zeros((Ny * Ny * Nt, Nx * Nt))          # rows t Ny^2 + a + Ny b of d cov[a][b] / dz_d
            M2[t * Ny * Ny:(t + 1) * Ny * Ny, t * Nx:(t + 1) * Nx] = d2c[t][:, :, :, e].transpose(1, 0, 2).reshape(Ny * Ny, Nx)
            exp[8][:, e + Nx * t] = M2.flatten(order='F')
            if method_name == 'TA':
                M3 = np.zeros((Ny * Ny * Nt, Nx * Nx * Nt))   # d (J_a[f] J_b[g]) / dz_e at column f + Nx g
                blk = np.einsum('af,bg->bagf', Hm[t][:, :, e], J[t]) + np.einsum('af,bg->bagf', J[t], Hm[t][:, :, e])
                M3[t * Ny * Ny:(t + 1) * Ny * Ny, t * Nx * Nx:(t + 1) * Nx * Nx] = blk.reshape(Ny * Ny, Nx * Nx)
                exp[12][:, e + Nx * t] = M3.flatten(order='F')
        if method_name == 'TA':
            for f in range(Nx):
                for gg in range(Nx):                   # d (d cov[a][b] / dz_d) / d Sigma_t[f][g]
                    M2 = np.zeros((Ny * Ny * Nt, Nx * Nt))
                    blk = np.einsum('ad,b->bad', Hm[t][:, f, :], J[t][:, gg]) + np.einsum('a,bd->bad', J[t][:, f], Hm[t][:, gg, :])
                    M2[t * Ny * Ny:(t + 1) * Ny * Ny, t * Nx:(t + 1) * Nx] = blk.reshape(Ny * Ny, Nx)
                    exp[9][:, f + Nx * (t * Nx + gg)] = M2.flatten(order='F')
    for k in range(16):
        D = _dense(pats[k], outs[k])
        if k in (0, 8):
            assert np.array_equal(D, exp[k]), k                                   # copies of the engine's values
        elif k in nonempty:
            assert relinf(D, exp[k]) < 1e-14, k                                    # products formed on the host
        else:
            assert not D.any(), k
    lib.gp_b200_unbind()
    assert not lib.jac_jac_gp_b200_sparsity_out(0)
    eng.close()


@pytest.mark.gpu
def test_gp_predict_batch_hess_vs_differences_of_predict_batch_grad():
    """GP.predict_batch_hess on the tank fixture (normalize=True) in the caller's units against central differences
    of predict_batch_grad; its first-order entries equal predict_batch_grad's."""
    import gp_mpc_b200
    m = load_fixture('tank')
    kw = dict(mean_func='zero', gp_method='TA', normalize=m['normalize'],
              hyper=dict(hyper=m['hyper'], invK=m['invK'], alpha=m['alpha'], chol=m['chol'],
                         length_scale=m['length_scale'], signal_var=m['signal_var'],
                         noise_var=m['noise_var'], mean=m['mean']))
    if m['normalize']:
        kw.update(meta=m['meta'], xlb=m['xlb'], xub=m['xub'], ulb=m['ulb'], uub=m['uub'])
    gp = gp_mpc_b200.GP(m['X'], m['Y'], **kw)
    d = load_golden('derived', 'tank')
    xs = np.tile(d['x0'], (3, 1)) * (1 + 0.02 * np.arange(3)[:, None]); us = np.tile(d['u0'], (3, 1))
    Ny = xs.shape[1]
    for method in ('TA', 'ME'):
        gh = gp.predict_batch_hess(xs, us, d['Sigma'], method=method)
        gg = gp.predict_batch_grad(xs, us, d['Sigma'], method=method)
        for k in gg:
            assert np.array_equal(gh[k], gg[k]), k
        zs = np.hstack([xs, us])
        for e in range(zs.shape[1]):
            h = 1e-4 * max(1.0, abs(zs[0, e]))
            zp = zs.copy(); zp[:, e] += h
            zm = zs.copy(); zm[:, e] -= h
            gp_ = gp.predict_batch_grad(zp[:, :Ny], zp[:, Ny:], d['Sigma'], method=method)
            gm_ = gp.predict_batch_grad(zm[:, :Ny], zm[:, Ny:], d['Sigma'], method=method)
            e_m = relinf(gh['d2mean_dz2'][..., e], (gp_['dmean_dz'] - gm_['dmean_dz']) / (2 * h))
            e_c = relinf(gh['d2cov_dz2'][..., e], (gp_['dcov_dz'] - gm_['dcov_dz']) / (2 * h))
            e_s = relinf(gh['d2cov_dzdSigma_factor'][..., e], (gp_['dcov_dSigma_factor'] - gm_['dcov_dSigma_factor']) / (2 * h))
            print('[hess] gp %s e=%d d2mean %.2e d2cov %.2e factor %.2e' % (method, e, e_m, e_c, e_s))
            assert e_m < 1e-5 and e_c < 1e-4 and e_s < 1e-5
    gp.close()
