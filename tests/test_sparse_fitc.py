"""FITC sparse GPs (gpmpc_fitc, Engine.fitc, GP(..., inducing=...), GP.sparse).

CPU: the three oracle forms of tests/_fitc_oracle.py agree; FITC with U = X and a tiny jitter is the dense GP; the dense
closed-form derivatives evaluated with (U, alpha_s, Ltilde) are the derivatives of the FITC prediction.
GPU: the engine's build against the direct form on the reference fixtures, against the Woodbury form with several panels
and beyond the dense engine's capacity; determinism; every consumer of the factor slabs on a sparse handle; refusals.
Achieved errors are printed ('[fitc] ...', visible with -s)."""
import ctypes as C

import numpy as np
import pytest

from oracle import gp_oracle as orc
from tests import _fitc_oracle as fo
from tests._hess_oracle import predict_grad_closed, predict_hess_closed
from tests._util import load_fixture, relinf

PANEL = 4096           # the engine's default panel width (option "fitc_panel")


def _synthetic(N, Nx, Ny, seed):
    """Smooth targets with noise sn = 0.1 and length scales 1.5..3 (standardised inputs)."""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((N, Nx))
    W = rng.standard_normal((Nx, Ny)) / np.sqrt(Nx)
    Y = np.sin(X @ W) + 0.1 * rng.standard_normal((N, Ny))
    hyper = np.column_stack([rng.uniform(1.5, 3.0, (Ny, Nx)), np.ones(Ny), np.full(Ny, 0.1)])
    return X, Y, hyper


def _dense_case():
    """Well conditioned (cond K ~ 1.2e3, sn = 0.1) so that U = X with jitter 1e-10 is the dense GP."""
    rng = np.random.default_rng(5)
    X = rng.standard_normal((150, 4))
    Y = np.sin(X @ rng.standard_normal((4, 2)))
    hyper = np.column_stack([np.full((2, 4), 0.7), np.ones(2), np.full(2, 0.1)])
    return X, Y, hyper, 0.5 * rng.standard_normal((9, 4))


# U = X, jitter 1e-10: FITC differs from the dense GP by the jitter alone.  Measured on the CPU: 2.7e-10 (mean),
# 1.3e-9 (var), 1e-14 (nll) relative, i.e. about 13 x jitter; the bound leaves a decade for the GPU's rounding.
DENSE_JITTER, DENSE_TOL = 1e-10, 1e-8


# ------------------------------------------------------------------ CPU
@pytest.mark.parametrize('shape', [(1500, 120, 5, 2), (3000, 200, 10, 3)])
def test_oracle_forms_agree(shape):
    """direct (N x N) = Woodbury (M x M) = the restated build, for mean, var and nll.  Measured: <= 2.6e-10 between
    the Woodbury form and the others (its Kuu + Kuf Lambda^-1 Kfu is the worst conditioned matrix of the three)."""
    N, M, Nx, Ny = shape
    X, Y, hyper = _synthetic(N, Nx, Ny, N)
    U = X[fo.seeded_subset(N, M)]
    Z = 0.5 * np.random.default_rng(1).standard_normal((9, Nx))
    md, vd, nd = fo.predict('direct', U, X, Y, hyper, Z)
    mw, vw, nw = fo.predict('woodbury', U, X, Y, hyper, Z, chunk=700)
    b = fo.model(U, X, Y, hyper, chunk=1000)
    mb, vb = orc.gp_mean_var(U, hyper, b['alpha'], b['chol'], Z)
    assert relinf(mw, md) < 2e-9 and relinf(vw, vd) < 2e-9 and relinf(nw, nd) < 1e-10
    assert relinf(mb, md) < 1e-10 and relinf(vb, vd) < 1e-10 and relinf(b['nll'], nd) < 1e-10
    assert np.allclose(np.einsum('aki,akj->aij', b['R'], b['R']), b['invK'])


@pytest.mark.parametrize('name,M', [('tank', 30), ('car', 100)])
def test_oracle_build_equals_direct_form_on_fixtures(name, M):
    m = load_fixture(name)
    X, Y, hyper = m['X'], m['Y'], m['hyper']
    U = X[fo.seeded_subset(X.shape[0], M)]
    Z = X[:7] + 0.1
    md, vd, nd = fo.predict('direct', U, X, Y, hyper, Z)
    b = fo.model(U, X, Y, hyper)
    mb, vb = orc.gp_mean_var(U, hyper, b['alpha'], b['chol'], Z)
    assert relinf(mb, md) < 1e-9 and relinf(vb, vd) < 1e-8 and relinf(b['nll'], nd) < 1e-10


def test_oracle_inducing_equal_training_is_dense():
    X, Y, hyper, Z = _dense_case()
    post = orc.postfit(X, Y, hyper, lapack_general_solve=False)
    mo, vo = orc.gp_mean_var(X, hyper, post['alpha'], post['chol'], Z)
    b = fo.model(X, X, Y, hyper, jitter=DENSE_JITTER)
    mb, vb = orc.gp_mean_var(X, hyper, b['alpha'], b['chol'], Z)
    nll = [orc.calc_NLL(hyper[a], X, Y[:, a], False) for a in range(2)]
    assert relinf(mb, mo) < DENSE_TOL and relinf(vb, vo) < DENSE_TOL and relinf(b['nll'], nll) < DENSE_TOL


def test_oracle_closed_forms_are_fitc_derivatives():
    """predict_grad_closed / predict_hess_closed with X -> U, alpha -> alpha_s, chol -> Ltilde against central
    differences of the direct-form FITC mean and variance."""
    X, Y, hyper = _synthetic(400, 3, 2, 17)
    U = X[fo.seeded_subset(400, 40)]
    b = fo.model(U, X, Y, hyper)
    Z = 0.4 * np.random.default_rng(3).standard_normal((4, 3))
    c = predict_hess_closed(U, hyper, b['alpha'], b['chol'], Z, np.zeros((3, 3)), 'ME')
    fdm = np.zeros_like(c['dmean']); fdv = np.zeros_like(c['dvar']); fdh = np.zeros_like(c['d2var'])
    for e in range(3):
        h = 1e-4
        Zp = Z.copy(); Zp[:, e] += h
        Zm = Z.copy(); Zm[:, e] -= h
        mp, vp, _ = fo.predict('direct', U, X, Y, hyper, Zp)
        mm, vm, _ = fo.predict('direct', U, X, Y, hyper, Zm)
        fdm[..., e] = (mp - mm) / (2 * h)
        fdv[..., e] = (vp - vm) / (2 * h)
        gp_ = predict_grad_closed(U, hyper, b['alpha'], b['chol'], Zp, None, 'ME')
        gm_ = predict_grad_closed(U, hyper, b['alpha'], b['chol'], Zm, None, 'ME')
        fdh[..., e] = (gp_['dvar'] - gm_['dvar']) / (2 * h)
    assert relinf(c['dmean'], fdm) < 1e-6 and relinf(c['dvar'], fdv) < 1e-6 and relinf(c['d2var'], fdh) < 1e-5


def test_gp_sparse_refusals_without_a_gpu():
    """A sharded GP refuses sparse(); an explicit inducing array needs hyper.  (No engine is created.)"""
    import gp_mpc_b200
    from tests._fake_engine import OracleEngine

    class TwoRankComm:
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
    with pytest.raises(NotImplementedError, match='one GPU'):
        gp.sparse(10)
    assert gp.inducing is None
    with pytest.raises(NotImplementedError, match='one GPU'):
        gp_mpc_b200.GP(p['X'], p['Y'], hyper=dict(hyper=p['hyper']), normalize=False, engine_factory=OracleEngine,
                       comm=TwoRankComm(), inducing=10)
    with pytest.raises(ValueError, match='needs hyper'):
        gp_mpc_b200.GP(p['X'], p['Y'], normalize=False, engine_factory=OracleEngine, inducing=p['X'][:5])


# ------------------------------------------------------------------ GPU
def _sparse_engine(U, X, Y, hyper, jitter=1e-6, panel=None):
    import gp_mpc_b200
    eng = gp_mpc_b200.Engine(U.shape[0], U.shape[1], Y.shape[1], device=0)
    if panel:
        eng.set_option('fitc_panel', panel)
    eng.set_data(U, np.zeros((U.shape[0], Y.shape[1])))
    eng.set_hyper(hyper)
    info, nll = eng.fitc(X, Y, jitter)
    return eng, info, nll


def _fixture_case(name):
    m = load_fixture(name)
    X, Y, hyper = m['X'], m['Y'], m['hyper']
    M = {'tank': 30, 'car': 100}[name]
    U = X[fo.seeded_subset(X.shape[0], M)]
    rng = np.random.default_rng(21)
    Z = X[:12] + 0.1 * rng.standard_normal((12, X.shape[1]))
    A = rng.standard_normal((X.shape[1],) * 2)
    S = 1e-3 * np.eye(X.shape[1]) + 1e-4 * A @ A.T
    return X, Y, hyper, U, Z, S


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['tank', 'car'])
def test_fitc_fixture_vs_direct_form(name):
    """M = 30 of 60 (tank) and 100 of 200 (car), neither a multiple of 128: mean, var, Jacobian, TA covariance and nll
    against the direct form (N x N algebra), with the dense suite's tolerances."""
    L = __import__('gp_mpc_b200')._lib
    X, Y, hyper, U, Z, S = _fixture_case(name)
    eng, info, nll = _sparse_engine(U, X, Y, hyper)
    md, vd, nd = fo.predict('direct', U, X, Y, hyper, Z)
    b = fo.model(U, X, Y, hyper)
    J = fo.jacobian(U, b['alpha'], hyper, Z)
    mean, var, cov, jac = eng.predict(Z, S, L.METHOD_TA)
    e = dict(mean=relinf(mean, md), var=relinf(var, vd), jac=relinf(jac, J), cov=relinf(cov, orc.ta_cov(vd, J, S)),
             nll=relinf(nll, nd))
    print('[fitc] %s vs direct form: %s' % (name, ' '.join('%s %.2e' % kv for kv in e.items())))
    assert not info.any()
    assert e['mean'] < 1e-6 and e['var'] < 1e-6 and e['jac'] < 1e-6 and e['cov'] < 1e-6 and e['nll'] < 1e-9
    # factors the C ABI exposes: alpha_s and R (lower, zeros above the diagonal)
    R = eng.get(L.GET_LINV, 0)
    assert relinf(eng.get(L.GET_ALPHA, 0), b['alpha'][0]) < 1e-6 and not np.triu(R, 1).any()
    eng.close()


@pytest.mark.gpu
def test_fitc_multi_panel_vs_woodbury():
    """Three panels, the last one partial (N = 2 * 4096 + 1500), M = 500, Nx = 10, Ny = 3, against the Woodbury form."""
    L = __import__('gp_mpc_b200')._lib
    N, M = 2 * PANEL + 1500, 500
    X, Y, hyper = _synthetic(N, 10, 3, 101)
    U = X[fo.seeded_subset(N, M)]
    Z = 0.5 * np.random.default_rng(2).standard_normal((20, 10))
    eng, info, nll = _sparse_engine(U, X, Y, hyper)
    mw, vw, nw = fo.predict('woodbury', U, X, Y, hyper, Z)
    mean, var, _, _ = eng.predict(Z, None, L.METHOD_ME, want_cov=False, want_jac=False)
    e = (relinf(mean, mw), relinf(var, vw), relinf(nll, nw))
    print('[fitc] 3 panels N=%d M=%d vs Woodbury: mean %.2e var %.2e nll %.2e' % ((N, M) + e))
    assert e[0] < 1e-6 and e[1] < 1e-6 and e[2] < 1e-9
    eng.close()


@pytest.mark.gpu
def test_fitc_beyond_dense_capacity():
    """N = 131072 (a dense model would need 137 GB per Npad^2 slab), M = 2048, Ny = 2 through
    GP(X, Y, hyper=..., inducing=2048): no engine larger than M points is ever created; against the Woodbury form."""
    import gp_mpc_b200
    N, M = 131072, 2048
    X, Y, hyper = _synthetic(N, 10, 2, 7)
    sizes = []

    def factory(*args):
        sizes.append(args[0])
        return gp_mpc_b200.Engine(*args)

    gp = gp_mpc_b200.GP(X, Y, hyper=dict(hyper=hyper), normalize=False, gp_method='ME', inducing=M,
                        engine_factory=factory)
    assert sizes == [M] and gp.inducing.shape == (M, 10) and gp.get_size()[0] == N
    U = X[fo.seeded_subset(N, M)]
    assert np.array_equal(gp.inducing, U)
    Z = 0.5 * np.random.default_rng(4).standard_normal((16, 10))
    mw, vw, _ = fo.predict('woodbury', U, X, Y, hyper, Z)
    mean, var, _, _ = gp.engine.predict(Z, None, 0, want_cov=False, want_jac=False)
    e = (relinf(mean, mw), relinf(var, vw))
    print('[fitc] N=%d M=%d vs Woodbury: mean %.2e var %.2e' % ((N, M) + e))
    assert e[0] < 1e-6 and e[1] < 1e-6
    gp.close()


@pytest.mark.gpu
def test_fitc_build_is_deterministic():
    L = __import__('gp_mpc_b200')._lib
    N, M = PANEL + 700, 300
    X, Y, hyper = _synthetic(N, 6, 2, 33)
    U = X[fo.seeded_subset(N, M)]
    Z = 0.5 * np.random.default_rng(5).standard_normal((10, 6))
    outs = []
    for _ in range(2):
        eng, info, nll = _sparse_engine(U, X, Y, hyper)
        outs.append((nll, eng.get(L.GET_ALPHA, 1), eng.get(L.GET_LINV, 1)) + eng.predict(Z, 1e-3 * np.eye(6), L.METHOD_TA))
        eng.close()
    for a, b in zip(*outs):
        assert np.array_equal(a, b)


@pytest.mark.gpu
def test_fitc_with_all_points_equals_dense_handle():
    """M = N, U = X, jitter 1e-10: the sparse handle matches a dense handle on the same data (tolerance from the CPU)."""
    import gp_mpc_b200
    L = gp_mpc_b200._lib
    X, Y, hyper, Z = _dense_case()
    S = 1e-3 * np.eye(4)
    eng, _, nll = _sparse_engine(X, X, Y, hyper, jitter=DENSE_JITTER)
    dense = gp_mpc_b200.Engine(150, 4, 2, device=0)
    dense.set_data(X, Y); dense.set_hyper(hyper); dense.factorize()
    a, b = eng.predict(Z, S, L.METHOD_TA), dense.predict(Z, S, L.METHOD_TA)
    e = [relinf(x, y) for x, y in zip(a, b)]
    nd = [dense.nlml(k, hyper[k], grad=False) for k in range(2)]
    print('[fitc] U = X vs dense handle: mean %.2e var %.2e cov %.2e jac %.2e nll %.2e' % tuple(e + [relinf(nll, nd)]))
    assert max(e) < DENSE_TOL and relinf(nll, nd) < DENSE_TOL
    eng.close(); dense.close()


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['tank', 'car'])
def test_fitc_derivatives_vs_closed_forms(name):
    """predict_grad / predict_hess on the sparse handle ('ME' and 'TA') against the dense closed forms evaluated with
    (U, alpha_s, Ltilde); predict_hess's first-order outputs equal predict_grad's bit for bit."""
    L = __import__('gp_mpc_b200')._lib
    X, Y, hyper, U, Z, S = _fixture_case(name)
    eng, _, _ = _sparse_engine(U, X, Y, hyper)
    b = fo.model(U, X, Y, hyper)
    tol = 1e-6 if name == 'tank' else 1e-4
    for method, mname, Sx in ((L.METHOD_TA, 'TA', S), (L.METHOD_ME, 'ME', None)):
        g = eng.predict_hess(Z, Sx, method)
        g1 = eng.predict_grad(Z, Sx, method, want_hess=True)
        for k in ('mean', 'var', 'cov', 'jac', 'dvar_dz', 'dcov_dz', 'hess'):
            assert np.array_equal(g[k], g1[k]), k
        c = predict_hess_closed(U, hyper, b['alpha'], b['chol'], Z, S, mname)
        e = dict(dmean=relinf(g['jac'], c['dmean']), dvar=relinf(g['dvar_dz'], c['dvar']),
                 dcov=relinf(g['dcov_dz'], c['dcov']), hess=relinf(g['hess'], c['hess']),
                 d2var=relinf(g['d2var_dz2'], c['d2var']), d2cov=relinf(g['d2cov_dz2'], c['d2cov']))
        print('[fitc] %s %s derivatives: %s' % (name, mname, ' '.join('%s %.2e' % kv for kv in e.items())))
        assert max(e.values()) < tol, e
    eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize('method_name', ['TA', 'ME'])
def test_fitc_jac_jac_gp_b200_equals_predict_hess(method_name):
    """casadi.external's jac_jac_gp_b200 bound to a sparse handle returns predict_hess's values on it."""
    from tests.test_predict_hess import _ccs, _dense
    Lb = __import__('gp_mpc_b200')._lib
    lib = Lb.load()
    method = Lb.METHOD_TA if method_name == 'TA' else Lb.METHOD_ME
    X, Y, hyper, U, Z, S = _fixture_case('tank')
    eng, _, _ = _sparse_engine(U, X, Y, hyper)
    Ny, Nx, Nt = 4, 6, 5
    Z = Z[:Nt]
    Sg = np.stack([S * (1 + 0.1 * t) for t in range(Nt)])
    assert lib.gp_b200_bind(eng.h, method, Nt) == 0
    jac_pats = [_ccs(lib.jac_gp_b200_sparsity_out(k)) for k in range(4)]
    pats = [_ccs(lib.jac_jac_gp_b200_sparsity_out(k)) for k in range(16)]
    dp = C.POINTER(C.c_double)
    ins = [np.ascontiguousarray(Z), np.ascontiguousarray(np.transpose(Sg, (0, 2, 1))), np.zeros(Nt * Ny),
           np.zeros(Nt * Ny * Ny)] + [np.zeros(max(1, p[2][-1])) for p in jac_pats]
    outs = [np.full(max(1, p[2][-1]), np.nan) for p in pats]
    arg = (dp * 8)(*[a.ctypes.data_as(dp) for a in ins])
    res = (dp * 16)(*[o.ctypes.data_as(dp) for o in outs])
    assert lib.jac_jac_gp_b200(arg, res, None, None, 0) == 0
    g = eng.predict_hess(Z, Sg if method_name == 'TA' else None, method)
    D0, D8 = _dense(pats[0], outs[0]), _dense(pats[8], outs[8])
    for t in range(Nt):
        for e in range(Nx):
            M0 = np.zeros((Ny * Nt, Nx * Nt)); M0[t * Ny:(t + 1) * Ny, t * Nx:(t + 1) * Nx] = g['hess'][t][:, :, e]
            assert np.array_equal(D0[:, e + Nx * t], M0.flatten(order='F'))
            M2 = np.zeros((Ny * Ny * Nt, Nx * Nt))
            M2[t * Ny * Ny:(t + 1) * Ny * Ny, t * Nx:(t + 1) * Nx] = \
                g['d2cov_dz2'][t][:, :, :, e].transpose(1, 0, 2).reshape(Ny * Ny, Nx)
            assert np.array_equal(D8[:, e + Nx * t], M2.flatten(order='F'))
    lib.gp_b200_unbind()
    eng.close()


def _sparse_gp_from_fixture(name, M):
    import gp_mpc_b200
    m = load_fixture(name)
    kw = dict(mean_func='zero', gp_method='TA', normalize=m['normalize'], hyper=dict(hyper=m['hyper']), inducing=M)
    if m['normalize']:
        kw.update(meta=m['meta'], xlb=m['xlb'], xub=m['xub'], ulb=m['ulb'], uub=m['uub'])
    return gp_mpc_b200.GP(m['X'], m['Y'], **kw), m


@pytest.mark.gpu
def test_fitc_gp_consumers():
    """On a sparse GP: the device rollout equals the host loop, 'EM' equals gp_exact_moment with invK = K~^-1 (the
    targets replaced by K~ alpha_s), GP.covar equals sf2 - (R ks)^T (R ks), and GP.sparse converts a dense GP in place
    to the same model."""
    from tests._util import load_golden
    gp, m = _sparse_gp_from_fixture('tank', 30)
    X, hyper = m['X'], m['hyper']
    U = gp.inducing
    assert np.array_equal(U, X[fo.seeded_subset(60, 30)])
    b = fo.model(U, X, m['Y'], hyper)
    d = load_golden('derived', 'tank')
    useq = np.tile(d['u0'], (12, 1)) * (1 + 0.02 * np.arange(12)[:, None])
    rm, rv = gp.rollout(d['x0'], useq, methods=['TA', 'ME'])
    rm_h, rv_h = gp.rollout(d['x0'], useq, methods=['TA', 'ME'], device_rollout=False)
    print('[fitc] rollout device vs host: %.2e %.2e' % (relinf(rm, rm_h), relinf(rv, rv_h)))
    assert relinf(rm, rm_h) < 1e-12 and relinf(rv, rv_h) < 1e-12 and (rv[:, 1:] > 0).all()
    # EM
    z = X[3] + 0.05
    Sig = 1e-3 * np.eye(6)
    mean, var, cov, _ = gp.engine.predict(z[None], Sig, 2, want_jac=False)
    mo, co = orc.gp_exact_moment(b['invK'], U, b['Yeff'], hyper, z, Sig)
    print('[fitc] EM vs gp_exact_moment: mean %.2e cov %.2e' % (relinf(mean[0], mo), relinf(cov[0], co)))
    assert relinf(mean[0], mo) < 1e-6 and relinf(cov[0], co) < 1e-5
    # covar
    Zc = X[:5] + 0.1
    cv = gp.covar(Zc)
    for a in range(4):
        v = np.linalg.solve(b['chol'][a], orc.covSEard(U, Zc, hyper[a, :6], hyper[a, 6] ** 2))
        assert relinf(cv[a], hyper[a, 6] ** 2 - v.T @ v) < 1e-6
    assert not cv[4:].any()
    # GP.sparse(M) on a dense GP gives the same model
    from tests.test_gpu_parity import _gp_from_fixture
    dense, _ = _gp_from_fixture('tank')
    assert dense.inducing is None
    dense.sparse(30)
    assert np.array_equal(dense.inducing, U)
    Zs = d['Zs'] if d['Zs'].ndim == 2 else d['Zs'][None]
    for k in range(3):
        a1, a2 = gp.engine.predict(Zs, Sig, 1)[k], dense.engine.predict(Zs, Sig, 1)[k]
        assert np.array_equal(a1, a2)
    gp.close(); dense.close()


@pytest.mark.gpu
def test_fitc_refusals():
    """GPMPC_ERR_STATE for CHOL / K / INVK / LOGDET, append and refine on a sparse handle; GPMPC_ERR_ARG for bad N;
    gpmpc_factorize turns the handle back into a dense GP; the GP methods that need the dense model raise."""
    import gp_mpc_b200
    L = gp_mpc_b200._lib
    X, Y, hyper, U, Z, S = _fixture_case('tank')
    eng, _, _ = _sparse_engine(U, X, Y, hyper)
    for what in (L.GET_CHOL, L.GET_K, L.GET_INVK, L.GET_LOGDET):
        with pytest.raises(L.GpmpcError) as ex:
            eng.get(what, 0)
        assert ex.value.code == L.ERR_STATE
    assert eng.append(X[0] + 0.1, Y[0]) is False
    assert eng.lib.gpmpc_append(eng.h, X[0].ctypes.data_as(C.POINTER(C.c_double)),
                                Y[0].ctypes.data_as(C.POINTER(C.c_double))) == L.ERR_STATE
    with pytest.raises(L.GpmpcError) as ex:
        eng.set_option('refine', 1)
    assert ex.value.code == L.ERR_STATE
    dp = C.POINTER(C.c_double)
    x, y = np.ascontiguousarray(X), np.ascontiguousarray(Y)
    for n in (0, -3, (1 << 30) + 1):
        assert eng.lib.gpmpc_fitc(eng.h, n, x.ctypes.data_as(dp), y.ctypes.data_as(dp), 1e-6, None, None) == L.ERR_ARG
    assert 'N <= ' in eng.lib.gpmpc_last_error(eng.h).decode()
    # back to a dense GP on the handle's own 30 points
    eng.factorize()
    post = orc.postfit(U, np.zeros((30, 4)), hyper, lapack_general_solve=False)
    assert relinf(eng.get(L.GET_CHOL, 0), post['chol'][0]) < 1e-9
    eng.close()
    gp, m = _sparse_gp_from_fixture('tank', 30)
    for call in (lambda: gp.optimize(), lambda: gp.update_data_all(m['X'][:2], m['Y'][:2]),
                 lambda: gp.replace_data_all(m['X'][:2], m['Y'][:2]), lambda: gp.append_data(m['X'][:1], m['Y'][:1]),
                 lambda: gp.save_model('/nonexistent/x'), lambda: gp.save_model_npz('/nonexistent/x'),
                 gp.get_chol, gp.get_invK):
        with pytest.raises(NotImplementedError, match='sparse'):
            call()
    gp.close()
