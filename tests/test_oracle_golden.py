"""Pin the CPU oracle: (1) against the reference's own stored model outputs,
(2) against the committed outputs of the reference's numpy functions run
verbatim, (3) against a recorded run of the reference at further test points,
(4) restated CasADi-only parts by finite differences / limiting cases."""
import numpy as np
import pytest

from oracle import gp_oracle as orc
from tests._util import load_fixture, load_golden, relinf

# tolerances: what re-running LAPACK on the stored (X,Y,hyper) reproduces
# (SURVEY 8c: chol 1e-12 / 2e-10, alpha 6e-13 / 3e-11, invK 4e-10 / 6e-7)
TOL = {'tank': dict(chol=1e-11, alpha=1e-7, invK=1e-7),
       'car': dict(chol=1e-9, alpha=1e-5, invK=1e-5)}


@pytest.mark.parametrize('name', ['tank', 'car'])
def test_postfit_reproduces_stored_model(name):
    m = load_fixture(name)
    out = orc.postfit(m['X'], m['Y'], m['hyper'])
    assert not out['jitter'].any()
    for a in range(m['hyper'].shape[0]):
        assert relinf(out['chol'][a], m['chol'][a]) < TOL[name]['chol']
        assert relinf(out['alpha'][a], m['alpha'][a]) < TOL[name]['alpha']
        assert relinf(out['invK'][a], m['invK'][a]) < TOL[name]['invK']
        # L L^T == K(hyper) to rounding
        K = orc.assemble_K(m['X'], m['hyper'][a])
        assert relinf(m['chol'][a] @ m['chol'][a].T, K) < 1e-13
        assert np.all(np.triu(m['chol'][a], 1) == 0.0)


@pytest.mark.parametrize('name', ['tank', 'car'])
def test_matches_reference_numpy_functions_golden(name):
    m = load_fixture(name)
    g = load_golden('ref_verbatim', name)
    N, Nx = m['X'].shape
    for a in range(m['hyper'].shape[0]):
        ell = m['hyper'][a, :Nx]; sf2 = m['hyper'][a, Nx] ** 2
        K = orc.calc_cov_matrix(m['X'], ell, sf2)
        assert K.sum() == pytest.approx(g['K_sum'][a], rel=1e-13)
        np.testing.assert_allclose(K[N // 3], g['K_row'][a], rtol=1e-13, atol=0)
        # direct-difference kernel (CasADi form) agrees with the expansion form (q13)
        Kd = orc.covSEard(m['X'], m['X'], ell, sf2)
        assert relinf(Kd, K) < 1e-12
        ks = orc.covSEard_expanded(m['X'], g['Zt'], ell, sf2)
        np.testing.assert_allclose(ks, g['ks'][a], rtol=1e-13, atol=1e-300)
        nll = orc.calc_NLL(m['hyper'][a], m['X'], m['Y'][:, a])
        assert nll == pytest.approx(g['nll'][a], rel=1e-12)
        nll_tri = orc.calc_NLL(m['hyper'][a], m['X'], m['Y'][:, a], lapack_general_solve=False)
        assert nll_tri == pytest.approx(g['nll'][a], rel=1e-9)
    cv = orc.covar(m, g['Zt'])
    assert cv.shape == g['covar'].shape
    Ny = m['hyper'].shape[0]
    # full posterior covariance between test points (cancellation-limited on car)
    for a in range(Ny):
        assert relinf(cv[a], g['covar'][a]) < (1e-9 if name == 'tank' else 1e-5)
    assert np.all(cv[Ny:] == 0.0)


@pytest.mark.parametrize('name', ['tank', 'car'])
def test_matches_live_reference(name):
    """Against a recorded run of the reference's calc_cov_matrix, calc_NLL_numpy and GP.covar
    at these test points (oracle/make_golden_live.py)."""
    ref = load_golden('ref_live', name)
    m = load_fixture(name)
    N, Nx = m['X'].shape
    rng = np.random.default_rng(5)
    Zt = m['X'][rng.integers(0, N, 7)] + 0.2 * rng.standard_normal((7, Nx)) * m['X'].std(0)
    np.testing.assert_array_equal(Zt, ref['Zt'])
    for a in range(m['hyper'].shape[0]):
        ell = m['hyper'][a, :Nx]; sf2 = m['hyper'][a, Nx] ** 2
        K = orc.calc_cov_matrix(m['X'], ell, sf2)
        np.testing.assert_allclose(K[ref['K_idx']], ref['K_rows'][a], rtol=1e-14)
        np.testing.assert_allclose(K.sum(1), ref['K_rowsum'][a], rtol=1e-14)
        assert orc.calc_NLL(m['hyper'][a], m['X'], m['Y'][:, a]) == pytest.approx(ref['nll'][a], rel=1e-13)
    np.testing.assert_allclose(orc.covar(m, Zt), ref['covar'], rtol=1e-9, atol=1e-12)
    # variance diag of GP.covar == gp_mean_var's var (LU vs triangular solve)
    _, var = orc.gp_mean_var(m['X'], m['hyper'], m['alpha'], m['chol'], Zt)
    cv = ref['covar']
    for a in range(m['hyper'].shape[0]):
        assert relinf(var[:, a], np.diag(cv[a])) < (1e-8 if name == 'tank' else 5e-6)


@pytest.mark.parametrize('name', ['tank', 'car'])
def test_derived_known_answers(name):
    """SURVEY.md 8(c) 'derived known answers' reproduced from the committed files."""
    m = load_fixture(name)
    d = load_golden('derived', name)
    mean_me, cov_me = orc.predict(m, d['x0'], d['u0'], d['Sigma'], 'ME')
    mean_ta, cov_ta = orc.predict(m, d['x0'], d['u0'], d['Sigma'], 'TA')
    np.testing.assert_allclose(mean_me, d['mean_me'], rtol=1e-12)
    np.testing.assert_allclose(cov_ta, d['cov_ta'], rtol=1e-9, atol=1e-18)
    if name == 'tank':
        np.testing.assert_allclose(mean_me.ravel(), [8.266752073463, 10.48810463329, 9.109971934416,
                                                     19.27473140379], rtol=1e-11)
        np.testing.assert_allclose(np.diag(cov_me), [3.298694845277e-06, 2.992691634063e-06,
                                                     2.279772830960e-06, 1.875281281372e-06], rtol=1e-7)
        np.testing.assert_allclose(np.diag(cov_ta), [1.408665144347e-05, 9.375589269445e-06,
                                                     8.563826033365e-06, 8.508391345415e-06], rtol=1e-8)
        assert cov_ta[0, 1] == pytest.approx(1.9612918544e-09, rel=1e-6)
        mean_em, cov_em = orc.predict(m, d['x0'], d['u0'], d['Sigma'], 'EM')
        np.testing.assert_allclose(np.diag(cov_em), [1.409425146282e-05, 9.386797059696e-06,
                                                     8.584099468967e-06, 8.457177247012e-06], rtol=1e-6)
    else:
        np.testing.assert_allclose(mean_me.ravel(), [13.88592412141, -6.941252728289e-05,
                                                     -4.368765672432e-05], rtol=1e-9)
        np.testing.assert_allclose(np.diag(cov_me), [8.884176168067e-07, 1.101415847415e-08,
                                                     3.437013518237e-08], rtol=2e-6)
        np.testing.assert_allclose(np.diag(cov_ta), [3.142999878963e-06, 3.054629214916e-06,
                                                     5.207704242658e-05], rtol=1e-6)


def test_jacobian_closed_form_vs_central_differences():
    m = load_fixture('tank')
    rng = np.random.default_rng(3)
    Z = 0.5 * rng.standard_normal((5, 6))
    J = orc.gp_mean_jac(m['X'], m['hyper'], m['alpha'], Z)
    h = 1e-4          # mean carries ~1e-11 cancellation noise: keep h well above it
    for d in range(6):
        Zp = Z.copy(); Zp[:, d] += h
        Zm = Z.copy(); Zm[:, d] -= h
        mp, _ = orc.gp_mean_var(m['X'], m['hyper'], m['alpha'], m['chol'], Zp)
        mm, _ = orc.gp_mean_var(m['X'], m['hyper'], m['alpha'], m['chol'], Zm)
        fd = (mp - mm) / (2 * h)
        assert relinf(J[:, :, d], fd) < 1e-5


def test_em_reduces_to_me_at_zero_input_covariance():
    m = load_fixture('tank')
    d = load_golden('derived', 'tank')
    mean_me, cov_me = orc.predict(m, d['x0'], d['u0'], None, 'ME')
    mean_em, cov_em = orc.predict(m, d['x0'], d['u0'], np.zeros((6, 6)), 'EM')
    assert relinf(mean_em, mean_me) < 1e-8
    # EM forms the variance from invK (gp_functions.py:410-411): sf2 - ks^T invK ks cancels ~6
    # digits, and the stored invK carries ~1e-9 relative error (cond 5e7) => only ~2-3 digits
    assert relinf(np.diag(cov_em), np.diag(cov_me)) < 2e-2


def test_nll_gradient_analytic_vs_fd():
    p = orc.synthetic_problem(120, 4, 2, config_id=11)
    for a in range(2):
        th = p['hyper'][a].copy()
        th[:4] *= 0.5
        g = orc.calc_NLL_grad_analytic(th, p['X'], p['Y'][:, a])
        gfd = orc.calc_NLL_grad_fd(th, p['X'], p['Y'][:, a])
        assert relinf(g, gfd) < 1e-5


def test_validate_and_linearize_shapes():
    m = load_fixture('tank')
    rng = np.random.default_rng(1)
    Xt = m['meta']['meanZ'] + m['meta']['stdZ'] * rng.standard_normal((20, 6)) * 0.5
    Yt = m['meta']['meanY'] + m['meta']['stdY'] * rng.standard_normal((20, 4)) * 0.5
    smse, mnlp = orc.validate(m, Xt, Yt)
    assert smse.shape == (4,) and mnlp.shape == (4,)
    d = load_golden('derived', 'tank')
    A, B = orc.discrete_linearize(m, d['x0'], d['u0'])
    assert A.shape == (4, 4) and B.shape == (4, 2)
    np.testing.assert_allclose(A[0], [0.992895022802, -0.001587231485, 0.057914859716, -0.002419994653],
                               rtol=1e-8)


def test_train_small_problem_recovers_low_nll():
    p = orc.synthetic_problem(40, 2, 1, config_id=21)
    out = orc.train_gp(p['X'], p['Y'])
    _, init = orc.train_bounds_init(p['X'], p['Y'][:, 0])
    assert orc.calc_NLL(out['hyper'][0], p['X'], p['Y'][:, 0]) < orc.calc_NLL(init, p['X'], p['Y'][:, 0])


def test_large_size_helpers_match_the_restatement():
    """factor_large / predict_large (BLAS-folded K, no invK -- used by the N >= 4096 GPU parity
    tests) agree with postfit / gp_mean_var / gp_mean_jac / calc_NLL, which are pinned above."""
    p = orc.synthetic_problem(700, 6, 2, config_id=9, H=9)
    post = orc.postfit(p['X'], p['Y'], p['hyper'], lapack_general_solve=False)
    mo, vo = orc.gp_mean_var(p['X'], p['hyper'], post['alpha'], post['chol'], p['Z'])
    Jo = orc.gp_mean_jac(p['X'], p['hyper'], post['alpha'], p['Z'])
    for a in range(2):
        f = orc.factor_large(p['X'], p['Y'][:, a], p['hyper'][a])
        assert relinf(f['chol'], post['chol'][a]) < 1e-11
        assert relinf(f['alpha'], post['alpha'][a]) < 1e-8
        assert f['nll'] == pytest.approx(orc.calc_NLL(p['hyper'][a], p['X'], p['Y'][:, a]), rel=1e-9)   # y.alpha and logdet cancel
        m, v, J = orc.predict_large(p['X'], p['hyper'][a], f['alpha'], f['chol'], p['Z'])
        assert relinf(m, mo[:, a]) < 1e-9 and relinf(v, vo[:, a]) < 1e-8 and relinf(J, Jo[:, a]) < 1e-9
    for name in ('tank', 'car'):
        m = load_fixture(name)
        f = orc.factor_large(m['X'], m['Y'][:, 0], m['hyper'][0])
        assert relinf(f['chol'], m['chol'][0]) < (1e-10 if name == 'tank' else 2e-9)   # the reference's stored factor


def test_fd_derivative_oracle_matches_closed_forms():
    """predict_grad_fd (the checker of gpmpc_predict_grad) against the closed forms evaluated in
    numpy on the tank fixture: d var/dz = -2 (K^-1 ks)^T d ks/dz, mean Hessian, d cov_TA/dz."""
    from scipy.linalg import solve_triangular
    m = load_fixture('tank'); X, Y, hyper = m['X'], m['Y'], m['hyper']
    Ny, Nx = Y.shape[1], X.shape[1]
    post = orc.postfit(X, Y, hyper, lapack_general_solve=False)
    rng = np.random.default_rng(5)
    Z = X[:3] + 0.05 * rng.standard_normal((3, Nx))
    A = rng.standard_normal((Nx, Nx)); S = 1e-3 * np.eye(Nx) + 1e-4 * A @ A.T
    fd = orc.predict_grad_fd(X, hyper, post['alpha'], post['chol'], Z, S, 'TA')
    mean, var = orc.gp_mean_var(X, hyper, post['alpha'], post['chol'], Z)
    J = orc.gp_mean_jac(X, hyper, post['alpha'], Z)
    dvar = np.zeros((3, Ny, Nx)); Hm = np.zeros((3, Ny, Nx, Nx))
    for a in range(Ny):
        ell = hyper[a, :Nx]
        ks = orc.covSEard(X, Z, ell, hyper[a, Nx] ** 2)
        v = solve_triangular(post['chol'][a], ks, lower=True)
        beta = solve_triangular(post['chol'][a], v, lower=True, trans='T')
        for h in range(3):
            s = (X - Z[h]) / ell ** 2
            dvar[h, a] = -2 * (beta[:, h] * ks[:, h]) @ s
            Hm[h, a] = (s * (post['alpha'][a] * ks[:, h])[:, None]).T @ s - np.diag(mean[h, a] / ell ** 2)
    dcov = np.einsum('hade,hbd->habe', Hm, np.einsum('de,hbe->hbd', S, J)) + np.einsum('had,hbde->habe', J @ S, Hm)
    for a in range(Ny):
        dcov[:, a, a, :] += dvar[:, a, :]
    assert relinf(J, fd['dmean']) < 1e-7 and relinf(Hm, fd['hess']) < 1e-6
    assert relinf(dvar, fd['dvar']) < 1e-5 and relinf(dcov, fd['dcov']) < 1e-5
