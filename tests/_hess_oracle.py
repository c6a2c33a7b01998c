"""Closed-form first and second derivatives of the restated GP prediction w.r.t. the test input -- the
checker for gpmpc_predict_hess (TEST INFRASTRUCTURE ONLY).

The prediction is the oracle's restatement of ``build_gp`` / ``build_TA_cov`` (``gp_functions.py:111-173``):
mean = ks^T alpha, var = sf2 - v^T v with v = L^-1 ks, cov = diag(var) [+ J Sigma J^T for 'TA'].  With
s_id = (X_id - z_d)/ell_d^2 and beta = K^-1 ks = L^-T v:
    J_d        = sum_i alpha_i ks_i s_id
    dvar_d     = -2 sum_i beta_i ks_i s_id
    Hm_de      = sum_i alpha_i ks_i s_id s_ie - delta_de mean/ell_d^2
    d2var_de   = -2 [ w_d^T w_e + sum_i beta_i ks_i s_id s_ie - delta_de (sf2 - var)/ell_d^2 ],  w_d = L^-1 (ks o s_.d)
    T_fde      = sum_i alpha_i ks_i s_if s_id s_ie - delta_fd J_e/ell_f^2 - delta_fe J_d/ell_f^2 - delta_de J_f/ell_d^2
    'TA' dcov_ab,d   = delta_ab dvar_a,d + sum_fg [Hm_a,fd Sigma_fg J_b,g + J_a,f Sigma_fg Hm_b,gd]
    'TA' d2cov_ab,de = delta_ab d2var_a,de + sum_fg [T_a,fde Sigma_fg J_b,g + Hm_a,fd Sigma_fg Hm_b,ge
                                                     + Hm_a,fe Sigma_fg Hm_b,gd + J_a,f Sigma_fg T_b,gde]
    'ME' dcov = diag(dvar), d2cov = diag(d2var)
Both functions use triangular solves on the factor ``oracle.gp_oracle.postfit`` returns; Sigma need not be
symmetric.  They are pinned against central differences of ``oracle.gp_oracle.predict_grad_fd`` and of each other
in tests/test_predict_hess.py.
"""
import numpy as np
from scipy.linalg import solve_triangular

from oracle import gp_oracle as orc


def _per_output(X, hyper_a, alpha_a, L_a, Z):
    """ks (N,H), s (H,N,Nx), mean (H,), var (H,), J (H,Nx), Hm (H,Nx,Nx), dvar (H,Nx), beta-weighted ks (N,H)."""
    Nx = X.shape[1]
    ell = hyper_a[:Nx]; sf2 = hyper_a[Nx] ** 2
    ks = orc.covSEard(X, Z, ell, sf2)                                   # (N,H)
    s = (X[None, :, :] - Z[:, None, :]) / ell ** 2                      # (H,N,Nx)
    v = solve_triangular(L_a, ks, lower=True)
    beta = solve_triangular(L_a, v, lower=True, trans='T')
    mean = ks.T @ alpha_a
    var = sf2 - np.sum(v * v, axis=0)
    wa = (ks * alpha_a[:, None]).T                                      # (H,N)
    wb = (ks * beta).T
    J = np.einsum('hi,hid->hd', wa, s)
    dvar = -2.0 * np.einsum('hi,hid->hd', wb, s)
    Hm = np.einsum('hi,hid,hie->hde', wa, s, s) - np.einsum('h,de->hde', mean, np.diag(1.0 / ell ** 2))
    return dict(ks=ks, s=s, mean=mean, var=var, J=J, Hm=Hm, dvar=dvar, wa=wa, wb=wb, ell=ell, sf2=sf2)


def _sigma(Sigma, H, Nx):
    S = np.asarray(Sigma, dtype=np.float64)
    return np.broadcast_to(S, (H, Nx, Nx)) if S.ndim == 2 else S


def predict_grad_closed(X, hyper, alpha, chol, Z, Sigma, method='TA'):
    """Closed forms of ``predict_grad_fd``: dict(dmean (H,Ny,Nx), dvar (H,Ny,Nx), dcov (H,Ny,Ny,Nx), hess (H,Ny,Nx,Nx))."""
    return _closed(X, hyper, alpha, chol, Z, Sigma, method, second=False)


def predict_hess_closed(X, hyper, alpha, chol, Z, Sigma, method='TA'):
    """``predict_grad_closed`` plus d2var (H,Ny,Nx,Nx) and d2cov (H,Ny,Ny,Nx,Nx)."""
    return _closed(X, hyper, alpha, chol, Z, Sigma, method, second=True)


def _closed(X, hyper, alpha, chol, Z, Sigma, method, second):
    X = np.asarray(X, dtype=np.float64)
    Z = np.atleast_2d(np.asarray(Z, dtype=np.float64))
    hyper = np.atleast_2d(np.asarray(hyper, dtype=np.float64))
    H, Nx = Z.shape
    Ny = hyper.shape[0]
    P = [_per_output(X, hyper[a], alpha[a], chol[a], Z) for a in range(Ny)]
    J = np.stack([p['J'] for p in P], 1)                                # (H,Ny,Nx)
    Hm = np.stack([p['Hm'] for p in P], 1)                              # (H,Ny,Nx,Nx)
    dvar = np.stack([p['dvar'] for p in P], 1)
    eye = np.eye(Ny)
    dcov = np.einsum('ab,had->habd', eye, dvar)
    if method == 'TA':
        S = _sigma(Sigma, H, Nx)
        dcov = dcov + np.einsum('hafd,hfg,hbg->habd', Hm, S, J) + np.einsum('haf,hfg,hbgd->habd', J, S, Hm)
    out = dict(dmean=J, dvar=dvar, dcov=dcov, hess=Hm)
    if not second:
        return out
    d2var = np.zeros((H, Ny, Nx, Nx)); T = np.zeros((H, Ny, Nx, Nx, Nx))
    for a, p in enumerate(P):
        ie2 = 1.0 / p['ell'] ** 2
        for h in range(H):
            dks = p['ks'][:, h][:, None] * p['s'][h]                     # (N,Nx)
            W = solve_triangular(chol[a], dks, lower=True)
            pb = np.einsum('i,id,ie->de', p['wb'][h], p['s'][h], p['s'][h])
            d2var[h, a] = -2.0 * (W.T @ W + pb - np.diag((p['sf2'] - p['var'][h]) * ie2))
            t = np.einsum('i,if,id,ie->fde', p['wa'][h], p['s'][h], p['s'][h], p['s'][h])
            Jh = p['J'][h]
            I = np.eye(Nx)
            t -= np.einsum('fd,e,f->fde', I, Jh, ie2) + np.einsum('fe,d,f->fde', I, Jh, ie2) \
                + np.einsum('de,f,d->fde', I, Jh, ie2)
            T[h, a] = t
    d2cov = np.einsum('ab,hade->habde', eye, d2var)
    if method == 'TA':
        S = _sigma(Sigma, H, Nx)
        d2cov = d2cov + np.einsum('hafde,hfg,hbg->habde', T, S, J) + np.einsum('hafd,hfg,hbge->habde', Hm, S, Hm) \
            + np.einsum('hafe,hfg,hbgd->habde', Hm, S, Hm) + np.einsum('haf,hfg,hbgde->habde', J, S, T)
    out.update(d2var=d2var, d2cov=d2cov)
    return out
