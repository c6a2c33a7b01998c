"""FITC sparse GP restated on the CPU in float64 -- the checker for gpmpc_fitc (TEST INFRASTRUCTURE ONLY).

Inducing points U (M), training set (X, y) (N), Kuu = k(U,U) + jitter sf2 I, Qff = Kfu Kuu^-1 Kuf,
Lambda = diag(Kff - Qff) + sn2 I (the diagonal clamped at 0 before sn2 is added, as the engine does).
Three independent forms of the same model:
  * direct:    an exact GP with prior covariance Qff + Lambda: N x N solves (N <= ~2000)
               mean = Qzf C^-1 y,  var = sf2 - Qzf C^-1 Qfz,  nll = 1/2 y^T C^-1 y + 1/2 log det C
  * Woodbury:  Sigma = (Kuu + Kuf Lambda^-1 Kfu)^-1, alpha_s = Sigma Kuf Lambda^-1 y, K~^-1 = Kuu^-1 - Sigma;
               only M x M solves, the training set in chunks (any N)
  * build:     the engine's algorithm (Luu, V = Luu^-1 Kuf, A = I + V Lambda^-1 V^T, B = I - A^-1, reverse Cholesky
               S^T S = B, R = S Luu^-1, alpha_s = Luu^-T LA^-T LA^-1 b)
The build returns (U, alpha_s, Ltilde = Luu S^-1): Ltilde^-1 = R, so the dense oracle functions (gp_mean_var, ta_cov,
predict_hess_closed, gp_exact_moment with invK = Ltilde^-T Ltilde^-1) evaluate the FITC model with X -> U,
alpha -> alpha_s and chol -> Ltilde.  All nll values follow the reference convention (no N/2 log 2 pi).
"""
import numpy as np
from scipy.linalg import cho_solve, cholesky, solve_triangular

from oracle import gp_oracle as orc


def _k(A, B, hyp_a):
    Nx = A.shape[1]
    return orc.covSEard(A, B, hyp_a[:Nx], hyp_a[Nx] ** 2)


def _luu(U, hyp_a, jitter):
    Nx = U.shape[1]
    return cholesky(_k(U, U, hyp_a) + jitter * hyp_a[Nx] ** 2 * np.eye(U.shape[0]), lower=True)


def _lam(V, hyp_a, Nx):
    q = np.sum(V * V, axis=0)
    return np.maximum(hyp_a[Nx] ** 2 - q, 0.0) + hyp_a[Nx + 1] ** 2


def _chunks(N, chunk):
    for c0 in range(0, N, chunk):
        yield slice(c0, min(N, c0 + chunk))


def direct(U, X, y, hyp_a, Z, jitter=1e-6):
    """mean (H,), var (H,), nll of one output from the exact GP with prior Qff + Lambda."""
    Nx = X.shape[1]
    sf2 = hyp_a[Nx] ** 2
    Luu = _luu(U, hyp_a, jitter)
    V = solve_triangular(Luu, _k(U, X, hyp_a), lower=True)             # (M,N)
    C = V.T @ V + np.diag(_lam(V, hyp_a, Nx))
    Lc = cholesky(C, lower=True)
    Qzf = solve_triangular(Luu, _k(U, Z, hyp_a), lower=True).T @ V       # (H,N)
    a = cho_solve((Lc, True), y)
    W = solve_triangular(Lc, Qzf.T, lower=True)
    nll = 0.5 * y @ a + np.sum(np.log(np.diag(Lc)))
    return Qzf @ a, sf2 - np.sum(W * W, axis=0), nll


def woodbury(U, X, y, hyp_a, Z, jitter=1e-6, chunk=8192):
    """mean (H,), var (H,), nll of one output with M x M solves only."""
    Nx, M = X.shape[1], U.shape[0]
    sf2 = hyp_a[Nx] ** 2
    Kuu = _k(U, U, hyp_a) + jitter * sf2 * np.eye(M)
    Luu = cholesky(Kuu, lower=True)
    P = np.zeros((M, M)); r = np.zeros(M); yly = 0.0; logl = 0.0
    for sl in _chunks(X.shape[0], chunk):
        Kuf = _k(U, X[sl], hyp_a)
        lam = _lam(solve_triangular(Luu, Kuf, lower=True), hyp_a, Nx)
        P += (Kuf / lam) @ Kuf.T
        r += Kuf @ (y[sl] / lam)
        yly += np.sum(y[sl] ** 2 / lam)
        logl += np.sum(np.log(lam))
    Ls = cholesky(Kuu + P, lower=True)
    alpha = cho_solve((Ls, True), r)
    I = np.eye(M)
    Kt = cho_solve((Luu, True), I) - cho_solve((Ls, True), I)
    ks = _k(U, Z, hyp_a)
    nll = 0.5 * (yly - r @ alpha) + 0.5 * logl + np.sum(np.log(np.diag(Ls))) - np.sum(np.log(np.diag(Luu)))
    return ks.T @ alpha, sf2 - np.einsum('ih,ij,jh->h', ks, Kt, ks), nll


def build(U, X, y, hyp_a, jitter=1e-6, chunk=8192, shift=1e-10):
    """The engine's algorithm restated: dict(alpha, R, Ltilde, nll, shifted) of one output."""
    Nx, M = X.shape[1], U.shape[0]
    Luu = _luu(U, hyp_a, jitter)
    I = np.eye(M)
    Luu_i = solve_triangular(Luu, I, lower=True)
    Phi = np.zeros((M, M)); b = np.zeros(M); yly = 0.0; logl = 0.0
    for sl in _chunks(X.shape[0], chunk):
        V = Luu_i @ _k(U, X[sl], hyp_a)
        lam = _lam(V, hyp_a, Nx)
        Vs = V / np.sqrt(lam)
        Phi += Vs @ Vs.T
        b += Vs @ (y[sl] / np.sqrt(lam))
        yly += np.sum(y[sl] ** 2 / lam)
        logl += np.sum(np.log(lam))
    LA = cholesky(I + Phi, lower=True)
    LA_i = solve_triangular(LA, I, lower=True)
    B = I - LA_i.T @ LA_i
    shifted = 0
    try:
        G = cholesky(B[::-1, ::-1], lower=True)
    except np.linalg.LinAlgError:
        shifted = 1
        G = cholesky(B[::-1, ::-1] + shift * I, lower=True)
    S = G.T[::-1, ::-1]                                                  # J G^T J: lower, S^T S = B
    t = LA_i @ b
    alpha = Luu_i.T @ (LA_i.T @ t)
    nll = 0.5 * (yly - t @ t) + 0.5 * (logl + 2.0 * np.sum(np.log(np.diag(LA))))
    return dict(alpha=alpha, R=S @ Luu_i, Ltilde=Luu @ solve_triangular(S, I, lower=True), nll=nll, shifted=shifted)


def model(U, X, Y, hyper, jitter=1e-6, chunk=8192):
    """All outputs: dict(U, alpha (Ny,M), chol = Ltilde (Ny,M,M), R (Ny,M,M), nll (Ny,), invK (Ny,M,M), Yeff (M,Ny)).
    invK = K~^-1 and Yeff = K~ alpha_s are what gp_exact_moment takes in place of K^-1 and the targets."""
    hyper = np.atleast_2d(hyper)
    outs = [build(U, X, Y[:, a], hyper[a], jitter, chunk) for a in range(hyper.shape[0])]
    chol = np.stack([o['Ltilde'] for o in outs])
    R = np.stack([o['R'] for o in outs])
    alpha = np.stack([o['alpha'] for o in outs])
    invK = np.einsum('aki,akj->aij', R, R)
    Yeff = np.stack([chol[a] @ (chol[a].T @ alpha[a]) for a in range(len(outs))], 1)
    return dict(U=U, alpha=alpha, chol=chol, R=R, nll=np.array([o['nll'] for o in outs]), invK=invK, Yeff=Yeff,
                shifted=np.array([o['shifted'] for o in outs]))


def predict(form, U, X, Y, hyper, Z, jitter=1e-6, **kw):
    """mean (H,Ny), var (H,Ny), nll (Ny,) from the direct or Woodbury form."""
    hyper = np.atleast_2d(hyper)
    f = direct if form == 'direct' else woodbury
    res = [f(U, X, Y[:, a], hyper[a], Z, jitter, **kw) for a in range(hyper.shape[0])]
    return (np.stack([r[0] for r in res], 1), np.stack([r[1] for r in res], 1), np.array([r[2] for r in res]))


def jacobian(U, alpha, hyper, Z):
    """d mean / d z (H,Ny,Nx): the dense closed form with X -> U, alpha -> alpha_s."""
    return orc.gp_mean_jac(U, hyper, alpha, Z)


def seeded_subset(N, M):
    """The inducing subset GP(..., inducing=M) / GP.sparse(M) picks."""
    return np.sort(np.random.default_rng(0).choice(N, M, replace=False))
