"""Small end-to-end pass over every kernel of the engine for compute-sanitizer
(memcheck / racecheck / synccheck / initcheck):  K build, leaf + DMMA GEMMs (cp.async and TMA
tensor-map feeds), alpha, NLML + gradient, the persistent stream-K predict kernel with tile
fix-ups (several grid sizes, lower and upper mode), predict_grad, predict_hess (W passes, pair sums), EM, rank-1 append, GP.covar, the FITC build.
    compute-sanitizer --tool racecheck python tools/sanitize_run.py"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import gp_mpc_b200
from gp_mpc_b200 import _lib as L
from oracle import gp_oracle as orc
from tests._util import relinf

N, Nx, Ny, H = int(os.environ.get('SAN_N', 700)), 5, 2, 21
p = orc.synthetic_problem(N, Nx, Ny, config_id=3, H=H)
eng = gp_mpc_b200.Engine(N, Nx, Ny, device=0)
eng.set_data(p['X'], p['Y']); eng.set_hyper(p['hyper'])
eng.set_option('small_tiles', 4)          # push the top-level products onto the TMA tensor-map GEMM as well
eng.factorize()
post = orc.postfit(p['X'], p['Y'], p['hyper'], lapack_general_solve=False)
print('chol', relinf(eng.get(L.GET_CHOL, 0), post['chol'][0]), flush=True)
mo, vo = orc.gp_mean_var(p['X'], p['hyper'], post['alpha'], post['chol'], p['Z'])
for ctas in (0, 1, 3, 37):
    eng.set_option('predict_ctas', ctas)
    mean, var, cov, jac = eng.predict(p['Z'], p['Sigma'], L.METHOD_TA)
    print('predict ctas=%d' % ctas, relinf(mean, mo), relinf(var, vo), flush=True)
eng.set_option('predict_ctas', 5)
g = eng.predict_grad(p['Z'], p['Sigma'], L.METHOD_TA, want_hess=True)
fd = orc.predict_grad_fd(p['X'], p['hyper'], post['alpha'], post['chol'], p['Z'], p['Sigma'], 'TA')
print('grad', relinf(g['dvar_dz'], fd['dvar']), relinf(g['dcov_dz'], fd['dcov']), flush=True)
from tests._hess_oracle import predict_hess_closed
for meth, name, S in ((L.METHOD_TA, 'TA', p['Sigma']), (L.METHOD_ME, 'ME', None)):
    g2 = eng.predict_hess(p['Z'], S, meth)
    c2 = predict_hess_closed(p['X'], p['hyper'], post['alpha'], post['chol'], p['Z'], p['Sigma'], name)
    print('hess', name, relinf(g2['d2var_dz2'], c2['d2var']), relinf(g2['d2cov_dz2'], c2['d2cov']), flush=True)
eng.set_option('refine', 1)
mean, var, _, _ = eng.predict(p['Z'], p['Sigma'], L.METHOD_TA)
print('refine', relinf(var, vo), flush=True)
eng.set_option('refine', 0)
m_em, v_em, c_em, _ = eng.predict(p['Z'][:2], 1e-4 * np.eye(Nx), L.METHOD_EM, want_jac=False)
print('em var>0', bool((v_em > 0).all()), flush=True)
pc = eng.posterior_cov(p['Z'][:5])
nll, gr = eng.nlml(0, p['hyper'][0] * 0.9, grad=True)
print('nlml', nll, orc.calc_NLL(p['hyper'][0] * 0.9, p['X'], p['Y'][:, 0], False), flush=True)
eng.factorize()
ok = eng.append(p['X'][0] + 0.3, p['Y'][0])
print('append', ok, flush=True)
eng.close()
# FITC build: three panels of 256 points (the last one partial), M = 150 (not a multiple of 128), then predict on it
from tests import _fitc_oracle as fo
U = p['X'][fo.seeded_subset(N, 150)]
sp = gp_mpc_b200.Engine(150, Nx, Ny, device=0)
sp.set_option('fitc_panel', 256)
sp.set_data(U, np.zeros((150, Ny))); sp.set_hyper(p['hyper'])
info, nll = sp.fitc(p['X'], p['Y'])
mw, vw, nw = fo.predict('direct', U, p['X'], p['Y'], p['hyper'], p['Z'])
mean, var, _, _ = sp.predict(p['Z'], p['Sigma'], L.METHOD_TA)
print('fitc', relinf(mean, mw), relinf(var, vw), relinf(nll, nw), flush=True)
sp.close()
print('done', flush=True)
