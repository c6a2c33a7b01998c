"""Generator of tests/golden/ref_live_{tank,car}.npz: what the reference's own numpy functions
return at the inputs of tests/test_oracle_golden.py::test_matches_live_reference, so that the
test runs without a reference checkout.  Needs the reference (oracle/ref_loader.py):

    GPMPC_REFERENCE_ROOT=<reference checkout> python oracle/make_golden_live.py

What is written, per fixture (calls executed verbatim in the reference package):
  Zt         the test's seeded test points (rng 5, 7 points near the data)
  nll        optimize.calc_NLL_numpy(hyper[a], X, Y[:, a]) per output
  K_rows     rows K_idx of optimize.calc_cov_matrix(X, ell_a, sf2_a) per output: 16 seeded rows
             of the N x N matrix keep the file small (the car fixture's three full K are ~1 MB)
  K_rowsum   the row sums of that matrix per output: every row is covered
  covar      GP.covar(Zt)
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_loader                # noqa: E402
from tests._util import load_fixture         # noqa: E402

N_ROWS = 16


def main():
    ref = ref_loader.load_reference()
    for name in ('tank', 'car'):
        m = load_fixture(name)
        N, Nx = m['X'].shape
        Ny = m['hyper'].shape[0]
        rng = np.random.default_rng(5)          # the test's points
        Zt = m['X'][rng.integers(0, N, 7)] + 0.2 * rng.standard_normal((7, Nx)) * m['X'].std(0)
        idx = np.sort(np.random.default_rng(17).choice(N, N_ROWS, replace=False))
        nll = np.zeros(Ny); K_rows = np.zeros((Ny, N_ROWS, N)); K_rowsum = np.zeros((Ny, N))
        for a in range(Ny):
            ell = m['hyper'][a, :Nx]; sf2 = m['hyper'][a, Nx] ** 2
            K = ref.optimize.calc_cov_matrix(m['X'].copy(), ell, sf2)
            K_rows[a] = K[idx]; K_rowsum[a] = K.sum(1)
            nll[a] = float(ref.optimize.calc_NLL_numpy(m['hyper'][a].copy(), m['X'].copy(), m['Y'][:, a].copy()))
        covar = ref_loader.reference_gp_shell(m).covar(Zt.copy())
        path = os.path.join(ROOT, 'tests', 'golden', 'ref_live_%s.npz' % name)
        np.savez_compressed(path, Zt=Zt, nll=nll, K_idx=idx, K_rows=K_rows, K_rowsum=K_rowsum, covar=covar)
        print(path, os.path.getsize(path))


if __name__ == '__main__':
    main()
