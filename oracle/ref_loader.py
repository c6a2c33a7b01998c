"""Import the UNMODIFIED reference package from /root/reference with its absent
third-party imports stubbed  --  TEST INFRASTRUCTURE ONLY (build container only).

Every reference module imports casadi at top level (gp_class.py:12,
gp_functions.py:12, optimize.py:14, mpc_class.py:13-14, model_class.py:14) and
casadi / pyDOE / matplotlib are not installed, so the package cannot be
imported as-is.  With empty stub modules in ``sys.modules`` the package imports
and its numpy-only functions run VERBATIM:

    optimize.calc_cov_matrix   (optimize.py:303-319)
    optimize.calc_NLL_numpy    (optimize.py:322-356)
    GP.covSEard                (gp_class.py:314-350)
    GP.covar                   (gp_class.py:353-381)
    optimize.standardize / normalize (optimize.py:561-587)

Nothing here is copied from the reference; the reference is executed where it
lies.  This module is only used by the golden-data generators
``oracle/make_golden.py`` and ``oracle/make_golden_live.py``, whose outputs are
committed under ``tests/golden/``; the test-suite never needs the reference.
"""
from __future__ import annotations

import os
import sys
import types

REFERENCE_ROOT = os.environ.get('GPMPC_REFERENCE_ROOT', '/root/reference')


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, 'gp_mpc'))


class _Anything(types.ModuleType):
    """Module whose every attribute is a harmless placeholder."""

    def __getattr__(self, name):
        if name.startswith('__'):
            raise AttributeError(name)
        return _Placeholder(name)


class _Placeholder:
    def __init__(self, name='x'):
        self._name = name

    def __call__(self, *a, **k):
        raise RuntimeError('stubbed third-party symbol %r was called: this reference '
                           'function needs CasADi/pyDOE/matplotlib' % self._name)

    def __getattr__(self, name):
        if name.startswith('__'):
            raise AttributeError(name)
        return _Placeholder(self._name + '.' + name)


def load_reference():
    """Return the reference ``gp_mpc`` package (imported under the private name
    ``_gpmpc_reference`` so it can never shadow the product)."""
    if '_gpmpc_reference' in sys.modules:
        return sys.modules['_gpmpc_reference']
    if not reference_available():
        raise ImportError('reference checkout not found at ' + REFERENCE_ROOT)
    stubs = ['casadi', 'casadi.tools', 'pyDOE', 'matplotlib', 'matplotlib.pyplot',
             'matplotlib.font_manager']
    saved = {n: sys.modules.get(n) for n in stubs}
    for n in stubs:
        if saved[n] is None:
            try:
                __import__(n)
            except Exception:
                sys.modules[n] = _Anything(n)
    import importlib.util
    import warnings
    pkg_dir = os.path.join(REFERENCE_ROOT, 'gp_mpc')
    spec = importlib.util.spec_from_file_location(
        '_gpmpc_reference', os.path.join(pkg_dir, '__init__.py'),
        submodule_search_locations=[pkg_dir])
    mod = importlib.util.module_from_spec(spec)
    sys.modules['_gpmpc_reference'] = mod
    dont = sys.dont_write_bytecode
    sys.dont_write_bytecode = True        # /root/reference is read-only
    try:
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')   # `is 'literal'` SyntaxWarnings (q6)
            spec.loader.exec_module(mod)
    finally:
        sys.dont_write_bytecode = dont
    return mod


def reference_gp_shell(model):
    """A reference ``GP`` instance WITHOUT running its constructor (which needs
    CasADi), with exactly the private attributes ``GP.covar`` reads
    (gp_class.py:373-379)."""
    import numpy as np
    ref = load_reference()
    GP = ref.GP
    g = GP.__new__(GP)
    hyper = np.atleast_2d(np.asarray(model['hyper'], dtype=np.float64))
    Nx = np.asarray(model['X']).shape[1]
    g._GP__Ny = hyper.shape[0]
    g._GP__X = np.asarray(model['X'], dtype=np.float64)
    g._GP__hyper_length_scales = hyper[:, :Nx]
    g._GP__hyper_signal_variance = hyper[:, Nx] ** 2
    g._GP__chol = np.asarray(model['chol'], dtype=np.float64)
    return g
