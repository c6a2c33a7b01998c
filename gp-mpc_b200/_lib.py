"""ctypes binding of libgpmpc.so (the C ABI in include/gpmpc.h).

There is deliberately NO fallback: if the CUDA library has not been built
(``python -c "import __graft_entry__ as g; g.build()"``) importing the engine
fails loudly, and ``gpmpc_create`` fails when no sm_100 device is present.
"""
from __future__ import annotations

import ctypes as C
import threading
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('GPMPC_LIB', os.path.join(_HERE, 'lib', 'libgpmpc.so'))

OK, ERR_ARG, ERR_CUDA, ERR_STATE, ERR_NCCL, ERR_NOTPD = 0, -1, -2, -3, -4, -5
METHOD_ME, METHOD_TA, METHOD_EM = 0, 1, 2
GET_CHOL, GET_ALPHA, GET_INVK, GET_K, GET_LOGDET, GET_LINV, GET_ALPHA_NLML = range(7)
PROF_KBUILD_FULL, PROF_KBUILD_LOWER, PROF_SYRK, PROF_FACTORIZE, PROF_TRIGEMM, PROF_KS, PROF_PREDICT_TAIL = range(7)

# every symbol include/gpmpc.h declares: (name, restype, argtypes)
_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_H = C.c_void_p
SYMBOLS = [
    ('gpmpc_version', C.c_int, []),
    ('gpmpc_create', C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_H)]),
    ('gpmpc_destroy', C.c_int, [_H]),
    ('gpmpc_last_error', C.c_char_p, [_H]),
    ('gpmpc_set_data', C.c_int, [_H, _dp, _dp]),
    ('gpmpc_set_hyper', C.c_int, [_H, _dp, C.c_int]),
    ('gpmpc_set_y', C.c_int, [_H, C.c_int, _dp]),
    ('gpmpc_build_K', C.c_int, [_H, C.c_int, _dp]),
    ('gpmpc_factorize', C.c_int, [_H, C.c_double, _ip]),
    ('gpmpc_fitc', C.c_int, [_H, C.c_int, _dp, _dp, C.c_double, _ip, _dp]),
    ('gpmpc_fitc_timings', C.c_int, [_H, _dp]),
    ('gpmpc_nlml', C.c_int, [_H, C.c_int, _dp, _dp, _dp]),
    ('gpmpc_predict', C.c_int, [_H, C.c_int, C.c_int, _dp, _dp, C.c_int, _dp, _dp, _dp, _dp]),
    ('gpmpc_predict_grad', C.c_int, [_H, C.c_int, C.c_int, _dp, _dp, C.c_int, _dp, _dp, _dp, _dp, _dp, _dp, _dp]),
    ('gpmpc_predict_hess', C.c_int, [_H, C.c_int, C.c_int, _dp, _dp, C.c_int, _dp, _dp, _dp, _dp, _dp, _dp, _dp, _dp, _dp]),
    ('gpmpc_get_size', C.c_int, [_H, _ip, _ip, _ip]),
    ('gpmpc_append', C.c_int, [_H, _dp, _dp]),
    ('gpmpc_posterior_cov', C.c_int, [_H, C.c_int, _dp, _dp]),
    ('gpmpc_rollout', C.c_int, [_H, C.c_int, C.c_int, _dp, _dp, _dp, _dp, _dp, _dp, _dp]),
    ('gpmpc_predict_device', C.c_int, [_H, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    ('gpmpc_get', C.c_int, [_H, C.c_int, C.c_int, _dp]),
    ('gpmpc_set_option', C.c_int, [_H, C.c_char_p, C.c_double]),
    ('gpmpc_comm_unique_id', C.c_int, [C.c_void_p]),
    ('gpmpc_comm_init', C.c_int, [_H, C.c_void_p, C.c_int, C.c_int]),
    ('gpmpc_peer_export', C.c_int, [_H, C.c_int, C.c_void_p]),
    ('gpmpc_peer_attach', C.c_int, [_H, C.c_void_p]),
    ('gpmpc_stream', C.c_void_p, [_H]),
    ('gpmpc_synchronize', C.c_int, [_H]),
    ('gpmpc_profile', C.c_int, [_H, C.c_int, C.c_int, C.c_int, _dp]),
    ('gpmpc_profile_balance', C.c_int, [_H, C.c_int, _dp]),
    ('gpmpc_profile_leaf', C.c_int, [_H, _dp]),
    ('gpmpc_profile_tail', C.c_int, [_H, C.c_int, _dp]),
]

_ll = C.c_longlong
_llp = C.POINTER(C.c_longlong)
_dpp = C.POINTER(_dp)
# include/gpmpc_casadi.h: the CasADi `external` family (function + its Jacobian)
for _f in ('gp_b200', 'jac_gp_b200'):
    SYMBOLS += [
        (_f + '_n_in', _ll, []), (_f + '_n_out', _ll, []),
        (_f + '_name_in', C.c_char_p, [_ll]), (_f + '_name_out', C.c_char_p, [_ll]),
        (_f + '_sparsity_in', _llp, [_ll]), (_f + '_sparsity_out', _llp, [_ll]),
        (_f + '_work', C.c_int, [_llp, _llp, _llp, _llp]),
        (_f, C.c_int, [_dpp, _dpp, _llp, _dp, C.c_int]),
    ]
SYMBOLS += [('gp_b200_bind', C.c_int, [_H, C.c_int, C.c_int]), ('gp_b200_unbind', None, []),
            ('gp_b200_incref', None, []), ('gp_b200_decref', None, [])]
# the next derivative level of that family: the Jacobian of jac_gp_b200, which CasADi looks up as jac_jac_gp_b200
_f = 'jac_jac_gp_b200'
SYMBOLS_HESS = [
    (_f + '_n_in', _ll, []), (_f + '_n_out', _ll, []),
    (_f + '_name_in', C.c_char_p, [_ll]), (_f + '_name_out', C.c_char_p, [_ll]),
    (_f + '_sparsity_in', _llp, [_ll]), (_f + '_sparsity_out', _llp, [_ll]),
    (_f + '_work', C.c_int, [_llp, _llp, _llp, _llp]),
    (_f, C.c_int, [_dpp, _dpp, _llp, _dp, C.c_int]),
]

_lib = None


class GpmpcError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__('gpmpc error %d: %s' % (code, msg))
        self.code = code


def load():
    """Load libgpmpc.so once; raises ImportError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            'libgpmpc.so not found at %s -- build it with `python -c "import __graft_entry__ as g; '
            'g.build()"` (nvcc, sm_100a).  This engine has no CPU fallback.' % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, res, args in SYMBOLS + SYMBOLS_HESS:
        fn = getattr(lib, name)      # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(_dp)


def _f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        a = a.reshape(shape)
    return a


class Engine:
    """One handle = one GPU.  Thin, typed veneer over the C ABI; all heavy work is CUDA."""

    def __init__(self, N, Nx, Ny, out_begin=0, out_count=None, device=0):
        self.lib = load()
        self.N, self.Nx, self.Ny = int(N), int(Nx), int(Ny)
        self._stage, self._stage_lock = {}, threading.Lock()     # predict(): per-shape host staging arrays + their pointers
        self.out_begin = int(out_begin)
        self.out_count = int(Ny - out_begin if out_count is None else out_count)
        self.device = int(device)
        self.h = _H()
        rc = self.lib.gpmpc_create(self.N, self.Nx, self.Ny, self.out_begin, self.out_count, self.device,
                                   C.byref(self.h))
        if rc != OK:
            msg = self.lib.gpmpc_last_error(None).decode()
            self.h = None
            raise GpmpcError(rc, msg)

    # -- plumbing ---------------------------------------------------------------------
    def _check(self, rc):
        if rc != OK:
            raise GpmpcError(rc, self.lib.gpmpc_last_error(self.h).decode())

    def close(self):
        if getattr(self, 'h', None):
            self.lib.gpmpc_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def local_outputs(self):
        return range(self.out_begin, self.out_begin + self.out_count)

    # -- model ------------------------------------------------------------------------
    def set_data(self, X, Y):
        X = _f64(X, (self.N, self.Nx)); Y = _f64(Y, (self.N, self.Ny))
        self._check(self.lib.gpmpc_set_data(self.h, _ptr(X), _ptr(Y)))

    def set_hyper(self, hyper):
        hyper = _f64(hyper)
        assert hyper.ndim == 2 and hyper.shape[0] == self.Ny and hyper.shape[1] >= self.Nx + 2
        self._check(self.lib.gpmpc_set_hyper(self.h, _ptr(hyper), hyper.shape[1]))

    def set_y(self, a, y):
        y = _f64(y, (self.N,))
        self._check(self.lib.gpmpc_set_y(self.h, int(a), _ptr(y)))

    def build_K(self, a):
        K = np.empty((self.N, self.N))
        self._check(self.lib.gpmpc_build_K(self.h, int(a), _ptr(K)))
        return K

    def factorize(self, jitter=1e-8):
        info = np.zeros(self.out_count, dtype=np.int32)
        rc = self.lib.gpmpc_factorize(self.h, float(jitter), info.ctypes.data_as(_ip))
        if rc == ERR_NOTPD:
            raise np.linalg.LinAlgError(self.lib.gpmpc_last_error(self.h).decode())
        self._check(rc)
        return info

    def fitc(self, X, Y, jitter=1e-6):
        """FITC sparse model (gpmpc_fitc): the handle's own points are the M inducing points, X:(N,Nx), Y:(N,Ny) the
        training set in the GP's input space.  Returns (info, nll) per owned output: info 1 = the B factor needed its
        retry shift, nll = FITC negative log marginal likelihood.  Afterwards every predict method evaluates FITC."""
        X = _f64(X); Y = _f64(Y)
        N = X.shape[0]
        X = X.reshape(N, self.Nx); Y = Y.reshape(N, self.Ny)
        info = np.zeros(self.out_count, dtype=np.int32)
        nll = np.zeros(self.out_count)
        rc = self.lib.gpmpc_fitc(self.h, int(N), _ptr(X), _ptr(Y), float(jitter), info.ctypes.data_as(_ip), _ptr(nll))
        if rc == ERR_NOTPD:
            raise np.linalg.LinAlgError(self.lib.gpmpc_last_error(self.h).decode())
        self._check(rc)
        return info, nll

    def fitc_timings(self):
        """Phase times (ms) of the last fitc build: dict(kuf, v_product, column_pass, syrk, factorisations)."""
        out = np.zeros(5)
        self._check(self.lib.gpmpc_fitc_timings(self.h, _ptr(out)))
        return dict(zip(('kuf', 'v_product', 'column_pass', 'syrk', 'factorisations'), out))

    def nlml(self, a, theta, grad=True):
        theta = _f64(theta, (self.Nx + 2,))
        nll = C.c_double(0.0)
        g = np.empty(self.Nx + 2) if grad else None
        rc = self.lib.gpmpc_nlml(self.h, int(a), _ptr(theta), C.byref(nll), _ptr(g))
        if rc == ERR_NOTPD:
            raise np.linalg.LinAlgError(self.lib.gpmpc_last_error(self.h).decode())
        self._check(rc)
        return (nll.value, g) if grad else nll.value

    def get(self, what, a):
        N = self.N
        shape = {GET_CHOL: (N, N), GET_LINV: (N, N), GET_INVK: (N, N), GET_K: (N, N),
                 GET_ALPHA: (N,), GET_ALPHA_NLML: (N,), GET_LOGDET: (1,)}[what]
        out = np.empty(shape)
        self._check(self.lib.gpmpc_get(self.h, int(what), int(a), _ptr(out)))
        return out

    def set_option(self, name, value):
        self._check(self.lib.gpmpc_set_option(self.h, name.encode(), float(value)))

    # -- predict ----------------------------------------------------------------------
    def predict(self, Z, Sigma=None, method=METHOD_TA, want_cov=True, want_jac=True):
        """Z:(H,Nx) -> mean:(H,Ny), var:(H,Ny), cov:(H,Ny,Ny)|None, jac:(H,Ny,Nx)|None (host arrays).
        The ctypes pointer objects cost 2.5 us each to build (six per call: 13 of the 61 us of a C2-sized call), so the call
        goes through per-shape staging arrays whose pointers are built once; the results are returned as fresh copies."""
        Z = _f64(Z).reshape(-1, self.Nx)
        H = Z.shape[0]
        spp = 0
        if Sigma is not None:
            Sigma = _f64(Sigma)
            if Sigma.ndim == 3:
                assert Sigma.shape == (H, self.Nx, self.Nx)
                spp = 1
            else:
                assert Sigma.shape == (self.Nx, self.Nx)
        key = (H, spp, Sigma is None, bool(want_cov), bool(want_jac))
        with self._stage_lock:
            st = self._stage.get(key)
            if st is None:
                if len(self._stage) >= 16:
                    self._stage.clear()
                arrs = dict(Z=np.empty((H, self.Nx)),
                            S=None if Sigma is None else np.empty(Sigma.shape),
                            mean=np.empty((H, self.Ny)), var=np.empty((H, self.Ny)),
                            cov=np.empty((H, self.Ny, self.Ny)) if want_cov else None,
                            jac=np.empty((H, self.Ny, self.Nx)) if want_jac else None)
                st = self._stage[key] = (arrs, {k: _ptr(v) for k, v in arrs.items()})
            arrs, ptrs = st
            np.copyto(arrs['Z'], Z)
            if Sigma is not None:
                np.copyto(arrs['S'], Sigma)
            self._check(self.lib.gpmpc_predict(self.h, int(method), H, ptrs['Z'], ptrs['S'], spp,
                                               ptrs['mean'], ptrs['var'], ptrs['cov'], ptrs['jac']))
            return (arrs['mean'].copy(), arrs['var'].copy(),
                    arrs['cov'].copy() if want_cov else None, arrs['jac'].copy() if want_jac else None)

    def rollout(self, z0, U, Sigma0, method=METHOD_TA, scale=None):
        """gpmpc_rollout: Nt open-loop steps with the state kept on the device.  z0:(Nx,), U:(Nt,Nu) (GP input units),
        Sigma0:(Nx,Nx), scale:(4,Ny)|None -> means (Nt,Ny), vars (Nt,Ny), cov_last (Ny,Ny) in GP output units."""
        Nu = self.Nx - self.Ny
        z0 = _f64(z0, (self.Nx,)); Sigma0 = _f64(Sigma0, (self.Nx, self.Nx))
        U = _f64(U).reshape(-1, Nu) if Nu > 0 else np.zeros((int(np.shape(U)[0]), 0))
        Nt = U.shape[0]
        if scale is not None:
            scale = _f64(scale, (4, self.Ny))
        means = np.empty((Nt, self.Ny)); var = np.empty((Nt, self.Ny)); cov = np.empty((self.Ny, self.Ny))
        self._check(self.lib.gpmpc_rollout(self.h, int(method), Nt, _ptr(z0), _ptr(U) if Nu > 0 else None, _ptr(Sigma0),
                                           _ptr(scale), _ptr(means), _ptr(var), _ptr(cov)))
        return means, var, cov

    def predict_grad(self, Z, Sigma=None, method=METHOD_TA, want_hess=False):
        """Predict + first derivatives w.r.t. the test inputs (gpmpc_predict_grad).
        Returns dict(mean (H,Ny), var, cov (H,Ny,Ny), jac = dmean_dz (H,Ny,Nx), dvar_dz (H,Ny,Nx),
        dcov_dz (H,Ny,Ny,Nx)[, hess (H,Ny,Nx,Nx)])."""
        Z = _f64(Z).reshape(-1, self.Nx)
        H = Z.shape[0]
        spp = 0
        if Sigma is not None:
            Sigma = _f64(Sigma)
            spp = 1 if Sigma.ndim == 3 else 0
            assert Sigma.shape == ((H, self.Nx, self.Nx) if spp else (self.Nx, self.Nx))
        out = dict(mean=np.empty((H, self.Ny)), var=np.empty((H, self.Ny)), cov=np.empty((H, self.Ny, self.Ny)),
                   jac=np.empty((H, self.Ny, self.Nx)), dvar_dz=np.empty((H, self.Ny, self.Nx)),
                   dcov_dz=np.empty((H, self.Ny, self.Ny, self.Nx)))
        if want_hess:
            out['hess'] = np.empty((H, self.Ny, self.Nx, self.Nx))
        self._check(self.lib.gpmpc_predict_grad(self.h, int(method), H, _ptr(Z), _ptr(Sigma), spp, _ptr(out['mean']),
                                                _ptr(out['var']), _ptr(out['cov']), _ptr(out['jac']), _ptr(out['dvar_dz']),
                                                _ptr(out['dcov_dz']), _ptr(out.get('hess'))))
        return out

    def predict_hess(self, Z, Sigma=None, method=METHOD_TA):
        """Predict + first and second derivatives w.r.t. the test inputs (gpmpc_predict_hess).
        Returns the predict_grad dict with hess (H,Ny,Nx,Nx) plus d2var_dz2 (H,Ny,Nx,Nx) and d2cov_dz2 (H,Ny,Ny,Nx,Nx)."""
        Z = _f64(Z).reshape(-1, self.Nx)
        H = Z.shape[0]
        spp = 0
        if Sigma is not None:
            Sigma = _f64(Sigma)
            spp = 1 if Sigma.ndim == 3 else 0
            assert Sigma.shape == ((H, self.Nx, self.Nx) if spp else (self.Nx, self.Nx))
        Ny, Nx = self.Ny, self.Nx
        out = dict(mean=np.empty((H, Ny)), var=np.empty((H, Ny)), cov=np.empty((H, Ny, Ny)), jac=np.empty((H, Ny, Nx)),
                   dvar_dz=np.empty((H, Ny, Nx)), dcov_dz=np.empty((H, Ny, Ny, Nx)), hess=np.empty((H, Ny, Nx, Nx)),
                   d2var_dz2=np.empty((H, Ny, Nx, Nx)), d2cov_dz2=np.empty((H, Ny, Ny, Nx, Nx)))
        self._check(self.lib.gpmpc_predict_hess(self.h, int(method), H, _ptr(Z), _ptr(Sigma), spp,
                                                *[_ptr(out[k]) for k in ('mean', 'var', 'cov', 'jac', 'dvar_dz', 'dcov_dz',
                                                                         'hess', 'd2var_dz2', 'd2cov_dz2')]))
        return out

    def append(self, x_new, y_new):
        """Rank-1 append of one training point; returns False when the padded capacity is full
        or positive definiteness is lost (caller refits), True on success."""
        x = _f64(x_new, (self.Nx,)); y = _f64(y_new, (self.Ny,))
        rc = self.lib.gpmpc_append(self.h, _ptr(x), _ptr(y))
        if rc in (ERR_STATE, ERR_NOTPD):
            return False
        self._check(rc)
        self.N += 1
        return True

    def posterior_cov(self, Z):
        """(out_count, H, H): sf2 - V^T V per owned output (GP.covar)."""
        Z = _f64(Z).reshape(-1, self.Nx)
        out = np.empty((self.out_count, Z.shape[0], Z.shape[0]))
        self._check(self.lib.gpmpc_posterior_cov(self.h, Z.shape[0], _ptr(Z), _ptr(out)))
        return out

    def predict_device(self, method, H, dZ, dSigma, spp, d_mean, d_var, d_cov, d_jac, sync=False):
        """Raw device-pointer variant (ints); enqueues on the handle's stream."""
        self._check(self.lib.gpmpc_predict_device(self.h, int(method), int(H), dZ, dSigma, int(spp),
                                                  d_mean, d_var, d_cov, d_jac, 1 if sync else 0))

    # -- multi-GPU --------------------------------------------------------------------
    @staticmethod
    def comm_unique_id():
        lib = load()
        buf = C.create_string_buffer(128)
        rc = lib.gpmpc_comm_unique_id(buf)
        if rc != OK:
            raise GpmpcError(rc, lib.gpmpc_last_error(None).decode())
        return bytes(buf.raw)

    def comm_init(self, uid, rank, world):
        buf = C.create_string_buffer(bytes(uid), 128)
        self._check(self.lib.gpmpc_comm_init(self.h, buf, int(rank), int(world)))

    def peer_export(self, Hcap=256):
        buf = C.create_string_buffer(64)
        self._check(self.lib.gpmpc_peer_export(self.h, int(Hcap), buf))
        return bytes(buf.raw)

    def peer_attach(self, handles):
        blob = b''.join(bytes(x) for x in handles)
        buf = C.create_string_buffer(blob, len(blob))
        self._check(self.lib.gpmpc_peer_attach(self.h, buf))

    def stream(self):
        return self.lib.gpmpc_stream(self.h)

    def synchronize(self):
        self._check(self.lib.gpmpc_synchronize(self.h))

    def profile_leaf(self):
        out = np.zeros(15)
        self._check(self.lib.gpmpc_profile_leaf(self.h, _ptr(out)))
        return out

    def profile_tail(self, H):
        out = np.zeros(8)
        self._check(self.lib.gpmpc_profile_tail(self.h, int(H), _ptr(out)))
        return dict(zip(('output_done', 'records', 'step_counter', 'staged', 'jsigma', 'written', 'kernel_span', 'tail_cta_span'), out))

    def profile_balance(self, H):
        out = np.zeros(4)
        self._check(self.lib.gpmpc_profile_balance(self.h, int(H), _ptr(out)))
        return dict(zip(('min_us', 'max_us', 'mean_us', 'span_us'), out))

    def profile(self, what, n=0, reps=5):
        ms = C.c_double(0.0)
        self._check(self.lib.gpmpc_profile(self.h, int(what), int(n), int(reps), C.byref(ms)))
        return ms.value
