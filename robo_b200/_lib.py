"""ctypes binding of include/gpk.h — the stub a RoBO maintainer would add (INTEGRATION.md).

There is deliberately NO CPU fallback: if libgpk.so cannot be loaded, or no CUDA device is
present, every compute call raises.  Status codes map to the exceptions the reference's
callers already handle (SURVEY.md section 8b "Error conventions"):
    GPK_NOT_PD     -> numpy.linalg.LinAlgError   (gaussian_process.py:120,156)
    GPK_BAD_ARG    -> ValueError
    GPK_CUDA_ERROR -> RuntimeError
"""
import ctypes as C
import os

import numpy as np

from . import _build

GPK_OK, GPK_NOT_PD, GPK_BAD_ARG, GPK_CUDA_ERROR, GPK_NOT_FITTED, GPK_NOT_APPLICABLE = range(6)
MATERN52, EXPSQUARED, MATERN32 = 0, 1, 2
ACQ_NONE, ACQ_EI, ACQ_LOG_EI, ACQ_PI, ACQ_LCB = range(5)
ACQ_KIND = {"ei": ACQ_EI, "log_ei": ACQ_LOG_EI, "pi": ACQ_PI, "lcb": ACQ_LCB, "none": ACQ_NONE}

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_lp = C.POINTER(C.c_long)
_vp = C.c_void_p

_SIGNATURES = {
    "gpk_create": [C.POINTER(_vp), C.c_int],
    "gpk_destroy": [_vp],
    "gpk_set_option": [_vp, C.c_char_p, C.c_long],
    "gpk_set_stream": [_vp, _vp],
    "gpk_synchronize": [_vp],
    "gpk_set_data": [_vp, _dp, _dp, C.c_int, C.c_int],
    "gpk_set_input_bounds": [_vp, _dp, _dp, C.c_int],
    "gpk_set_output_transform": [_vp, C.c_int, C.c_double, C.c_double],
    "gpk_set_kernel": [_vp, C.c_int, C.c_double, C.c_int, _ip, _ip, _dp],
    "gpk_fit": [_vp, C.c_double, C.c_double, _dp, _dp],
    "gpk_fit_begin": [_vp, C.c_double, C.c_double],
    "gpk_fit_end": [_vp, _dp, _dp],
    "gpk_fit_append": [_vp, _dp, _dp, C.c_int, C.c_int, C.c_double, C.c_double, _dp, _dp],
    "gpk_predict": [_vp, _dp, C.c_long, _dp, _dp],
    "gpk_predict_cov": [_vp, _dp, C.c_long, _dp, _dp],
    "gpk_posterior_cov": [_vp, _dp, C.c_long, _dp, _dp],
    "gpk_acq": [_vp, _dp, C.c_long, C.c_int, C.c_double, C.c_double, _dp, _dp, _dp, _dp, _lp, _lp],
    "gpk_acq_dev": [_vp, _vp, C.c_long, C.c_int, C.c_double, C.c_double, _vp, _vp, _vp, _vp],
    "gpk_predict_grad": [_vp, _dp, C.c_long, C.c_int, C.c_double, C.c_double, _dp, _dp, _dp, _dp, _dp, _dp],
    "gpk_maximize_random": [_vp, C.c_ulonglong, C.c_long, C.c_long, C.c_long, _dp, _dp, _dp, C.c_double, C.c_int,
                            C.c_double, C.c_double, _dp, _dp, _lp],
    "gpk_generate_candidates": [_vp, C.c_ulonglong, C.c_long, C.c_long, C.c_long, C.c_int, _dp, _dp, _dp, C.c_double, _dp],
    "gpk_acq_moments": [_vp, _dp, _dp, C.c_long, C.c_int, C.c_double, C.c_double, _dp, _lp],
    "gpk_kernel_matrix": [_vp, _dp, C.c_long, _dp, C.c_long, C.c_int, _dp],
    "gpk_reduce_models": [_vp, _dp, _dp, C.c_int, C.c_long, C.c_int, _dp, _dp],
    "gpk_acq_multi": [C.POINTER(_vp), C.c_int, _dp, C.c_long, C.c_int, C.c_int, _dp, C.c_double, _dp, _dp, _lp, _dp, _lp],
    "gpk_comm_unique_id": [_vp],
    "gpk_comm_init": [_vp, C.c_int, C.c_int, _vp],
    "gpk_comm_destroy": [_vp],
    "gpk_comm_info": [_vp, _ip, _ip, _ip],
    "gpk_shard_bounds": [C.c_long, C.c_int, C.c_int, _lp, _lp],
    "gpk_comm_argmax_pair": [_vp, C.c_double, C.c_long, _dp, _lp],
    "gpk_acq_argmax_sharded": [_vp, _dp, C.c_long, C.c_int, C.c_double, C.c_double, _dp, _lp],
    "gpk_acq_argmax_sharded_dev": [_vp, _vp, C.c_long, C.c_long, C.c_int, C.c_double, C.c_double, _vp],
    "gpk_maximize_random_sharded": [_vp, C.c_ulonglong, C.c_long, C.c_long, _dp, _dp, _dp, C.c_double, C.c_int,
                                    C.c_double, C.c_double, _dp, _dp, _lp],
    "gpk_nll_grad": [_vp, C.c_double, _dp],
    "gpk_measure_fp64_peaks": [_vp, _dp, _dp],
    "gpk_measure_int8_peak": [_vp, _dp],
    "gpk_measure_int8_peak_sustained": [_vp, C.c_double, C.c_int, _dp],
    "gpk_es_joint_min": [_vp, _dp, _dp, C.c_int, _dp, _dp, _dp, _dp, _ip],
    "gpk_es_update": [_vp, _dp, C.c_int, _dp, C.c_int, C.c_double, _dp],
    "gpk_es_compute": [_vp, _dp, C.c_long, _dp, _dp, _dp, _dp, _lp],
    "gpk_es_get_state": [_vp, _dp, _dp, _dp, _dp, _ip],
    "gpk_get_factor": [_vp, _dp],
    "gpk_get_linv": [_vp, _dp],
    "gpk_get_z": [_vp, _dp],
    "gpk_get_timings": [_vp, _dp],
    "gpk_get_diag_profile": [_vp, C.POINTER(C.c_longlong)],
    "gpk_get_oz_profile": [_vp, C.POINTER(C.c_longlong), C.c_int, C.POINTER(C.c_int)],
}

_lib = None


def library_path():
    return _build.LIB


def load(build_if_missing=True):
    """dlopen libgpk.so (building it first if the sources are newer). Raises if impossible."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if build_if_missing and os.environ.get("GPK_NO_BUILD") != "1":
        try:
            _build.build()
        except Exception as e:
            if not os.path.exists(path):
                raise
            # sources are newer than the binary and cannot be rebuilt (no nvcc on this box): the binary that travelled
            # with the tree is used, loudly; the ABI check below still refuses a library that lacks a declared symbol
            import warnings
            warnings.warn("libgpk.so is older than its sources and could not be rebuilt (%s); using the existing binary"
                          % str(e).splitlines()[0])
    if not os.path.exists(path):
        raise RuntimeError("libgpk.so is missing (%s) and could not be built; there is no CPU fallback" % path)
    lib = C.CDLL(path)
    for name, argtypes in _SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if a declared symbol is not exported
        fn.argtypes = argtypes
        fn.restype = C.c_int
    lib.gpk_last_error.argtypes = [_vp]
    lib.gpk_last_error.restype = C.c_char_p
    lib.gpk_version.argtypes = []
    lib.gpk_version.restype = C.c_char_p
    _lib = lib
    return lib


def exported_symbols():
    return sorted(list(_SIGNATURES) + ["gpk_last_error", "gpk_version"])


def _as_dp(a):
    return a.ctypes.data_as(_dp)


def f64(a):
    """C-contiguous float64 view/copy (the ABI takes plain double*)."""
    return np.ascontiguousarray(a, dtype=np.float64)


class Handle(object):
    """Owns one gpk_handle (one fitted GP on one GPU)."""

    def __init__(self, device=0):
        self.lib = load()
        self.device = int(device)
        h = _vp()
        rc = self.lib.gpk_create(C.byref(h), self.device)
        if rc != GPK_OK:
            raise RuntimeError("gpk_create failed on device %d (status %d): no usable CUDA device; "
                               "robo_b200 has no CPU fallback" % (self.device, rc))
        self._h = h
        # test/diagnostic overrides: GPK_LOADER=0|1 (cp.async | TMA staging), GPK_CHUNK=<multiple of 128>
        if os.environ.get("GPK_LOADER"):
            self.set_option("loader", int(os.environ["GPK_LOADER"]))
        if os.environ.get("GPK_DIAG"):
            self.set_option("diag", int(os.environ["GPK_DIAG"]))
        if os.environ.get("GPK_CHUNK"):
            self.set_option("chunk", int(os.environ["GPK_CHUNK"]))
        # implementation switches (all default-on variants have a cross-check twin): GPK_COV=1|2, GPK_PERSIST=0|1,
        # GPK_CHAINSPLIT=0|1, GPK_OZAKI=0|1
        for env, key in (("GPK_COV", "cov"), ("GPK_PERSIST", "persist"), ("GPK_CHAINSPLIT", "chainsplit"),
                         ("GPK_OZAKI", "ozaki"), ("GPK_GRAPH", "graph"), ("GPK_DEPTH2", "depth2"), ("GPK_OZFUSED", "ozfused"), ("GPK_OZTILE", "oztile"), ("GPK_OZPAIR", "ozpair"), ("GPK_OZPERSIST", "ozpersist"), ("GPK_OZPDL", "ozpdl"), ("GPK_COVCTAS", "covctas")):
            if os.environ.get(env):
                self.set_option(key, int(os.environ[env]))

    # -- plumbing -----------------------------------------------------------------
    def close(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            try:
                self.lib.gpk_destroy(h)
            except Exception:
                pass

    def __del__(self):
        self.close()

    def _check(self, rc):
        if rc == GPK_OK:
            return
        msg = self.lib.gpk_last_error(self._h)
        msg = msg.decode("utf-8", "replace") if msg else ""
        if rc == GPK_NOT_PD:
            raise np.linalg.LinAlgError(msg or "Matrix is not positive definite")
        if rc == GPK_BAD_ARG:
            raise ValueError(msg)
        if rc == GPK_NOT_FITTED:
            raise RuntimeError(msg or "model not fitted")
        raise RuntimeError("gpk: " + msg)

    def set_option(self, key, value):
        self._check(self.lib.gpk_set_option(self._h, key.encode(), int(value)))

    def set_stream(self, cuda_stream_ptr):
        self._check(self.lib.gpk_set_stream(self._h, _vp(cuda_stream_ptr or 0)))

    def synchronize(self):
        self._check(self.lib.gpk_synchronize(self._h))

    # -- model state ----------------------------------------------------------------
    def set_data(self, X, y):
        X, y = f64(X), f64(y)
        n, d = X.shape
        self._check(self.lib.gpk_set_data(self._h, _as_dp(X), _as_dp(y), n, d))

    def set_input_bounds(self, lower, upper):
        if lower is None or upper is None:
            self._check(self.lib.gpk_set_input_bounds(self._h, None, None, 0))
            return
        lo, up = f64(lower).ravel(), f64(upper).ravel()
        self._check(self.lib.gpk_set_input_bounds(self._h, _as_dp(lo), _as_dp(up), lo.size))

    def set_output_transform(self, enabled, y_mean=0.0, y_std=1.0):
        self._check(self.lib.gpk_set_output_transform(self._h, int(bool(enabled)), float(y_mean), float(y_std)))

    def set_kernel(self, family, log_amp, axis, group, log_metric):
        axis = np.ascontiguousarray(axis, dtype=np.int32)
        group = np.ascontiguousarray(group, dtype=np.int32)
        lm = f64(log_metric)
        self._check(self.lib.gpk_set_kernel(self._h, int(family), float(log_amp), axis.size,
                                            axis.ctypes.data_as(_ip), group.ctypes.data_as(_ip), _as_dp(lm)))

    def fit(self, diag_add, mean):
        logdet, ll = C.c_double(), C.c_double()
        self._check(self.lib.gpk_fit(self._h, float(diag_add), float(mean), C.byref(logdet), C.byref(ll)))
        return logdet.value, ll.value

    def fit_append(self, X, y, diag_add, mean):
        """Incremental refit after rows were appended (gpk_fit_append).  Returns (logdet, loglik), or None when the
        library reports that the shortcut does not apply (the model is untouched: run set_data + fit)."""
        X, y = f64(X), f64(y)
        n, d = X.shape
        logdet, ll = C.c_double(), C.c_double()
        rc = self.lib.gpk_fit_append(self._h, _as_dp(X), _as_dp(y), n, d, float(diag_add), float(mean),
                                     C.byref(logdet), C.byref(ll))
        if rc == GPK_NOT_APPLICABLE:
            return None
        self._check(rc)
        return logdet.value, ll.value

    def fit_begin(self, diag_add, mean):
        self._check(self.lib.gpk_fit_begin(self._h, float(diag_add), float(mean)))

    def fit_end(self):
        logdet, ll = C.c_double(), C.c_double()
        self._check(self.lib.gpk_fit_end(self._h, C.byref(logdet), C.byref(ll)))
        return logdet.value, ll.value

    # -- scoring ----------------------------------------------------------------------
    def predict(self, Xs):
        Xs = f64(Xs)
        m = Xs.shape[0]
        mu, var = np.empty(m), np.empty(m)
        self._check(self.lib.gpk_predict(self._h, _as_dp(Xs), m, _as_dp(mu), _as_dp(var)))
        return mu, var

    def predict_cov(self, Xs):
        Xs = f64(Xs)
        m = Xs.shape[0]
        mu, cov = np.empty(m), np.empty((m, m))
        self._check(self.lib.gpk_predict_cov(self._h, _as_dp(Xs), m, _as_dp(mu), _as_dp(cov)))
        return mu, cov

    def posterior_cov(self, Xs):
        """(mu, cov) with the raw, unclipped posterior covariance (sampling; gpk_posterior_cov)."""
        Xs = f64(Xs)
        m = Xs.shape[0]
        mu, cov = np.empty(m), np.empty((m, m))
        self._check(self.lib.gpk_posterior_cov(self._h, _as_dp(Xs), m, _as_dp(mu), _as_dp(cov)))
        return mu, cov

    def acq(self, Xs, kind, eta=0.0, par=0.0, want_values=True, want_moments=False):
        """-> dict(values, mu, var, best_val, best_idx, n_negative)"""
        Xs = f64(Xs)
        m = Xs.shape[0]
        out = np.empty(m) if want_values else None
        mu = np.empty(m) if want_moments else None
        var = np.empty(m) if want_moments else None
        bv, bi, nn = C.c_double(), C.c_long(-1), C.c_long(0)
        self._check(self.lib.gpk_acq(self._h, _as_dp(Xs), m, int(kind), float(eta), float(par),
                                     _as_dp(out) if want_values else None,
                                     _as_dp(mu) if want_moments else None,
                                     _as_dp(var) if want_moments else None,
                                     C.byref(bv), C.byref(bi), C.byref(nn)))
        return dict(values=out, mu=mu, var=var, best_val=bv.value, best_idx=bi.value, n_negative=nn.value)

    def acq_dev(self, d_Xs_ptr, m, kind, eta, par, d_out_ptr=0, d_mu_ptr=0, d_var_ptr=0, d_best_ptr=0):
        """Device-pointer variant (asynchronous on the handle's stream)."""
        self._check(self.lib.gpk_acq_dev(self._h, _vp(d_Xs_ptr), int(m), int(kind), float(eta), float(par),
                                         _vp(d_out_ptr or 0), _vp(d_mu_ptr or 0), _vp(d_var_ptr or 0),
                                         _vp(d_best_ptr or 0)))

    def predict_grad(self, Xs, kind=ACQ_NONE, eta=0.0, par=0.0):
        """-> dict(mu, var, dmu (m,d), dvar (m,d)[, f, df]) — moments and their input gradients."""
        Xs = f64(Xs)
        m, d = Xs.shape
        mu, var, dmu, dvar = np.empty(m), np.empty(m), np.empty((m, d)), np.empty((m, d))
        f = np.empty(m) if kind != ACQ_NONE else None
        df = np.empty((m, d)) if kind != ACQ_NONE else None
        self._check(self.lib.gpk_predict_grad(self._h, _as_dp(Xs), m, int(kind), float(eta), float(par), _as_dp(mu),
                                              _as_dp(var), _as_dp(dmu), _as_dp(dvar),
                                              _as_dp(f) if f is not None else None,
                                              _as_dp(df) if df is not None else None))
        return dict(mu=mu, var=var, dmu=dmu, dvar=dvar, f=f, df=df)

    def maximize_random(self, seed, first, count, n_uniform, lower, upper, incumbent, scale, kind, eta=0.0, par=0.0):
        """-> (best_x (d,), best_val, best_global_idx) over device-generated candidates [first, first+count)."""
        lo, up, inc = f64(lower).ravel(), f64(upper).ravel(), f64(incumbent).ravel()
        bx = np.empty(lo.size)
        bv, bi = C.c_double(), C.c_long(-1)
        self._check(self.lib.gpk_maximize_random(self._h, int(seed), int(first), int(count), int(n_uniform), _as_dp(lo),
                                                 _as_dp(up), _as_dp(inc), float(scale), int(kind), float(eta), float(par),
                                                 _as_dp(bx), C.byref(bv), C.byref(bi)))
        return bx, bv.value, bi.value

    def generate_candidates(self, seed, first, count, n_uniform, lower, upper, incumbent, scale):
        lo, up, inc = f64(lower).ravel(), f64(upper).ravel(), f64(incumbent).ravel()
        out = np.empty((count, lo.size))
        self._check(self.lib.gpk_generate_candidates(self._h, int(seed), int(first), int(count), int(n_uniform), lo.size,
                                                     _as_dp(lo), _as_dp(up), _as_dp(inc), float(scale), _as_dp(out)))
        return out

    # -- multi-GPU (gpk_comm_*) -----------------------------------------------------------
    def comm_init(self, rank, world, unique_id=None):
        """Collective over all ranks.  unique_id: the 128 bytes of comm_unique_id() made on rank 0."""
        buf = C.create_string_buffer(bytes(unique_id), 128) if unique_id is not None else None
        self._check(self.lib.gpk_comm_init(self._h, int(rank), int(world), C.cast(buf, _vp) if buf is not None else None))

    def comm_destroy(self):
        self._check(self.lib.gpk_comm_destroy(self._h))

    def comm_info(self):
        r, w, v = C.c_int(), C.c_int(), C.c_int()
        self._check(self.lib.gpk_comm_info(self._h, C.byref(r), C.byref(w), C.byref(v)))
        return dict(rank=r.value, world=w.value, nccl_version=v.value)

    def comm_argmax_pair(self, val, idx):
        """Exchange only: this rank's (value, global index) -> the merged winner on every rank."""
        bv, bi = C.c_double(), C.c_long(-1)
        self._check(self.lib.gpk_comm_argmax_pair(self._h, float(val), int(idx), C.byref(bv), C.byref(bi)))
        return bv.value, bi.value

    def acq_argmax_sharded(self, Xs_all, kind, eta=0.0, par=0.0):
        """Xs_all: the full batch, identical on every rank -> (best value, best GLOBAL index) on every rank."""
        Xs_all = f64(Xs_all)
        bv, bi = C.c_double(), C.c_long(-1)
        self._check(self.lib.gpk_acq_argmax_sharded(self._h, _as_dp(Xs_all), Xs_all.shape[0], int(kind), float(eta),
                                                    float(par), C.byref(bv), C.byref(bi)))
        return bv.value, bi.value

    def acq_argmax_sharded_dev(self, d_Xs_ptr, m_shard, first_global, kind, eta, par, d_best_ptr=0):
        self._check(self.lib.gpk_acq_argmax_sharded_dev(self._h, _vp(d_Xs_ptr or 0), int(m_shard), int(first_global),
                                                        int(kind), float(eta), float(par), _vp(d_best_ptr or 0)))

    def maximize_random_sharded(self, seed, n_total, n_uniform, lower, upper, incumbent, scale, kind, eta=0.0, par=0.0):
        lo, up, inc = f64(lower).ravel(), f64(upper).ravel(), f64(incumbent).ravel()
        bx = np.empty(lo.size)
        bv, bi = C.c_double(), C.c_long(-1)
        self._check(self.lib.gpk_maximize_random_sharded(self._h, int(seed), int(n_total), int(n_uniform), _as_dp(lo),
                                                         _as_dp(up), _as_dp(inc), float(scale), int(kind), float(eta),
                                                         float(par), _as_dp(bx), C.byref(bv), C.byref(bi)))
        return bx, bv.value, bi.value

    def acq_moments(self, mu, var, kind, eta=0.0, par=0.0):
        mu, var = f64(mu).ravel(), f64(var).ravel()
        out = np.empty(mu.size)
        nn = C.c_long(0)
        self._check(self.lib.gpk_acq_moments(self._h, _as_dp(mu), _as_dp(var), mu.size, int(kind), float(eta),
                                             float(par), _as_dp(out), C.byref(nn)))
        return out, nn.value

    def nll_grad(self, noise_var, n_terms):
        """d(-loglik)/d[log_amp, log_metric_t..., log sigma^2] of the current fit."""
        g = np.empty(n_terms + 2)
        self._check(self.lib.gpk_nll_grad(self._h, float(noise_var), _as_dp(g)))
        return g

    def reduce_models(self, A, B=None):
        """mean over models (B None) or GP-MCMC mixture moments (mean, var) (B = per-model variances)."""
        A = f64(A)
        n, m = A.shape
        out1 = np.empty(m)
        if B is None:
            self._check(self.lib.gpk_reduce_models(self._h, _as_dp(A), None, n, m, 0, _as_dp(out1), None))
            return out1
        B = f64(B)
        out2 = np.empty(m)
        self._check(self.lib.gpk_reduce_models(self._h, _as_dp(A), _as_dp(B), n, m, 1, _as_dp(out1), _as_dp(out2)))
        return out1, out2

    def kernel_matrix(self, X1, X2):
        X1, X2 = f64(X1), f64(X2)
        out = np.empty((X1.shape[0], X2.shape[0]))
        self._check(self.lib.gpk_kernel_matrix(self._h, _as_dp(X1), X1.shape[0], _as_dp(X2), X2.shape[0],
                                               X1.shape[1], _as_dp(out)))
        return out

    def measure_fp64_peaks(self):
        """-> (DMMA tensor-pipe TFLOP/s, DFMA vector-pipe TFLOP/s) measured on this GPU."""
        a, b = C.c_double(), C.c_double()
        self._check(self.lib.gpk_measure_fp64_peaks(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def measure_int8_peak(self):
        """-> int8 tensor-pipe issue-rate peak in TOP/s (tcgen05 kind::i8) measured on this GPU."""
        a = C.c_double()
        self._check(self.lib.gpk_measure_int8_peak(self._h, C.byref(a)))
        return a.value

    def measure_int8_peak_sustained(self, seconds=0.4, random_operands=True):
        """-> the same issue rate held for `seconds` (second half timed): what the power limit leaves of the burst figure.
        random_operands: pseudo-random operand bytes (switching activity of real digit slices) instead of a constant pattern."""
        a = C.c_double()
        self._check(self.lib.gpk_measure_int8_peak_sustained(self._h, float(seconds), 1 if random_operands else 0, C.byref(a)))
        return a.value

    # -- entropy search (gpk_es_*) ----------------------------------------------------------
    def _es_out(self, nb):
        return dict(logP=np.empty(nb), dlogPdMu=np.empty((nb, nb)), dlogPdSigma=np.empty((nb, nb * (nb + 1) // 2)),
                    dlogPdMudMu=np.empty((nb, nb, nb)), sweeps=np.empty(nb, dtype=np.int32))

    def es_joint_min(self, mu, V):
        """epmgp.joint_min(mu, V, with_derivatives=True) on the device -> dict(logP, dlogPdMu, dlogPdSigma,
        dlogPdMudMu, sweeps)."""
        mu, V = f64(mu).ravel(), f64(V)
        nb = mu.size
        r = self._es_out(nb)
        self._check(self.lib.gpk_es_joint_min(self._h, _as_dp(mu), _as_dp(V), nb, _as_dp(r["logP"]), _as_dp(r["dlogPdMu"]),
                                              _as_dp(r["dlogPdSigma"]), _as_dp(r["dlogPdMudMu"]),
                                              r["sweeps"].ctypes.data_as(_ip)))
        return r

    def es_update(self, zb, lmb, np_grid, sn2):
        """Entropy-search state for representer points zb (raw inputs) -> logP (nb,)."""
        zb, lmb = f64(zb), f64(lmb).ravel()
        logP = np.empty(lmb.size)
        self._check(self.lib.gpk_es_update(self._h, _as_dp(zb), lmb.size, _as_dp(lmb), int(np_grid), float(sn2),
                                           _as_dp(logP)))
        return logP

    def es_compute(self, Xs, lower=None, upper=None, want_values=True):
        """-> dict(values, best_val, best_idx) of the information gain at raw candidates Xs."""
        Xs = f64(Xs)
        m = Xs.shape[0]
        out = np.empty(m) if want_values else None
        lo = None if lower is None else f64(lower).ravel()
        up = None if upper is None else f64(upper).ravel()
        bv, bi = C.c_double(), C.c_long(-1)
        self._check(self.lib.gpk_es_compute(self._h, _as_dp(Xs), m, _as_dp(lo) if lo is not None else None,
                                            _as_dp(up) if up is not None else None,
                                            _as_dp(out) if want_values else None, C.byref(bv), C.byref(bi)))
        return dict(values=out, best_val=bv.value, best_idx=bi.value)

    def es_get_state(self, nb):
        r = self._es_out(nb)
        self._check(self.lib.gpk_es_get_state(self._h, _as_dp(r["logP"]), _as_dp(r["dlogPdMu"]), _as_dp(r["dlogPdSigma"]),
                                              _as_dp(r["dlogPdMudMu"]), r["sweeps"].ctypes.data_as(_ip)))
        return r

    # -- introspection ----------------------------------------------------------------
    def get_factor(self, n):
        L = np.empty((n, n))
        self._check(self.lib.gpk_get_factor(self._h, _as_dp(L)))
        return L

    def get_linv(self, n):
        L = np.empty((n, n))
        self._check(self.lib.gpk_get_linv(self._h, _as_dp(L)))
        return L

    def get_z(self, n):
        z = np.empty(n)
        self._check(self.lib.gpk_get_z(self._h, _as_dp(z)))
        return z

    def diag_profile(self):
        t = np.zeros(64, dtype=np.int64)
        self._check(self.lib.gpk_get_diag_profile(self._h, t.ctypes.data_as(C.POINTER(C.c_longlong))))
        return t

    def oz_profile(self, max_ctas=16384):
        """(n_ctas, 8) clock64() sums of the last persistent int8 contraction (option "ozprof")."""
        buf = (C.c_longlong * (8 * max_ctas))()
        n = C.c_int(0)
        self._check(self.lib.gpk_get_oz_profile(self._h, buf, int(max_ctas), C.byref(n)))
        return np.frombuffer(buf, dtype=np.int64, count=8 * n.value).reshape(n.value, 8).copy()

    def timings(self):
        t = np.zeros(16)
        self._check(self.lib.gpk_get_timings(self._h, _as_dp(t)))
        keys = ["fit_ms", "kbuild_ms", "potrf_ms", "linv_ms", "score_ms", "kstar_ms", "vargemm_ms", "finish_ms",
                "launches_vargemm", "launches_total", "launches_ozaki", "ozaki_max_row_exponent", "persist",
                "ozaki_slice_pairs", "ozaki_kernel_variant"]
        return dict(zip(keys, t.tolist()))


def comm_unique_id():
    """128-byte NCCL id (rank 0 makes it and ships it to the other ranks by any means: file, pipe, MPI, a
    torch.distributed store ...)."""
    lib = load()
    buf = C.create_string_buffer(128)
    if lib.gpk_comm_unique_id(C.cast(buf, _vp)) != GPK_OK:
        raise RuntimeError("gpk_comm_unique_id failed: NCCL (libnccl.so.2) is not available")
    return buf.raw


def shard_bounds(m, rank, world):
    lib = load()
    lo, hi = C.c_long(), C.c_long()
    if lib.gpk_shard_bounds(int(m), int(rank), int(world), C.byref(lo), C.byref(hi)) != GPK_OK:
        raise ValueError("shard_bounds: bad arguments")
    return lo.value, hi.value


def acq_multi(handles, Xs, mode, kind=ACQ_NONE, eta=None, par=0.0, want_argmax=False):
    """gpk_acq_multi over ``handles`` (all fitted, same device).  mode 0 -> dict(values, n_negative, best_val,
    best_idx); mode 1 -> dict(mean, var)."""
    h0 = handles[0]
    Xs = f64(Xs)
    m = Xs.shape[0]
    arr = (_vp * len(handles))(*[h._h for h in handles])
    out1 = np.empty(m)
    out2 = np.empty(m) if mode == 1 else None
    etas = f64(np.zeros(len(handles)) if eta is None else np.broadcast_to(np.asarray(eta, dtype=np.float64), (len(handles),)))
    nn, bv, bi = C.c_long(0), C.c_double(), C.c_long(-1)
    h0._check(h0.lib.gpk_acq_multi(arr, len(handles), _as_dp(Xs), m, int(mode), int(kind), _as_dp(etas), float(par),
                                   _as_dp(out1), _as_dp(out2) if out2 is not None else None, C.byref(nn),
                                   C.byref(bv) if want_argmax else None, C.byref(bi) if want_argmax else None))
    if mode == 1:
        return dict(mean=out1, var=out2)
    return dict(values=out1, n_negative=nn.value, best_val=bv.value, best_idx=bi.value)


_moments_handle = {}


def moments_handle(device=0):
    """Shared handle for gpk_acq_moments (acquisition on non-GPU models)."""
    if device not in _moments_handle:
        _moments_handle[device] = Handle(device)
    return _moments_handle[device]
