"""DeviceGP — the george.GP object of the reference, backed by one gpk handle.

The reference keeps a ``george.GP`` in ``GaussianProcess.gp`` (gaussian_process.py:106) and
drives it with compute / log_likelihood / predict.  This class offers the same verbs; all
arithmetic happens in libgpk.so on the GPU:

    compute(X, yerr)          K build + blocked Cholesky + forward solve + log-det  (gpk_fit)
    log_likelihood(y)         the value gpk_fit already produced (needs the same y)
    predict / predict_cov     fused K* build, L^-1 K*^T contraction, moments       (gpk_predict*)
    score                     ... plus the acquisition closed form and arg-max     (gpk_acq)

george adds yerr^2 + exp(white_noise) to the diagonal, white_noise = log(1.25e-12) by default
(SURVEY.md Appendix A); the same value is computed here on the host and handed to gpk_fit.
"""
import numpy as np

from . import _lib

TINY = 1.25e-12


class DeviceGP(object):
    def __init__(self, kernel, mean=0.0, device=0, white_noise=None):
        self.kernel = kernel
        self.mean = float(mean)
        self.device = int(device)
        self.white_noise = np.log(TINY) if white_noise is None else white_noise
        self._handle = None
        self._x = None
        self._y = None
        self._data_dirty = True
        self._yerr = None
        self._bounds = None
        self._out = (False, 0.0, 1.0)
        self._cfg_dirty = True
        self.computed = False
        self.log_determinant = None
        self._ll = None
        # incremental refit (gpk_fit_append, SURVEY.md 8f-4): what the handle's factorisation was computed for
        self.incremental = True
        self._fit_x = None
        self._fit_sig = None
        self.n_appends = 0

    # ---- handle lifetime: handles do not survive pickling / deepcopy -----------------
    def __getstate__(self):
        st = self.__dict__.copy()
        st["_handle"] = None
        st["_data_dirty"] = True
        st["_cfg_dirty"] = True
        was_computed = st["computed"]
        st["computed"] = False
        st["_recompute"] = bool(was_computed)
        st["_fit_x"] = None
        st["_fit_sig"] = None
        return st

    def __setstate__(self, st):
        self.__dict__.update(st)

    @property
    def handle(self):
        if self._handle is None:
            self._handle = _lib.Handle(self.device)
            self._data_dirty = True
            self._cfg_dirty = True
            self._fit_x = None
        return self._handle

    def _restore(self):
        """After deepcopy/unpickle: rebuild the device state lazily from host state."""
        if getattr(self, "_recompute", False) and not self.computed and self._x is not None:
            self._recompute = False
            self.compute(self._x, self._yerr)

    # ---- configuration -------------------------------------------------------------------
    def set_data(self, X, y):
        self._x = _lib.f64(X)
        self._y = _lib.f64(y)
        self._data_dirty = True
        self.computed = False

    def set_input_bounds(self, lower, upper):
        self._bounds = None if lower is None else (_lib.f64(lower).ravel(), _lib.f64(upper).ravel())
        self._cfg_dirty = True

    def set_output_transform(self, enabled, y_mean=0.0, y_std=1.0):
        self._out = (bool(enabled), float(y_mean), float(y_std))
        self._cfg_dirty = True

    def _push_cfg(self):
        h = self.handle
        if self._cfg_dirty:
            if self._bounds is None:
                h.set_input_bounds(None, None)
            else:
                h.set_input_bounds(*self._bounds)
            h.set_output_transform(*self._out)
            self._cfg_dirty = False

    # ---- george verbs ----------------------------------------------------------------------
    def compute(self, x=None, yerr=0.0, **kwargs):
        """K = k(X,X) + (yerr^2 + TINY) I ; factorise.  Raises numpy.linalg.LinAlgError when
        K is not positive definite, like george's BasicSolver (scipy.linalg.cholesky)."""
        if x is not None and (self._x is None or x is not self._x):
            x = _lib.f64(x)
            if self._x is None or x.shape != self._x.shape or not np.array_equal(x, self._x):
                if self._y is None or len(self._y) != len(x):
                    raise ValueError("DeviceGP.compute: call set_data(X, y) first (y enters the factorisation)")
                self._x = x
                self._data_dirty = True
        if self._x is None or self._y is None:
            raise ValueError("DeviceGP.compute: no training data")
        h = self.handle
        f = self.kernel.flatten()
        self._yerr = float(yerr)
        yerr_tot = np.sqrt(np.float64(self._yerr) ** 2 + np.exp(self.white_noise))
        diag_add = float(yerr_tot ** 2)
        sig = (int(f["family"]), float(f["log_amp"]), tuple(int(a) for a in f["axis"]),
               tuple(int(g) for g in f["group"]), tuple(float(v) for v in np.asarray(f["log_metric"]).ravel()), diag_add)
        self.computed = False
        # Rows appended to an already factorised training set with the same kernel and noise (BaseModel.update /
        # train(do_optimize=False) inside the solver loop): only the last block row of the factor changes.
        fx = self._fit_x
        if (self.incremental and self._data_dirty and fx is not None and self._fit_sig == sig
                and self._x.ndim == 2 and self._x.shape[1] == fx.shape[1] and len(self._x) > len(fx)
                and np.array_equal(self._x[:len(fx)], fx)):
            self._push_cfg()
            self._fit_x = None                       # a failed attempt leaves the handle to be refitted
            res = h.fit_append(self._x, self._y, diag_add, self.mean)
            if res is not None:
                self.log_determinant, self._ll = res
                self._data_dirty = False
                self._fit_x = self._x.copy()
                self.n_appends += 1
                self.computed = True
                return
        self._fit_x = None
        if self._data_dirty:
            h.set_data(self._x, self._y)
            self._data_dirty = False
        self._push_cfg()
        h.set_kernel(f["family"], f["log_amp"], f["axis"], f["group"], f["log_metric"])
        self.log_determinant, self._ll = h.fit(diag_add, self.mean)
        self._fit_x = self._x.copy()
        self._fit_sig = sig
        self.computed = True

    # the same factorisation in two halves (gpk_fit_begin / gpk_fit_end): several DeviceGPs — the n_hypers sub-models of
    # a GaussianProcessMCMC, gaussian_process_mcmc.py:149-164 — enqueue their fits first and collect afterwards, so the
    # latency-bound Cholesky chains overlap on the GPU instead of running one after the other
    def compute_begin(self, x=None, yerr=0.0):
        if x is not None and (self._x is None or x is not self._x):
            x = _lib.f64(x)
            if self._x is None or x.shape != self._x.shape or not np.array_equal(x, self._x):
                if self._y is None or len(self._y) != len(x):
                    raise ValueError("DeviceGP.compute_begin: call set_data(X, y) first")
                self._x = x
                self._data_dirty = True
        if self._x is None or self._y is None:
            raise ValueError("DeviceGP.compute_begin: no training data")
        h = self.handle
        f = self.kernel.flatten()
        self._yerr = float(yerr)
        yerr_tot = np.sqrt(np.float64(self._yerr) ** 2 + np.exp(self.white_noise))
        diag_add = float(yerr_tot ** 2)
        self._pending_sig = (int(f["family"]), float(f["log_amp"]), tuple(int(a) for a in f["axis"]),
                             tuple(int(g) for g in f["group"]),
                             tuple(float(v) for v in np.asarray(f["log_metric"]).ravel()), diag_add)
        self.computed = False
        self._fit_x = None
        if self._data_dirty:
            h.set_data(self._x, self._y)
            self._data_dirty = False
        self._push_cfg()
        h.set_kernel(f["family"], f["log_amp"], f["axis"], f["group"], f["log_metric"])
        h.fit_begin(diag_add, self.mean)

    def compute_end(self):
        """Collects compute_begin(); raises numpy.linalg.LinAlgError like compute()."""
        self.log_determinant, self._ll = self.handle.fit_end()
        self._fit_x = self._x.copy()
        self._fit_sig = self._pending_sig
        self.computed = True

    def log_likelihood(self, y=None, quiet=False):
        if y is not None and self._y is not None and y is not self._y and not np.array_equal(y, self._y):
            # different targets: refit with them (the forward solve is part of the factorisation)
            self.set_data(self._x, y)
            try:
                self.compute(None, self._yerr)
            except np.linalg.LinAlgError:
                if quiet:
                    return -np.inf
                raise
        if not self.computed:
            self._restore()
        if not self.computed:
            raise RuntimeError("You need to compute the model first")
        return self._ll if np.isfinite(self._ll) else -np.inf

    lnlikelihood = log_likelihood

    def grad_neg_log_likelihood(self, noise_var):
        """d(-loglik)/d theta for theta = [kernel parameter vector ..., log sigma^2] of the current
        factorisation (gpk_nll_grad), mapped from the device's per-term layout back onto the george
        parameter vector (isotropic kernels sum their terms; every ConstantKernel factor receives
        the amplitude derivative)."""
        if not self.computed:
            self._restore()
        if not self.computed:
            raise RuntimeError("You need to compute the model first")
        f = self.kernel.flatten()
        g = self.handle.nll_grad(noise_var, len(f["axis"]))
        out = np.empty(len(f["slots"]) + 1)
        for p, (kind, terms) in enumerate(f["slots"]):
            out[p] = g[0] if kind == "amp" else sum(g[1 + t] for t in terms)
        out[-1] = g[-1]
        return out

    def predict(self, y, t, return_cov=False, return_var=True):
        self._restore()
        if return_cov:
            return self.predict_cov(t)
        return self.predict_moments(t)

    def predict_moments(self, Xs):
        self._restore()
        self._push_cfg()
        return self.handle.predict(Xs)

    def predict_cov(self, Xs):
        self._restore()
        self._push_cfg()
        return self.handle.predict_cov(Xs)

    def posterior_cov(self, Xs):
        """(mu, cov) with the raw posterior covariance K** - K* K^-1 K*^T: no clip, negative off-diagonal entries
        kept.  george's GP.predict returns exactly this; the reference clips afterwards in its own predict()
        (gaussian_process.py:290-294) and samples from the raw matrix (:324)."""
        self._restore()
        self._push_cfg()
        return self.handle.posterior_cov(Xs)

    def predict_grad(self, Xs, kind=0, eta=0.0, par=0.0):
        self._restore()
        self._push_cfg()
        return self.handle.predict_grad(Xs, kind, eta, par)

    def score(self, Xs, kind, eta=0.0, par=0.0, want_values=True, want_moments=False):
        self._restore()
        self._push_cfg()
        return self.handle.acq(Xs, kind, eta, par, want_values, want_moments)

    def es_update(self, zb, lmb, np_grid, sn2):
        """Entropy-search state of this model on the device (gpk_es_update) -> logP."""
        self._restore()
        self._push_cfg()
        return self.handle.es_update(zb, lmb, np_grid, sn2)

    def es_compute(self, Xs, lower=None, upper=None, want_values=True):
        self._restore()
        self._push_cfg()
        return self.handle.es_compute(Xs, lower, upper, want_values)

    def sample_conditional(self, y, t, size=1):
        mu, cov = self.posterior_cov(t)
        if size > 1:
            return np.random.multivariate_normal(mu, cov, size=size)
        return np.random.multivariate_normal(mu, cov)
