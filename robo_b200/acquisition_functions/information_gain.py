"""InformationGain (robo/acquisition_functions/information_gain.py): entropy search of Hennig & Schuler (JMLR 2012).

Same constructor, attributes and update / compute as the reference class.  Where the arithmetic runs:

  reference (CPU, per candidate)                      here (GPU, libgpk.so, gpk_es_*)
  --------------------------------------------------  ---------------------------------------------------------
  epmgp.joint_min: EP in Python per representer pt    gpk_es_ep_kernel, one CTA per representer point
  predict(x) + predict_variance(zb, x) per candidate  the scoring pass's variance + S = k(zb, X*) - B^T K*^T (DMMA)
  dlogPdSigma . vech, trace term, stochastic term     F . vech(s s^T) on DMMA, vech generated in shared memory
  Np x Nb log-sum-exp and entropy change              one warp per candidate, one exp per (i, p)

The representer points are sampled like the reference (50 steps of an affine-invariant ensemble sampler over the
sampling acquisition, EI in the facades); each half-ensemble is one fused acquisition call.  Sampling parity with the
reference is statistical (robo_b200.util.ensemble_sampler).  ``derivative=True`` raises NotImplementedError: the
reference's finite-difference loop flips the gradient's sign inside the loop, so there is no behaviour to match.
"""
import itertools
import logging

import numpy as np
import scipy.stats

from robo_b200.acquisition_functions.base_acquisition import BaseAcquisitionFunction
from robo_b200.acquisition_functions.log_ei import LogEI
from robo_b200.util.ensemble_sampler import EnsembleSampler

logger = logging.getLogger(__name__)

_STATE_IDS = itertools.count(1)


class InformationGain(BaseAcquisitionFunction):

    def __init__(self, model, lower, upper, Nb=50, Np=400, sampling_acquisition=None,
                 sampling_acquisition_kw={"par": 0.0}, rng=None, **kwargs):
        self.Nb = Nb
        super(InformationGain, self).__init__(model)
        self.lower = lower
        self.upper = upper
        self.D = self.lower.shape[0]
        self.sn2 = None
        if sampling_acquisition is None:
            sampling_acquisition = LogEI
        self.sampling_acquisition = sampling_acquisition(model, **sampling_acquisition_kw)
        self.Np = Np
        if rng is None:
            self.rng = np.random.RandomState(np.random.randint(0, 10000))
        else:
            self.rng = rng
        self.zb = self.lmb = self.logP = self.dlogPdMu = self.dlogPdSigma = self.dlogPdMudMu = self.W = None
        self._state_id = None

    # ---- representer points (information_gain.py:127-151) ---------------------------------------------------
    def sampling_acquisition_wrapper(self, x):
        if np.any(x < self.lower) or np.any(x > self.upper):
            return -np.inf
        return self.sampling_acquisition(np.array([x]))[0]

    def _sampling_lower_upper(self):
        return self.lower, self.upper

    def _project(self, X):
        return X

    def sampling_acquisition_batch(self, X):
        """The wrapper above for a half-ensemble of proposals: rows outside the bounds get -inf, the others are scored
        in one call of the sampling acquisition."""
        X = np.atleast_2d(np.asarray(X, dtype=np.float64))
        lower, upper = self._sampling_lower_upper()
        inside = np.all((X >= lower) & (X <= upper), axis=1)
        out = np.full(X.shape[0], -np.inf)
        if inside.any():
            out[inside] = np.asarray(self.sampling_acquisition(self._project(X[inside])), dtype=np.float64).ravel()
        return out

    def _restarts(self, lower, upper):
        return lower + (upper - lower) * self.rng.uniform(size=(self.Nb, lower.shape[0]))

    def sample_representer_points(self):
        self.sampling_acquisition.update(self.model)
        lower, upper = self._sampling_lower_upper()
        for i in range(5):
            restarts = self._restarts(lower, upper)
            sampler = EnsembleSampler(self.Nb, lower.shape[0], self.sampling_acquisition_wrapper,
                                      batch_lnpostfn=self.sampling_acquisition_batch)
            # zb are the representer points and lmb their sampling-acquisition values
            self.zb, self.lmb, _ = sampler.run_mcmc(restarts, 50, rstate0=self.rng)
            if not np.any(np.isinf(self.lmb)):
                break
            logger.info("Infinity")
        if len(self.zb.shape) == 1:
            self.zb = self.zb[:, None]
        if len(self.lmb.shape) == 1:
            self.lmb = self.lmb[:, None]

    # ---- update / compute ------------------------------------------------------------------------------------
    def update(self, model):
        """information_gain.py:153-167: representer points, then EP and the per-update device state."""
        self.model = model
        self.sn2 = self.model.get_noise()
        self.sample_representer_points()
        self.W = scipy.stats.norm.ppf(np.linspace(1. / (self.Np + 1), 1 - 1. / (self.Np + 1), self.Np))[np.newaxis, :]
        self._state_id = None
        self.logP = self.dlogPdMu = self.dlogPdSigma = self.dlogPdMudMu = None
        if not np.all(np.isfinite(self.lmb)):
            return                       # compute() raises ValueError, like the reference (:207-211)
        self._send_state()
        st = self._gp().handle.es_get_state(self.Nb)
        self.logP = st["logP"].reshape(-1, 1)
        self.dlogPdMu, self.dlogPdSigma, self.dlogPdMudMu = st["dlogPdMu"], st["dlogPdSigma"], st["dlogPdMudMu"]

    def _gp(self):
        gp = getattr(self.model, "gp", None)
        if gp is None or not hasattr(gp, "es_update") or not hasattr(self.model, "device_inputs"):
            raise NotImplementedError("InformationGain runs on the device: it needs a robo_b200 GaussianProcess model")
        return gp

    def _send_state(self):
        gp = self._gp()
        zb = self.model.device_inputs(np.asarray(self.zb, dtype=np.float64))
        gp.es_update(zb, np.asarray(self.lmb, dtype=np.float64).ravel(), self.Np, float(self.sn2))
        self._state_id = next(_STATE_IDS)
        gp.handle.es_owner = self._state_id

    def _scores(self, X, want_values=True):
        if self.lmb is None or not np.all(np.isfinite(self.lmb)):
            raise ValueError("lmb should not be infinite.")
        gp = self._gp()
        if self._state_id is None or getattr(gp.handle, "es_owner", None) != self._state_id:
            self._send_state()           # another acquisition object used this model's handle in between
        X = np.atleast_2d(np.asarray(X, dtype=np.float64))
        Xd = self.model.device_inputs(X)
        if Xd is X:
            return gp.es_compute(X, self.lower, self.upper, want_values)
        # inputs transformed on the host (FabolasGP): the bounds rule applies to the raw candidates
        r = gp.es_compute(Xd, None, None, True)
        outside = np.any((X < self.lower) | (X > self.upper), axis=1)
        r["values"][outside] = np.spacing(1)
        r["best_idx"] = int(np.argmax(r["values"]))
        return r

    def compute(self, X_test, derivative=False, **kwargs):
        """Change of the entropy of p_min per candidate, shape (N,) (information_gain.py:87-125)."""
        if derivative:
            raise NotImplementedError("InformationGain: derivative=True is not supported")
        return self._scores(X_test)["values"]

    def argmax(self, X):
        """numpy.argmax of compute(X), taken on the device."""
        return int(self._scores(X, want_values=False)["best_idx"])
