"""Entropy-search methods of the oracle-backed FakeHandle (TEST INFRASTRUCTURE ONLY): the gpk_es_* surface of
robo_b200._lib.Handle with the arithmetic of oracle/es_oracle.py, so the CPU suite drives InformationGain /
InformationGainPerUnitCost / MarginalizationGPMCMC through the same calls the GPU runs."""
import numpy as np
import scipy.linalg as spla

from oracle import es_oracle as E
from oracle import robo_oracle as O
from tests import fake_gpk


class FakeESHandle(fake_gpk.FakeHandle):
    n_es_updates = 0

    def es_joint_min(self, mu, V):
        logP, dMu, dSig, dMuMu, sweeps = E.joint_min(mu, V)
        self.es = dict(logP=logP, dlogPdMu=dMu, dlogPdSigma=dSig, dlogPdMudMu=dMuMu, sweeps=sweeps)
        self.es_ready = False
        return dict(self.es)

    def es_update(self, zb, lmb, np_grid, sn2):
        lmb = np.asarray(lmb, dtype=np.float64).ravel()
        if not np.all(np.isfinite(lmb)):
            raise ValueError("lmb should not be infinite")
        if not (2 <= len(lmb) <= 128) or np_grid < 1:
            raise ValueError("bad entropy-search sizes")
        mu_b, V_b = self.predict_cov(zb)
        self.es_joint_min(mu_b, V_b)
        self.es.update(lmb=lmb, W=E.grid(np_grid), sn2=float(sn2), zb=np.array(zb, dtype=np.float64))
        self.es_ready = True
        FakeESHandle.n_es_updates += 1
        return self.es["logP"].copy()

    def es_compute(self, Xs, lower=None, upper=None, want_values=True):
        if not getattr(self, "es_ready", False):
            raise ValueError("no entropy-search state")
        Xs = np.asarray(Xs, dtype=np.float64)
        zbn, Xn = self._norm(self.es["zb"]), self._norm(Xs)
        B = spla.cho_solve((self.L, True), self.kernel.get_value(self.X, zbn))
        s = self.kernel.get_value(Xn, zbn) - self.kernel.get_value(Xn, self.X) @ B
        on, _, ys = self.out
        if on:
            s = s * ys ** 2
        s = np.clip(s, O.EPS, np.inf)
        v = self.predict(Xs)[1]
        vals = E.information_gain(self.es, s, v, Xs, lower, upper)
        bi = int(np.argmax(vals))
        return dict(values=vals if want_values else None, best_val=float(vals[bi]), best_idx=bi)

    def es_get_state(self, nb):
        return {k: np.array(self.es[k]) for k in ("logP", "dlogPdMu", "dlogPdSigma", "dlogPdMudMu", "sweeps")}


def install(monkeypatch):
    from robo_b200 import _lib
    fake_gpk.install(monkeypatch)
    monkeypatch.setattr(_lib, "Handle", FakeESHandle)
    return FakeESHandle
