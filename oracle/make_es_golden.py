"""Generate tests/golden/es_*.npz by running the REAL reference entropy-search code (TEST INFRASTRUCTURE ONLY).

Runs verbatim from a RoBO checkout (ROBO_REFERENCE, read-only, via sys.path): robo/util/epmgp.py joint_min and the
InformationGain / InformationGainPerUnitCost classes.  Their model is the george restatement of oracle/ behind the
reference GaussianProcess's predict / predict_variance contract; emcee is replaced by a stub because the representer
points are fixed by overriding sample_representer_points on the instance.  The numpy restatement (oracle/es_oracle.py)
must reproduce every recorded array to rtol 1e-12, so the vectors pin the restatement to the reference's own code.

    ROBO_REFERENCE=<RoBO checkout> python oracle/make_es_golden.py
"""
import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("ROBO_REFERENCE")
if not REF:
    raise SystemExit("set ROBO_REFERENCE to a RoBO checkout")
sys.path.insert(0, ROOT)
sys.path.insert(0, REF)
sys.modules.setdefault("emcee", types.ModuleType("emcee"))
for _alias, _value in (("NAN", np.nan), ("Infinity", np.inf)):     # names the reference uses that numpy 2 removed
    if not hasattr(np, _alias):
        setattr(np, _alias, _value)

from oracle import es_oracle as E          # noqa: E402
from oracle import robo_oracle as O        # noqa: E402
from robo.util import epmgp                # noqa: E402
from robo.acquisition_functions.information_gain import InformationGain                     # noqa: E402
from robo.acquisition_functions.information_gain_per_unit_cost import InformationGainPerUnitCost  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


def same(a, b, what, rtol=1e-12):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    scale = max(np.max(np.abs(a)), 1e-300)
    if a.shape != b.shape or np.max(np.abs(a - b)) > rtol * scale:
        raise AssertionError("restatement != reference for %s" % what)


class OracleModel(object):
    """The reference GaussianProcess contract (predict with full_cov, predict_variance, get_noise) on an oracle state."""
    def __init__(self, st, noise):
        self.st, self.noise = st, noise

    def predict(self, X, full_cov=False, **kw):
        return O.gp_predict(self.st, X, full_cov=full_cov)

    def predict_variance(self, x1, X2):
        _, var = self.predict(np.concatenate((x1, X2)), full_cov=True)
        return var[-1, :-1, np.newaxis]

    def get_noise(self):
        return self.noise

    def update(self, *a, **k):
        pass


class ConstModel(object):
    def __init__(self, c):
        self.c = c

    def predict(self, X, **kw):
        return np.full(X.shape[0], self.c), np.ones(X.shape[0])


def ep_case(name, mu, S):
    ref = epmgp.joint_min(mu, S, with_derivatives=True)
    got = E.joint_min(mu, S)
    for r, g, n in zip(ref, got, ("logP", "dlogPdMu", "dlogPdSigma", "dlogPdMudMu")):
        same(r, g, name + " " + n)
    np.savez_compressed(os.path.join(GOLDEN, "es_ep_%s.npz" % name), mu=mu, V=S, logP=ref[0], dlogPdMu=ref[1],
                        dlogPdSigma=ref[2], dlogPdMudMu=ref[3], sweeps=got[4])


def gp_problem(normalize_output, N=60, D=2, seed=3):
    rng = np.random.RandomState(seed)
    X = rng.rand(N, D)
    y = np.sin(6 * X[:, 0]) + np.cos(4 * X[:, 1]) + 0.05 * rng.randn(N)
    theta = np.array([0.3, np.log(0.1), np.log(0.2)])
    noise = 1e-3
    st = O.gp_fit(O.make_kernel("matern52", D, theta), X, y, noise=noise, normalize_input=True,
                  normalize_output=normalize_output, lower=np.zeros(D), upper=np.ones(D))
    return X, y, theta, noise, st


def compute_case(name, normalize_output, Nb=50, Np=400, M=256):
    X, y, theta, noise, st = gp_problem(normalize_output)
    D = X.shape[1]
    rng = np.random.RandomState(7)
    zb = rng.rand(Nb, D)
    lmb = np.log(rng.rand(Nb) + 0.1)[:, None]
    lower, upper = np.zeros(D), np.ones(D)
    model = OracleModel(st, noise)
    ig = InformationGain(model, lower, upper, Nb=Nb, Np=Np, sampling_acquisition=lambda m, **kw: ConstModel(0.0))
    ig.sample_representer_points = lambda: setattr(ig, "zb", zb) or setattr(ig, "lmb", lmb)
    ig.update(model)
    Xs = rng.uniform(-0.05, 1.05, size=(M, D))          # a few rows fall outside [0, 1]
    # ig.compute raises on a row outside the bounds (dh_fun returns its (value, gradient) pair there even without
    # derivative=True, :219-222): those rows take dh_fun's value, np.spacing(1)
    outside = np.any((Xs < lower) | (Xs > upper), axis=1)
    ref = np.empty(M)
    ref[~outside] = ig.compute(Xs[~outside])
    ref[outside] = [ig.dh_fun(x[None, :])[0][0, 0] for x in Xs[outside]]
    mu_b, V_b, s, v = E.gp_es_inputs(st, O.gp_predict, zb, Xs)
    logP, dMu, dSig, dMuMu, sweeps = E.joint_min(mu_b, V_b)
    same(ig.logP.ravel(), logP, name + " logP")
    state = dict(logP=logP, dlogPdMu=dMu, dlogPdSigma=dSig, dlogPdMudMu=dMuMu, lmb=lmb, W=E.grid(Np), sn2=noise)
    got = E.information_gain(state, s, v, Xs, lower, upper)
    same(ref, got, name + " dH", rtol=1e-10)
    np.savez_compressed(os.path.join(GOLDEN, "es_compute_%s.npz" % name), X=X, y=y, theta=theta, noise=noise,
                        normalize_output=normalize_output, zb=zb, lmb=lmb.ravel(), Np=Np, Xs=Xs, dH=ref,
                        logP=ig.logP.ravel(), H=-np.sum(np.exp(logP) * (logP + lmb.ravel())))


def per_unit_cost_case():
    """InformationGainPerUnitCost on a FabolasGP-style input (last column = dataset fraction): dh / (exp(cost) + oh)."""
    X, y, theta, noise, st = gp_problem(False, seed=5)
    Xc, yc = X, 0.5 + X[:, 1]
    stc = O.gp_fit(O.make_kernel("matern52", 2, np.array([0.0, 0.0, 0.0])), Xc, yc, noise=1e-3, normalize_input=True,
                   lower=np.zeros(2), upper=np.ones(2))
    model, cost = OracleModel(st, noise), OracleModel(stc, 1e-3)
    lower, upper, is_env = np.zeros(2), np.ones(2), np.array([0, 1])
    ig = InformationGainPerUnitCost(model, cost, lower, upper, is_env, sampling_acquisition=lambda m, **kw: ConstModel(0.0),
                                    n_representer=20)
    rng = np.random.RandomState(11)
    zb = np.concatenate([rng.rand(20, 1), np.ones((20, 1))], axis=1)      # what sample_representer_points leaves
    lmb = np.log(rng.rand(20) + 0.1)[:, None]
    ig.sample_representer_points = lambda: setattr(ig, "zb", zb) or setattr(ig, "lmb", lmb)
    ig.update(model, cost, overhead=0.25)
    Xs = rng.rand(64, 2)
    ref = np.array([ig.compute(x[None, :])[0] for x in Xs])
    np.savez_compressed(os.path.join(GOLDEN, "es_cost.npz"), X=X, y=y, theta=theta, noise=noise, Xc=Xc, yc=yc, zb=zb,
                        lmb=lmb.ravel(), Xs=Xs, overhead=0.25, value=ref)


def main():
    rng = np.random.RandomState(0)
    ep_case("uniform", np.zeros(10), np.eye(10))                          # test/test_util/test_epmgp.py style cases
    S = np.full((10, 10), 1e-8) + np.eye(10) * 1e-3
    ep_case("dirac", np.concatenate([[-5.0], np.zeros(9)]), S)
    X, y, theta, noise, st = gp_problem(True)
    zb = rng.rand(24, 2)
    mu_b, V_b = O.gp_predict(st, zb, full_cov=True)
    ep_case("gp24", mu_b, V_b)
    compute_case("norm", True)
    compute_case("raw", False)
    per_unit_cost_case()
    print("es goldens written")


if __name__ == "__main__":
    main()
