"""Entropy search on the B200 (gpk_es_*, robo_b200.acquisition_functions.InformationGain): EP against the reference's
own epmgp.joint_min (tests/golden/es_ep_*.npz) and the numpy restatement, the information gain against the
reference's InformationGain (tests/golden/es_compute_*.npz) and the restatement at N = 1024 / 4096, chunking,
MarginalizationGPMCMC over sub-models, and the entropy_search facade."""
import os

import numpy as np
import pytest
import scipy.linalg as spla

from oracle import es_oracle as E
from oracle import robo_oracle as O

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _load(name):
    return dict(np.load(os.path.join(GOLDEN, name)))


def _rel(a, b):
    return np.max(np.abs(np.asarray(a) - np.asarray(b))) / max(np.max(np.abs(b)), 1e-300)


@pytest.mark.parametrize("case", ["uniform", "dirac", "gp24"])
def test_joint_min_matches_reference_golden(case):
    from robo_b200 import _lib
    g = _load("es_ep_%s.npz" % case)
    h = _lib.Handle(0)
    r = h.es_joint_min(g["mu"], g["V"])
    for key in ("logP", "dlogPdMu", "dlogPdSigma", "dlogPdMudMu"):
        assert _rel(r[key], g[key]) < 1e-10, (key, _rel(r[key], g[key]))
    assert np.array_equal(r["sweeps"], g["sweeps"])
    h.close()


@pytest.mark.parametrize("nb", [2, 50, 128])
def test_joint_min_matches_oracle(nb):
    from robo_b200 import _lib
    rng = np.random.RandomState(nb)
    Z = rng.rand(nb, 3)
    S = np.exp(-((Z[:, None] - Z[None]) ** 2).sum(-1) / 0.3) + 1e-4 * np.eye(nb)
    mu = 0.3 * rng.randn(nb)
    ref = E.joint_min(mu, S)
    h = _lib.Handle(0)
    r = h.es_joint_min(mu, S)
    for key, want in zip(("logP", "dlogPdMu", "dlogPdSigma", "dlogPdMudMu"), ref[:4]):
        assert _rel(r[key], want) < 1e-10, (key, _rel(r[key], want))
    assert np.array_equal(r["sweeps"], ref[4])
    with pytest.raises(ValueError):
        h.es_joint_min(np.zeros(129), np.eye(129))
    h.close()


def _model(X, y, theta, noise, normalize_output, D):
    from robo_b200 import kernels as K
    from robo_b200.models.gaussian_process import GaussianProcess
    kernel = K.Product(K.ConstantKernel(theta[0], ndim=D), K.Matern52Kernel(np.exp(theta[1:]), ndim=D))
    m = GaussianProcess(kernel, noise=noise, normalize_input=True, normalize_output=normalize_output,
                        lower=np.zeros(D), upper=np.ones(D))
    m.train(X, y, do_optimize=False)
    return m


def _ig(model, zb, lmb, Np=400):
    from robo_b200.acquisition_functions import InformationGain
    D = zb.shape[1]
    ig = InformationGain(model, np.zeros(D), np.ones(D), Nb=zb.shape[0], Np=Np)
    ig.sample_representer_points = lambda: (setattr(ig, "zb", zb), setattr(ig, "lmb", lmb[:, None]))
    ig.update(model)
    return ig


@pytest.mark.parametrize("case", ["norm", "raw"])
def test_compute_matches_reference_golden(case):
    g = _load("es_compute_%s.npz" % case)
    D = g["X"].shape[1]
    model = _model(g["X"], g["y"], g["theta"], float(g["noise"]), bool(g["normalize_output"]), D)
    ig = _ig(model, g["zb"], g["lmb"], int(g["Np"]))
    assert _rel(ig.logP.ravel(), g["logP"]) < 1e-10
    got = ig.compute(g["Xs"])
    tol = 1e-8 * max(np.max(np.abs(g["dH"])), abs(float(g["H"])))
    assert np.max(np.abs(got - g["dH"])) < tol
    assert ig.argmax(g["Xs"]) == int(np.argmax(g["dH"]))
    outside = np.any((g["Xs"] < 0) | (g["Xs"] > 1), axis=1)
    assert outside.any() and np.all(got[outside] == np.spacing(1))


def _oracle_dH(X, y, theta, noise, zb, lmb, Xs, Np=400):
    """Restatement of compute at sizes where the reference's full joint covariance does not fit: s from the explicit
    K^-1 k(X, zb), in chunks."""
    D = X.shape[1]
    k = O.make_kernel("matern52", D, theta)
    st = O.gp_fit(k, X, y, noise=noise, normalize_input=True, lower=np.zeros(D), upper=np.ones(D))
    mu_b, V_b = O.gp_predict(st, zb, full_cov=True)
    logP, dMu, dSig, dMuMu, _ = E.joint_min(mu_b, V_b)
    Kxx = k.get_value(X) + (noise + 1.25e-12) * np.eye(len(X))
    cf = spla.cho_factor(Kxx, lower=True)
    B = spla.cho_solve(cf, k.get_value(X, zb))
    state = dict(logP=logP, dlogPdMu=dMu, dlogPdSigma=dSig, dlogPdMudMu=dMuMu, lmb=lmb, W=E.grid(Np), sn2=noise)
    out = []
    for i in range(0, len(Xs), 1000):
        C = Xs[i:i + 1000]
        s = np.clip(k.get_value(C, zb) - k.get_value(C, X) @ B, O.EPS, np.inf)
        v = O.gp_predict_var_only_fast(st, C)[1]
        out.append(E.information_gain(state, s, v, C, np.zeros(D), np.ones(D)))
    H = -np.sum(np.exp(logP) * (logP + lmb))
    return np.concatenate(out), H


@pytest.mark.parametrize("N,D,M", [(1024, 8, 1000), (1024, 8, 20000), (4096, 16, 1000), (4096, 16, 20000)])
def test_compute_matches_oracle_at_scale(N, D, M):
    X, y, _, theta, noise = O.synthetic_problem(N, D, 1)
    rng = np.random.RandomState(N + M)
    zb, lmb = rng.rand(50, D), np.log(rng.rand(50) + 0.05)
    Xs = rng.rand(M, D)
    model = _model(X, y, theta, noise, False, D)
    ig = _ig(model, zb, lmb)
    got = ig.compute(Xs)
    ref, H = _oracle_dH(X, y, theta, noise, zb, lmb, Xs)
    assert np.max(np.abs(got - ref)) < 1e-8 * max(np.max(np.abs(ref)), abs(H))
    assert ig.argmax(Xs) == int(np.argmax(got))


def test_chunk_size_invariance_and_two_objects_on_one_model():
    X, y, _, theta, noise = O.synthetic_problem(700, 4, 1)
    rng = np.random.RandomState(1)
    Xs = rng.rand(5000, 4)
    model = _model(X, y, theta, noise, True, 4)
    a = _ig(model, rng.rand(50, 4), np.log(rng.rand(50) + 0.1))
    b = _ig(model, rng.rand(30, 4), np.log(rng.rand(30) + 0.1))        # b's state now sits on the handle

    def tol(ig, v):
        return 1e-8 * max(np.max(np.abs(v)), abs(float(-np.sum(np.exp(ig.logP) * (ig.logP + ig.lmb)))))

    va = a.compute(Xs)                                                # a re-sends its own state
    vb = b.compute(Xs)
    # chunks of 1024 candidates: the variance runs on the fp64 kernel instead of the int8 one (batches < 2048)
    model.gp.handle.set_option("chunk", 1024)
    assert np.max(np.abs(a.compute(Xs) - va)) <= tol(a, va)
    assert np.max(np.abs(b.compute(Xs) - vb)) <= tol(b, vb)
    assert a.argmax(Xs) == int(np.argmax(va))
    model.gp.handle.set_option("chunk", 0)
    assert np.array_equal(a.compute(Xs), va) and np.array_equal(b.compute(Xs), vb)


def test_marginalisation_over_sub_models_is_the_mean_of_oracle_values(monkeypatch):
    from robo_b200.acquisition_functions import InformationGain, MarginalizationGPMCMC
    X, y, _, theta0, noise = O.synthetic_problem(300, 3, 1)
    rng = np.random.RandomState(5)
    thetas = [theta0 + 0.2 * rng.randn(theta0.size) for _ in range(10)]
    models = [_model(X, y, t, noise, False, 3) for t in thetas]

    class Mixture(object):
        def __init__(self, models):
            self.models = models

    zb, lmb = rng.rand(40, 3), np.log(rng.rand(40) + 0.1)
    monkeypatch.setattr(InformationGain, "sample_representer_points",
                        lambda self: (setattr(self, "zb", zb), setattr(self, "lmb", lmb[:, None])))
    mix = Mixture(models)
    acq = MarginalizationGPMCMC(InformationGain(mix, np.zeros(3), np.ones(3), Nb=40))
    acq.update(mix)
    Xs = rng.rand(800, 3)
    got = acq.compute(Xs)
    refs = [_oracle_dH(X, y, t, noise, zb, lmb, Xs) for t in thetas]
    ref = np.mean([r for r, _ in refs], axis=0)
    scale = max(np.max(np.abs(ref)), max(abs(H) for _, H in refs))
    assert np.max(np.abs(got - ref)) < 1e-8 * scale


@pytest.mark.parametrize("model_type", ["gp", "gp_mcmc"])
def test_entropy_search_facade_on_branin(model_type):
    from robo_b200.fmin import entropy_search

    def branin(x):
        x1, x2 = x[0], x[1]
        return (x2 - 5.1 / (4 * np.pi ** 2) * x1 ** 2 + 5 / np.pi * x1 - 6) ** 2 \
            + 10 * (1 - 1 / (8 * np.pi)) * np.cos(x1) + 10

    lower, upper = np.array([-5.0, 0.0]), np.array([10.0, 15.0])
    res = entropy_search(branin, lower, upper, num_iterations=6, model=model_type, n_init=3,
                         rng=np.random.RandomState(0), chain_length=20, burnin_steps=10)
    assert len(res["y"]) == 6 and np.isfinite(res["f_opt"]) and np.all(np.isfinite(res["y"]))
    assert np.all(np.array(res["X"]) >= lower) and np.all(np.array(res["X"]) <= upper)
