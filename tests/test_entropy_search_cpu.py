"""Entropy search without a GPU: the numpy restatement against the reference's own outputs
(tests/golden/es_*.npz), the vech layouts, and the host classes (InformationGain, InformationGainPerUnitCost,
MarginalizationGPMCMC, the entropy_search facade) on the oracle-backed fake handle."""
import os

import numpy as np
import pytest

from oracle import es_oracle as E
from oracle import robo_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _load(name):
    return dict(np.load(os.path.join(GOLDEN, name)))


def _rel(a, b):
    return np.max(np.abs(np.asarray(a) - np.asarray(b))) / max(np.max(np.abs(b)), 1e-300)


@pytest.fixture
def fake(monkeypatch):
    from tests import fake_gpk_es
    return fake_gpk_es.install(monkeypatch)


@pytest.mark.parametrize("case", ["uniform", "dirac", "gp24"])
def test_ep_restatement_matches_reference_golden(case):
    g = _load("es_ep_%s.npz" % case)
    got = E.joint_min(g["mu"], g["V"])
    for key, val in zip(("logP", "dlogPdMu", "dlogPdSigma", "dlogPdMudMu"), got[:4]):
        assert _rel(val, g[key]) < 1e-12, key
    assert np.array_equal(got[4], g["sweeps"])


@pytest.mark.parametrize("case", ["norm", "raw"])
def test_information_gain_restatement_matches_reference_golden(case):
    g = _load("es_compute_%s.npz" % case)
    D = g["X"].shape[1]
    st = O.gp_fit(O.make_kernel("matern52", D, g["theta"]), g["X"], g["y"], noise=float(g["noise"]),
                  normalize_input=True, normalize_output=bool(g["normalize_output"]), lower=np.zeros(D), upper=np.ones(D))
    mu_b, V_b, s, v = E.gp_es_inputs(st, O.gp_predict, g["zb"], g["Xs"])
    logP, dMu, dSig, dMuMu, _ = E.joint_min(mu_b, V_b)
    state = dict(logP=logP, dlogPdMu=dMu, dlogPdSigma=dSig, dlogPdMudMu=dMuMu, lmb=g["lmb"], W=E.grid(int(g["Np"])),
                 sn2=float(g["noise"]))
    got = E.information_gain(state, s, v, g["Xs"], np.zeros(D), np.ones(D))
    assert _rel(got, g["dH"]) < 1e-10


def test_vech_layouts_of_the_reference_agree():
    D = 6
    M = np.arange(D * D, dtype=float).reshape(D, D)
    a = M[np.triu(np.ones((D, D))).T.astype(bool)]                     # information_gain.py:177
    b = np.rot90(M, k=2)[np.triu_indices(D)][::-1]                     # epmgp.py:168
    r, c = E.vech_index(D)
    assert np.array_equal(a, M[r, c]) and np.array_equal(b, M[r, c])
    assert list(zip(r[:4], c[:4])) == [(0, 0), (1, 0), (1, 1), (2, 0)]


def _gp(X, y, theta, noise, normalize_output, D):
    from robo_b200 import kernels as K
    from robo_b200.models.gaussian_process import GaussianProcess
    kernel = K.Product(K.ConstantKernel(theta[0], ndim=D), K.Matern52Kernel(np.exp(theta[1:]), ndim=D))
    m = GaussianProcess(kernel, noise=noise, normalize_input=True, normalize_output=normalize_output,
                        lower=np.zeros(D), upper=np.ones(D))
    m.train(X, y, do_optimize=False)
    return m


def _fix(ig, zb, lmb):
    ig.sample_representer_points = lambda: (setattr(ig, "zb", zb), setattr(ig, "lmb", np.asarray(lmb)[:, None]))


def test_information_gain_host_class_on_fake(fake):
    from robo_b200.acquisition_functions import InformationGain
    g = _load("es_compute_norm.npz")
    model = _gp(g["X"], g["y"], g["theta"], float(g["noise"]), True, 2)
    ig = InformationGain(model, np.zeros(2), np.ones(2), Nb=50, Np=int(g["Np"]))
    _fix(ig, g["zb"], g["lmb"])
    ig.update(model)
    assert ig.logP.shape == (50, 1) and ig.dlogPdSigma.shape == (50, 1275) and ig.W.shape == (1, 400)
    vals = ig.compute(g["Xs"])
    assert _rel(vals, g["dH"]) < 1e-10
    outside = np.any((g["Xs"] < 0) | (g["Xs"] > 1), axis=1)
    assert np.all(vals[outside] == np.spacing(1))
    assert ig.argmax(g["Xs"]) == int(np.argmax(g["dH"]))
    with pytest.raises(NotImplementedError):
        ig.compute(g["Xs"], derivative=True)
    # a non-finite sampling-acquisition value: update keeps going, compute raises like the reference
    lmb = g["lmb"].copy()
    lmb[3] = -np.inf
    _fix(ig, g["zb"], lmb)
    ig.update(model)
    with pytest.raises(ValueError):
        ig.compute(g["Xs"])


def test_two_objects_share_one_model(fake):
    from robo_b200.acquisition_functions import InformationGain
    X, y, Xs, theta, noise = O.synthetic_problem(80, 2, 64)
    model = _gp(X, y, theta, noise, False, 2)
    rng = np.random.RandomState(0)
    a = InformationGain(model, np.zeros(2), np.ones(2), Nb=20, Np=50)
    b = InformationGain(model, np.zeros(2), np.ones(2), Nb=10, Np=50)
    _fix(a, rng.rand(20, 2), np.log(rng.rand(20) + 0.1))
    _fix(b, rng.rand(10, 2), np.log(rng.rand(10) + 0.1))
    a.update(model)
    va = a.compute(Xs)
    b.update(model)
    vb = b.compute(Xs)
    n = fake.n_es_updates
    assert np.array_equal(a.compute(Xs), va)            # a's state is sent again ...
    assert fake.n_es_updates == n + 1
    assert np.array_equal(a.compute(Xs), va)            # ... once
    assert fake.n_es_updates == n + 1
    assert np.array_equal(b.compute(Xs), vb)


def test_per_unit_cost_division_and_projection(fake):
    from robo_b200.acquisition_functions import InformationGainPerUnitCost
    g = _load("es_cost.npz")
    model = _gp(g["X"], g["y"], g["theta"], float(g["noise"]), False, 2)
    cost = _gp(g["Xc"], g["yc"], np.zeros(3), 1e-3, False, 2)
    ig = InformationGainPerUnitCost(model, cost, np.zeros(2), np.ones(2), np.array([0, 1]), n_representer=20)
    _fix(ig, g["zb"], g["lmb"])
    ig.update(model, cost, overhead=float(g["overhead"]))
    assert _rel(ig.compute(g["Xs"]), g["value"]) < 1e-10
    # representer points: sampled over the configuration columns, environment column = number of env columns
    ig2 = InformationGainPerUnitCost(model, cost, np.zeros(3), np.ones(3) * 2, np.array([0, 0, 1]), n_representer=10)
    seen = []
    ig2.sampling_acquisition = lambda X: (seen.append(np.array(X)), np.zeros(len(X)))[1]
    ig2.sampling_acquisition.update = lambda m: None
    ig2.model = model
    ig2.sample_representer_points()
    assert ig2.zb.shape == (10, 3) and np.all(ig2.zb[:, 2] == 1.0)
    assert all(np.all(x[:, 2] == 2.0) for x in seen)          # the sampling acquisition sees upper in env columns


def test_marginalised_mean_and_cost_model_plumbing(fake):
    from robo_b200.acquisition_functions import InformationGain, InformationGainPerUnitCost, MarginalizationGPMCMC
    X, y, Xs, theta, noise = O.synthetic_problem(60, 2, 40)
    rng = np.random.RandomState(2)
    models = [_gp(X, y, theta + 0.1 * rng.randn(3), noise, False, 2) for _ in range(3)]
    costs = [_gp(X, X[:, 1], np.zeros(3), 1e-3, False, 2) for _ in range(3)]

    class Mix(object):
        def __init__(self, ms):
            self.models = ms

    zb, lmb = rng.rand(12, 2), np.log(rng.rand(12) + 0.1)
    mix, cmix = Mix(models), Mix(costs)
    ig = InformationGain(mix, np.zeros(2), np.ones(2), Nb=12, Np=40)
    ig.sample_representer_points = None
    acq = MarginalizationGPMCMC(ig)
    for e in acq.estimators:
        _fix(e, zb, lmb)
    acq.update(mix)
    per = [e.compute(Xs) for e in acq.estimators]
    assert np.allclose(acq.compute(Xs), np.mean(per, axis=0), rtol=1e-14, atol=0)
    assert [e.model for e in acq.estimators] == models
    pc = InformationGainPerUnitCost(mix, cmix, np.zeros(2), np.ones(2), np.array([0, 1]), n_representer=12)
    acq2 = MarginalizationGPMCMC(pc)
    for e in acq2.estimators:
        _fix(e, zb, lmb)
    acq2.update(mix, cmix, overhead=0.5)
    assert [e.cost_model for e in acq2.estimators] == costs
    per2 = [e.compute(Xs) for e in acq2.estimators]
    assert np.allclose(acq2.compute(Xs), np.mean(per2, axis=0), rtol=1e-14, atol=0)
    for e, q in zip(acq2.estimators, per2):
        dh = InformationGain.compute(e, Xs)
        assert np.allclose(q, dh / (np.exp(e.cost_model.predict(Xs)[0]) + 0.5), rtol=1e-12, atol=0)


def test_entropy_search_facade_on_fake(fake):
    from robo_b200.fmin import entropy_search

    def f(x):
        return float(np.sum((x - 0.3) ** 2))

    lower, upper = np.zeros(2), np.ones(2)
    res = entropy_search(f, lower, upper, num_iterations=5, model="gp", n_init=3, rng=np.random.RandomState(0))
    assert len(res["y"]) == 5 and res["f_opt"] == min(res["y"])
    with pytest.raises(ValueError):
        entropy_search(f, lower, upper, num_iterations=4, model="rf")
