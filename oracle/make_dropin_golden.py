#!/usr/bin/env python
"""Generate tests/golden/dropin_*.npz by running the UNMODIFIED RoBO reference on the robo_b200 host layer.

TEST INFRASTRUCTURE ONLY.  Needs a checkout of the reference (automl/RoBO, the commit DESIGN.md cites):

    python oracle/make_dropin_golden.py <path of the RoBO checkout>

Each scenario runs the reference's own solver, fmin facade, maximizers and model classes with ``george`` and ``emcee``
replaced by the robo_b200.compat shims and the device library replaced by tests/fake_gpk.FakeHandle (oracle
arithmetic, so this runs without a GPU).  tests/dropin_trace.Recorder logs every call the reference makes into the
shims; tests/test_dropin_reference_cpu.py replays them.  Scenario results that the product's own classes must
reproduce are stored beside the trace (``extra.*``).
"""
import copy
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, "tests", "golden")

from tests import fake_gpk                                         # noqa: E402
from tests.dropin_trace import Recorder                            # noqa: E402
from robo_b200 import compat                                       # noqa: E402
from robo_b200 import kernels as K                                 # noqa: E402


def branin(x):
    x1, x2 = x[0], x[1]
    return (x2 - 5.1 / (4 * np.pi ** 2) * x1 ** 2 + 5 / np.pi * x1 - 6) ** 2 + 10 * (1 - 1 / (8 * np.pi)) * np.cos(x1) + 10


def solver_calls(rec):
    """The reference's BayesianOptimization solver driving the product's model / acquisition / maximizer: its calls
    into them are logged."""
    from robo.solver.bayesian_optimization import BayesianOptimization
    from robo_b200.acquisition_functions import LCB
    from robo_b200.maximizers import RandomSampling
    from robo_b200.models import GaussianProcess
    lower, upper = np.zeros(1), np.ones(1) * 6
    model = GaussianProcess(K.Matern52Kernel(np.ones(1), ndim=1), noise=1e-3, lower=lower, upper=upper,
                            rng=np.random.RandomState(2))
    acq = LCB(model)
    maximizer = RandomSampling(acq, lower, upper, rng=np.random.RandomState(1))
    rec.log_calls(model, "train")
    rec.log_calls(acq, "update")
    rec.log_calls(maximizer, "maximize")
    solver = BayesianOptimization(lambda x: np.sin(3 * x[0]) * 4 * (x[0] - 1) * (x[0] + 2), lower, upper, acq, model,
                                  maximizer, rng=np.random.RandomState(0))
    np.random.seed(7)                       # RandomSampling draws its candidates from numpy's global generator
    solver.run(num_iterations=6)
    return dict(X=np.array(solver.X), y=np.array(solver.y), incumbents=np.array(solver.incumbents),
                incumbents_values=np.array(solver.incumbents_values))


def fmin_gp(maximizer):
    from robo.fmin import bayesian_optimization
    res = bayesian_optimization(branin, np.array([-5.0, 0.0]), np.array([10.0, 15.0]), num_iterations=7,
                                maximizer=maximizer, acquisition_func="ei", model_type="gp", n_init=3,
                                rng=np.random.RandomState(2))
    return dict(X=np.array(res["X"]), y=np.array(res["y"]))


def fmin_gp_mcmc_log_ei():
    import robo.fmin  # noqa: F401
    facade = sys.modules["robo.fmin.bayesian_optimization"]
    real = facade.GaussianProcessMCMC

    def short_chains(*a, **kw):
        kw.update(chain_length=6, burnin_steps=4)
        return real(*a, **kw)
    facade.GaussianProcessMCMC = short_chains
    try:
        res = facade.bayesian_optimization(branin, np.array([-5.0, 0.0]), np.array([10.0, 15.0]), num_iterations=5,
                                           n_init=3, rng=np.random.RandomState(3))
    finally:
        facade.GaussianProcessMCMC = real
    return dict(X=np.array(res["X"]), y=np.array(res["y"]))


def gp_class_branin_ny1():
    import george
    from robo.models.gaussian_process import GaussianProcess
    from robo.acquisition_functions.ei import EI
    from robo.priors.default_priors import DefaultPrior
    d = np.load(os.path.join(OUT, "gp_branin_ny1.npz"))
    k = 2 * george.kernels.Matern52Kernel(np.ones(2), ndim=2)
    k.set_parameter_vector(np.array([np.log(1.7), np.log(0.15), np.log(0.4)]))
    model = GaussianProcess(k, prior=DefaultPrior(len(k) + 1), noise=float(d["noise"]), normalize_input=True,
                            normalize_output=True, lower=d["lower"], upper=d["upper"], rng=np.random.RandomState(0))
    model.train(d["X"], d["y"], do_optimize=False)
    mu, var = model.predict(d["Xs"])
    return dict(mu=mu, var=var, acq_ei=EI(model).compute(d["Xs"]), nll_vals=np.array([model.nll(t) for t in d["nll_thetas"]]))


def fabolas_problem():
    rng = np.random.RandomState(5)
    lower, upper = np.array([-1.0, 2.0]), np.array([3.0, 5.0])
    X = np.concatenate((lower + (upper - lower) * rng.rand(25, 2), rng.rand(25, 1)), axis=1)
    y = np.sin(X[:, 0]) + 0.3 * X[:, 1] + (1 - X[:, 2]) ** 2
    Xt = np.concatenate((lower + (upper - lower) * rng.rand(9, 2), rng.rand(9, 1)), axis=1)
    return lower, upper, X, y, Xt


def fabolas():
    """robo/models/fabolas_gp.py FabolasGP and FabolasGPMCMC on the shims."""
    import george
    from robo.models.fabolas_gp import FabolasGP, FabolasGPMCMC
    from robo.acquisition_functions.ei import EI
    lower, upper, X, y, Xt = fabolas_problem()

    def basis(s):
        return (1 - s) ** 2

    k = 1.3 * george.kernels.Matern52Kernel(np.ones(1) * 0.4, ndim=3, axes=0)
    k *= george.kernels.Matern52Kernel(np.ones(1) * 0.6, ndim=3, axes=1)
    k *= george.kernels.Matern52Kernel(np.ones(1) * 0.9, ndim=3, axes=2)
    ref = FabolasGP(copy.deepcopy(k), basis_function=basis, noise=1e-3, lower=lower, upper=upper,
                    rng=np.random.RandomState(0))
    ref.train(X, y, do_optimize=False)
    mu, var = ref.predict(Xt)
    ei = EI(ref).compute(Xt)

    class Prior(object):
        def __init__(self, r):
            self.r = r

        def lnprob(self, t):
            return 0.0 if np.all(np.abs(t) < 6) else -np.inf

        def sample_from_prior(self, n):
            return self.r.uniform(-2, 1, size=(n, 5))
    refm = FabolasGPMCMC(copy.deepcopy(k), basis_func=basis, prior=Prior(np.random.RandomState(1)), n_hypers=10,
                         chain_length=4, burnin_steps=3, lower=lower, upper=upper, rng=np.random.RandomState(2))
    refm.train(X, y, do_optimize=True)
    mm, vm = refm.predict(Xt)
    return dict(mu=mu, var=var, acq_ei=ei, mcmc_hypers=np.array(refm.hypers), mcmc_mu=mm, mcmc_var=vm)


SCENARIOS = [
    ("dropin_solver", None, solver_calls),
    ("dropin_fmin_gp_random", "branin", lambda rec: fmin_gp("random")),
    ("dropin_fmin_gp_scipy", "branin", lambda rec: fmin_gp("scipy")),
    ("dropin_fmin_gp_differential_evolution", "branin", lambda rec: fmin_gp("differential_evolution")),
    ("dropin_fmin_gp_mcmc_log_ei", "branin", lambda rec: fmin_gp_mcmc_log_ei()),
    ("dropin_gp_class_branin_ny1", "branin", lambda rec: gp_class_branin_ny1()),
    ("dropin_fabolas", "fabolas", lambda rec: fabolas()),
]


def main():
    if len(sys.argv) != 2 or not os.path.isdir(os.path.join(sys.argv[1], "robo")):
        sys.exit("usage: python oracle/make_dropin_golden.py <path of the RoBO checkout>")
    sys.path.insert(0, os.path.abspath(sys.argv[1]))
    mp = pytest.MonkeyPatch()
    fake_gpk.install(mp)
    compat.install(force_emcee=True)
    for name, kernel, fn in SCENARIOS:
        with Recorder(kernel) as rec:
            extra = fn(rec)
        path = os.path.join(OUT, name + ".npz")
        rec.save(path, **extra)
        print("%s: %d calls, %d bytes" % (path, len(rec.ops), os.path.getsize(path)))
    mp.undo()


if __name__ == "__main__":
    main()
