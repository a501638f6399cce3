"""Drop-in boundary, CPU side: the UNMODIFIED reference (solver, fmin facade, maximizers, its own
GaussianProcess / GaussianProcessMCMC / FabolasGP classes) on top of the robo_b200 host layer.

The reference drives robo_b200 through the ``george`` and ``emcee`` shims of robo_b200.compat.  Its calls into them,
with their answers, were recorded by oracle/make_dropin_golden.py (tests/golden/dropin_*.npz; tests/dropin_trace.py);
these tests issue the same calls to the shims of this tree and require the same answers, so the reference would take
the same path through them as it did when it was recorded.  libgpk.so cannot execute without a GPU, so ``_lib.Handle``
is replaced by tests/fake_gpk.FakeHandle (oracle arithmetic, same method surface); the GPU suite covers the same
surface against the real library."""
import os

import numpy as np
import pytest

from tests import dropin_trace


@pytest.fixture
def fake(monkeypatch):
    from tests import fake_gpk
    return fake_gpk.install(monkeypatch)


def branin_kernel():
    from robo_b200 import kernels as K
    return 2 * K.Matern52Kernel(np.ones(2), ndim=2)                # robo/fmin/bayesian_optimization.py:75-81


def fabolas_kernel():
    from robo_b200 import kernels as K
    k = 1.3 * K.Matern52Kernel(np.ones(1) * 0.4, ndim=3, axes=0)
    k *= K.Matern52Kernel(np.ones(1) * 0.6, ndim=3, axes=1)
    k *= K.Matern52Kernel(np.ones(1) * 0.9, ndim=3, axes=2)
    return k


KERNELS = {"branin": branin_kernel, "fabolas": fabolas_kernel}


def replay_matches(golden_dir, scenario):
    """Every recorded call gives the recorded answer (LinAlgError where the reference met one).  Returns the number
    of calls checked and the scenario's stored results."""
    path = os.path.join(golden_dir, scenario + ".npz")
    n = 0
    for i, op, rec, got in dropin_trace.replay(path, KERNELS):
        assert set(rec) == set(got), (i, op["op"])
        for k in rec:
            r, g = np.asarray(rec[k], dtype=np.float64), np.asarray(got[k], dtype=np.float64)
            assert r.shape == g.shape, (i, op["op"], k)
            scale = np.max(np.abs(r[np.isfinite(r)]), initial=1.0)
            np.testing.assert_allclose(g, r, rtol=1e-9, atol=1e-12 * scale, err_msg="call %d (%s) %s" % (i, op["op"], k))
        n += 1
    return n, dropin_trace.load(path)[1]


def test_reference_solver_drives_robo_b200_objects(fake, golden_dir):
    """test/test_solver/test_bayesian_optimization.py:28-49: the reference's own BayesianOptimization solver drove the
    product's model / acquisition / maximizer; its recorded calls (train, update, maximize) on fresh objects give the
    recorded next points."""
    from robo_b200 import kernels as K
    from robo_b200.acquisition_functions import LCB
    from robo_b200.maximizers import RandomSampling
    from robo_b200.models import GaussianProcess
    ops, ref = dropin_trace.load(os.path.join(golden_dir, "dropin_solver.npz"))
    lower, upper = np.zeros(1), np.ones(1) * 6
    model = GaussianProcess(K.Matern52Kernel(np.ones(1), ndim=1), noise=1e-3, lower=lower, upper=upper,
                            rng=np.random.RandomState(2))
    acq = LCB(model)
    maximizer = RandomSampling(acq, lower, upper, rng=np.random.RandomState(1))
    assert [op["op"] for op in ops] == ["train", "update", "maximize"] * 3
    state = np.random.get_state()
    np.random.seed(7)                       # RandomSampling draws its candidates from numpy's global generator
    try:
        for op in ops:
            arr = op["arrays"]
            if op["op"] == "train":
                model.train(arr["arg0"], arr["arg1"], **op["kw"])
            elif op["op"] == "update":
                acq.update(model)
            else:
                x = maximizer.maximize()
                assert np.all(x >= lower) and np.all(x <= upper)
                np.testing.assert_allclose(x, arr["out"], rtol=1e-9, atol=1e-12)
    finally:
        np.random.set_state(state)
    assert len(ref["incumbents"]) == 6 and len(ref["incumbents_values"]) == 6
    assert model.gp.handle.n_fits >= 3


@pytest.mark.parametrize("maximizer", ["random", "scipy", "differential_evolution"])
def test_unmodified_reference_fmin_gp(fake, golden_dir, maximizer):
    """robo.fmin.bayesian_optimization (reference facade + solver + maximizers + the reference's own
    GaussianProcess class) with george replaced by the robo_b200 shim."""
    n, res = replay_matches(golden_dir, "dropin_fmin_gp_" + maximizer)
    assert n > 100
    lower, upper = np.array([-5.0, 0.0]), np.array([10.0, 15.0])
    assert len(res["y"]) == 7 and np.all(res["X"] >= lower) and np.all(res["X"] <= upper)


def test_unmodified_reference_fmin_gp_mcmc_log_ei(fake, golden_dir):
    """the facade's default path: GaussianProcessMCMC (reference class, emcee shim) + MarginalizationGPMCMC(LogEI),
    with short chains (chain_length=6, burnin_steps=4)."""
    ops = dropin_trace.load(os.path.join(golden_dir, "dropin_fmin_gp_mcmc_log_ei.npz"))[0]
    assert sum(op["op"] == "run_mcmc" for op in ops) >= 2
    n, res = replay_matches(golden_dir, "dropin_fmin_gp_mcmc_log_ei")
    lower, upper = np.array([-5.0, 0.0]), np.array([10.0, 15.0])
    assert len(res["y"]) == 5 and np.all(res["X"] >= lower) and np.all(res["X"] <= upper)


def test_reference_gp_class_on_shim_matches_golden(fake, golden_dir):
    """The reference's own GaussianProcess on the george shim reproduced the golden vectors that were generated with
    the same class on the oracle (the shim is a faithful george.GP for RoBO's call pattern), and the shim still
    answers that call pattern the same way."""
    replay_matches(golden_dir, "dropin_gp_class_branin_ny1")
    ref = dropin_trace.load(os.path.join(golden_dir, "dropin_gp_class_branin_ny1.npz"))[1]
    d = np.load(os.path.join(golden_dir, "gp_branin_ny1.npz"))
    np.testing.assert_allclose(ref["mu"], d["mu"], rtol=1e-9)
    np.testing.assert_allclose(ref["var"], d["var"], rtol=1e-8)
    np.testing.assert_allclose(ref["acq_ei"], d["acq_ei"], rtol=1e-7, atol=1e-12)
    for v, t in zip(ref["nll_vals"], d["nll_vals"]):
        assert abs(v - t) <= 1e-9 * abs(t) or t == 1e25


def test_product_host_layer_on_fake_handle_matches_golden(fake, golden_dir):
    """robo_b200's own classes (host logic: normalisation, hypers bookkeeping, incumbent, retry, EI quirks)
    against the golden vectors, with the C library substituted by the oracle."""
    from tests.golden_cases import kernel_spec, load_case
    from tests.product_cases import product_model
    from robo_b200.acquisition_functions import EI, LCB, PI, LogEI
    for name in ("gp_unit", "gp_branin_ny0", "gp_autobounds", "gp_prod1d"):
        d, _ = load_case(name)
        family, theta = kernel_spec(name)
        model = product_model(d, family, theta)
        model.train(d["X"], d["y"], do_optimize=False)
        mu, var = model.predict(d["Xs"])
        np.testing.assert_allclose(mu, d["mu"], rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(var, d["var"], rtol=1e-7)
        np.testing.assert_allclose(model.hypers, d["hypers"], rtol=1e-15)
        np.testing.assert_allclose(model.get_incumbent()[0], d["inc_x"], rtol=1e-15)
        for cls, key in ((EI, "acq_ei"), (PI, "acq_pi"), (LCB, "acq_lcb"), (LogEI, "acq_log_ei")):
            np.testing.assert_allclose(cls(model).compute(d["Xs"]), d[key], rtol=1e-6, atol=1e-10)


def test_fabolas_subclasses_ride_the_path(fake, golden_dir):
    """robo/models/fabolas_gp.py (FabolasGP, FabolasGPMCMC) UNMODIFIED on the george / emcee shims (replayed), next to
    the product's own FabolasGP / FabolasGPMCMC (robo_b200/models/fabolas_gp.py): same predictions as the reference
    class gave, since both are the base classes plus the input transform of fabolas_gp.py:122-126."""
    from oracle.make_dropin_golden import fabolas_problem
    from robo_b200.acquisition_functions import EI, MarginalizationGPMCMC
    from robo_b200.models import FabolasGP, FabolasGPMCMC
    replay_matches(golden_dir, "dropin_fabolas")
    ref = dropin_trace.load(os.path.join(golden_dir, "dropin_fabolas.npz"))[1]
    assert ref["mcmc_hypers"].shape == (10, 5) and ref["mcmc_mu"].shape == (9,)
    lower, upper, X, y, Xt = fabolas_problem()

    def basis(s):
        return (1 - s) ** 2                                   # fabolas.py:96-98

    own = FabolasGP(fabolas_kernel(), basis_function=basis, noise=1e-3, lower=lower, upper=upper,
                    rng=np.random.RandomState(0))
    own.train(X, y, do_optimize=False)
    m2, v2 = own.predict(Xt)
    np.testing.assert_allclose(m2, ref["mu"], rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(v2, ref["var"], rtol=1e-7)
    np.testing.assert_allclose(EI(own).compute(Xt), ref["acq_ei"], rtol=1e-6, atol=1e-12)
    # MCMC variant: short chains; the product's sub-models are FabolasGP on the device path and the marginalised
    # acquisition goes through the fused multi-model call on transformed inputs
    class Prior(object):
        def __init__(self, r):
            self.r = r

        def lnprob(self, t):
            return 0.0 if np.all(np.abs(t) < 6) else -np.inf

        def sample_from_prior(self, n):
            return self.r.uniform(-2, 1, size=(n, 5))
    ownm = FabolasGPMCMC(fabolas_kernel(), basis_func=basis, prior=Prior(np.random.RandomState(1)), n_hypers=10,
                         chain_length=4, burnin_steps=3, lower=lower, upper=upper, rng=np.random.RandomState(2))
    ownm.train(X, y, do_optimize=True)
    assert len(ownm.models) == 10 and all(isinstance(m, FabolasGP) for m in ownm.models)
    m, v = ownm.predict(Xt)
    mus = np.array([sub.predict(Xt)[0] for sub in ownm.models])
    vs = np.array([sub.predict(Xt)[1] for sub in ownm.models])
    np.testing.assert_allclose(m, mus.mean(axis=0), rtol=1e-12)
    np.testing.assert_allclose(v, np.clip(mus.var(axis=0) + vs.mean(axis=0), np.finfo(float).eps, np.inf), rtol=1e-10)
    acq = MarginalizationGPMCMC(EI(ownm))
    assert acq._fused_spec() is not None
    np.testing.assert_allclose(acq.compute(Xt), np.mean([EI(s).compute(Xt) for s in ownm.models], axis=0), rtol=1e-12)
    hyp = [list(hh) for hh in ownm.hypers]
    ownm.train(X, y, do_optimize=False)                       # fabolas_gp.py:77-81: samples are kept
    assert [list(hh) for hh in ownm.hypers] == hyp
