"""``entropy_search`` facade with the signature and object wiring of robo/fmin/entropy_search.py:20-131: the same
kernel (cov_amp * Matern52), DefaultPrior, n_hypers rule, InformationGain with EI as the sampling acquisition,
MarginalizationGPMCMC wrapping for ``gp_mcmc`` and result dict — built from the robo_b200 classes, so the
information gain of every candidate is scored on the GPU.  Orchestration only."""
import numpy as np

from robo_b200 import kernels
from robo_b200.acquisition_functions import EI, InformationGain, MarginalizationGPMCMC
from robo_b200.initial_design import init_latin_hypercube_sampling
from robo_b200.maximizers import RandomSampling
from robo_b200.models import GaussianProcess, GaussianProcessMCMC
from robo_b200.priors import DefaultPrior
from robo_b200.solver import BayesianOptimization


def entropy_search(objective_function, lower, upper, num_iterations=30, maximizer="random", model="gp_mcmc",
                   X_init=None, Y_init=None, n_init=3, output_path=None, rng=None,
                   chain_length=200, burnin_steps=100):
    assert upper.shape[0] == lower.shape[0], "Dimension miss match"
    assert np.all(lower < upper), "Lower bound >= upper bound"
    assert n_init <= num_iterations, "Number of initial design point has to be <= than the number of iterations"
    if rng is None:
        rng = np.random.RandomState(np.random.randint(0, 10000))

    cov_amp = 2
    n_dims = lower.shape[0]
    kernel = cov_amp * kernels.Matern52Kernel(np.ones([n_dims]), ndim=n_dims)
    prior = DefaultPrior(len(kernel) + 1)
    n_hypers = 3 * len(kernel)
    if n_hypers % 2 == 1:
        n_hypers += 1

    if model == "gp":
        gp = GaussianProcess(kernel, prior=prior, rng=rng, normalize_output=False, normalize_input=True,
                             lower=lower, upper=upper)
    elif model == "gp_mcmc":
        gp = GaussianProcessMCMC(kernel, prior=prior, n_hypers=n_hypers, chain_length=chain_length,
                                 burnin_steps=burnin_steps, normalize_input=True, normalize_output=False,
                                 rng=rng, lower=lower, upper=upper)
    else:
        raise ValueError("'{}' is not a valid model on the B200 path (gp, gp_mcmc)".format(model))

    a = InformationGain(gp, lower=lower, upper=upper, sampling_acquisition=EI, rng=rng)
    acquisition_func = MarginalizationGPMCMC(a) if model == "gp_mcmc" else a

    if maximizer == "random":
        max_func = RandomSampling(acquisition_func, lower, upper, rng=rng)
    else:
        raise ValueError("'{}' is not accelerated on the B200 path; use 'random' or pass the robo_b200 "
                         "objects to the reference's own maximizers".format(maximizer))

    bo = BayesianOptimization(objective_function, lower, upper, acquisition_func, gp, max_func,
                              initial_design=init_latin_hypercube_sampling, initial_points=n_init, rng=rng,
                              output_path=output_path)
    x_best, f_min = bo.run(num_iterations, X=X_init, y=Y_init)

    results = dict()
    results["x_opt"] = x_best
    results["f_opt"] = f_min
    results["incumbents"] = [inc for inc in bo.incumbents]
    results["incumbent_values"] = [val for val in bo.incumbents_values]
    results["runtime"] = bo.runtime
    results["overhead"] = bo.time_overhead
    results["X"] = [x.tolist() for x in bo.X]
    results["y"] = [y for y in bo.y]
    return results
