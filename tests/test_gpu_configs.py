"""-m gpu parity on the EXACT BASELINE.json configurations (SURVEY.md section 8 "Config sizes"), through the C ABI:

  C2  N=4096  D=16              8192 candidates: mu, var 1e-10, EI 1e-8, arg-max equal to the oracle's
  C3  N=1024  D=8   M=2^20      every one of the 2^20 EI values, the arg-max index and the top-k against the oracle
  C4  N=2048  20 theta          product-of-1-D Matern-5/2 (Fabolas shape): 20 log-likelihoods, batched == sequential
                                == oracle; marginalised EI over the 20 sub-models in ONE fused call (gpk_acq_multi)
  C5  N=8192  D=32              log-likelihood 1e-10 and the full analytic gradient (H = 34) against the oracle
  a7  sample_functions          on the device path (raw posterior covariance), against the oracle's draw

The oracle (oracle/, numpy + the threaded C restatement oracle/kmat.c) is the checker; tolerances are the north_star's
(tests/product_cases.py states the denominators).  CPU time is dominated by the oracle (about two minutes in total).
"""
import os

import numpy as np
import pytest

from oracle import george_oracle as G
from oracle import robo_oracle as O
from tests.product_cases import assert_acq_close, assert_mean_close, assert_var_close, product_kernel

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    for k in ("GPK_LOADER", "GPK_CHUNK", "GPK_DIAG"):
        os.environ.pop(k, None)


def _diag_add(noise):
    return float(np.sqrt(np.float64(np.sqrt(noise)) ** 2 + 1.25e-12) ** 2)


def _fitted_handle(family, theta, X, y, noise, D):
    from robo_b200 import _lib
    h = _lib.Handle(0)
    h.set_data(X, y)
    f = product_kernel(family, theta, D).flatten()
    h.set_kernel(f["family"], f["log_amp"], f["axis"], f["group"], f["log_metric"])
    mean = float(np.mean(y))
    logdet, ll = h.fit(_diag_add(noise), mean)
    return h, logdet, ll, mean, f


# ------------------------------------------------------------------------------------------------ C2
def test_c2_exact_config_8192_candidates_against_oracle():
    """configs[1]: GP posterior N=4096, D=16, Matern-5/2 fp64: K build + Cholesky + predict + EI + arg-max."""
    from robo_b200 import _lib
    N, D, M = 4096, 16, 8192
    X, y, Xs, theta, noise = O.synthetic_problem(N, D, M)
    h, logdet, ll, mean, _ = _fitted_handle("matern52", theta, X, y, noise, D)
    eta = float(np.min(y))
    r = h.acq(Xs, _lib.ACQ_EI, eta, 0.0, want_values=True, want_moments=True)
    st = O.gp_fit(O.make_kernel("matern52", D, theta), X, y, noise=noise, normalize_input=False)
    ll_ref, logdet_ref = O.gp_loglik_terms(st)
    assert abs(ll - ll_ref) <= 1e-10 * abs(ll_ref) and abs(logdet - logdet_ref) <= 1e-10 * abs(logdet_ref)
    mu_ref, var_ref = O.gp_predict_var_only_fast(st, Xs)
    amp = float(np.exp(theta[0]))
    assert_mean_close(r["mu"], mu_ref, y)
    assert_var_close(r["var"], var_ref, amp)
    ei_ref = O.acq_ei(mu_ref, var_ref, eta)
    assert_acq_close(r["values"], ei_ref, rtol=1e-8, atol=1e-13)
    assert r["best_idx"] == int(np.argmax(ei_ref)) == int(np.argmax(r["values"]))
    assert r["n_negative"] == 0
    # the reference-faithful path (full M x M covariance, gaussian_process.py:280-286) on a slice agrees too
    mu_f, var_f = O.gp_predict(st, Xs[:256])
    assert_mean_close(r["mu"][:256], mu_f, y)
    assert_var_close(r["var"][:256], var_f, amp)
    h.close()


# ------------------------------------------------------------------------------------------------ C3
def test_c3_exact_config_2pow20_candidates_argmax_and_values():
    """configs[2]: batched EI over 2^20 candidates, N=1024, D=8 (the natural batched entry is
    robo/maximizers/random_sampling.py:38-50).  EVERY candidate is compared with the oracle."""
    from robo_b200 import _lib
    N, D, M = 1024, 8, 2 ** 20
    X, y, Xs, theta, noise = O.synthetic_problem(N, D, M)
    h, logdet, ll, mean, _ = _fitted_handle("matern52", theta, X, y, noise, D)
    eta = float(np.min(y))
    r = h.acq(Xs, _lib.ACQ_EI, eta, 0.0, want_values=True, want_moments=True)      # pageable host batch, 67 MB
    st = O.gp_fit(O.make_kernel("matern52", D, theta), X, y, noise=noise, normalize_input=False)
    mu_ref, var_ref = O.gp_predict_var_only_fast(st, Xs)
    amp = float(np.exp(theta[0]))
    assert_mean_close(r["mu"], mu_ref, y)
    assert_var_close(r["var"], var_ref, amp)
    ei_ref = O.acq_ei(mu_ref, var_ref, eta)
    assert_acq_close(r["values"], ei_ref, rtol=1e-8, atol=1e-13)
    best_ref = int(np.argmax(ei_ref))
    assert r["best_idx"] == best_ref == int(np.argmax(r["values"]))
    assert abs(r["best_val"] - ei_ref[best_ref]) <= 1e-8 * ei_ref[best_ref]
    top_ref = np.argsort(-ei_ref, kind="stable")[:64]
    top_gpu = np.argsort(-r["values"], kind="stable")[:64]
    # top-k as a set and in order wherever neighbouring oracle values differ by more than the tolerance
    assert set(top_ref.tolist()) == set(top_gpu.tolist())
    gaps = np.abs(np.diff(ei_ref[top_ref])) > 4e-8 * ei_ref[top_ref][:-1]
    assert np.array_equal(top_ref[:-1][gaps], top_gpu[:-1][gaps])
    # arg-max only (values never leave the device) and a different chunking give the same winner
    r2 = h.acq(Xs, _lib.ACQ_EI, eta, 0.0, want_values=False)
    assert r2["best_idx"] == best_ref and r2["best_val"] == r["best_val"]
    h.set_option("chunk", 65536)
    r3 = h.acq(Xs, _lib.ACQ_EI, eta, 0.0, want_values=False)
    assert r3["best_idx"] == best_ref and r3["best_val"] == r["best_val"]
    # the same maximisation with the candidates generated on the device (Philox by global index): the candidate the
    # device reports is the oracle's arg-max over the oracle's restatement of the generator
    lower, upper = np.zeros(D), np.ones(D)
    inc = X[np.argmin(y)]
    n_uniform = int(M * 0.7)
    bx, bv, bi = h.maximize_random(1234567, 0, M, n_uniform, lower, upper, inc, 0.1, _lib.ACQ_EI, eta, 0.0)
    C = h.generate_candidates(1234567, 0, M, n_uniform, lower, upper, inc, 0.1)
    for a, b in ((0, 2048), (n_uniform - 1024, n_uniform + 1024), (M - 2048, M)):
        ref_c = O.generate_candidates(1234567, a, b - a, n_uniform, lower, upper, inc, 0.1)
        nu_loc = max(0, min(b, n_uniform) - a)
        np.testing.assert_array_equal(C[a:a + nu_loc], ref_c[:nu_loc])          # uniform part: bit-exact
        np.testing.assert_allclose(C[a + nu_loc:b], ref_c[nu_loc:], rtol=0, atol=1e-13)   # Gaussian part: to rounding
    mu_c, var_c = O.gp_predict_var_only_fast(st, C)
    ei_c = O.acq_ei(mu_c, var_c, eta)
    assert bi == int(np.argmax(ei_c))
    np.testing.assert_array_equal(bx, C[bi])
    assert abs(bv - ei_c[bi]) <= 1e-8 * ei_c[bi]
    h.close()


# ------------------------------------------------------------------------------------------------ C4
def _c4_problem():
    """SURVEY.md 8d C4: N=2048, 2 configuration columns + 1 environment column s mapped through (1-s)^2
    (fabolas_gp.py:122-126), kernel = c * Matern52_1D(x0) * Matern52_1D(x1) * Matern52_1D(env column); 20 theta drawn
    like EnvPrior.sample_from_prior (env_priors.py:56-79: amplitude lognormal(-2, 1) used as the log-parameter,
    log-metrics uniform on [-10, 2], noise from the horseshoe sampler base_prior.py:213-216), RandomState(7)."""
    rng = np.random.RandomState(7)
    N, D = 2048, 3
    X = rng.rand(N, D)
    X[:, 2] = (1.0 - X[:, 2]) ** 2
    y = np.sinc(X[:, :2] * 10 - 5).sum(axis=1) * (0.5 + X[:, 2]) + 0.01 * rng.randn(N)
    thetas = np.zeros((20, D + 2))
    thetas[:, 0] = rng.lognormal(mean=-2, sigma=1.0, size=20)
    thetas[:, 1:D + 1] = rng.uniform(-10, 2, size=(20, D))
    lamda = np.abs(rng.standard_cauchy(size=20))
    thetas[:, -1] = np.log(np.abs(rng.randn() * lamda * 0.001))
    return X, y, thetas


def _oracle_prod1d(theta, D):
    k = G.ConstantKernel(theta[0], ndim=D)
    for d in range(D):
        k = G.Product(k, G.Matern52Kernel(np.exp(theta[1 + d:2 + d]), ndim=D, axes=d))
    return k


def test_c4_exact_config_20_thetas_n2048_loglik_and_marginalised_ei():
    """configs[3]: GP-MCMC with 20 hyper-parameter samples at N=2048 (GaussianProcessMCMC.loglikelihood,
    gaussian_process_mcmc.py:168-202; MarginalizationGPMCMC.compute, marginalization.py:115-121)."""
    from robo_b200 import _lib
    from robo_b200 import kernels as K
    from robo_b200.acquisition_functions import EI, MarginalizationGPMCMC
    from robo_b200.models import GaussianProcessMCMC
    from robo_b200.models.gaussian_process import GaussianProcess
    from robo_b200.models.gaussian_process_mcmc import _LikelihoodPool
    X, y, thetas = _c4_problem()
    N, D = X.shape
    kernel = product_kernel("prod1d_matern52", thetas[0, :-1], D)
    model = GaussianProcessMCMC(kernel, prior=None, n_hypers=20, chain_length=1, burnin_steps=1, normalize_input=False,
                                normalize_output=False, rng=np.random.RandomState(1))
    # log-likelihoods: one-at-a-time, and batched in half-ensembles of 10 concurrent handles (as emcee's stretch move
    # evaluates them), against the oracle
    model.X, model.y, model.mean = X, y, np.mean(y)
    from robo_b200.device_gp import DeviceGP
    model.gp = DeviceGP(model.kernel, mean=model.mean)
    model.gp.set_data(X, y)
    seq = np.array([model.loglikelihood(t) for t in thetas])
    model._pool = _LikelihoodPool(kernel, X, y, model.mean, 10)
    bat = np.concatenate([model.loglikelihood_batch(thetas[:10]), model.loglikelihood_batch(thetas[10:])])
    model._pool.close()
    model._pool = None
    np.testing.assert_array_equal(seq, bat)
    refs = []
    for t in thetas:
        st = O.gp_fit(_oracle_prod1d(t[:-1], D), X, y, noise=float(np.exp(t[-1])), normalize_input=False)
        refs.append(-O.gp_nll(st, t))
    refs = np.array(refs)
    fin = refs != -1e25
    assert fin.sum() >= 15
    assert np.all(seq[~fin] == -np.inf)
    assert np.max(np.abs(seq[fin] - refs[fin]) / np.abs(refs[fin])) <= 1e-10
    # the 20 sub-models (train(do_optimize=False) per sample, gaussian_process_mcmc.py:149-164) and the marginalised EI
    good = thetas[fin]
    model.hypers = good
    model.models = []
    for t in good:
        sub = GaussianProcess(product_kernel("prod1d_matern52", t[:-1], D), noise=float(np.exp(t[-1])),
                              normalize_input=False, normalize_output=False, rng=np.random.RandomState(0))
        sub.train(X, y, do_optimize=False)
        model.models.append(sub)
    model.is_trained = True
    Xc = np.random.RandomState(11).rand(500, D)
    acq = MarginalizationGPMCMC(EI(model))
    assert acq._fused_spec() is not None, "the fused multi-model path must be the one that runs"
    a = acq.compute(Xc)
    per_model, mus, vs = [], [], []
    for t in good:
        st = O.gp_fit(_oracle_prod1d(t[:-1], D), X, y, noise=float(np.exp(t[-1])), normalize_input=False)
        m_ref, v_ref = O.gp_predict_var_only_fast(st, Xc)
        mus.append(m_ref)
        vs.append(v_ref)
        per_model.append(O.acq_ei(m_ref, v_ref, float(np.min(y))))
    ref = O.marginalised_acquisition(np.array(per_model))
    assert_acq_close(a, ref, rtol=1e-8, atol=1e-13)
    assert acq.argmax(Xc) == int(np.argmax(ref))
    # fused == the reference's loop over estimators (per-model compute, values through the host)
    loop = np.mean([est.compute(Xc) for est in acq.estimators], axis=0)
    np.testing.assert_allclose(a, loop, rtol=1e-13, atol=1e-300)
    # mixture moments (gaussian_process_mcmc.py:235-247) through the same fused call
    m, v = model.predict(Xc)
    m_ref, v_ref = O.mcmc_mixture_moments(np.array(mus), np.array(vs))
    assert_mean_close(m, m_ref, y)
    assert np.max(np.abs(v - v_ref) / np.maximum(v_ref, 1e-6 * np.exp(good[:, 0]).max())) <= 1e-10


# ------------------------------------------------------------------------------------------------ C5
def test_c5_exact_config_n8192_d32_loglik_and_gradient():
    """configs[4]: marginal log-likelihood + gradient at N=8192, D=32 (gaussian_process.py:129-191, gradient with the
    corrected noise term).  The oracle evaluates the einsum of :186 without the 18 GB (N, N, H) array."""
    from robo_b200 import _lib
    N, D = 8192, 32
    X, y, _, theta, noise = O.synthetic_problem(N, D, 1)
    theta = theta + 0.05 * np.random.RandomState(5).randn(D + 1)
    h, logdet, ll, mean, f = _fitted_handle("matern52", theta, X, y, noise, D)
    g = h.nll_grad(noise, D)
    st = O.gp_fit(O.make_kernel("matern52", D, theta), X, y, noise=noise, normalize_input=False)
    ll_ref, logdet_ref = O.gp_loglik_terms(st)
    assert abs(ll - ll_ref) <= 1e-10 * abs(ll_ref)
    assert abs(logdet - logdet_ref) <= 1e-10 * abs(logdet_ref)
    g_ref = O.gp_grad_nll_terms_fast(st, np.append(theta, np.log(noise)), recompute=False)
    assert g.shape == g_ref.shape == (D + 2,)
    assert np.max(np.abs(g - g_ref) / np.maximum(1.0, np.abs(g_ref))) <= 1e-8
    # and against central differences of the device's own nll for two components
    def nll_at(th):
        ff = product_kernel("matern52", th, D).flatten()
        h.set_kernel(ff["family"], ff["log_amp"], ff["axis"], ff["group"], ff["log_metric"])
        return -h.fit(_diag_add(noise), mean)[1]
    for p in (0, 17):
        tp, tm = theta.copy(), theta.copy()
        tp[p] += 1e-5
        tm[p] -= 1e-5
        fd = (nll_at(tp) - nll_at(tm)) / 2e-5
        assert abs(g[p] - fd) <= 1e-5 * max(1.0, abs(fd))
    h.close()


# ------------------------------------------------------------------------------------------------ a7
def test_sample_functions_on_device_path_uses_raw_covariance():
    """GaussianProcess.sample_functions (gaussian_process.py:298-332): george's sample_conditional draws from the RAW
    posterior covariance; only predict() clips.  Negative posterior correlations must survive."""
    from robo_b200.models.gaussian_process import GaussianProcess
    rng = np.random.RandomState(3)
    N, D, M = 40, 2, 12
    X = rng.rand(N, D)
    y = np.sinc(X * 10 - 5).sum(axis=1)
    Xt = rng.rand(M, D)
    theta = np.array([0.1, -1.5, -1.0])
    for norm_out in (False, True):
        model = GaussianProcess(product_kernel("matern52", theta, D), noise=1e-3, normalize_input=True,
                                normalize_output=norm_out, lower=np.zeros(D), upper=np.ones(D),
                                rng=np.random.RandomState(0))
        model.train(X, y, do_optimize=False)
        st = O.gp_fit(O.make_kernel("matern52", D, theta), X, y, noise=1e-3, normalize_input=True,
                      normalize_output=norm_out, lower=np.zeros(D), upper=np.ones(D))
        Xn, _, _ = O.zero_one_normalization(Xt, st["lower"], st["upper"])
        mu_ref, cov_ref = st["gp"].predict(st["y"], Xn)                 # raw george moments (normalised outputs)
        if norm_out:
            mu_u, cov_u = mu_ref * st["y_std"] + st["y_mean"], cov_ref * st["y_std"] ** 2
        else:
            mu_u, cov_u = mu_ref, cov_ref
        assert cov_ref.min() < -1e-8, "the test needs negative posterior covariances"
        mu, cov = model.gp.posterior_cov(Xt)
        assert_mean_close(mu, mu_u, y)
        scale = np.sqrt(np.outer(np.diag(cov_u), np.diag(cov_u)))
        assert np.max(np.abs(cov - cov_u) / np.maximum(scale, 1e-6 * np.exp(theta[0]))) <= 1e-9
        assert cov.min() < 0
        # predict(full_cov=True) keeps the reference's clip
        _, cov_clip = model.predict(Xt, full_cov=True)
        assert cov_clip.min() >= np.finfo(float).eps
        # the draw itself is numpy's, like george's (np.random.multivariate_normal on the raw moments, global RNG),
        # followed by the reference's output un-normalisation (:326-327); with the same seed the samples are the
        # ones numpy makes from the device moments, and they agree with the draw from the oracle's moments
        np.random.seed(99)
        funcs = model.sample_functions(Xt, n_funcs=5)
        np.random.seed(99)
        same = np.random.multivariate_normal(mu, cov, 5)
        assert funcs.shape == (5, M)
        np.testing.assert_array_equal(funcs, same)
        np.random.seed(99)
        ref = np.random.multivariate_normal(mu_ref, cov_ref, size=5)
        if norm_out:
            ref = ref * st["y_std"] + st["y_mean"]
        # SVD-based draw: continuous in (mu, cov) for separated singular values; tolerance reflects that only
        assert np.max(np.abs(funcs - ref)) <= 1e-4 * np.abs(ref).max()
        np.random.seed(5)
        one = model.sample_functions(Xt, n_funcs=1)
        assert one.shape == (1, M)


def test_bench_dump_outputs_of_the_last_timed_step(tmp_path):
    """bench.py --dump-outputs: the merged arg-max of the device path and the EI values of the e2e path, as float64
    arrays that agree with each other and with the JSON line."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    m = 4096
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "2", "--warmup", "1", "--m", str(m),
                          "--no-c3", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["argmax_check"] is True
    best = np.load(os.path.join(str(tmp_path), "argmax.npy"))
    ei = np.load(os.path.join(str(tmp_path), "ei_values.npy"))
    assert best.dtype == ei.dtype == np.float64 and best.shape == (2,) and ei.shape == (m,)
    assert best[0] == line["argmax"]["merged"]["value"] and int(best[1]) == line["argmax"]["merged"]["index"]
    assert int(np.argmax(ei)) == int(best[1]) and abs(ei[int(best[1])] - best[0]) <= 1e-12 * abs(best[0])
