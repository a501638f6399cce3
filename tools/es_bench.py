"""Entropy search on the GPU: one JSON line with the EP time, the whole update() time, compute throughput split into
the EI-equivalent scoring pass and the entropy-search extra, the CPU cost of the reference-faithful numpy restatement
(labelled as such), and the deviation from that restatement on a subset of the timed batch.

    python tools/es_bench.py [--nb 50] [--np 400] [--m 131072] [--cpu-candidates 200]

Needs a CUDA device (no CPU fallback).  Writes nothing into the tree."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import es_oracle as E            # noqa: E402
from oracle import robo_oracle as O          # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout
        name, power = [x.strip() for x in out.splitlines()[0].split(",")]
        return name, power
    except Exception:
        return "unknown", "unknown"


def timed(fn, reps):
    fn()
    t0 = time.perf_counter()
    for _ in range(reps):
        r = fn()
    return (time.perf_counter() - t0) / reps, r


def case(N, D, nb, Np, M, n_cpu, rng):
    from robo_b200 import kernels as K
    from robo_b200.acquisition_functions import EI, InformationGain
    from robo_b200.models.gaussian_process import GaussianProcess
    X, y, _, theta, noise = O.synthetic_problem(N, D, 1)
    kernel = K.Product(K.ConstantKernel(theta[0], ndim=D), K.Matern52Kernel(np.exp(theta[1:]), ndim=D))
    model = GaussianProcess(kernel, noise=noise, normalize_input=True, lower=np.zeros(D), upper=np.ones(D))
    model.train(X, y, do_optimize=False)
    zb, lmb = rng.rand(nb, D), np.log(rng.rand(nb) + 0.05)
    ig = InformationGain(model, np.zeros(D), np.ones(D), Nb=nb, Np=Np, sampling_acquisition=EI)
    h = model.gp.handle
    mu_b, V_b = model.predict(zb, full_cov=True)
    t_ep, _ = timed(lambda: h.es_joint_min(mu_b, V_b), 5)
    t_update, _ = timed(lambda: ig.update(model), 2)                 # representer sampling + EP + device prep
    ig.sample_representer_points = lambda: (setattr(ig, "zb", zb), setattr(ig, "lmb", lmb[:, None]))
    ig.update(model)
    Xs = rng.rand(M, D)
    ei = EI(model)
    t_ei, _ = timed(lambda: ei.argmax(Xs), 3)
    t_es, _ = timed(lambda: ig.argmax(Xs), 3)
    vals = ig.compute(Xs)
    # restatement on a subset, and its per-candidate CPU time
    import scipy.linalg as spla
    k = O.make_kernel("matern52", D, theta)
    st = O.gp_fit(k, X, y, noise=noise, normalize_input=True, lower=np.zeros(D), upper=np.ones(D))
    t0 = time.perf_counter()
    logP, dMu, dSig, dMuMu, _ = E.joint_min(*O.gp_predict(st, zb, full_cov=True))
    t_cpu_ep = time.perf_counter() - t0
    cf = spla.cho_factor(k.get_value(X) + (noise + 1.25e-12) * np.eye(N), lower=True)
    B = spla.cho_solve(cf, k.get_value(X, zb))
    state = dict(logP=logP, dlogPdMu=dMu, dlogPdSigma=dSig, dlogPdMudMu=dMuMu, lmb=lmb, W=E.grid(Np), sn2=noise)
    sub = Xs[:n_cpu]
    t0 = time.perf_counter()
    ref = np.concatenate([E.information_gain(state, np.clip(k.get_value(x[None], zb) - k.get_value(x[None], X) @ B,
                                                            O.EPS, np.inf),
                                             O.gp_predict(st, x[None])[1], x[None], np.zeros(D), np.ones(D))
                          for x in sub])
    t_cpu = (time.perf_counter() - t0) / n_cpu
    H = -np.sum(np.exp(logP) * (logP + lmb))
    dev = float(np.max(np.abs(vals[:n_cpu] - ref)) / max(np.max(np.abs(ref)), abs(H)))
    return {"N": N, "D": D, "Nb": nb, "Np": Np, "M": M,
            "ep_ms": 1e3 * t_ep, "update_ms": 1e3 * t_update,
            "ei_scoring_cands_per_s": M / t_ei, "es_cands_per_s": M / t_es,
            "es_extra_ms": 1e3 * (t_es - t_ei), "ei_scoring_ms": 1e3 * t_ei,
            "cpu_restatement_per_candidate_ms": 1e3 * t_cpu, "cpu_restatement_ep_ms": 1e3 * t_cpu_ep,
            "max_rel_dev_vs_restatement": dev}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nb", type=int, default=50)
    ap.add_argument("--np", type=int, default=400)
    ap.add_argument("--m", type=int, default=131072)
    ap.add_argument("--cpu-candidates", type=int, default=200)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("es_bench.py needs a CUDA device")
    name, power = gpu_info()
    rng = np.random.RandomState(0)
    res = [case(N, D, a.nb, a.np, a.m, a.cpu_candidates, rng) for N, D in ((1024, 8), (4096, 16))]
    print(json.dumps({"gpu": name, "power_limit": power, "cases": res}))


if __name__ == "__main__":
    main()
