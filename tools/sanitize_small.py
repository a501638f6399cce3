"""Small end-to-end pass over every kernel (all staging variants) for compute-sanitizer runs."""
import os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from robo_b200 import _lib
from robo_b200 import kernels as K

rng = np.random.RandomState(0)
N, D, M = 300, 3, 700
X, y, Xs = rng.rand(N, D), rng.rand(N), rng.rand(M, D)
f = K.Product(K.ConstantKernel(0.1, ndim=D), K.Matern52Kernel(np.array([0.3, 0.5, 0.8]), ndim=D)).flatten()
for loader, diag in ((2, 4), (1, 3), (0, 2)):
    h = _lib.Handle(0)
    h.set_option("loader", loader)
    h.set_option("diag", diag)
    h.set_option("chunk", 256)
    h.set_data(X, y)
    h.set_input_bounds(np.zeros(D), np.ones(D))
    h.set_output_transform(True, 0.5, 2.0)
    h.set_kernel(f["family"], f["log_amp"], f["axis"], f["group"], f["log_metric"])
    print("loader", loader, "fit", h.fit(1e-3 + 1.25e-12, float(y.mean())))
    r = h.acq(Xs, _lib.ACQ_EI, float(y.min()), 0.0, want_values=True, want_moments=True)
    print(" acq best", r["best_idx"], r["best_val"], "neg", r["n_negative"])
    for kind in (_lib.ACQ_LOG_EI, _lib.ACQ_PI, _lib.ACQ_LCB):
        h.acq(Xs[:300], kind, float(y.min()), 0.1)
    mu, cov = h.predict_cov(Xs[:150])
    g = h.nll_grad(1e-3, D)
    pg = h.predict_grad(Xs[:5], _lib.ACQ_EI, float(y.min()), 0.0)
    bx, bv, bi = h.maximize_random(7, 0, 1000, 700, np.zeros(D), np.ones(D), X[0], 0.1, _lib.ACQ_EI, float(y.min()), 0.0)
    km = h.kernel_matrix(Xs[:40], X[:50])
    print(" cov", cov.shape, "grad", np.round(g, 3), "dmu", pg["dmu"].shape, "max idx", bi, km.shape)
    # incremental refit: 300 -> 310 rows inside the last 128-row block (NP = 384)
    X2, y2 = np.vstack([X, rng.rand(10, D)]), np.concatenate([y, rng.rand(10)])
    print(" append", h.fit_append(X2, y2, 1e-3 + 1.25e-12, float(y2.mean())), h.predict(Xs[:64])[0][:2])
    h.close()
# round-2 kernels: int8 contraction (fused and unfused digit builders, several chunks), persistent fp64 contraction,
# split chain replayed from a CUDA graph, depth-2 trailing updates, fused multi-model scoring, raw posterior covariance
Xb = rng.rand(2304, D)
hs = []
for opts in ({"ozaki": 1, "ozfused": 1}, {"ozaki": 1, "ozfused": 0}, {"ozaki": 0, "persist": 1},
             {"ozaki": 0, "chainsplit": 1, "graph": 1, "depth2": 1},
             # int8 contraction variants: one pass / CTA pair / two passes / persistent walk / resident builder + dependent launch
             {"ozaki": 1, "oztile": 64, "ozpair": 0}, {"ozaki": 1, "oztile": 64, "ozpair": 1}, {"ozaki": 1, "oztile": 128, "ozpair": 0},
             {"ozaki": 1, "oztile": 64, "ozpair": 0, "ozpersist": 1}, {"ozaki": 1, "oztile": 64, "ozpair": 1, "ozpersist": 1},
             {"ozaki": 1, "ozpersist": 1}, {"ozaki": 1, "ozpdl": 1}):
    h = _lib.Handle(0)
    for k, v in opts.items():
        h.set_option(k, v)
    h.set_option("chunk", 1024)
    Xt, yt = (X, y) if len(hs) < 4 else (X[:250], y[:250])       # 250 rows = 2 row blocks: the CTA-pair kernels apply
    h.set_data(Xt, yt)
    h.set_kernel(f["family"], f["log_amp"], f["axis"], f["group"], f["log_metric"])
    for _ in range(2):
        ll = h.fit(1e-3 + 1.25e-12, float(yt.mean()))
    r = h.acq(Xb, _lib.ACQ_EI, float(y.min()), 0.0, want_values=True, want_moments=True)
    t = h.timings()
    print(opts, "fit", ll, "best", r["best_idx"], "oz launches", t["launches_ozaki"], "variant", t["ozaki_kernel_variant"])
    mu, cov = h.posterior_cov(Xs[:100])
    hs.append(h)
rm = _lib.acq_multi(hs[:3], Xs[:300], 0, _lib.ACQ_EI, [float(y.min())] * 3, 0.0, want_argmax=True)
rp = _lib.acq_multi(hs[:3], Xs[:300], 1)
print("multi", rm["best_idx"], rp["var"][:2])
for h in hs:
    h.close()
h = _lib.moments_handle()
print(h.acq_moments(rng.randn(100), rng.rand(100) + 0.1, _lib.ACQ_LOG_EI, 0.0, 0.0)[0][:3])
print(h.reduce_models(rng.rand(4, 50), rng.rand(4, 50))[1][:3])
# entropy search: EP (gpk_es_ep_kernel, gpk_es_renorm_kernel), per-update prep (gpk_es_pack_kernel, gpk_es_grid_kernel,
# gpk_es_gemm_kernel) and two scoring chunks (gpk_es_gemm_kernel, gpk_es_score_kernel)
h = _lib.Handle(0)
h.set_option("chunk", 256)
h.set_data(X, y)
h.set_input_bounds(np.zeros(D), np.ones(D))
h.set_output_transform(True, 0.5, 2.0)
h.set_kernel(f["family"], f["log_amp"], f["axis"], f["group"], f["log_metric"])
h.fit(1e-3 + 1.25e-12, float(y.mean()))
print("es logP", h.es_update(rng.rand(20, D), np.log(rng.rand(20) + 0.1), 40, 1e-3)[:3])
r = h.es_compute(Xs[:400], np.zeros(D), np.ones(D))
print("es best", r["best_idx"], h.es_joint_min(np.zeros(5), np.eye(5))["sweeps"])
h.close()
print("done")
