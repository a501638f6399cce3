#!/usr/bin/env python
"""bench.py — EI evaluations / second + GP fit time on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--m M] [--dump-outputs DIR]

Workload (BASELINE.json configs[1] / SURVEY.md section 8d "C2"): GP posterior with N = 4096
training points, D = 16, amp * ARD Matern-5/2, fp64, synthetic seeded data; one *step* scores a
batch of M candidates per GPU (predict -> EI -> arg-max) against the fitted model.

Our arm (default)
  value   candidates scored per second, candidates resident in HBM (gpk_acq_argmax_sharded_dev: scoring, NCCL
          exchange and merge on the handle's stream, no host synchronisation inside the timed region), CUDA events on
          the launching stream, max over ranks.
  e2e     the same through the RoBO-facing classes: EI(model).compute(X) on a PAGEABLE numpy array with the values
          returned to the host + numpy arg-max (+ the 16-byte exchange at N > 1) — what
          robo/maximizers/random_sampling.py:48-50 does.  `e2e_pinned_argmax_only` keeps the round-1 figure
          (pinned host buffer, arg-max only) beside it.
  multi-GPU  one process per GPU (torchrun); ALL ranks hold the same candidate list of world x M rows, rank r scores
          the contiguous shard gpk_shard_bounds gives it (weak scaling), the fit state is replicated, and the arg-max
          is exchanged by libgpk.so itself (NCCL bound behind the C ABI; torch.distributed only launches the processes,
          ships the 128-byte NCCL id and reduces the timings).  Outside the timed region rank 0 scores the FULL list on
          one GPU and the merged (value, global index) must equal that arg-max: "argmax_check".
  --dump-outputs DIR  rank 0 writes what the timed paths returned in their last step, float64: DIR/argmax.npy = the
          merged (EI value, global candidate index) of the device path, DIR/ei_values.npy = the EI values of the rank's
          shard that EI(model).compute returned on the e2e path.  Inputs are seeded, so two builds run with the same
          arguments can be compared output for output.
  configs.c3  BASELINE.json configs[2] (2^20 candidates, N = 1024, D = 8) STRONG scaling: the 2^20 candidates are
          split over the ranks; wall time of one whole maximisation including the replicated fit, from a pageable
          host array and from on-device Philox candidates.

Reference arm (--impl reference): the reference's CPU implementation of the same path.  george is an un-vendored
third-party dependency that cannot be installed here (SURVEY.md section 0), so the arm runs the oracle port
(oracle/robo_oracle.py: reference-faithful predict with the full M x M covariance, then EI —
gaussian_process.py:280-294 + ei.py:65-78) on the host cores with all BLAS threads, in the reference's own batch size
of 500 candidates (random_sampling.py:9).  Both arms also report `cpu_baseline_optimised`: variance-only predict
through one triangular solve (no M x M) with a threaded K* build, i.e. what a sane CPU implementation would do.
"""
import argparse
import csv
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_TRAIN, DIM = 4096, 16
METRIC = "EI evals/sec (GP N=4096, D=16, fp64)"
FP64_PEAK_TFLOPS = 37.0      # SURVEY.md section 8d "P64": B200 FP64 / FP64-tensor datasheet (296 TF per 8-GPU HGX)
VARGEMM_NCU_CSV = os.path.join("profiles", "r02_vargemm_fp64_ncu_full_raw.csv")
OZ_NCU_CSV = os.path.join("profiles", "r02_oz_pair2_ncu_full_raw.csv")
OZ_KERNELS = {1: "gpk_oz_vargemm_kernel (128 x 64 tile per CTA, one pass)", 2: "gpk_oz_pair_kernel (CTA pair, 256 x 64, one pass)",
              3: "gpk_oz2_vargemm_kernel (128 x 128 per CTA, two passes)",
              4: "gpk_oz_pair2_kernel (CTA pair, tcgen05 cta_group::2: 256 x 128 per pair, two passes)"}


def train_problem(n=N_TRAIN, d=DIM):
    """SURVEY.md section 8d synthetic inputs (restated here so the product arm does not import oracle/)."""
    rng = np.random.RandomState(1234)
    X = rng.rand(n, d)
    y = np.sinc(X * 10 - 5).sum(axis=1) + 0.01 * rng.randn(n)
    theta = np.concatenate(([0.0], np.full(d, np.log(d / 4.0))))
    return X, y, theta, 1e-3


def candidates(m, d=DIM, seed=4321):
    return np.random.RandomState(seed).rand(m, d)


def problem(m, seed_cand=4321):
    X, y, theta, noise = train_problem()
    return X, y, candidates(m, DIM, seed_cand), theta, noise


def diag_add_of(noise):
    return float(np.sqrt(np.float64(np.sqrt(noise)) ** 2 + 1.25e-12) ** 2)


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.lines, self.proc, self.gpu, self.t_timed = [], None, gpu_index, None

    def mark_timed_region(self):
        self.t_timed = time.time()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        timed = [ln for t, ln in self.lines if self.t_timed is None or t >= self.t_timed]
        for ln in (timed if timed else [ln for _, ln in self.lines]):
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------------------------
# CPU arms (the only place bench.py executes oracle/)
# ---------------------------------------------------------------------------------------------------------------
def host_threads():
    """(os.cpu_count(), size of the BLAS pool scipy.linalg uses) — stated separately, SURVEY.md 8d."""
    import threadpoolctl
    cpus = os.cpu_count()
    blas = None
    try:
        import scipy.linalg  # noqa: F401  (loads scipy's own OpenBLAS)
        for p in threadpoolctl.threadpool_info():
            if p.get("user_api") == "blas" and "scipy" in os.path.basename(os.path.dirname(p.get("filepath", ""))):
                blas = p.get("num_threads")
        if blas is None:
            blas = max(p.get("num_threads", 1) for p in threadpoolctl.threadpool_info() if p.get("user_api") == "blas")
    except Exception:
        blas = cpus
    return cpus, int(blas)


def cpu_reference_rate(n_batches, batch=500):
    """Reference-faithful path on the host cores via the oracle port: predict (full M x M covariance) + EI per batch
    of 500.  Returns the fit split into the numpy K build (george's own K build is single-threaded C++ and cannot be
    timed here) and LAPACK (Cholesky + solve), and the per-batch times."""
    import scipy.linalg as spla
    from oracle import robo_oracle as O
    X, y, Xs, theta, noise = problem(batch * max(n_batches, 1))
    kernel = O.make_kernel("matern52", DIM, theta)
    t0 = time.perf_counter()
    K = kernel.get_value(X)
    kbuild_s = time.perf_counter() - t0
    K[np.diag_indices_from(K)] += diag_add_of(noise)
    t0 = time.perf_counter()
    L = spla.cholesky(K, lower=True, overwrite_a=True, check_finite=False)
    spla.cho_solve((L, True), y - y.mean(), check_finite=False)
    lapack_s = time.perf_counter() - t0
    del K, L
    t0 = time.perf_counter()
    st = O.gp_fit(kernel, X, y, noise=noise, normalize_input=False)
    fit_s = time.perf_counter() - t0
    eta = O.gp_get_incumbent(st)[1]
    times = []
    for b in range(n_batches):
        t0 = time.perf_counter()
        m, v = O.gp_predict(st, Xs[b * batch:(b + 1) * batch])
        ei = O.acq_ei(m, v, eta)
        int(np.argmax(ei))
        times.append(time.perf_counter() - t0)
    return dict(fit_s=fit_s, kbuild_numpy_s=kbuild_s, lapack_s=lapack_s, times=times, state=st)


def cpu_optimised_rate(st, m=8192, reps=2):
    """What a sane CPU implementation does (BASELINE.md section 3 row ii): variance only through ONE triangular solve
    (no M x M covariance), K* from the threaded C restatement, all cores."""
    from oracle import robo_oracle as O
    X, y, theta, noise = train_problem()
    Xs = candidates(m)
    eta = O.gp_get_incumbent(st)[1]
    t0 = time.perf_counter()
    O.kmat_fast(st["gp"].kernel, X, X)
    kbuild_c_s = time.perf_counter() - t0
    best = None
    for _ in range(reps):
        t0 = time.perf_counter()
        mu, var = O.gp_predict_var_only_fast(st, Xs)
        ei = O.acq_ei(mu, var, eta)
        int(np.argmax(ei))
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return dict(value=m / best, seconds=best, m=m, kbuild_threaded_c_s=kbuild_c_s)


def cpu_rows(n_batches, warm):
    """Both CPU rows + the thread counts, as JSON-ready dicts."""
    import threadpoolctl
    cpus, blas = host_threads()
    with threadpoolctl.threadpool_limits(limits=cpus):
        cpus, blas = host_threads()
        ref = cpu_reference_rate(n_batches)
        timed = ref["times"][warm:]
        total = float(np.sum(timed))
        opt = cpu_optimised_rate(ref["state"])
    faithful = {"value": 500 * len(timed) / total, "unit": "EI evals/s", "cores": blas, "host_cpus": cpus,
                "blas_threads_scipy": blas, "kind": "port",
                "fit_ms": 1e3 * ref["fit_s"], "fit_kbuild_numpy_ms": 1e3 * ref["kbuild_numpy_s"],
                "fit_lapack_cholesky_solve_ms": 1e3 * ref["lapack_s"],
                "sample": "%d batches of 500 candidates (reference batch size random_sampling.py:9, full M x M covariance "
                          "per batch as gaussian_process.py:280-286), N=4096 D=16, oracle port of "
                          "gaussian_process.py:280-294 + ei.py:65-78; fit not included" % len(timed)}
    optimised = {"value": opt["value"], "unit": "EI evals/s", "cores": blas, "host_cpus": cpus, "kind": "port",
                 "fit_kbuild_threaded_c_ms": 1e3 * opt["kbuild_threaded_c_s"],
                 "fit_lapack_cholesky_solve_ms": 1e3 * ref["lapack_s"],
                 "sample": "%d candidates in one batch, variance-only predict (one triangular solve, no M x M "
                           "covariance: oracle.gp_predict_var_only_fast), K* by the threaded C restatement "
                           "(oracle/kmat.c, OpenMP), EI + arg-max; best of 2" % opt["m"]}
    return faithful, optimised, total, timed


def run_reference(args, rank):
    if rank != 0:
        return
    faithful, optimised, total, timed = cpu_rows(args.warmup + args.steps, args.warmup)
    value = faithful["value"]
    faithful = dict(faithful, sample=faithful["sample"])
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "EI evals/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(timed),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "GP posterior N=4096 D=16 Matern52 fp64: predict + EI + argmax (configs[1])",
                   "n_train": N_TRAIN, "dim": DIM, "candidates_per_step": 500,
                   "note": "reference CPU path (oracle port of gaussian_process.py:280-294 + ei.py:65-78, full "
                           "M x M covariance per 500-candidate batch as random_sampling.py:9); george itself is "
                           "not installable here"},
        "cpu_baseline": faithful, "cpu_baseline_optimised": optimised,
        "e2e": {"value": value, "unit": "EI evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "fit_ms": faithful["fit_ms"], "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------
# product arm
# ---------------------------------------------------------------------------------------------------------------
def ncu_dram_bytes(path, kernel_substring):
    """dram__bytes_read.sum + dram__bytes_write.sum (bytes) of the first launch of `kernel_substring` in a committed
    `ncu --page raw --csv` export (row 0 names, row 1 units)."""
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    try:
        with open(os.path.join(ROOT, path), newline="") as f:
            rows = list(csv.reader(f))
        names, units = rows[0], rows[1]
        ik = names.index("Kernel Name")
        ir, iw = names.index("dram__bytes_read.sum"), names.index("dram__bytes_write.sum")
        for r in rows[2:]:
            if kernel_substring in r[ik]:
                return float(r[ir]) * unit[units[ir]] + float(r[iw]) * unit[units[iw]]
    except Exception:
        return None
    return None


def measure_dgemm_tflops(torch, dev):
    """cuBLAS DGEMM on this GPU as the practical fp64 tensor-pipe reference (reported, not on our path)."""
    n = 8192
    a = torch.randn(n, n, dtype=torch.float64, device=dev)
    b = torch.randn(n, n, dtype=torch.float64, device=dev)
    torch.matmul(a, b)
    torch.cuda.synchronize()
    best = 0.0
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize()
        best = max(best, 2.0 * n ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    del a, b
    return best


def unpack_pair(t):
    import torch
    host = t.detach().cpu()
    return float(host[0]), int(host[1:].view(torch.int64)[0])


def c3_block(torch, dist, _lib, K, rank, world, local_rank, stream, barrier, max_over_ranks, reps=5, warm=2):
    """BASELINE.json configs[2]: batched EI over 2^20 candidates, N=1024, D=8, split over `world` GPUs (STRONG scaling).
    One maximisation = replicated fit (K build + Cholesky + L^-1 on every rank, no communication) + scoring of the rank's
    shard + the NCCL exchange + D2H of the winner; timed as wall time (blocking C-ABI call, barrier + synchronize on both
    sides, max over ranks)."""
    from robo_b200.distributed import init_comm
    N3, D3, M3 = 1024, 8, 2 ** 20
    X, y, theta, noise = train_problem(N3, D3)
    Xs_all = candidates(M3, D3)                              # pageable numpy array, identical on every rank
    h = _lib.Handle(local_rank)
    h.set_stream(stream.cuda_stream)
    h.set_data(X, y)
    f = K.Product(K.ConstantKernel(theta[0], ndim=D3), K.Matern52Kernel(np.exp(theta[1:]), ndim=D3)).flatten()
    dadd, mean, eta = diag_add_of(noise), float(np.mean(y)), float(np.min(y))
    init_comm(h, rank, world)
    lower, upper, inc = np.zeros(D3), np.ones(D3), X[int(np.argmin(y))]
    n_uniform = int(M3 * 0.7)

    def refit():
        h.set_kernel(f["family"], f["log_amp"], f["axis"], f["group"], f["log_metric"])    # invalidates the factor
        h.fit(dadd, mean)

    def from_host():
        refit()
        return h.acq_argmax_sharded(Xs_all, _lib.ACQ_EI, eta, 0.0)

    def from_device():
        refit()
        _, v, i = h.maximize_random_sharded(20260923, M3, n_uniform, lower, upper, inc, 0.1, _lib.ACQ_EI, eta, 0.0)
        return v, i

    out = {}
    for name, fn in (("host_pageable", from_host), ("device_philox", from_device)):
        for _ in range(warm):
            res = fn()
        walls, parts = [], []
        for _ in range(reps):
            barrier()
            t0 = time.perf_counter()
            res = fn()
            torch.cuda.synchronize()
            walls.append(max_over_ranks(1e3 * (time.perf_counter() - t0)))
            t = h.timings()
            parts.append((t["fit_ms"], t["linv_ms"], t["score_ms"]))
        wall = float(np.median(walls))
        out[name] = {"wall_ms": wall, "wall_ms_min": float(np.min(walls)), "ei_per_s": M3 / (wall * 1e-3),
                     "rank0_fit_ms": float(np.median([p[0] for p in parts])),
                     "rank0_linv_ms": float(np.median([p[1] for p in parts])),
                     "rank0_score_ms_last_call": float(np.median([p[2] for p in parts])),
                     "argmax": {"value": res[0], "index": int(res[1])}}
    # answers, outside the timed region: rank 0 alone over the full list
    check = None
    if rank == 0:
        g = _lib.Handle(local_rank)
        g.set_data(X, y)
        g.set_kernel(f["family"], f["log_amp"], f["axis"], f["group"], f["log_metric"])
        g.fit(dadd, mean)
        r = g.acq(Xs_all, _lib.ACQ_EI, eta, 0.0, want_values=False)
        _, v1, i1 = g.maximize_random(20260923, 0, M3, n_uniform, lower, upper, inc, 0.1, _lib.ACQ_EI, eta, 0.0)
        check = bool((r["best_val"], r["best_idx"]) == (out["host_pageable"]["argmax"]["value"],
                                                        out["host_pageable"]["argmax"]["index"])
                     and (v1, i1) == (out["device_philox"]["argmax"]["value"], out["device_philox"]["argmax"]["index"]))
        g.close()
    h.comm_destroy()
    h.close()
    f_ei = N3 ** 2 + N3 * (3 * D3 + 40) + 2 * N3          # SURVEY.md 8d: 1.116 MFLOP per EI evaluation
    roof = FP64_PEAK_TFLOPS * 1e12 / f_ei                  # 33.1 M EI/s per GPU
    for v in out.values():
        v["frac_of_roofline_all_gpus"] = v["ei_per_s"] / (roof * world)
    return {"workload": "configs[2]: EI over 2^20 candidates, N=1024, D=8, sharded over %d GPU(s): STRONG scaling; one "
                        "maximise = replicated fit + shard scoring + NCCL arg-max exchange + D2H of the winner" % world,
            "candidates_total": M3, "n_train": N3, "dim": D3, "reps": reps, "flop_per_ei": f_ei,
            "roofline_ei_per_s_per_gpu": roof, "h2d_bytes_per_rank_host_pageable": int(M3 // world * D3 * 8),
            "argmax_check": check, **out}


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from robo_b200 import _lib
    from robo_b200 import kernels as K
    from robo_b200.acquisition_functions import EI
    from robo_b200.distributed import init_comm
    from robo_b200.models.gaussian_process import GaussianProcess

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (no CPU fallback in the product path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    M = args.m
    M_total = world * M
    X, y, theta, noise = train_problem()
    Xs_all = candidates(M_total)                      # the same pageable array on every rank
    lo, hi = _lib.shard_bounds(M_total, rank, world)

    h = _lib.Handle(local_rank)
    # a real (non-default) torch stream: the handle launches on it, and torch.cuda.Event timing sees it
    # high priority like the handle's own stream: the single-CTA kernels of the Cholesky chain must not queue behind the
    # trailing-update tiles the handle launches on its low-priority side stream
    stream = torch.cuda.Stream(device=dev, priority=-1)
    torch.cuda.set_stream(stream)
    h.set_stream(stream.cuda_stream)
    h.set_option("chunk", args.chunk)
    h.set_data(X, y)
    f = K.Product(K.ConstantKernel(theta[0], ndim=DIM), K.Matern52Kernel(np.exp(theta[1:]), ndim=DIM)).flatten()
    h.set_kernel(f["family"], f["log_amp"], f["axis"], f["group"], f["log_metric"])
    diag_add = diag_add_of(noise)
    mean = float(np.mean(y))
    eta = float(np.min(y))
    init_comm(h, rank, world)                         # NCCL communicator inside libgpk.so (no-op at world = 1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- GP fit (K build + Cholesky + forward solve + log-det), then L^-1 for scoring ----
    fit_ms = []
    for _ in range(4):
        logdet, ll = h.fit(diag_add, mean)
        fit_ms.append(h.timings()["fit_ms"])
    d_X = torch.from_numpy(np.ascontiguousarray(Xs_all[lo:hi])).to(dev)
    d_best = torch.zeros(2, dtype=torch.float64, device=dev)
    h.acq_dev(d_X.data_ptr(), min(hi - lo, 1024), _lib.ACQ_EI, eta, 0.0, 0, 0, 0, 0)              # builds L^-1
    torch.cuda.synchronize()
    t_fit = h.timings()

    def step_dev():
        # scoring of this rank's shard, ncclAllGather of the 16-byte pairs and the merge: all on `stream`, no host sync
        h.acq_argmax_sharded_dev(d_X.data_ptr(), hi - lo, lo, _lib.ACQ_EI, eta, 0.0, d_best.data_ptr())

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()            # started before the warm-up so that samples exist even for short timed regions
    for _ in range(args.warmup):
        step_dev()
    launches0 = h.timings()["launches_total"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.mark_timed_region()
    e0.record(stream)
    for _ in range(args.steps):
        step_dev()
    e1.record(stream)
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop() if rank == 0 else None
    tim = h.timings()
    launches = tim["launches_total"] - launches0
    value = M_total * args.steps / (ms * 1e-3)
    merged = unpack_pair(d_best)
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "argmax.npy"), np.array(merged, dtype=np.float64))

    # ---- roofline of the dominant kernel (variance GEMM), measured live with CUDA events ----
    # algorithmic flops per launch: every candidate row of the chunk contracts with the lower
    # triangle of L^-1 (N^2/2 FMA = N^2 flop) plus the mean reduction (2N)   [SURVEY.md 8d: F_ei ~ N^2]
    rows = min(args.chunk, ((M + 127) // 128) * 128)
    last_rows = rows if M > rows else M          # timings() averages the full-size chunk launches of the last step
    gemm_ms = tim["vargemm_ms"]
    flops = float(last_rows) * (N_TRAIN ** 2 + 2 * N_TRAIN)
    achieved = flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0

    # ---- answer check (outside the timed region): rank 0 scores the FULL list alone ----
    argmax_check, single = None, None
    if rank == 0:
        r = h.acq(Xs_all, _lib.ACQ_EI, eta, 0.0, want_values=False)         # host-batch path, no communicator involved
        single = (r["best_val"], r["best_idx"])
        argmax_check = bool(single == merged)
    barrier()

    # ---- end to end through the RoBO-facing classes: pageable numpy in, acquisition values out ----
    kernel = K.Product(K.ConstantKernel(theta[0], ndim=DIM), K.Matern52Kernel(np.exp(theta[1:]), ndim=DIM))
    model = GaussianProcess(kernel, noise=noise, normalize_input=True, normalize_output=False,
                            lower=np.zeros(DIM), upper=np.ones(DIM), rng=np.random.RandomState(0), device=local_rank)
    model.train(X, y, do_optimize=False)
    mh = model.gp.handle
    mh.set_stream(stream.cuda_stream)
    mh.set_option("chunk", args.chunk)
    init_comm(mh, rank, world)
    acq = EI(model)
    X_shard = np.array(Xs_all[lo:hi], copy=True)      # plain (pageable) numpy array, as a RoBO maximizer would hold

    last_vals = [None]

    def step_e2e():
        vals = acq.compute(X_shard)                   # H2D of the shard, scoring, D2H of M values (blocking)
        last_vals[0] = vals
        i = int(np.argmax(vals))                      # random_sampling.py:50
        if world > 1:
            return mh.comm_argmax_pair(vals[i], lo + i)
        return float(vals[i]), lo + i

    for _ in range(max(1, args.warmup // 2)):
        e2e_res = step_e2e()
    barrier()
    t0 = time.perf_counter()
    e0.record(stream)
    for _ in range(args.steps):
        e2e_res = step_e2e()
    e1.record(stream)
    barrier()
    wall_e2e = max_over_ranks(1e3 * (time.perf_counter() - t0))
    ms_e2e = max_over_ranks(e0.elapsed_time(e1))
    e2e_value = M_total * args.steps / (ms_e2e * 1e-3)
    e2e_ok = bool(e2e_res[1] == merged[1] and abs(e2e_res[0] - merged[0]) <= 1e-12 * abs(merged[0]))
    if args.dump_outputs and rank == 0:
        np.save(os.path.join(args.dump_outputs, "ei_values.npy"), np.asarray(last_vals[0], dtype=np.float64))

    # second key: the round-1 figure (pinned host candidates, arg-max only: 24 bytes back)
    Xs_pinned = torch.from_numpy(X_shard).pin_memory()
    Xp = Xs_pinned.numpy()

    def step_pinned():
        r = h.acq(Xp, _lib.ACQ_EI, eta, 0.0, want_values=False)
        if world > 1:
            h.comm_argmax_pair(r["best_val"], lo + r["best_idx"])

    step_pinned()
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        step_pinned()
    e1.record(stream)
    barrier()
    ms_pinned = max_over_ranks(e0.elapsed_time(e1))

    # ---- configs[2]: strong scaling of one whole maximisation over 2^20 candidates ----
    c3 = None
    if not args.no_c3:
        c3 = c3_block(torch, dist, _lib, K, rank, world, local_rank, stream, barrier, max_over_ranks)

    mh.comm_destroy()
    h.comm_destroy()
    if rank != 0:
        return
    dgemm = measure_dgemm_tflops(torch, dev)
    dmma_peak, dfma_peak = h.measure_fp64_peaks()
    used_int8 = tim.get("launches_ozaki", 0) > 0
    int8_peak = h.measure_int8_peak() if used_int8 else None
    int8_peak_sustained = h.measure_int8_peak_sustained(0.5, True) if used_int8 else None
    int8_peak_sustained_const = h.measure_int8_peak_sustained(0.5, False) if used_int8 else None
    # ---- CPU baselines on this box's host cores (bounded sample; rank 0, N = 1 only) ----
    cpu, cpu_opt = None, None
    if world == 1 and not args.no_cpu_baseline:
        cpu, cpu_opt, _, _ = cpu_rows(6, 1)
    # incremental refit (gpk_fit_append): the last 8 rows appended to a model fitted on N - 8 rows (extra info, untimed
    # with respect to the headline; rank 0 only)
    append_ms = None
    try:
        for rep in range(2):                                 # the first pass loads the kernels of this path
            h2 = _lib.Handle(dev.index or 0)
            h2.set_data(X[:N_TRAIN - 8], y[:N_TRAIN - 8])
            h2.set_kernel(f["family"], f["log_amp"], f["axis"], f["group"], f["log_metric"])
            h2.fit(diag_add, float(np.mean(y[:N_TRAIN - 8])))
            h2.predict(Xs_all[:128])
            res = h2.fit_append(X, y, diag_add, mean)
            if res is not None:
                append_ms = h2.timings()["fit_ms"]
                assert abs(res[1] - ll) <= 1e-10 * abs(ll), "incremental refit disagrees with the full fit"
            h2.close()
    except Exception as e:                                   # noqa: BLE001
        print("fit_append timing skipped: %r" % (e,), file=sys.stderr)
    traffic = ncu_dram_bytes(VARGEMM_NCU_CSV, "gpk_gemm_ws_kernel<1>") if last_rows == 16384 else None
    fp64_block = {"fp64_equivalent_tflops": achieved, "dmma_peak_tflops": dmma_peak, "frac_of_dmma_peak": achieved / dmma_peak,
                  "frac_of_datasheet_fp64": achieved / FP64_PEAK_TFLOPS, "dfma_vector_peak_tflops": dfma_peak,
                  "dgemm_cublas_tflops": dgemm, "frac_of_cublas_dgemm": achieved / dgemm if dgemm > 0 else None,
                  "launch_ms": gemm_ms, "launch_candidates": int(last_rows),
                  "launches_averaged": int(max(1, (M + rows - 1) // rows - 1)) if M > rows else 1}
    if used_int8:
        # the contraction ran on the int8 tensor pipe: `pairs` exact slice-pair products per fp64 product over the lower
        # triangle of L^-1 in 128-row blocks = pairs (N^2 + 128 N) int8 multiply-adds x 2 per candidate row
        pairs = float(tim.get("ozaki_slice_pairs") or 28.0)
        int8_ops = float(last_rows) * pairs * (N_TRAIN ** 2 + 128 * N_TRAIN)
        oz_traffic = (ncu_dram_bytes(OZ_NCU_CSV, "gpk_oz_pair2")
                      if last_rows == 16384 and int(tim.get("ozaki_kernel_variant", 0)) == 4 else None)
        int8_achieved = int8_ops / (gemm_ms * 1e-3) / 1e12
        roofline = dict(fp64_block, bound="tensor",
                        kernel="%s%s: L^-1 K*^T as %d int8 slice-pair products, tcgen05.mma kind::i8, TMEM accumulators, TMA-staged "
                               "swizzled slices" % (OZ_KERNELS.get(int(tim.get("ozaki_kernel_variant", 0)) & 7, "int8 contraction"),
                                                    ", persistent tile walk" if int(tim.get("ozaki_kernel_variant", 0)) & 8 else "", int(pairs)),
                        achieved=int8_achieved, peak=int8_peak_sustained, unit="TFLOP/s", frac=int8_achieved / int8_peak_sustained,
                        peak_burst=int8_peak, frac_of_burst_peak=int8_achieved / int8_peak,
                        peak_sustained_constant_operands=int8_peak_sustained_const,
                        ops="int8 multiply-accumulate counted as 2 ops (TOP/s)",
                        peak_source="measured live on this GPU: tcgen05.mma kind::i8 128x128x32 issue rate from shared memory, "
                                    "pseudo-random operand bytes, launched back to back for 0.5 s, second half timed "
                                    "(gpk_measure_int8_peak_sustained): the contraction is timed inside a long step and the int8 pipe "
                                    "runs into sw_power_cap, so the sustained figure is the denominator (as MEASURED_PEAKS.json does "
                                    "for bf16: 1376 sustained / 1667 burst); peak_sustained_constant_operands = the same with a "
                                    "constant operand pattern (no switching activity); peak_burst = one 0.3 ms launch "
                                    "(gpk_measure_int8_peak); nominal dense int8 = 4500 TOP/s",
                        traffic=oz_traffic,
                        traffic_source="read at run time from the committed capture %s (ncu --set full, one 16384-candidate "
                                       "launch); algorithmic minimum = %d slices x (L^-1 lower triangle 8.4 MB + K* 67 MB) "
                                       "read once" % (OZ_NCU_CSV, 7))
    else:
        roofline = dict(fp64_block, bound="tensor",
                        kernel="%s (L^-1 K*^T contraction, fp64 DMMA, warp-specialised TMA)"
                               % ("gpk_vargemm_persistent_kernel" if tim.get("persist") else "gpk_gemm_ws_kernel<EPI_COLREDUCE>"),
                        achieved=achieved, peak=dmma_peak, unit="TFLOP/s", frac=achieved / dmma_peak,
                        peak_source="measured live on this GPU: register-resident DMMA m8n8k4 issue rate "
                                    "(gpk_measure_fp64_peaks); MEASURED_PEAKS.json has no fp64 figure; datasheet "
                                    "FP64-tensor = %.0f TF/s (SURVEY 8d P64)" % FP64_PEAK_TFLOPS,
                        traffic=traffic,
                        traffic_source="read at run time from the committed capture %s (ncu --set full, one 16384-candidate "
                                       "launch: dram__bytes_read.sum + dram__bytes_write.sum); algorithmic minimum 0.60e9 "
                                       "(L^-1 lower triangle 67 MB + K* 537 MB read once)" % VARGEMM_NCU_CSV)
    line = {
        "metric": METRIC, "value": value, "unit": "EI evals/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "GP posterior N=4096 D=16 Matern52 fp64: predict + EI + argmax (configs[1])",
                   "n_train": N_TRAIN, "dim": DIM, "candidates_per_step_per_gpu": M, "candidates_per_step": M_total,
                   "chunk": args.chunk,
                   "parallelism": "common candidate list of %d rows, contiguous shards x%d (gpk_shard_bounds), fit state "
                                  "replicated, one 16-byte ncclAllGather + device merge per step inside libgpk.so"
                                  % (M_total, world),
                   "l2": ("working set per step (int8 digit slices: L^-1 %d MB + K* %d MB per chunk, %d chunks per step) exceeds "
                          "the 126 MB L2; no flush needed"
                          % (7 * N_TRAIN * N_TRAIN // 2 ** 20, 7 * rows * N_TRAIN // 2 ** 20, (M + rows - 1) // rows)) if used_int8 else
                         ("working set per step (L^-1 134 MB + K* chunk %d MB) exceeds the 126 MB L2; no flush needed"
                          % (rows * N_TRAIN * 8 // 2 ** 20))},
        "fit_ms": float(np.median(fit_ms[1:])), "fit_breakdown_ms": {k: t_fit[k] for k in ("kbuild_ms", "potrf_ms", "linv_ms")},
        "loglik": ll, "fit_append_8rows_ms": append_ms,
        "argmax_check": argmax_check,
        "argmax": {"merged": {"value": merged[0], "index": merged[1]},
                   "single_gpu_full_list": {"value": single[0], "index": single[1]},
                   "e2e_path_agrees": e2e_ok},
        "e2e": {"value": e2e_value, "unit": "EI evals/s", "h2d_bytes_per_step": int((hi - lo) * DIM * 8),
                "d2h_bytes_per_step": int((hi - lo) * 8 + 24), "ms_per_step": ms_e2e / args.steps,
                "wall_ms_per_step": wall_e2e / args.steps,
                "call": "robo_b200.acquisition_functions.EI(model).compute(X) on a pageable numpy array, values returned "
                        "to the host, numpy arg-max" + (", gpk_comm_argmax_pair" if world > 1 else "")},
        "e2e_pinned_argmax_only": {"value": M_total * args.steps / (ms_pinned * 1e-3), "unit": "EI evals/s",
                                   "h2d_bytes_per_step": int((hi - lo) * DIM * 8), "d2h_bytes_per_step": 24,
                                   "ms_per_step": ms_pinned / args.steps,
                                   "call": "gpk_acq on a page-locked host buffer, arg-max only (round-1 e2e)"},
        "gpu_launches": int(launches),
        "roofline": roofline,
        "kernel_ms_last_chunk": {k: tim[k] for k in ("kstar_ms", "vargemm_ms", "finish_ms")},
        "configs": {"c3": c3},
        "cpu_baseline": cpu, "cpu_baseline_optimised": cpu_opt, "clocks": clocks,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--m", type=int, default=131072, help="candidates per step per GPU")
    ap.add_argument("--chunk", type=int, default=16384)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c3", action="store_true", help="skip the configs[2] strong-scaling block")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 0:
        ap.error("--warmup must not be negative")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
