/* gpk.h — C ABI of libgpk.so: B200-native (sm_100a) GP posterior + acquisition kernels.
 *
 * This is the drop-in boundary for RoBO's hot path (SURVEY.md section 8b).  Every entry
 * point replaces a call the reference makes into george / scipy-LAPACK / scipy.stats from
 *   robo/models/gaussian_process.py          (train / nll / predict)
 *   robo/acquisition_functions/{ei,log_ei,pi,lcb}.py   (compute)
 *   robo/acquisition_functions/information_gain{,_per_unit_cost}.py and robo/util/epmgp.py (entropy search)
 * The reference is pure Python; its "FFI" for this path is george's Cython bridge, so the
 * binding a RoBO maintainer would add is a ctypes stub (see INTEGRATION.md and
 * robo_b200/_lib.py, which is exactly that stub).
 *
 * Conventions
 *   - plain C: pointers + sizes, no torch / numpy types.  All floating point is IEEE fp64.
 *   - host pointers are caller-owned, C-contiguous, read/written only during the call.
 *   - `*_dev` entry points take device pointers (e.g. torch.Tensor.data_ptr()) and are
 *     asynchronous on the handle's stream.
 *   - every function returns a gpk_status; nothing throws or aborts.  The Python side maps
 *     GPK_NOT_PD -> numpy.linalg.LinAlgError (caught at gaussian_process.py:120,156 and by
 *     the bare except at gaussian_process_mcmc.py:196), GPK_BAD_ARG -> ValueError,
 *     GPK_CUDA_ERROR -> RuntimeError.
 *   - one CUDA stream per handle; calls on one handle are not re-entrant.
 */
#ifndef GPK_H_
#define GPK_H_

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gpk_handle gpk_handle;

typedef enum {
    GPK_OK = 0,
    GPK_NOT_PD = 1,        /* Cholesky pivot <= 0 or NaN: numpy.linalg.LinAlgError in the reference */
    GPK_BAD_ARG = 2,
    GPK_CUDA_ERROR = 3,
    GPK_NOT_FITTED = 4,
    GPK_NOT_APPLICABLE = 5 /* gpk_fit_append: preconditions not met, nothing was changed; do a full fit */
} gpk_status;

/* stationary radial families, george names (oracle/george_oracle.py) */
typedef enum {
    GPK_MATERN52 = 0,      /* george.kernels.Matern52Kernel   */
    GPK_EXPSQUARED = 1,    /* george.kernels.ExpSquaredKernel */
    GPK_MATERN32 = 2       /* george.kernels.Matern32Kernel   */
} gpk_family;

typedef enum {
    GPK_ACQ_NONE = 0,      /* posterior moments only                              */
    GPK_ACQ_EI = 1,        /* robo/acquisition_functions/ei.py:65-78              */
    GPK_ACQ_LOG_EI = 2,    /* robo/acquisition_functions/log_ei.py:67-122         */
    GPK_ACQ_PI = 3,        /* robo/acquisition_functions/pi.py:58-63              */
    GPK_ACQ_LCB = 4        /* robo/acquisition_functions/lcb.py:62-65             */
} gpk_acq_kind;

#define GPK_MAX_TERMS 64   /* metric entries (input dims x product factors) per kernel */

/* ---- lifetime ---------------------------------------------------------------------- */
int gpk_create(gpk_handle** h, int device);
int gpk_destroy(gpk_handle* h);
const char* gpk_last_error(gpk_handle* h);
const char* gpk_version(void);
/* key in
 *   "loader"    operand staging of the GEMM tile engine: 2 = TMA with a dedicated producer warp and
 *               full/empty mbarriers [default], 1 = TMA issued by a consumer thread, 0 = cp.async (cross-check)
 *   "chunk"     candidates per scoring pass (multiple of 128); 0 = automatic [default]: the K* buffer is kept near
 *               512 MB (16384 candidates at N = 4096, 65536 at N <= 1024)
 *   "cov"       covariance builder: 2 = TMA-staged, pre-scaled term-major operands [default], 1 = round-1 kernel
 *   "graph"     1 = the split-chain schedule of a factorisation (~600 launches / event records / stream waits at
 *               N = 4096) is captured once per layout into a CUDA graph and replayed per fit [default]; 0 = enqueue
 *               every call directly
 *   "ozaki"     1 = variance contraction on the int8 tensor pipe (tcgen05 kind::i8, TMEM accumulators) through an
 *               error-free split of L^-1 and K* into 7 balanced base-256 digits each, 28 digit-pair products
 *               (gpk_ozaki.cuh); used while max |L^-1| < 64 and N <= 16384, otherwise the fp64 kernel runs [default;
 *               batches of >= 2048 candidates]; 0 = always fp64 DMMA.  The posterior mean never goes through the digits
 *               (fp64 K* alpha)
 *   "oztile"    128 = two passes over the contraction (levels 4..6, then 0..3), 128 candidates per tile [default];
 *               64 = one pass, 64 candidates per tile, 7 accumulators of 64 TMEM columns
 *   "ozpair"    1 = CTA pairs (tcgen05 cta_group::2, cluster of 2): 256 rows of L^-1 per pair, each CTA stages half of the
 *               K* slice tiles [default, with "oztile" 128: gpk_oz_pair2_kernel; needs an even number of 128-row blocks,
 *               otherwise the one-pass single-CTA kernel runs]; 0 = one CTA per tile
 *   "ozpersist" 0 = one CTA (pair) per tile; 1 = one CTA (pair) per SM walks the tile list; 2 = the persistent kernel
 *               launched with one tile per CTA (profiling aid); 3 = automatic [default]: persistent for N <= 3072, where a
 *               scoring pass is 7 - 13 % shorter (the resident grid lets the next chunk's K* builder run beside it;
 *               profiles/r02_persistent_walk_by_n.json, configs[2] maximisation 23.6 -> 22.1 ms), one tile per CTA above
 *               (N = 4096, D = 16, sustained: 3.5 % slower, profiles/r02_int8_variants_bench.txt)
 *   "ozpdl"     1 = the look-ahead K* builder runs as a small resident grid ("covctas" CTAs per SM) that triggers a
 *               programmatic dependent launch of the contraction behind it on the same stream (the two really co-run);
 *               0 = builder on the side stream (the block scheduler places it in the contraction's tail) [default: the
 *               co-running contraction loses more than the builder costs]
 *   "ozfused"   1 = with "ozaki": the covariance builder writes the int8 digits and the mean partials itself, no fp64
 *               K* in HBM [default]; 0 = fp64 K* + split kernel + mean dot
 *   "ozprof"    1 = the persistent int8 kernel accumulates clock64() sums per role (gpk_get_oz_profile)
 *   "persist"   1 = persistent fp64 variance contraction (one CTA per SM, dynamic tile counter); 0 = one CTA per tile
 *               [default: the persistent variant measured 2 % slower at N = 4096 and equal at N = 1024]
 *   "depth2"    1 = trailing updates of two consecutive panels in one K = 256 contraction (odd steps; even steps update
 *               only the next-but-one block column); 0 = one K = 128 update per step (bit-identical factor);
 *               2 = automatic [default]: on for N >= 6144, where the trailing updates gate the fit (5 % at N = 8192)
 *   "chainsplit" 1 = split Cholesky chain: diag(k+1) waits only for block row k+1 of step k (one launch on
 *               four 32-row tiles), the rows below run on a second high-priority stream, trailing update with
 *               look-ahead 2 (measured neutral against the plain schedule: profiles/r02_fit_compare_*.jsonl);
 *               0 = plain look-ahead schedule [default] (bit-identical factor)
 *   "diag"      diagonal-block Cholesky + inverse kernel: 4 = 16-column panels, square-root-free pivot chain in one warp,
 *               substitutions in four, rank-16 updates on the fp64 tensor pipe [default]; 3 = the same with DFMA register
 *               tiles; 2 = column-by-column register-tiled kernel; 0 = simple shared-memory version (cross-checks)
 *   "diagprof"  1 = the blocked diagonal kernels record clock64() stamps per phase (gpk_get_diag_profile)
 *   "lookahead" 1 = trailing updates on a side stream, overlapped with the next diag/panel [default]
 *   "smalltile" 1 = 32-row tiles for the panel solve / next-panel update [default], 2 = 16-row tiles, 0 = 128-row tiles
 *   "fusechain" 1 = panel solve + next-panel update of a step in one launch (measured neutral; default 0)
 *   "pdl"       1 = programmatic dependent launch for the kernels of the Cholesky chain [default]
 *   "overlap"   1 = build K* of chunk i+1 on the side stream while chunk i contracts [default] */
int gpk_set_option(gpk_handle* h, const char* key, long value);
/* run on an existing CUDA stream (cudaStream_t passed as void*); NULL = the handle's own.  The handle's own stream has
 * the highest priority and its side stream (trailing updates, K* look-ahead) the lowest: give an external stream a high
 * priority too, or the single-CTA kernels of the Cholesky chain queue behind the side stream's tiles (fit 2.6 instead of
 * 2.3 ms at N = 4096). */
int gpk_set_stream(gpk_handle* h, void* cuda_stream);
int gpk_synchronize(gpk_handle* h);

/* ---- model state ------------------------------------------------------------------- */
/* Training inputs as the reference hands them to george: X already scaled by
 * zero_one_normalization (gaussian_process.py:89-93), y already standardised if
 * normalize_output (:95-101).  X is (n, d) row-major. */
int gpk_set_data(gpk_handle* h, const double* X, const double* y, int n, int d);

/* Test-input scaling fused into the scoring kernels: x <- (x - lower) / (upper - lower)
 * (robo/util/normalization.py:11, applied at gaussian_process.py:276).  NULL disables. */
int gpk_set_input_bounds(gpk_handle* h, const double* lower, const double* upper, int d);

/* Output un-normalisation fused into the scoring kernels (gaussian_process.py:282-284):
 * mu <- mu * y_std + y_mean ; var <- var * y_std^2.  enabled = 0 disables. */
int gpk_set_output_transform(gpk_handle* h, int enabled, double y_mean, double y_std);

/* k(x, x') = exp(log_amp) * prod_g f( sum_{t in g} (x[axis_t] - x'[axis_t])^2 / exp(log_metric_t) )
 * Terms are listed group by group (group[] non-decreasing from 0).  One group over all
 * columns = george's axis-aligned (ARD) kernel; one group per column = the product of 1-D
 * kernels built at robo/fmin/fabolas.py:104-110.  Replaces kernel.set_parameter_vector
 * (gaussian_process.py:110,151). */
int gpk_set_kernel(gpk_handle* h, int family, double log_amp, int n_terms,
                   const int* axis, const int* group, const double* log_metric);

/* ---- fit: K build + Cholesky + forward solve + log-det ------------------------------- */
/* Replaces george GP.compute + GP.log_likelihood (gaussian_process.py:119,155,159):
 *   K = k(X, X) + diag_add * I ; K = L L^T ; z = L^-1 (y - mean)
 *   logdet = 2 sum log L_ii ; loglik = -1/2 z^T z - 1/2 logdet - n/2 log(2 pi)
 * diag_add is the value george adds to the diagonal, yerr^2 + 1.25e-12, computed by the host
 * exactly as george does.  Returns GPK_NOT_PD where scipy.linalg.cholesky would raise. */
int gpk_fit(gpk_handle* h, double diag_add, double mean, double* logdet, double* loglik);

/* The same in two halves, for evaluating many hyper-parameter vectors at once: gpk_fit_begin only
 * enqueues the work on the handle's stream and returns; gpk_fit_end waits and returns the
 * results.  With one handle per theta (each on its own stream) the latency-bound Cholesky chains
 * of several thetas overlap on the GPU: this is how GaussianProcessMCMC.loglikelihood
 * (gaussian_process_mcmc.py:168-202) is served for a half-ensemble of emcee walkers per step. */
int gpk_fit_begin(gpk_handle* h, double diag_add, double mean);
int gpk_fit_end(gpk_handle* h, double* logdet, double* loglik);

/* Incremental refit after rows were appended (robo/models/base_model.py:30-45 `update`, and
 * robo/solver/bayesian_optimization.py:161-167 train(do_optimize=False) when hyper-parameters are frozen).
 * X (n x d) and y (n) are the full new training set; its first rows must be the ones of the last fit, the kernel
 * and diag_add unchanged.  Requires a fitted handle whose L^-1 has been built (any predict / acq call) and the new
 * rows to fall into the last 128-row block of the padded layout; otherwise returns GPK_NOT_APPLICABLE without
 * touching the model.  O(N^2): only the last block row of the factor and of its inverse is recomputed. */
int gpk_fit_append(gpk_handle* h, const double* X, const double* y, int n, int d, double diag_add, double mean,
                   double* logdet, double* loglik);

/* ---- posterior + acquisition over a candidate batch -------------------------------- */
/* Replaces george GP.predict + np.diag + clip (gaussian_process.py:276-294):
 * mu[m], var[m] (var clipped to >= DBL_EPSILON).  Xs is (m, d) row-major, raw (un-scaled). */
int gpk_predict(gpk_handle* h, const double* Xs, long m, double* mu, double* var);

/* full_cov=True path (gaussian_process.py:280-294): cov is (m, m) row-major, every entry
 * clipped to >= DBL_EPSILON like the reference does. */
int gpk_predict_cov(gpk_handle* h, const double* Xs, long m, double* mu, double* cov);

/* The same without the clip: the raw posterior covariance K** - K* K^-1 K*^T (negative off-diagonal entries kept,
 * output transform applied).  This is what george's GP.sample_conditional draws from at gaussian_process.py:324
 * (sample_functions); only predict() clips (:290-294). */
int gpk_posterior_cov(gpk_handle* h, const double* Xs, long m, double* mu, double* cov);

/* Fused predict -> acquisition -> argmax.  out (m values) may be NULL when only the argmax
 * is wanted.  best_idx follows numpy.argmax (first maximum; NaN counts as maximum) as used at
 * robo/maximizers/random_sampling.py:50.  n_negative counts EI values < 0 (the reference
 * raises ValueError on any, ei.py:86-88).  mu/var may be NULL. */
int gpk_acq(gpk_handle* h, const double* Xs, long m, int acq_kind, double eta, double par,
            double* out, double* mu, double* var,
            double* best_val, long* best_idx, long* n_negative);

/* Device-pointer variant, asynchronous on the handle's stream.  d_Xs: (m, d) fp64 row-major
 * on the device.  d_out/d_mu/d_var (m doubles each) may be NULL.  d_best: 16 bytes
 * {double value; long long index}.  */
int gpk_acq_dev(gpk_handle* h, const void* d_Xs, long m, int acq_kind, double eta, double par,
                void* d_out, void* d_mu, void* d_var, void* d_best);

/* Predictive gradients and acquisition gradients (SURVEY.md section 8f rank 3).  The reference's
 * acquisition functions call model.predictive_gradients when derivative=True (ei.py:80-85, pi.py:65-71,
 * lcb.py:66-69) but none of its models implements it.  Xs: (m, d) raw inputs; mu, var: (m); dmu, dvar:
 * (m, d) = d mu / d x, d var / d x (chain rules of the input scaling and output transform included).
 * acq_kind = GPK_ACQ_NONE, or EI / PI / LCB to also get f (m) and df (m, d) = d acquisition / d x. */
int gpk_predict_grad(gpk_handle* h, const double* Xs, long m, int acq_kind, double eta, double par,
                     double* mu, double* var, double* dmu, double* dvar, double* f, double* df);

/* RandomSampling.maximize with the candidates generated on the device
 * (robo/maximizers/random_sampling.py:38-50; SURVEY.md section 8f rank 2).  Candidate i (global index) is
 *   i < n_uniform : lower + (upper - lower) * U[0,1)^d
 *   otherwise     : clip(incumbent + scale * N(0,1)^d, lower, upper)
 * from Philox4x32-10 keyed by (seed, i, coordinate pair): independent of chunking and of how the range
 * [first, first+count) is split over GPUs.  Returns the best candidate of the range (numpy.argmax
 * tie-breaking), its acquisition value and its GLOBAL index; no candidate or value crosses PCIe. */
int gpk_maximize_random(gpk_handle* h, unsigned long long seed, long first, long count, long n_uniform,
                        const double* lower, const double* upper, const double* incumbent, double scale,
                        int acq_kind, double eta, double par,
                        double* best_x, double* best_val, long* best_idx);
/* the same generator, candidates copied to the host (out: count x d row-major); tests and re-creating
 * the winning point on another rank */
int gpk_generate_candidates(gpk_handle* h, unsigned long long seed, long first, long count, long n_uniform, int d,
                            const double* lower, const double* upper, const double* incumbent, double scale,
                            double* out);

/* Acquisition closed forms on caller-supplied moments (host arrays), evaluated by the same
 * device function as the fused path.  Serves models that are not GPU GPs (e.g. the
 * reference's test/dummy_model.py).  No handle state is used except the device/stream. */
int gpk_acq_moments(gpk_handle* h, const double* mu, const double* var, long m, int acq_kind,
                    double eta, double par, double* out, long* n_negative);

/* Reductions over the n_models hyper-parameter samples of a GP-MCMC model; A, B are
 * (n_models, m) row-major host arrays.
 *   mode 0: out1 = mean_i A_i                      MarginalizationGPMCMC.compute (marginalization.py:115-121)
 *   mode 1: out1 = mean_i A_i, out2 = var_i(A_i) + mean_i(B_i) clipped at DBL_EPSILON
 *                                                  GaussianProcessMCMC.predict (gaussian_process_mcmc.py:235-247) */
int gpk_reduce_models(gpk_handle* h, const double* A, const double* B, int n_models, long m, int mode,
                      double* out1, double* out2);

/* One candidate batch against the n_models fitted handles of a GP-MCMC model (all on one device, same input
 * dimension), reduced over the models ON THE DEVICE: the batch goes H2D once, every model scores it on its own stream
 * (the small launches overlap), and only the reduced vectors come back.  Xs: (m, d) raw host inputs.
 *   mode 0: out1 = mean_i acq_i(x)  with eta[i] the incumbent of model i      MarginalizationGPMCMC.compute
 *           (robo/acquisition_functions/marginalization.py:115-121); best_val/best_idx = numpy.argmax of out1 (may be
 *           NULL); n_negative = EI values < 0 over all models (ei.py:86-88 raises on any)
 *   mode 1: out1 = mean_i mu_i, out2 = var_i(mu_i) + mean_i var_i clipped at DBL_EPSILON   GaussianProcessMCMC.predict
 *           (robo/models/gaussian_process_mcmc.py:235-247); acq_kind / eta / par ignored */
int gpk_acq_multi(gpk_handle* const* models, int n_models, const double* Xs, long m, int mode, int acq_kind,
                  const double* eta, double par, double* out1, double* out2, long* n_negative, double* best_val,
                  long* best_idx);

/* kernel.get_value(X1, X2) (test/test_models/test_gaussian_process.py:44-46) with the
 * handle's current kernel; no input scaling.  out is (n1, n2) row-major. */
int gpk_kernel_matrix(gpk_handle* h, const double* X1, long n1, const double* X2, long n2,
                      int d, double* out);

/* ---- multi-GPU: candidate shards, one 16-byte exchange per arg-max (SURVEY.md section 8e) -------------------- */
/* One process per GPU, one handle per process.  The fit state is replicated (every rank calls gpk_set_data /
 * gpk_set_kernel / gpk_fit with the same inputs: zero communication), rank r scores the contiguous slice
 * gpk_shard_bounds(m, r, world) of the candidate list, and the ranks agree on numpy.argmax of the whole list
 * (robo/maximizers/random_sampling.py:50: first maximum, NaN first) through ONE ncclAllGather of the 16-byte
 * {value, global index} pair on the handle's stream followed by a deterministic merge on the device.  NCCL is bound at
 * run time (dlopen of libnccl.so.2; GPK_NCCL_LIB overrides), so the library itself links cudart only. */
int gpk_comm_unique_id(void* id128);           /* rank 0: ncclGetUniqueId; ship the 128 bytes to the other ranks */
int gpk_comm_init(gpk_handle* h, int rank, int world, const void* id128);    /* collective over all ranks */
int gpk_comm_destroy(gpk_handle* h);
int gpk_comm_info(gpk_handle* h, int* rank, int* world, int* nccl_version);
int gpk_shard_bounds(long m, int rank, int world, long* lo, long* hi);       /* sizes differ by at most one */
/* The exchange alone: this rank's best {value, GLOBAL index} (index < 0: nothing to offer) in, the merged winner out on
 * every rank.  For callers that scored their shard themselves (e.g. EI.compute on a slice, values wanted on the host). */
int gpk_comm_argmax_pair(gpk_handle* h, double val, long idx, double* best_val, long* best_idx);
/* Xs: the FULL candidate batch (m_total, d), identical host array on every rank; each rank copies and scores only its
 * slice.  Returns the global arg-max on every rank. */
int gpk_acq_argmax_sharded(gpk_handle* h, const double* Xs, long m_total, int acq_kind, double eta, double par,
                           double* best_val, long* best_idx);
/* Device-resident shard, asynchronous on the handle's stream, no host synchronisation: d_Xs_shard is this rank's
 * (m_shard, d) slice whose first row has global index first_global (m_shard may be 0); d_best (16 bytes, device)
 * receives the merged {double value; long long global index}. */
int gpk_acq_argmax_sharded_dev(gpk_handle* h, const void* d_Xs_shard, long m_shard, long first_global, int acq_kind,
                               double eta, double par, void* d_best);
/* gpk_maximize_random over n_total device-generated candidates split across the ranks (Philox keyed by the global
 * index: the result does not depend on the number of GPUs); best_x is re-created on every rank from the winning index. */
int gpk_maximize_random_sharded(gpk_handle* h, unsigned long long seed, long n_total, long n_uniform,
                                const double* lower, const double* upper, const double* incumbent, double scale,
                                int acq_kind, double eta, double par,
                                double* best_x, double* best_val, long* best_idx);

/* ---- marginal-likelihood gradient (gaussian_process.py:168-191, corrected noise term) -- */
/* grad[n_terms + 2] = d(-loglik)/d[log_amp, log_metric_t..., log sigma^2]; requires a
 * preceding successful gpk_fit with the same parameters.  noise_var = sigma^2. */
int gpk_nll_grad(gpk_handle* h, double noise_var, double* grad);

/* fp64 issue-rate peaks of this GPU in TFLOP/s, measured with register-resident operands: the DMMA
 * m8n8k4 tensor pipe (every GEMM of the library) and the DFMA vector pipe (covariance builder).  bench.py
 * uses the DMMA figure as the roofline denominator (MEASURED_PEAKS.json has no fp64 entry). */
int gpk_measure_fp64_peaks(gpk_handle* h, double* dmma_tflops, double* dfma_tflops);

/* int8 tensor-pipe issue-rate peak in TOP/s (tcgen05.mma kind::i8, 128 x 128 x 32, operands in shared memory,
 * accumulator in TMEM): the roofline denominator of the option-"ozaki" contraction. */
int gpk_measure_int8_peak(gpk_handle* h, double* tops);
/* the same kernel launched back to back for `seconds` (<= 10); reports the rate of the second half, i.e. at the SM clock
 * the board's power limit allows for this pipe: the denominator for a kernel timed inside a long step.
 * random_operands = 0: constant operand pattern (no switching activity: does not reach the power limit); 1: pseudo-random
 * bytes, the statistics of real digit slices. */
int gpk_measure_int8_peak_sustained(gpk_handle* h, double seconds, int random_operands, double* tops);

/* ---- entropy search (robo/acquisition_functions/information_gain.py, robo/util/epmgp.py) ----------------------- */
/* epmgp.joint_min(mu, V, with_derivatives=True) (epmgp.py:11-81) on caller-supplied moments: expectation propagation
 * per representer point (sweeps in the reference's order, stop at |diff| < 1e-3 or after 50), log Z and its
 * derivatives, then the renormalisation.  mu (nb), V (nb x nb) host arrays, 2 <= nb <= 128.  Outputs (any may be NULL):
 * logP (nb), dlogPdMu (nb x nb), dlogPdSigma (nb x nb(nb+1)/2, lower triangle row-major per row), dlogPdMudMu
 * (nb x nb x nb), sweeps (nb ints: EP sweeps run per point).  Uses the buffers of the handle's entropy-search state:
 * a later gpk_es_compute needs a new gpk_es_update.  GPK_NOT_PD when I + R^T Sigma R stays indefinite after the
 * 1e-10 / 1e-6 jitter retries (:147-153), GPK_BAD_ARG when an update yields NaN variances (:204-207). */
int gpk_es_joint_min(gpk_handle* h, const double* mu, const double* V, int nb, double* logP, double* dlogPdMu,
                     double* dlogPdSigma, double* dlogPdMudMu, int* sweeps);
/* InformationGain.update after the representer points were sampled (information_gain.py:153-167): zb (nb x d) raw
 * inputs, lmb (nb) their sampling-acquisition values, np_grid hallucinated values (Np), sn2 = model.get_noise().
 * Runs predict(zb, full_cov=True) with its eps clip, EP, and prepares B = K^-1 k(X, zb), the packed quadratic-form
 * operand, W = norm.ppf(linspace(1/(Np+1), 1-1/(Np+1), Np)) and the current entropy H on the device.  One state per
 * handle.  logP_out (nb) may be NULL.  GPK_NOT_FITTED without a fit; GPK_BAD_ARG when lmb is not finite (the reference
 * raises ValueError in compute, :207-211), nb is outside 2..128 or np_grid < 1. */
int gpk_es_update(gpk_handle* h, const double* zb, int nb, const double* lmb, int np_grid, double sn2, double* logP_out);
/* InformationGain.compute(X) (information_gain.py:87-125, 169-203, 253-272) for m raw candidates: out (m, may be NULL)
 * = the change of entropy of p_min per candidate; NaN or +inf become -DBL_MAX; with lower / upper (d each, the
 * acquisition's bounds, NULL: no rule) a candidate outside them scores np.spacing(1).  best_val / best_idx: numpy.argmax
 * of out.  GPK_NOT_FITTED when the model was refitted after gpk_es_update. */
int gpk_es_compute(gpk_handle* h, const double* Xs, long m, const double* lower, const double* upper, double* out,
                   double* best_val, long* best_idx);
/* The EP outputs of the last gpk_es_update or gpk_es_joint_min (shapes as there; any may be NULL). */
int gpk_es_get_state(gpk_handle* h, double* logP, double* dlogPdMu, double* dlogPdSigma, double* dlogPdMudMu, int* sweeps);

/* ---- introspection (tests / debugging) ----------------------------------------------- */
int gpk_get_factor(gpk_handle* h, double* L /* n x n row-major, lower */);
int gpk_get_linv(gpk_handle* h, double* Linv /* n x n row-major, lower */);
int gpk_get_z(gpk_handle* h, double* z /* n */);
/* last fit/score timings measured with CUDA events on the handle's stream, milliseconds:
 * out[0] fit total, [1] K build, [2] Cholesky, [3] L^-1, [4] last score call total,
 * [5] K* build and [7] epilogue of the last candidate chunk, [6] variance GEMM averaged over the
 * full-size chunk launches of that call;
 * out[8] = variance-GEMM launches so far,
 * out[9] = total kernel launches so far,
 * out[10] = of those, launches of the int8 (Ozaki) contraction; out[11] = largest row exponent of L^-1 seen by it
 * (option "ozaki"); out[12] = option "persist"; out[13] = int8 slice-pair products the int8 contraction spends per
 * fp64 product (28: 7 balanced base-256 digits per operand); out[14] = which int8 kernel ran last (1 one pass, 2 one pass on
 * CTA pairs, 3 two passes, 4 two passes on CTA pairs = the default; + 8: persistent tile walk); out[15] reserved (zero). */
int gpk_get_timings(gpk_handle* h, double* out16);
/* diagnostics of the persistent int8 contraction (option "ozprof" = 1): per CTA of its last launch 8 clock64() sums:
 * [0] MMA issuer loop, [1] of it waiting for staged operands, [2] waiting for the epilogue to drain TMEM, [3] TMA producer
 * waiting for a free stage, [4] epilogue waiting for final accumulators, [5] epilogue draining TMEM, [6] tiles, [7] 0. */
int gpk_get_oz_profile(gpk_handle* h, long long* out, int max_ctas, int* n_ctas);
/* diagnostics of the blocked diagonal-block kernel (option "diagprof" = 1): clock64() stamps of the last
 * launched block: out[0] start, out[1] tiles loaded, out[2+2p] panel p factorised + solved, out[3+2p] panel p's
 * rank-16 update applied and panel p+1 published, out[33] end, out[34..41] finer stamps inside panel 3. */
int gpk_get_diag_profile(gpk_handle* h, long long* out64);

#ifdef __cplusplus
}
#endif
#endif /* GPK_H_ */
