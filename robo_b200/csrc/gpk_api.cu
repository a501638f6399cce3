// gpk_api.cu — C ABI (include/gpk.h) and host orchestration of the sm_100a kernels.
//
// Data layout in HBM (all fp64, row-major, NP = n rounded up to 128, nb = NP / 128):
//   Xt    [d][NP]        training inputs, transposed (coalesced reads in the covariance builder)
//   Kbuf  [NP+128][NP]   K, overwritten in place by its lower Cholesky factor L; block row nb is
//                        the augmented right-hand side: after the factorisation row NP holds
//                        z = L^-1 (y - mean), so the log-likelihood needs no separate solve
//   P     [NP][NP]       L^-1   (lower; diagonal blocks come out of the Cholesky diag kernel)
//   Q     [NP][NP]       L^-T   (upper) — only needed while building P, and for alpha
//   W     [NP][NP]       scratch of the recursive triangular inverse
//   Kstar [chunk][NP]    K(X*, X) of the current candidate chunk
//   part_mu/part_ssq [nb][chunk]  per-row-block partial sums of the variance contraction
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <dlfcn.h>
#include <string>
#include <vector>

#include "gpk_gemm.cuh"
#include "gpk_kernels.cuh"
#include "gpk_diag16.cuh"
#include "gpk_chain.cuh"
#include "gpk_ozaki.cuh"

namespace {

constexpr int APP_KC = 512;          // split-K chunk of gpk_fit_append's long contractions

struct Range { int off = 0, cnt = 0; };

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
};

}  // namespace

struct gpk_handle {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t own_stream = nullptr;
    cudaStream_t side_stream = nullptr;     // trailing updates of the look-ahead Cholesky
    std::vector<cudaEvent_t> ev_panel, ev_rest;
    cudaStream_t panel_stream = nullptr;    // split chain: panel solve / next-panel update of the rows below block row k+1
    std::vector<cudaEvent_t> ev_cs;         // split chain: 5 events per step (diag, X, trsm', pu', rest_a)
    // variance contraction on the int8 tensor pipe (gpk_ozaki.cuh); 0 = fp64 DMMA kernels
    int ozaki = 1;
    DevBuf oz_Pq, oz_Kq, oz_Kq2, oz_eP, oz_emax, oz_mu, oz_mu2, oz_pmu2;
    int oz_tile = 128;              // 128: two passes, 128 candidates per tile (with oz_pair: 256 x 128 per CTA pair, gpk_oz_pair2_kernel:
                                    // the default; an odd row-block count falls back to the one-pass single-CTA kernel); 64: one pass
    DevBuf oz_scratch;
    CUtensorMap mapOzP32, mapOzK32, mapOzK32b;
    long oz_rows32 = 0, oz_rows32b = 0;
    int oz_pdl = 0;                 // 1: look-ahead K* builder = small resident grid that triggers the dependent launch of the
                                    //    contraction behind it on the SAME stream (real overlap); 0: side stream (tail overlap only)
    int cov_ctas = 2;               // CTAs per SM of that resident builder grid
    int oz_last_variant = 0;        // contraction kernel of the last int8 launch: 1 one pass, 2 one pass CTA pair, 3 two passes, 4 two passes
                                    // CTA pair; + 8 when the persistent tile walk ran
    int oz_prof = 0;                // 1: gpk_oz_persist_kernel accumulates clock64() wait sums per CTA (gpk_get_oz_profile)
    DevBuf oz_profbuf;
    int oz_prof_ctas = 0;
    int oz_persist = 3;             // 1: one CTA (pair) per SM walks the tile list; 0: one CTA (pair) per tile; 2: the persistent kernel with one
                                    // tile per CTA (profiling); 3 = automatic [default]: persistent for N <= 3072 (a scoring pass is 7 - 13 %
                                    // shorter, profiles/r02_persistent_walk_by_n.json), one tile per CTA above (N = 4096, sustained: 3.5 % slower)
    int oz_pair = 1;                // 1: CTA pairs (tcgen05 cta_group::2) when the row-block count is even
    CUtensorMap mapOzKh, mapOzKh2;  // K* slices in 32-row boxes (the half tiles of a pair)
    int oz_fused = 1;               // 1: K* leaves the covariance builder as int8 digits (gpk_cov_oz_kernel); 0: fp64 K* + split + dot
    long oz_linv_serial = -1;       // linv_serial the slices of L^-1 were made for
    long linv_serial = 0;           // bumped whenever L^-1 is (re)built
    int oz_emax_host = 0;
    long oz_rows = 0, oz_rows2 = 0;
    CUtensorMap mapOzP, mapOzK, mapOzK2;
    double oz_launches = 0;
    int persist = 0;                // 1: persistent variance contraction (gpk_vargemm_persistent_kernel); measured 2 % slower than one CTA per tile
    DevBuf tile_cnt;
    int n_sm = 0;
    int use_graph = 1;              // split chain: one CUDA graph per layout, replayed per fit
    cudaGraphExec_t fit_graph = nullptr;
    double fit_graph_launches = 0;
    int chainsplit = 0;             // 1: diag(k+1) waits only for block row k+1 of step k (gpk_chain_step_kernel on 4 CTAs)
    int lookahead = 1;
    int smalltile = 1;              // 32-row tiles for the panel solve / next-panel update
    int pdl = 1;                    // programmatic dependent launch on the Cholesky chain
    int fusechain = 0;              // 1: panel solve + next-panel update of a step in one launch (gpk_chain.cuh)
    DevBuf chain_cnt;
    char err[1024] = {0};
    int loader = LOADER_TMA_WS;
    long chunk = 16384;
    bool chunk_user = false;        // false: candidates per scoring pass chosen from N (chunk_rows)
    int diag_kernel = 4;          // 4 = blocked 16-column panels, DMMA updates (default); 3 = same with DFMA register tiles, 2 = column-by-column register-tiled, 0 = simple shared-memory version
    int diag_prof = 0;            // 1: the blocked diagonal kernel records clock64() stamps per phase (diagnostics)
    DevBuf dprof;

    // model
    int n = 0, d = 0, NP = 0, nb = 0;
    bool has_data = false, has_spec = false, fitted = false, linv_ready = false, alpha_ready = false;
    KSpec spec;
    double log_amp = 0.0;
    std::vector<double> log_metric;
    bool has_bounds = false;
    int norm_out = 0;
    double y_mean = 0.0, y_std = 1.0, mean = 0.0, diag_add = 0.0;

    // device buffers
    DevBuf Xrow, Xt, y, Kbuf, P, Q, W, lower, upper, logdet_part, scal, status, jobs;
    DevBuf Kstar2, cand2;
    DevBuf Xts;                     // training inputs, term-major and pre-scaled (operand of gpk_cov_tma_kernel)
    int cov_kernel = 2;             // 2 = TMA-staged, pre-scaled operands [default]; 1 = the round-1 kernel (cross-check)
    cudaStream_t copy_stream = nullptr;
    std::vector<cudaEvent_t> ev_copied, ev_scored;
    std::vector<cudaEvent_t> ev_g0, ev_g1;    // timed pairs around every variance-GEMM launch of the last scoring call
    int last_nchunks = 0;
    DevBuf cand, Kstar, part_mu, part_ssq, out_mu, out_var, out_acq, block_best, best, nneg;
    DevBuf Vt, cov, XsT, tmpjobs, alpha, tmp1, tmp2, tmp3;
    int layout_NP = -1;           // NP the P/Q/W buffers were zeroed for
    int jobs_nb = -1;

    // job tables
    std::vector<Range> trsm_r, syrk_r, tri1_r, tri2_r, trsm32_r, pu32_r, trsm16_r, pu16_r;
    std::vector<Range> syrk2_r;     // depth-2 trailing update: columns >= k+2 with panels k-1 and k in one contraction (K = 256)
    int depth2 = 2;                 // 0 / 1, or 2 = automatic: on for nb >= 48 (trailing updates gate the fit only there)
    Range kinv_r;
    Range app_row_r, app_syrk_r, app_t_r, app_p_r;      // gpk_fit_append (last block row only)
    Range app_row2_r, app_t2_r;                         // split-K versions of the two long contractions

    // tensor maps
    CUtensorMap mapK, mapP, mapQ, mapW, mapKs, mapVt;
    CUtensorMap mapK32, mapK16, mapKs2;
    long mapKs2_rows = 0;
    std::vector<cudaEvent_t> ev_cov, ev_gemm;
    int overlap = 1;                // build K* of chunk i+1 on the side stream while chunk i contracts            // Kbuf with a 32-row box: A operand of the small-tile chain GEMMs
    bool maps_ok = false;
    long mapKs_rows = 0, mapVt_rows = 0;

    // timing
    cudaEvent_t ev[16];
    cudaEvent_t ev_order = nullptr;
    bool ev_ok = false;
    bool fit_timed = false, score_timed = false;
    double launches_total = 0, launches_var = 0;
    long last_chunk_rows = 0;
    double* pin = nullptr;        // pinned host: [0..1] z^T z, logdet ; [2] status (as int) for async fits
    double* stage[2] = {nullptr, nullptr};    // pinned staging of pageable candidate batches (gpk_acq)
    size_t stage_cap = 0;
    bool fit_pending = false;

    // several models, one batch (gpk_acq_multi): buffers owned by the first handle of the call
    DevBuf multi_cand, multi_A, multi_B, multi_out, multi_bb;
    cudaEvent_t ev_multi = nullptr;
    // multi-GPU (gpk_comm_*): NCCL communicator bound at run time, one 16-byte pair per rank
    void* comm = nullptr;
    int rank = 0, world = 1;
    DevBuf gather, best_global;

    // entropy search (gpk_es.cuh): one state per handle, written by gpk_es_update
    DevBuf es_raw, es_scr, es_logP, es_dmu, es_dsig, es_dmumu, es_sweeps, es_F, es_jl, es_Bt, es_zb, es_zbop, es_W, es_lmb,
           es_cand, es_var, es_KZ, es_S, es_bb, es_best, es_lo, es_up;
    bool es_ready = false;
    int es_nb = 0, es_np = 0;
    double es_sn2 = 0.0, es_H = 0.0;
    long es_linv_serial = -1;
};

namespace {

void set_err(gpk_handle* h, const char* fmt, ...) {
    if (!h) return;
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(h->err, sizeof(h->err), fmt, ap);
    va_end(ap);
}

#define CK(call)                                                                                 \
    do {                                                                                         \
        cudaError_t e_ = (call);                                                                 \
        if (e_ != cudaSuccess) {                                                                 \
            set_err(h, "%s -> %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__);   \
            return GPK_CUDA_ERROR;                                                               \
        }                                                                                        \
    } while (0)

#define CKL()                                                                                    \
    do {                                                                                         \
        cudaError_t e_ = cudaGetLastError();                                                     \
        if (e_ != cudaSuccess) {                                                                 \
            set_err(h, "kernel launch -> %s (%s:%d)", cudaGetErrorString(e_), __FILE__, __LINE__); \
            return GPK_CUDA_ERROR;                                                               \
        }                                                                                        \
        h->launches_total += 1;                                                                  \
    } while (0)

#define BAD(...)                           \
    do {                                   \
        set_err(h, __VA_ARGS__);           \
        return GPK_BAD_ARG;                \
    } while (0)

int ensure(gpk_handle* h, DevBuf& b, size_t bytes, bool* grew = nullptr) {
    if (grew) *grew = false;
    if (bytes <= b.cap && b.p) return GPK_OK;
    if (b.p) CK(cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
    size_t want = std::max<size_t>(bytes, 256);
    CK(cudaMalloc(&b.p, want));
    b.cap = want;
    if (grew) *grew = true;
    return GPK_OK;
}

template <typename T> T* ptr(const DevBuf& b) { return reinterpret_cast<T*>(b.p); }

inline long round_up(long x, long m) { return (x + m - 1) / m * m; }

// ---- tensor maps ---------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// fp64 row-major matrix [rows][ld]; box = 128 rows x 16 doubles (128 B), 128B swizzle.
int make_map(gpk_handle* h, CUtensorMap* map, void* base, long rows, long cols, long ld, int box_rows = BM) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) {
        set_err(h, "cuTensorMapEncodeTiled entry point not available");
        return GPK_CUDA_ERROR;
    }
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 8};
    cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, base, dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_err(h, "cuTensorMapEncodeTiled failed with CUresult %d (rows=%ld cols=%ld ld=%ld)", (int)r, rows, cols, ld);
        return GPK_CUDA_ERROR;
    }
    return GPK_OK;
}

// term-major operand [n_terms][ld] of the covariance builder: box = n_terms rows x 128 columns, no swizzle
int make_cov_map(gpk_handle* h, CUtensorMap* map, void* base, int n_terms, long ld) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) {
        set_err(h, "cuTensorMapEncodeTiled entry point not available");
        return GPK_CUDA_ERROR;
    }
    cuuint64_t dims[2] = {(cuuint64_t)ld, (cuuint64_t)n_terms};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 8};
    cuuint32_t box[2] = {128u, (cuuint32_t)n_terms};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_err(h, "cuTensorMapEncodeTiled (covariance operand) failed with CUresult %d (terms=%d ld=%ld)", (int)r, n_terms, ld);
        return GPK_CUDA_ERROR;
    }
    return GPK_OK;
}

inline bool cov_tma(const gpk_handle* h) { return h->cov_kernel == 2 && h->loader != LOADER_CPASYNC; }

// "Transposed" operand of the covariance builder for n points X (row-major, n x d) into dst with ld columns:
// term-major + pre-scaled for the TMA kernel (dst needs n_terms x ld doubles), axis-major for the round-1 kernel
// (d x ld doubles).  lo / up: input bounds to apply first (NULL: none).
int build_cov_operand(gpk_handle* h, cudaStream_t st, const double* X, long n, int d, const double* lo, const double* up,
                      double* dst, long ld) {
    if (cov_tma(h)) {
        const long total = (long)h->spec.n_terms * ld;
        gpk_termmajor_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(h->spec, X, n, d, lo, up, dst, ld);
    } else {
        const long total = (long)d * ld;
        gpk_transpose_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(X, n, d, lo, up, dst, ld);
    }
    CKL();
    return GPK_OK;
}
inline size_t cov_operand_rows(const gpk_handle* h, int d) { return (size_t)std::max(d, h->spec.n_terms); }

// out[c][j] = k(cand_c, point_j) for m candidates (row-major raw inputs, bounds lo / up applied on the fly) against
// the n points of `operand` (built by build_cov_operand, ld = ldx columns); out has ldo columns and at least
// round_up(m, tile) rows.  small: the 128 x 16 tile variant that fits next to a resident variance-GEMM CTA.
int launch_cov_tiles(gpk_handle* h, cudaStream_t st, const double* operand, long ldx, int n, const double* cand, int dc,
                     long m, long m_padded, const double* lo, const double* up, double* out, long ldo, int tri, bool small) {
    const unsigned gx = (unsigned)(ldx / 128);
    if (cov_tma(h)) {
        CUtensorMap map;
        int rc = make_cov_map(h, &map, (void*)operand, h->spec.n_terms, ldx);
        if (rc) return rc;
        if (small)
            gpk_cov_tma_kernel<4><<<dim3(gx, (unsigned)(m_padded / 16)), 256, cov_tma_smem_bytes(h->spec.n_terms, 4), st>>>(
                map, h->spec, n, cand, dc, m, lo, up, out, ldo, tri);
        else
            gpk_cov_tma_kernel<8><<<dim3(gx, (unsigned)(m_padded / 32)), 256, cov_tma_smem_bytes(h->spec.n_terms, 8), st>>>(
                map, h->spec, n, cand, dc, m, lo, up, out, ldo, tri);
    } else if (small) {
        gpk_cov_kernel<8><<<dim3(gx, (unsigned)(m_padded / 16)), 256, 0, st>>>(h->spec, operand, ldx, n, cand, dc, m, lo, up, out, ldo, tri);
    } else {
        gpk_cov_kernel<16><<<dim3(gx, (unsigned)(m_padded / 32)), 256, 0, st>>>(h->spec, operand, ldx, n, cand, dc, m, lo, up, out, ldo, tri);
    }
    CKL();
    return GPK_OK;
}
inline const double* train_operand(const gpk_handle* h) { return cov_tma(h) ? ptr<double>(h->Xts) : ptr<double>(h->Xt); }

// ---- GEMM launch ---------------------------------------------------------------------------
// Launch with the programmatic-stream-serialization attribute (PDL): the kernel's launch latency and prologue
// overlap the tail of the previous kernel on the stream; the kernels call cudaGridDependencySynchronize().
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args... args) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// int8 contraction launch: optional CTA pair (cluster of 2) and optional programmatic dependency on the kernel launched
// just before it on the stream (the resident look-ahead K* builder, which triggers at its start)
template <typename... KArgs, typename... Args>
cudaError_t launch_oz(void (*kernel)(KArgs...), unsigned grid, size_t smem, cudaStream_t stream, bool pair, bool dependent, Args... args) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(OZ_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[2];
    int na = 0;
    if (pair) {
        attr[na].id = cudaLaunchAttributeClusterDimension;
        attr[na].val.clusterDim.x = 2; attr[na].val.clusterDim.y = 1; attr[na].val.clusterDim.z = 1;
        ++na;
    }
    if (dependent) {
        attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[na].val.programmaticStreamSerializationAllowed = 1;
        ++na;
    }
    cfg.attrs = attr;
    cfg.numAttrs = na;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

template <int EPI, int MI = 8>
int launch_gemm(gpk_handle* h, const CUtensorMap& mA, const CUtensorMap& mB, const GemmArgs& a, int njobs,
                cudaStream_t stream = nullptr, bool pdl = false) {
    if (njobs <= 0) return GPK_OK;
    if (stream == nullptr) stream = h->stream;
    if (pdl && h->pdl && h->loader != LOADER_CPASYNC && MI <= 2) {
        CK(launch_pdl(gpk_gemm_nt_kernel<EPI, LOADER_TMA, MI>, dim3(njobs), dim3(GEMM_THREADS),
                      (size_t)gemm_smem_bytes(LOADER_TMA, MI), stream, mA, mB, a));
        h->launches_total += 1;
        return GPK_OK;
    }
    if (h->loader == LOADER_TMA_WS && MI == 8)
        gpk_gemm_ws_kernel<EPI><<<njobs, WS_THREADS, GEMM_SMEM_TMA, stream>>>(mA, mB, a);
    else if (h->loader != LOADER_CPASYNC)
        gpk_gemm_nt_kernel<EPI, LOADER_TMA, MI><<<njobs, GEMM_THREADS, gemm_smem_bytes(LOADER_TMA, MI), stream>>>(mA, mB, a);
    else
        gpk_gemm_nt_kernel<EPI, LOADER_CPASYNC, MI><<<njobs, GEMM_THREADS, gemm_smem_bytes(LOADER_CPASYNC, MI), stream>>>(mA, mB, a);
    CKL();
    return GPK_OK;
}

int set_kernel_attrs(gpk_handle* h) {
    CK(cudaFuncSetAttribute(gpk_gemm_nt_kernel<EPI_STORE, LOADER_TMA, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_TMA));
    CK(cudaFuncSetAttribute(gpk_gemm_nt_kernel<EPI_COLREDUCE, LOADER_TMA, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_TMA));
    CK(cudaFuncSetAttribute(gpk_gemm_nt_kernel<EPI_STORE, LOADER_CPASYNC, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_PAD));
    CK(cudaFuncSetAttribute(gpk_gemm_nt_kernel<EPI_COLREDUCE, LOADER_CPASYNC, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_PAD));
    CK(cudaFuncSetAttribute(gpk_gemm_ws_kernel<EPI_STORE>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_TMA));
    CK(cudaFuncSetAttribute(gpk_gemm_ws_kernel<EPI_COLREDUCE>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_TMA));
    CK(cudaFuncSetAttribute(gpk_gemm_nt_kernel<EPI_STORE, LOADER_TMA, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, gemm_smem_bytes(LOADER_TMA, 2)));
    CK(cudaFuncSetAttribute(gpk_gemm_nt_kernel<EPI_STORE, LOADER_CPASYNC, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, gemm_smem_bytes(LOADER_CPASYNC, 2)));
    CK(cudaFuncSetAttribute(gpk_gemm_nt_kernel<EPI_STORE, LOADER_CPASYNC, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, gemm_smem_bytes(LOADER_CPASYNC, 1)));
    CK(cudaFuncSetAttribute(gpk_gemm_nt_kernel<EPI_STORE, LOADER_TMA, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, gemm_smem_bytes(LOADER_TMA, 1)));
    CK(cudaFuncSetAttribute(gpk_oz_vargemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, OZ_SMEM));
    CK(cudaFuncSetAttribute(gpk_oz_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, OZP_SMEM));
    CK(cudaFuncSetAttribute(gpk_oz_pair2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, OZQ_SMEM));
    CK(cudaFuncSetAttribute(gpk_oz_persist_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, OZ_PERSIST_SMEM));
    CK(cudaFuncSetAttribute(gpk_oz_persist_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, OZP_PERSIST_SMEM));
    CK(cudaFuncSetAttribute(gpk_oz2_vargemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, OZ2_SMEM));
    CK(cudaFuncSetAttribute(gpk_cov_oz_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cov_oz_smem_bytes(GPK_MAX_TERMS, 8)));
    CK(cudaFuncSetAttribute(gpk_cov_oz_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cov_oz_smem_bytes(GPK_MAX_TERMS, 4)));
    CK(cudaFuncSetAttribute(gpk_vargemm_persistent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PV_SMEM));
    {
        cudaDeviceProp prop;
        CK(cudaGetDeviceProperties(&prop, h->device));
        h->n_sm = prop.multiProcessorCount;
    }
    CK(cudaFuncSetAttribute(gpk_cov_tma_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cov_tma_smem_bytes(GPK_MAX_TERMS, 8)));
    CK(cudaFuncSetAttribute(gpk_cov_tma_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cov_tma_smem_bytes(GPK_MAX_TERMS, 4)));
    CK(cudaFuncSetAttribute(gpk_potrf_diag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DIAG_SMEM));
    CK(cudaFuncSetAttribute(gpk_potrf_diag_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DIAG2_SMEM));
    CK(cudaFuncSetAttribute(gpk_chain_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, CH_SMEM));
    CK(cudaFuncSetAttribute(gpk_potrf_diag_blocked_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DIAG3_SMEM));
    CK(cudaFuncSetAttribute(gpk_potrf_diag_dmma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DIAG4_SMEM));
    return GPK_OK;
}

// ---- job tables ----------------------------------------------------------------------------
struct Node { int lo, mid, hi, height; };

int build_nodes(int lo, int hi, std::vector<Node>& nodes) {
    if (hi - lo <= 1) return 0;
    int mid = lo + (hi - lo + 1) / 2;
    int hl = build_nodes(lo, mid, nodes);
    int hr = build_nodes(mid, hi, nodes);
    int ht = 1 + std::max(hl, hr);
    nodes.push_back({lo, mid, hi, ht});
    return ht;
}

int build_job_tables(gpk_handle* h) {
    const int nb = h->nb;
    if (h->jobs_nb == nb) return GPK_OK;
    std::vector<GemmJob> jobs;
    h->trsm_r.assign(nb, Range());
    h->syrk_r.assign(nb, Range());
    for (int k = 0; k < nb; ++k) {
        h->trsm_r[k].off = (int)jobs.size();
        for (int i = k + 1; i <= nb; ++i)          // i == nb: augmented rhs block row
            jobs.push_back({i * BM, k * BM, k * BM, (k + 1) * BM, i * BM, k * BM, 0, 0});
        h->trsm_r[k].cnt = (int)jobs.size() - h->trsm_r[k].off;
        h->syrk_r[k].off = (int)jobs.size();
        for (int j = k + 1; j < nb; ++j)
            for (int i = j; i <= nb; ++i)
                jobs.push_back({i * BM, j * BM, k * BM, (k + 1) * BM, i * BM, j * BM, 0, 0});
        h->syrk_r[k].cnt = (int)jobs.size() - h->syrk_r[k].off;
    }
    // depth-2 trailing update (odd steps k >= 1): tile (i, j), j >= k+2, receives panels k-1 and k in ONE contraction
    // over the 256 columns [(k-1)*128, (k+1)*128): same arithmetic, in the same order, as the two separate updates
    h->syrk2_r.assign(nb, Range());
    for (int k = 1; k < nb; k += 2) {
        h->syrk2_r[k].off = (int)jobs.size();
        for (int j = k + 2; j < nb; ++j)
            for (int i = j; i <= nb; ++i)
                jobs.push_back({i * BM, j * BM, (k - 1) * BM, (k + 1) * BM, i * BM, j * BM, 0, 0});
        h->syrk2_r[k].cnt = (int)jobs.size() - h->syrk2_r[k].off;
    }
    // 32-row versions of the two GEMMs on the critical chain (row split only: the in-place panel solve
    // stays race-free because every CTA reads and writes its own rows)
    h->trsm32_r.assign(nb, Range());
    h->pu32_r.assign(nb, Range());
    for (int k = 0; k < nb; ++k) {
        h->trsm32_r[k].off = (int)jobs.size();
        for (int i = k + 1; i <= nb; ++i)
            for (int q = 0; q < 4; ++q) {
                if (i == nb && q > 0) break;         // augmented block: only its first rows are non-zero
                jobs.push_back({i * BM + 32 * q, k * BM, k * BM, (k + 1) * BM, i * BM + 32 * q, k * BM, 0, 0});
            }
        h->trsm32_r[k].cnt = (int)jobs.size() - h->trsm32_r[k].off;
        h->pu32_r[k].off = (int)jobs.size();
        if (k + 1 < nb)
            for (int i = k + 1; i <= nb; ++i)
                for (int q = 0; q < 4; ++q) {
                    if (i == nb && q > 0) break;
                    jobs.push_back({i * BM + 32 * q, (k + 1) * BM, k * BM, (k + 1) * BM, i * BM + 32 * q, (k + 1) * BM, 0, 0});
                }
        h->pu32_r[k].cnt = (int)jobs.size() - h->pu32_r[k].off;
    }
    // 16-row versions (option smalltile = 2): twice the CTAs, half the arithmetic per CTA on the chain
    h->trsm16_r.assign(nb, Range());
    h->pu16_r.assign(nb, Range());
    for (int k = 0; k < nb; ++k) {
        h->trsm16_r[k].off = (int)jobs.size();
        for (int i = k + 1; i <= nb; ++i)
            for (int q = 0; q < 8; ++q) {
                if (i == nb && q > 0) break;
                jobs.push_back({i * BM + 16 * q, k * BM, k * BM, (k + 1) * BM, i * BM + 16 * q, k * BM, 0, 0});
            }
        h->trsm16_r[k].cnt = (int)jobs.size() - h->trsm16_r[k].off;
        h->pu16_r[k].off = (int)jobs.size();
        if (k + 1 < nb)
            for (int i = k + 1; i <= nb; ++i)
                for (int q = 0; q < 8; ++q) {
                    if (i == nb && q > 0) break;
                    jobs.push_back({i * BM + 16 * q, (k + 1) * BM, k * BM, (k + 1) * BM, i * BM + 16 * q, (k + 1) * BM, 0, 0});
                }
        h->pu16_r[k].cnt = (int)jobs.size() - h->pu16_r[k].off;
    }
    std::vector<Node> nodes;
    int hmax = build_nodes(0, nb, nodes);
    h->tri1_r.assign(hmax + 1, Range());
    h->tri2_r.assign(hmax + 1, Range());
    auto by_len = [](const GemmJob& a, const GemmJob& b) { return (a.k1 - a.k0) > (b.k1 - b.k0); };
    for (int ht = 1; ht <= hmax; ++ht) {
        size_t s1 = jobs.size();
        for (const Node& nd : nodes) {
            if (nd.height != ht) continue;
            for (int c = nd.lo; c < nd.mid; ++c)
                for (int i = nd.mid; i < nd.hi; ++i)   // T'[c][i] = sum_{k=c..mid} Q[c][k] L[i][k]
                    jobs.push_back({c * BM, i * BM, c * BM, nd.mid * BM, c * BM, i * BM, 0, 0});
        }
        std::stable_sort(jobs.begin() + s1, jobs.end(), by_len);
        h->tri1_r[ht].off = (int)s1;
        h->tri1_r[ht].cnt = (int)(jobs.size() - s1);
        size_t s2 = jobs.size();
        for (const Node& nd : nodes) {
            if (nd.height != ht) continue;
            for (int i = nd.mid; i < nd.hi; ++i)
                for (int c = nd.lo; c < nd.mid; ++c)   // R[i][c] = -sum_{k=mid..i} P[i][k] T'[c][k]
                    jobs.push_back({i * BM, c * BM, nd.mid * BM, (i + 1) * BM, i * BM, c * BM, 0, 0});
        }
        std::stable_sort(jobs.begin() + s2, jobs.end(), by_len);
        h->tri2_r[ht].off = (int)s2;
        h->tri2_r[ht].cnt = (int)(jobs.size() - s2);
    }
    // K^-1 = Q Q^T (lower tiles), Q = L^-T upper: K^-1[i][j] = sum_{k >= i} Q[i][k] Q[j][k], i >= j
    h->kinv_r.off = (int)jobs.size();
    for (int j = 0; j < nb; ++j)
        for (int i = j; i < nb; ++i)
            jobs.push_back({i * BM, j * BM, i * BM, nb * BM, i * BM, j * BM, 0, 0});
    std::stable_sort(jobs.begin() + h->kinv_r.off, jobs.end(), by_len);
    h->kinv_r.cnt = (int)jobs.size() - h->kinv_r.off;
    // gpk_fit_append: only block row b = nb-1 changes.  N1 = b*128 leading rows keep their factor L11 and inverse P11.
    {
        const int b = nb - 1, N1 = b * BM;
        // L_row = K[b, 0:N1] P11^T, 32-row tiles (the contraction is up to N1 long: more, shorter CTAs)
        h->app_row_r.off = (int)jobs.size();
        for (int j = b - 1; j >= 0; --j)
            for (int q = 0; q < 4; ++q)
                jobs.push_back({N1 + 32 * q, j * BM, 0, (j + 1) * BM, N1 + 32 * q, j * BM, 0, 0});
        h->app_row_r.cnt = (int)jobs.size() - h->app_row_r.off;
        // partial Gram tiles  T_s = L_row[:, s] L_row[:, s]^T  into the free tiles (s, b) of W; summed in fixed order
        h->app_syrk_r.off = (int)jobs.size();
        for (int sblk = 0; sblk < b; ++sblk)
            jobs.push_back({N1, N1, sblk * BM, (sblk + 1) * BM, sblk * BM, N1, 0, 0});
        h->app_syrk_r.cnt = (int)jobs.size() - h->app_syrk_r.off;
        // T = L_row P11 (= L_row Q11^T in NT form), 32-row tiles, stored to P[b, :] and transposed to Q[:, b]
        h->app_t_r.off = (int)jobs.size();
        for (int j = 0; j < b; ++j)
            for (int q = 0; q < 4; ++q)
                jobs.push_back({N1 + 32 * q, j * BM, j * BM, N1, N1 + 32 * q, j * BM, 0, 0});
        h->app_t_r.cnt = (int)jobs.size() - h->app_t_r.off;
        // split-K versions (default): 128-row tiles, the contraction cut into chunks of APP_KC columns, partial tile
        // (chunk c, column block j) -> scratch tile W(c, j); summed in fixed order by gpk_append_reduce_kernel
        h->app_row2_r.off = (int)jobs.size();
        for (int j = b - 1; j >= 0; --j)
            for (int c = 0, k0 = 0; k0 < (j + 1) * BM; ++c, k0 += APP_KC)
                jobs.push_back({N1, j * BM, k0, std::min(k0 + APP_KC, (j + 1) * BM), c * BM, j * BM, 0, 0});
        h->app_row2_r.cnt = (int)jobs.size() - h->app_row2_r.off;
        h->app_t2_r.off = (int)jobs.size();
        for (int j = 0; j < b; ++j)
            for (int c = 0, k0 = j * BM; k0 < N1; ++c, k0 += APP_KC)
                jobs.push_back({N1, j * BM, k0, std::min(k0 + APP_KC, N1), c * BM, j * BM, 0, 0});
        h->app_t2_r.cnt = (int)jobs.size() - h->app_t2_r.off;
        // P[b, j] = -P_bb T[:, j]
        h->app_p_r.off = (int)jobs.size();
        for (int j = 0; j < b; ++j)
            jobs.push_back({N1, j * BM, N1, nb * BM, N1, j * BM, 0, 0});
        h->app_p_r.cnt = (int)jobs.size() - h->app_p_r.off;
    }
    if (jobs.empty()) jobs.push_back({0, 0, 0, 0, 0, 0, 0, 0});
    int rc = ensure(h, h->jobs, jobs.size() * sizeof(GemmJob));
    if (rc) return rc;
    CK(cudaMemcpyAsync(h->jobs.p, jobs.data(), jobs.size() * sizeof(GemmJob), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->jobs_nb = nb;
    return GPK_OK;
}

int rebuild_maps(gpk_handle* h) {
    if (h->loader == LOADER_CPASYNC) { h->maps_ok = true; return GPK_OK; }
    const long NP = h->NP;
    int rc;
    if ((rc = make_map(h, &h->mapK, h->Kbuf.p, NP + BM, NP, NP))) return rc;
    if ((rc = make_map(h, &h->mapK32, h->Kbuf.p, NP + BM, NP, NP, 32))) return rc;
    if ((rc = make_map(h, &h->mapK16, h->Kbuf.p, NP + BM, NP, NP, 16))) return rc;
    if ((rc = make_map(h, &h->mapP, h->P.p, NP, NP, NP))) return rc;
    if ((rc = make_map(h, &h->mapQ, h->Q.p, NP, NP, NP))) return rc;
    if ((rc = make_map(h, &h->mapW, h->W.p, NP, NP, NP))) return rc;
    h->mapKs_rows = 0;
    h->mapKs2_rows = 0;
    h->mapVt_rows = 0;
    h->maps_ok = true;
    return GPK_OK;
}

// scratch for scoring `rows` (multiple of 128) candidates at once
int ensure_score_scratch(gpk_handle* h, long rows) {
    const long NP = h->NP;
    bool grew = false;
    int rc;
    if ((rc = ensure(h, h->Kstar, (size_t)rows * NP * 8, &grew))) return rc;
    if (grew || h->mapKs_rows != rows) {
        if (h->loader != LOADER_CPASYNC && (rc = make_map(h, &h->mapKs, h->Kstar.p, rows, NP, NP))) return rc;
        h->mapKs_rows = rows;
    }
    if (h->overlap) {
        if ((rc = ensure(h, h->Kstar2, (size_t)rows * NP * 8, &grew))) return rc;
        if (grew || h->mapKs2_rows != rows) {
            if (h->loader != LOADER_CPASYNC && (rc = make_map(h, &h->mapKs2, h->Kstar2.p, rows, NP, NP))) return rc;
            h->mapKs2_rows = rows;
        }
    }
    if ((rc = ensure(h, h->part_mu, (size_t)h->nb * rows * 8))) return rc;
    if ((rc = ensure(h, h->part_ssq, (size_t)h->nb * rows * 8))) return rc;
    if ((rc = ensure(h, h->block_best, (size_t)(rows / 256 + 1) * sizeof(BestPair)))) return rc;
    if ((rc = ensure(h, h->best, sizeof(BestPair)))) return rc;
    if ((rc = ensure(h, h->nneg, 8))) return rc;
    return GPK_OK;
}

__global__ void gpk_fit_reduce_kernel(const double* __restrict__ z, int n, const double* __restrict__ logdet_part,
                                      int nb, double* __restrict__ out2) {
    // single block, fixed summation order: out2[0] = z^T z, out2[1] = 2 * sum log diag
    __shared__ double sh[256];
    double s = 0.0;
    for (int i = threadIdx.x; i < n; i += 256) s = fma(z[i], z[i], s);
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        out2[0] = sh[0];
        double l = 0.0;
        for (int k = 0; k < nb; ++k) l += logdet_part[k];
        out2[1] = 2.0 * l;
    }
}

// mu_c = sum_k M[c][k] * z[k] over k in [k_lo(c), NP): one warp per row (tri: k >= c)
__global__ void gpk_rowdot_kernel(const double* __restrict__ M, long ld, long rows, int NP, int tri,
                                  const double* __restrict__ z, double* __restrict__ out) {
    long row = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (row >= rows) return;
    double s = 0.0;
    int kstart = tri ? (int)(row & ~31L) : 0;
    for (int k = kstart + lane; k < NP; k += 32)
        if (!tri || k >= row) s = fma(M[row * ld + k], z[k], s);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    if (lane == 0) out[row] = s;
}

__global__ void gpk_mu_finish_kernel(double* __restrict__ mu, long m, double mean, int norm_out, double y_mean,
                                     double y_std) {
    long c = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= m) return;
    double v = mu[c] + mean;
    if (norm_out) v = v * y_std + y_mean;
    mu[c] = v;
}

// gpk_fit_append helpers -------------------------------------------------------------------
// diagonal of the rows [i0, NP): += diag_add for training rows, unit diagonal on padding rows
__global__ void gpk_kfix_rows_kernel(double* __restrict__ K, long ld, int n, int NP, double diag_add, int i0) {
    int i = i0 + blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= NP) return;
    K[(long)i * ld + i] = (i < n) ? K[(long)i * ld + i] + diag_add : 1.0;
}

// dst[:, j-block] = sum_c W(c, j) over the nc(j) partial tiles of column block j (c ascending: deterministic);
// mode 0: nc = ceil((j + 1) * 128 / APP_KC) (L_row), mode 1: nc = ceil((b - j) * 128 / APP_KC) (L_row P11).
// dstT (may be NULL) receives the transpose: dstT[j*128 + c][r].  grid = (b, 64), 256 threads, one element each.
__global__ void gpk_append_reduce_kernel(const double* __restrict__ W, long ld, int b, int mode, double* __restrict__ dst,
                                         long ldd, double* __restrict__ dstT, long lddT, int tcol0) {
    const int j = blockIdx.x;
    const int e = blockIdx.y * 256 + threadIdx.x;              // 0 .. 128*128-1
    const int r = e >> 7, c = e & 127;
    const int len = mode == 0 ? (j + 1) * 128 : (b - j) * 128;
    const int nc = (len + APP_KC - 1) / APP_KC;
    double acc = 0.0;
    for (int q = 0; q < nc; ++q) acc += W[(long)(q * 128 + r) * ld + j * 128 + c];
    dst[(long)r * ldd + j * 128 + c] = acc;
    if (dstT != nullptr) dstT[(long)(j * 128 + c) * lddT + tcol0 + r] = acc;
}

// K[b,b] -= sum_s T_s with T_s = W tile (s, b), s ascending (deterministic); one thread per element
__global__ void gpk_append_schur_kernel(double* __restrict__ K, const double* __restrict__ W, long ld, int N1, int nparts) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;         // 0 .. 128*128-1
    const int i = e >> 7, c = e & 127;
    double acc = 0.0;
    for (int sblk = 0; sblk < nparts; ++sblk) acc += W[(long)(sblk * 128 + i) * ld + N1 + c];
    K[(long)(N1 + i) * ld + N1 + c] -= acc;
}

__global__ void gpk_resid_kernel(const double* __restrict__ y, double mean, int n, int NP, double* __restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < NP) out[i] = (i < n) ? y[i] - mean : 0.0;
}

int require(gpk_handle* h, bool data, bool spec, bool fitted) {
    if (!h) return GPK_BAD_ARG;
    if (data && !h->has_data) { set_err(h, "gpk_set_data has not been called"); return GPK_BAD_ARG; }
    if (spec && !h->has_spec) { set_err(h, "gpk_set_kernel has not been called"); return GPK_BAD_ARG; }
    if (fitted && !h->fitted) { set_err(h, "model is not fitted (gpk_fit)"); return GPK_NOT_FITTED; }
    return GPK_OK;
}

// L^-1 by recursive block inversion (P lower, Q = P^T upper), after a successful fit.
int build_linv(gpk_handle* h) {
    if (h->linv_ready) return GPK_OK;
    CK(cudaEventRecord(h->ev[4], h->stream));
    const long NP = h->NP;
    const int hmax = (int)h->tri1_r.size() - 1;
    for (int ht = 1; ht <= hmax; ++ht) {
        GemmArgs a;
        memset(&a, 0, sizeof(a));
        a.A = ptr<double>(h->Q); a.lda = NP;
        a.B = ptr<double>(h->Kbuf); a.ldb = NP;
        a.C = ptr<double>(h->W); a.ldc = NP;
        a.alpha = 1.0; a.beta = 0;
        a.jobs = ptr<GemmJob>(h->jobs) + h->tri1_r[ht].off;
        a.job_mode = JOBS_TABLE;
        int rc = launch_gemm<EPI_STORE>(h, h->mapQ, h->mapK, a, h->tri1_r[ht].cnt);
        if (rc) return rc;
        GemmArgs b;
        memset(&b, 0, sizeof(b));
        b.A = ptr<double>(h->P); b.lda = NP;
        b.B = ptr<double>(h->W); b.ldb = NP;
        b.C = ptr<double>(h->P); b.ldc = NP;
        b.Ct = ptr<double>(h->Q); b.ldct = NP;
        b.alpha = -1.0; b.beta = 0;
        b.jobs = ptr<GemmJob>(h->jobs) + h->tri2_r[ht].off;
        b.job_mode = JOBS_TABLE;
        rc = launch_gemm<EPI_STORE>(h, h->mapP, h->mapW, b, h->tri2_r[ht].cnt);
        if (rc) return rc;
    }
    CK(cudaEventRecord(h->ev[5], h->stream));
    h->linv_ready = true;
    h->linv_serial += 1;
    return GPK_OK;
}

// int8 tensor map over S stacked slice matrices [S * rows][cols] (int8, K contiguous): box = 64 bytes x box_rows, 64B swizzle
int make_oz_map(gpk_handle* h, CUtensorMap* map, void* base, long rows_total, long cols, int box_rows, int box_bytes = OZ_KB) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) { set_err(h, "cuTensorMapEncodeTiled entry point not available"); return GPK_CUDA_ERROR; }
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows_total};
    cuuint64_t strides[1] = {(cuuint64_t)cols};
    cuuint32_t box[2] = {(cuuint32_t)box_bytes, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    box_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_err(h, "cuTensorMapEncodeTiled (int8 slices) failed with CUresult %d", (int)r); return GPK_CUDA_ERROR; }
    return GPK_OK;
}

// Slices of L^-1 for the int8 contraction, once per factorisation.  Returns true in *usable when the factor is
// conditioned well enough for S = 8 slices (row exponents <= OZ_MAX_EXP) and the sizes fit the int32 accumulators.
int prepare_ozaki(gpk_handle* h, bool* usable) {
    *usable = false;
    if (!h->ozaki || h->loader == LOADER_CPASYNC || h->NP > 16384) return GPK_OK;
    const long NP = h->NP;
    if (h->oz_linv_serial != h->linv_serial) {
        int rc;
        if ((rc = ensure(h, h->oz_Pq, (size_t)OZ_S * NP * NP))) return rc;
        if ((rc = ensure(h, h->oz_eP, (size_t)NP * 4))) return rc;
        if ((rc = ensure(h, h->oz_emax, 4))) return rc;
        const int lowest = -100000;
        CK(cudaMemcpyAsync(h->oz_emax.p, &lowest, 4, cudaMemcpyHostToDevice, h->stream));
        gpk_oz_rowexp_kernel<<<(unsigned)NP, 256, 0, h->stream>>>(ptr<double>(h->P), NP, (int)NP, ptr<int>(h->oz_eP), ptr<int>(h->oz_emax));
        CKL();
        gpk_oz_split_kernel<<<(unsigned)((NP * NP + 255) / 256), 256, 0, h->stream>>>(ptr<double>(h->P), NP, NP, ptr<int>(h->oz_eP), 0,
                                                                                   ptr<int8_t>(h->oz_Pq), NP * NP);
        CKL();
        // alpha = L^-T z (Q = L^-T is upper triangular): the mean goes through fp64, mu - mean = K* alpha
        if ((rc = ensure(h, h->alpha, (size_t)NP * 8))) return rc;
        gpk_rowdot_kernel<<<(unsigned)((NP + 7) / 8), 256, 0, h->stream>>>(ptr<double>(h->Q), NP, NP, (int)NP, 1,
                                                                           ptr<double>(h->Kbuf) + NP * NP, ptr<double>(h->alpha));
        CKL();
        CK(cudaMemcpyAsync(&h->oz_emax_host, h->oz_emax.p, 4, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        if ((rc = make_oz_map(h, &h->mapOzP, h->oz_Pq.p, (long)OZ_S * NP, NP, OZ_TM))) return rc;
        h->oz_linv_serial = h->linv_serial;
    }
    *usable = h->oz_emax_host <= OZ_MAX_EXP;
    return GPK_OK;
}

// Candidates per scoring pass.  Unless the caller fixed it ("chunk" option) the K* buffer is kept at about 512 MB:
// 16384 candidates at N = 4096, 65536 at N <= 1024 (fewer, longer launches where a candidate costs only N^2 = 1 MFLOP).
long chunk_rows(const gpk_handle* h) {
    if (h->chunk_user) return h->chunk;
    long c = ((1L << 26) / std::max(h->NP, 128)) / BM * BM;
    return std::min<long>(65536, std::max<long>(4096, c));
}

// Host batches are fed to score_dev chunk by chunk: ready(lo, hi, st) makes sure the candidate rows [lo, hi) are on
// their way to the device buffer and lets stream `st` wait for them (gpk_acq: H2D of chunk i+1, and for pageable memory
// the host staging copy, overlap the scoring of chunk i inside ONE scoring pass with full K* look-ahead).
struct Feeder {
    virtual int ready(long lo, long hi, cudaStream_t st) = 0;
    virtual ~Feeder() {}
};

// Score m candidates resident on the device.  All output pointers are device pointers or NULL.
// index_offset: position of dX[0] in the caller's batch (offset into the output arrays and into the arg-max index);
// global_base: added to the arg-max index only (first index of this rank's shard in a sharded batch); reset: start a
// new running arg-max / negative-EI count (false when a host batch is fed in several pieces)
int score_dev(gpk_handle* h, const double* dX, long m, int kind, double eta, double par, double* d_out,
              double* d_mu, double* d_var, BestPair* d_best, unsigned long long* d_nneg,
              long index_offset = 0, bool reset = true, long global_base = 0, Feeder* feeder = nullptr) {
    int rc = build_linv(h);
    if (rc) return rc;
    const long NP = h->NP;
    const long cap = std::min<long>(chunk_rows(h), round_up(std::max<long>(m, 1), BM));
    if ((rc = ensure_score_scratch(h, cap))) return rc;
    // int8 path only for batches that amortise slicing L^-1 (once per fit, ~0.4 ms at N = 4096)
    bool use_oz = false;
    if (m >= 2048 && (rc = prepare_ozaki(h, &use_oz))) return rc;
    int oz_eK = 0;
    const bool oz_fused = use_oz && h->oz_fused && cov_tma(h);
    if (use_oz) {
        // slices of K* per chunk buffer: [S][cap][NP] int8; one exponent for the whole matrix (0 < k <= amp)
        // (the tensor maps are re-encoded per call: a few microseconds, and they depend on the buffer, cap and NP)
        if ((rc = ensure(h, h->oz_Kq, (size_t)OZ_S * cap * NP))) return rc;
        if (h->overlap && (rc = ensure(h, h->oz_Kq2, (size_t)OZ_S * cap * NP))) return rc;
        if ((rc = make_oz_map(h, &h->mapOzK, h->oz_Kq.p, (long)OZ_S * cap, NP, OZ_TN))) return rc;
        if (h->overlap && (rc = make_oz_map(h, &h->mapOzK2, h->oz_Kq2.p, (long)OZ_S * cap, NP, OZ_TN))) return rc;
        if (h->oz_tile == 128) {
            if ((rc = ensure(h, h->oz_scratch, (size_t)OZ2_SCRATCH_SLOTS * OZ2_T * OZ2_T * 8))) return rc;
            if ((rc = make_oz_map(h, &h->mapOzP32, h->oz_Pq.p, (long)OZ_S * NP, NP, OZ2_T, OZ2_KB))) return rc;
            if ((rc = make_oz_map(h, &h->mapOzK32, h->oz_Kq.p, (long)OZ_S * cap, NP, OZ2_T, OZ2_KB))) return rc;
            if (h->overlap && (rc = make_oz_map(h, &h->mapOzK32b, h->oz_Kq2.p, (long)OZ_S * cap, NP, OZ2_T, OZ2_KB))) return rc;
        } else {
            if (h->oz_pair) {
                if ((rc = make_oz_map(h, &h->mapOzKh, h->oz_Kq.p, (long)OZ_S * cap, NP, OZP_BH))) return rc;
                if (h->overlap && (rc = make_oz_map(h, &h->mapOzKh2, h->oz_Kq2.p, (long)OZ_S * cap, NP, OZP_BH))) return rc;
            }
        }
        if ((rc = ensure(h, h->oz_mu, (size_t)cap * 8))) return rc;
        if (h->overlap && (rc = ensure(h, h->oz_mu2, (size_t)cap * 8))) return rc;
        if (h->overlap && (rc = ensure(h, h->oz_pmu2, (size_t)h->nb * cap * 8))) return rc;
        oz_eK = oz_exponent(h->spec.amp);
    }
    if (d_best == nullptr) d_best = ptr<BestPair>(h->best);
    if (d_nneg == nullptr) d_nneg = ptr<unsigned long long>(h->nneg);
    if (reset) {
        CK(cudaMemsetAsync(d_best, 0xFF, sizeof(BestPair), h->stream));
        CK(cudaMemsetAsync(d_nneg, 0, 8, h->stream));
    }
    CK(cudaEventRecord(h->ev[6], h->stream));
    const int nchunks = (int)((m + cap - 1) / cap);
    // With more than one chunk, K* of chunk i+1 is built on the low-priority side stream (8 candidates
    // per thread, ~60 registers: its CTAs fit next to the resident GEMM CTAs and use the FP64 ALUs while
    // the GEMM keeps the DMMA pipe busy); two K* buffers alternate.
    const bool pipelined = h->overlap && nchunks > 1;
    if (pipelined) {
        while ((int)h->ev_cov.size() < nchunks) {
            cudaEvent_t e1, e2;
            CK(cudaEventCreateWithFlags(&e1, cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&e2, cudaEventDisableTiming));
            h->ev_cov.push_back(e1);
            h->ev_gemm.push_back(e2);
        }
    }
    while ((int)h->ev_g0.size() < nchunks) {
        cudaEvent_t e1, e2;
        CK(cudaEventCreate(&e1));
        CK(cudaEventCreate(&e2));
        h->ev_g0.push_back(e1);
        h->ev_g1.push_back(e2);
    }
    h->last_nchunks = nchunks;
    auto launch_cov = [&](int ci, cudaStream_t st, bool small, bool resident = false) -> int {
        const long base = (long)ci * cap;
        const long mc = std::min(cap, m - base);
        const long mcp = round_up(mc, BM);
        double* dst = (pipelined && (ci & 1)) ? ptr<double>(h->Kstar2) : ptr<double>(h->Kstar);
        if (feeder) {
            int frc = feeder->ready(base, base + mc, st);
            if (frc) return frc;
        }
        const double* lo = h->has_bounds ? ptr<double>(h->lower) : nullptr;
        const double* up = h->has_bounds ? ptr<double>(h->upper) : nullptr;
        int8_t* qdst = (pipelined && (ci & 1)) ? ptr<int8_t>(h->oz_Kq2) : ptr<int8_t>(h->oz_Kq);
        if (use_oz && oz_fused) {
            // K* never reaches HBM in fp64: digits + this tile's share of the mean straight out of the builder
            CUtensorMap map;
            int mrc = make_cov_map(h, &map, (void*)train_operand(h), h->spec.n_terms, NP);
            if (mrc) return mrc;
            double* pmu = (pipelined && (ci & 1)) ? ptr<double>(h->oz_pmu2) : ptr<double>(h->part_mu);
            const int gx = (int)(NP / 128);
            if (small) {
                const int gy = (int)(mcp / 16);
                const long items = (long)gx * gy;
                const unsigned grid = resident ? (unsigned)std::min<long>(items, (long)std::max(h->n_sm, 1) * h->cov_ctas) : (unsigned)items;
                gpk_cov_oz_kernel<4><<<grid, 256, cov_oz_smem_bytes(h->spec.n_terms, 4), st>>>(
                    map, h->spec, h->n, dX + base * h->d, h->d, mc, lo, up, ptr<double>(h->alpha), oz_eK, qdst, NP, cap * NP, pmu, cap,
                    gx, gy, resident ? 1 : 0);
            } else {
                const int gy = (int)(mcp / 32);
                gpk_cov_oz_kernel<8><<<(unsigned)((long)gx * gy), 256, cov_oz_smem_bytes(h->spec.n_terms, 8), st>>>(
                    map, h->spec, h->n, dX + base * h->d, h->d, mc, lo, up, ptr<double>(h->alpha), oz_eK, qdst, NP, cap * NP, pmu, cap,
                    gx, gy, 0);
            }
            CKL();
            return GPK_OK;
        }
        int crc = launch_cov_tiles(h, st, train_operand(h), NP, h->n, dX + base * h->d, h->d, mc, mcp, lo, up, dst, NP, 0, small);
        if (crc || !use_oz) return crc;
        // int8 slices of this chunk's K* (rows beyond mc are exact zeros in K*, so are their digits)
        gpk_oz_split_kernel<<<(unsigned)((mcp * NP + 255) / 256), 256, 0, st>>>(dst, mcp, NP, nullptr, oz_eK, qdst, cap * NP);
        CKL();
        // the mean of this chunk in fp64: one warp per candidate, K*[c, :] . alpha
        double* mdst = (pipelined && (ci & 1)) ? ptr<double>(h->oz_mu2) : ptr<double>(h->oz_mu);
        gpk_rowdot_kernel<<<(unsigned)((mcp + 7) / 8), 256, 0, st>>>(dst, NP, mcp, (int)NP, 0, ptr<double>(h->alpha), mdst);
        CKL();
        return GPK_OK;
    };
    // int8 path with the fused builder: everything on ONE stream.  The builder of chunk i+1 is a small resident grid
    // (cov_ctas CTAs per SM) that triggers its dependents at once; the contraction of chunk i behind it is launched with
    // the programmatic-stream-serialization attribute, so it starts while the builder runs and the two share the SMs
    // (FP64 ALU + tensor pipe).  With two streams the block scheduler only placed the builder in the contraction's tail.
    const bool chained = pipelined && oz_fused && h->oz_pdl;
    if (chained) {
        if ((rc = launch_cov(0, h->stream, false))) return rc;
    } else if (pipelined) {
        CK(cudaEventRecord(h->ev_order, h->stream));          // side stream starts after all prior work
        CK(cudaStreamWaitEvent(h->side_stream, h->ev_order, 0));
        if ((rc = launch_cov(0, h->side_stream, false))) return rc;
        CK(cudaEventRecord(h->ev_cov[0], h->side_stream));
    }
    for (int ci = 0; ci < nchunks; ++ci) {
        const long base = (long)ci * cap;
        const long mc = std::min(cap, m - base);
        const long mcp = round_up(mc, BM);
        const bool last = ci == nchunks - 1;
        if (last) CK(cudaEventRecord(h->ev[8], h->stream));
        bool dependent = false;                                 // the contraction below is the dependent of a resident builder
        if (chained) {
            if (last) CK(cudaEventRecord(h->ev[10], h->stream));
            CK(cudaEventRecord(h->ev_g0[ci], h->stream));       // nothing may sit between the builder and its dependent
            if (ci + 1 < nchunks) {
                if ((rc = launch_cov(ci + 1, h->stream, true, true))) return rc;
                dependent = true;
            }
        } else if (pipelined) {
            CK(cudaStreamWaitEvent(h->stream, h->ev_cov[ci], 0));
            if (ci + 1 < nchunks) {
                if (ci >= 1) CK(cudaStreamWaitEvent(h->side_stream, h->ev_gemm[ci - 1], 0));   // buffer (ci+1)&1 is free
                if ((rc = launch_cov(ci + 1, h->side_stream, true))) return rc;
                CK(cudaEventRecord(h->ev_cov[ci + 1], h->side_stream));
            }
        } else {
            if ((rc = launch_cov(ci, h->stream, false))) return rc;
        }
        const bool second = pipelined && (ci & 1);
        GemmArgs a;
        memset(&a, 0, sizeof(a));
        a.A = ptr<double>(h->P); a.lda = NP;
        a.B = second ? ptr<double>(h->Kstar2) : ptr<double>(h->Kstar); a.ldb = NP;
        a.alpha = 1.0;
        a.job_mode = JOBS_VARIANCE;
        a.nb = h->nb; a.mcb = (int)(mcp / BN);
        a.z = ptr<double>(h->Kbuf) + NP * NP;
        a.part_mu = ptr<double>(h->part_mu);
        a.part_ssq = ptr<double>(h->part_ssq);
        a.ldpart = cap;
        if (!chained) {
            if (last) CK(cudaEventRecord(h->ev[10], h->stream));
            CK(cudaEventRecord(h->ev_g0[ci], h->stream));
        }
        const bool oz_pair_ok = h->oz_pair && (h->nb % 2) == 0;
        const int oz_persist = h->oz_persist == 3 ? (h->nb <= 24 ? 1 : 0) : h->oz_persist;
        if (use_oz && h->oz_tile == 128 && (oz_pair_ok || !h->oz_pair)) {
            Oz2Args o;
            o.nb = h->nb; o.ncb = (int)(mcp / OZ2_T); o.NP = (int)NP; o.rows = (int)cap;
            o.group = (int)std::min<long>(64, std::max<long>(2, ((long)64 << 20) / ((long)OZ2_T * NP * OZ_S)));
            o.eP = ptr<int>(h->oz_eP); o.eK = oz_eK;
            o.part_ssq = a.part_ssq; o.ldpart = a.ldpart; o.scratch = ptr<double>(h->oz_scratch);
            o.prof = nullptr;
            h->oz_last_variant = oz_pair_ok ? 4 + (oz_persist == 1 ? 8 : 0) : 3;
            if (oz_pair_ok) {
                // CTA pair, 256 x 128 per pair in two passes; its K* half tile (64 rows x 64 B) is the box of mapOzK
                const int tiles = (o.nb / 2) * o.ncb;
                const unsigned grid = (unsigned)(2 * (oz_persist == 1 ? std::min(tiles, std::max(h->n_sm, 2) / 2) : tiles));
                if (h->oz_prof) {
                    if ((rc = ensure(h, h->oz_profbuf, (size_t)grid * 64))) return rc;
                    CK(cudaMemsetAsync(h->oz_profbuf.p, 0, (size_t)grid * 64, h->stream));
                    o.prof = ptr<long long>(h->oz_profbuf);
                    h->oz_prof_ctas = (int)grid;
                }
                CK(launch_oz(gpk_oz_pair2_kernel, grid, (size_t)OZQ_SMEM, h->stream, true, dependent, h->mapOzP, second ? h->mapOzK2 : h->mapOzK, o));
            } else
                CK(launch_oz(gpk_oz2_vargemm_kernel, (unsigned)(o.nb * o.ncb), (size_t)OZ2_SMEM, h->stream, false, dependent,
                             h->mapOzP32, second ? h->mapOzK32b : h->mapOzK32, o));
            CKL();
            h->oz_launches += 1;
        } else if (use_oz) {
            OzArgs o;
            o.nb = h->nb; o.ncb = (int)(mcp / OZ_TN); o.NP = (int)NP; o.rows = (int)cap;
            o.group = (int)std::min<long>(128, std::max<long>(4, ((long)64 << 20) / ((long)OZ_TN * NP * OZ_S)));
            o.eP = ptr<int>(h->oz_eP); o.eK = oz_eK;
            o.part_ssq = a.part_ssq; o.ldpart = a.ldpart;
            o.prof = nullptr;
            const bool pair = oz_pair_ok && h->oz_tile != 128;
            const CUtensorMap& mk = pair ? (second ? h->mapOzKh2 : h->mapOzKh) : (second ? h->mapOzK2 : h->mapOzK);
            const int tiles = pair ? (o.nb / 2) * o.ncb : o.nb * o.ncb;
            const int sms = std::max(h->n_sm, 2);
            // "ozpersist" 1: one CTA (pair) per SM walks the tile list; 2: the same kernel, one tile per CTA (pair); 0: the
            // one-tile kernels
            const int units = oz_persist == 1 ? std::min(tiles, pair ? sms / 2 : sms) : tiles;
            h->oz_last_variant = (pair ? 2 : 1) + (oz_persist == 1 ? 8 : 0);
            if (h->oz_prof && oz_persist) {
                const int ctas = pair ? 2 * units : units;
                if ((rc = ensure(h, h->oz_profbuf, (size_t)ctas * 64))) return rc;
                CK(cudaMemsetAsync(h->oz_profbuf.p, 0, (size_t)ctas * 64, h->stream));
                o.prof = ptr<long long>(h->oz_profbuf);
                h->oz_prof_ctas = ctas;
            }
            if (pair && oz_persist)
                CK(launch_oz(gpk_oz_persist_kernel<true>, (unsigned)(2 * units), (size_t)OZP_PERSIST_SMEM, h->stream, true, dependent, h->mapOzP, mk, o));
            else if (pair)
                CK(launch_oz(gpk_oz_pair_kernel, (unsigned)(2 * units), (size_t)OZP_SMEM, h->stream, true, dependent, h->mapOzP, mk, o));
            else if (oz_persist)
                CK(launch_oz(gpk_oz_persist_kernel<false>, (unsigned)units, (size_t)OZ_PERSIST_SMEM, h->stream, false, dependent, h->mapOzP, mk, o));
            else
                CK(launch_oz(gpk_oz_vargemm_kernel, (unsigned)tiles, (size_t)OZ_SMEM, h->stream, false, dependent, h->mapOzP, mk, o));
            CKL();
            h->oz_launches += 1;
        } else if (h->persist && h->loader == LOADER_TMA_WS) {
            // one CTA per SM, tiles handed out by a counter (zeroed in stream order before every launch)
            if ((rc = ensure(h, h->tile_cnt, 4))) return rc;
            CK(cudaMemsetAsync(h->tile_cnt.p, 0, 4, h->stream));
            VarArgs v;
            v.nb = a.nb; v.mcb = a.mcb; v.z = a.z; v.part_mu = a.part_mu; v.part_ssq = a.part_ssq; v.ldpart = a.ldpart;
            v.counter = ptr<int>(h->tile_cnt);
            const int grid = std::min(h->nb * a.mcb, std::max(h->n_sm, 1));
            gpk_vargemm_persistent_kernel<<<grid, WS_THREADS, PV_SMEM, h->stream>>>(h->mapP, second ? h->mapKs2 : h->mapKs, v);
            CKL();
        } else if ((rc = launch_gemm<EPI_COLREDUCE>(h, h->mapP, second ? h->mapKs2 : h->mapKs, a, h->nb * a.mcb))) return rc;
        CK(cudaEventRecord(h->ev_g1[ci], h->stream));
        if (last) CK(cudaEventRecord(h->ev[11], h->stream));
        if (pipelined && !chained && !oz_fused) CK(cudaEventRecord(h->ev_gemm[ci], h->stream));
        h->launches_var += 1;
        h->last_chunk_rows = mcp;
        FinishArgs f;
        memset(&f, 0, sizeof(f));
        f.part_mu = ptr<double>(h->part_mu); f.part_ssq = ptr<double>(h->part_ssq);
        f.ldpart = cap; f.nparts = h->nb; f.m = mc; f.base = global_base + index_offset + base;
        f.kss = h->spec.amp; f.mean = h->mean;
        f.norm_out = h->norm_out; f.y_mean = h->y_mean; f.y_std = h->y_std;
        f.acq_kind = kind; f.eta = eta; f.par = par;
        f.out_mu = d_mu ? d_mu + index_offset + base : nullptr;
        f.out_var = d_var ? d_var + index_offset + base : nullptr;
        f.out_acq = d_out ? d_out + index_offset + base : nullptr;
        f.block_best = ptr<BestPair>(h->block_best);
        f.n_negative = d_nneg;
        f.mu_direct = (use_oz && !oz_fused) ? (second ? ptr<double>(h->oz_mu2) : ptr<double>(h->oz_mu)) : nullptr;
        if (oz_fused && second) f.part_mu = ptr<double>(h->oz_pmu2);
        const int fb = (int)((mc + 255) / 256);
        gpk_finish_kernel<<<fb, 256, 0, h->stream>>>(f);
        CKL();
        if (kind != GPK_ACQ_NONE) {
            gpk_argmax_final_kernel<<<1, 256, 0, h->stream>>>(ptr<BestPair>(h->block_best), fb, d_best);
            CKL();
        }
        // fused int8 builder: it also writes this parity's mean partials, which the finish kernel above still reads
        if (pipelined && !chained && oz_fused) CK(cudaEventRecord(h->ev_gemm[ci], h->stream));
        if (last) CK(cudaEventRecord(h->ev[12], h->stream));
    }
    CK(cudaEventRecord(h->ev[7], h->stream));
    h->score_timed = true;
    return GPK_OK;
}

}  // namespace

// =============================================================================================
// C ABI
// =============================================================================================
extern "C" {

int gpk_comm_destroy(gpk_handle* h);

static void drop_fit_graph(gpk_handle* h) {
    if (h->fit_graph) { cudaGraphExecDestroy(h->fit_graph); h->fit_graph = nullptr; }
}

const char* gpk_version(void) { return "gpk 0.2 (sm_100a, fp64 DMMA + TMA)"; }

const char* gpk_last_error(gpk_handle* h) { return h ? h->err : "null handle"; }

int gpk_create(gpk_handle** out, int device) {
    if (!out) return GPK_BAD_ARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) return GPK_CUDA_ERROR;
    gpk_handle* h = new gpk_handle();
    h->device = device;
    memset(&h->spec, 0, sizeof(h->spec));
    if (cudaSetDevice(device) != cudaSuccess) { delete h; return GPK_CUDA_ERROR; }
    {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);      // hi = numerically smallest = highest priority
        if (cudaStreamCreateWithPriority(&h->own_stream, cudaStreamNonBlocking, hi) != cudaSuccess) { delete h; return GPK_CUDA_ERROR; }
        if (cudaStreamCreateWithPriority(&h->side_stream, cudaStreamNonBlocking, lo) != cudaSuccess) { delete h; return GPK_CUDA_ERROR; }
        if (cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking) != cudaSuccess) { delete h; return GPK_CUDA_ERROR; }
        if (cudaStreamCreateWithPriority(&h->panel_stream, cudaStreamNonBlocking, hi) != cudaSuccess) { delete h; return GPK_CUDA_ERROR; }
    }
    h->stream = h->own_stream;
    for (int i = 0; i < 16; ++i)
        if (cudaEventCreate(&h->ev[i]) != cudaSuccess) { delete h; return GPK_CUDA_ERROR; }
    h->ev_ok = true;
    if (cudaEventCreateWithFlags(&h->ev_order, cudaEventDisableTiming) != cudaSuccess) { delete h; return GPK_CUDA_ERROR; }
    int rc = set_kernel_attrs(h);
    if (rc) { fprintf(stderr, "gpk_create: %s\n", h->err); delete h; return rc; }
    rc = ensure(h, h->status, 4);
    if (!rc) rc = ensure(h, h->scal, 64);
    if (rc) { delete h; return rc; }
    if (cudaMallocHost((void**)&h->pin, 64) != cudaSuccess) { delete h; return GPK_CUDA_ERROR; }
    if (get_encode_fn() == nullptr) h->loader = LOADER_CPASYNC;
    *out = h;
    return GPK_OK;
}

int gpk_destroy(gpk_handle* h) {
    if (!h) return GPK_OK;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    drop_fit_graph(h);
    gpk_comm_destroy(h);
    if (h->ev_multi) cudaEventDestroy(h->ev_multi);
    DevBuf* bufs[] = {&h->Xrow, &h->Xt, &h->y, &h->Kbuf, &h->P, &h->Q, &h->W, &h->lower, &h->upper, &h->logdet_part,
                      &h->scal, &h->status, &h->jobs, &h->cand, &h->Kstar, &h->Kstar2, &h->cand2, &h->part_mu, &h->part_ssq, &h->out_mu,
                      &h->out_var, &h->out_acq, &h->block_best, &h->best, &h->nneg, &h->Vt, &h->cov, &h->XsT,
                      &h->tmpjobs, &h->alpha, &h->tmp1, &h->tmp2, &h->tmp3, &h->chain_cnt, &h->dprof, &h->Xts, &h->tile_cnt, &h->oz_Pq, &h->oz_Kq, &h->oz_Kq2, &h->oz_eP, &h->oz_emax, &h->oz_mu, &h->oz_mu2, &h->oz_pmu2, &h->oz_scratch,
                      &h->multi_cand, &h->multi_A, &h->multi_B, &h->multi_out, &h->multi_bb, &h->gather, &h->best_global,
                      &h->es_raw, &h->es_scr, &h->es_logP, &h->es_dmu, &h->es_dsig, &h->es_dmumu, &h->es_sweeps, &h->es_F,
                      &h->es_jl, &h->es_Bt, &h->es_zb, &h->es_zbop, &h->es_W, &h->es_lmb, &h->es_cand, &h->es_var, &h->es_KZ,
                      &h->es_S, &h->es_bb, &h->es_best, &h->es_lo, &h->es_up};
    for (DevBuf* b : bufs)
        if (b->p) cudaFree(b->p);
    if (h->ev_ok)
        for (int i = 0; i < 16; ++i) cudaEventDestroy(h->ev[i]);
    if (h->ev_order) cudaEventDestroy(h->ev_order);
    for (int i = 0; i < 2; ++i)
        if (h->stage[i]) cudaFreeHost(h->stage[i]);
    for (cudaEvent_t e : h->ev_cs) cudaEventDestroy(e);
    if (h->panel_stream) cudaStreamDestroy(h->panel_stream);
    for (cudaEvent_t e : h->ev_panel) cudaEventDestroy(e);
    for (cudaEvent_t e : h->ev_rest) cudaEventDestroy(e);
    for (cudaEvent_t e : h->ev_cov) cudaEventDestroy(e);
    for (cudaEvent_t e : h->ev_g0) cudaEventDestroy(e);
    for (cudaEvent_t e : h->ev_g1) cudaEventDestroy(e);
    for (cudaEvent_t e : h->ev_copied) cudaEventDestroy(e);
    for (cudaEvent_t e : h->ev_scored) cudaEventDestroy(e);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    for (cudaEvent_t e : h->ev_gemm) cudaEventDestroy(e);
    if (h->side_stream) cudaStreamDestroy(h->side_stream);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    if (h->pin) cudaFreeHost(h->pin);
    delete h;
    return GPK_OK;
}

int gpk_set_option(gpk_handle* h, const char* key, long value) {
    if (!h || !key) return GPK_BAD_ARG;
    drop_fit_graph(h);                       // every switch may change what a factorisation launches
    if (!strcmp(key, "graph")) {
        if (value != 0 && value != 1) BAD("graph must be 0 or 1");
        h->use_graph = (int)value;
        return GPK_OK;
    }
    if (!strcmp(key, "loader")) {
        if (value < LOADER_CPASYNC || value > LOADER_TMA_WS) BAD("loader must be 0 (cp.async), 1 (TMA) or 2 (TMA, warp-specialised)");
        if (value != LOADER_CPASYNC && get_encode_fn() == nullptr) BAD("TMA descriptors unavailable on this driver");
        h->loader = (int)value;
        h->maps_ok = false;
        h->mapKs_rows = 0;
        h->mapVt_rows = 0;
        return GPK_OK;
    }
    if (!strcmp(key, "oztile")) {
        if (value != 64 && value != 128) BAD("oztile must be 64 (one pass, 128 x 64 tiles) or 128 (two passes, 128 x 128 tiles)");
        h->oz_tile = (int)value;
        return GPK_OK;
    }
    if (!strcmp(key, "ozpersist")) {
        if (value < 0 || value > 3) BAD("ozpersist must be 0, 1, 2 or 3");
        h->oz_persist = (int)value;
        return GPK_OK;
    }
    if (!strcmp(key, "ozpdl")) {
        h->oz_pdl = (int)value;
        return GPK_OK;
    }
    if (!strcmp(key, "covctas")) {
        if (value < 1 || value > 8) BAD("covctas must be 1..8");
        h->cov_ctas = (int)value;
        return GPK_OK;
    }
    if (!strcmp(key, "ozprof")) {
        h->oz_prof = (int)value;
        return GPK_OK;
    }
    if (!strcmp(key, "ozpair")) {
        h->oz_pair = (int)value;
        return GPK_OK;
    }
    if (!strcmp(key, "ozfused")) {
        if (value != 0 && value != 1) BAD("ozfused must be 0 or 1");
        h->oz_fused = (int)value;
        return GPK_OK;
    }
    if (!strcmp(key, "ozaki")) {
        if (value != 0 && value != 1) BAD("ozaki must be 0 (fp64 DMMA) or 1 (int8 tensor pipe, error-free split)");
        h->ozaki = (int)value;
        return GPK_OK;
    }
    if (!strcmp(key, "persist")) {
        if (value != 0 && value != 1) BAD("persist must be 0 or 1");
        h->persist = (int)value;
        return GPK_OK;
    }
    if (!strcmp(key, "depth2")) {
        if (value < 0 || value > 2) BAD("depth2 must be 0, 1 or 2 (automatic)");
        h->depth2 = (int)value;
        return GPK_OK;
    }
    if (!strcmp(key, "chainsplit")) {
        if (value != 0 && value != 1) BAD("chainsplit must be 0 or 1");
        h->chainsplit = (int)value;
        return GPK_OK;
    }
    if (!strcmp(key, "fusechain")) {
        if (value != 0 && value != 1) BAD("fusechain must be 0 or 1");
        h->fusechain = (int)value;
        return GPK_OK;
    }
    if (!strcmp(key, "pdl")) {
        if (value != 0 && value != 1) BAD("pdl must be 0 or 1");
        h->pdl = (int)value;
        return GPK_OK;
    }
    if (!strcmp(key, "overlap")) {
        if (value != 0 && value != 1) BAD("overlap must be 0 or 1");
        h->overlap = (int)value;
        return GPK_OK;
    }
    if (!strcmp(key, "smalltile")) {
        if (value < 0 || value > 2) BAD("smalltile must be 0 (128-row chain tiles), 1 (32 rows) or 2 (16 rows)");
        h->smalltile = (int)value;
        return GPK_OK;
    }
    if (!strcmp(key, "lookahead")) {
        if (value != 0 && value != 1) BAD("lookahead must be 0 or 1");
        h->lookahead = (int)value;
        return GPK_OK;
    }
    if (!strcmp(key, "diagprof")) {                 // 1: stamps; 2: stamps + skip the kernel's global stores (timing only)
        h->diag_prof = value != 0;
        if (h->diag_prof) {
            int rc = ensure(h, h->dprof, 64 * 8);
            if (rc) return rc;
            CK(cudaMemset(h->dprof.p, 0, 64 * 8));
            if (value == 2) {
                const long long one = 1;
                CK(cudaMemcpy((char*)h->dprof.p + 63 * 8, &one, 8, cudaMemcpyHostToDevice));
            }
        }
        return GPK_OK;
    }
    if (!strcmp(key, "diag")) {
        if (value != 0 && value != 2 && value != 3 && value != 4)
            BAD("diag must be 4 (blocked panels, DMMA updates), 3 (blocked panels, DFMA register tiles), 2 (column-by-column "
                "register-tiled kernel) or 0 (simple shared-memory kernel)");
        h->diag_kernel = (int)value;
        return GPK_OK;
    }
    if (!strcmp(key, "cov")) {
        if (value != 1 && value != 2) BAD("cov must be 2 (TMA-staged covariance builder, pre-scaled operands) or 1 (round-1 kernel)");
        h->cov_kernel = (int)value;
        h->fitted = false;
        h->linv_ready = false;
        return GPK_OK;
    }
    if (!strcmp(key, "chunk")) {
        if (value == 0) { h->chunk_user = false; return GPK_OK; }          // back to the automatic choice
        if (value < BM || value % BM) BAD("chunk must be a positive multiple of 128 (0 = automatic)");
        h->chunk = value;
        h->chunk_user = true;
        return GPK_OK;
    }
    BAD("unknown option '%s'", key);
}

int gpk_set_stream(gpk_handle* h, void* s) {
    if (!h) return GPK_BAD_ARG;
    cudaStreamSynchronize(h->stream);
    h->stream = s ? (cudaStream_t)s : h->own_stream;
    return GPK_OK;
}

int gpk_synchronize(gpk_handle* h) {
    if (!h) return GPK_BAD_ARG;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    return GPK_OK;
}

int gpk_set_data(gpk_handle* h, const double* X, const double* y, int n, int d) {
    if (!h) return GPK_BAD_ARG;
    if (!X || !y || n <= 0 || d <= 0) BAD("gpk_set_data: need X, y, n > 0, d > 0");
    if (d > GPK_MAX_TERMS) BAD("gpk_set_data: d = %d exceeds GPK_MAX_TERMS = %d", d, GPK_MAX_TERMS);
    CK(cudaSetDevice(h->device));
    const long NP = round_up(n, BM);
    int rc;
    bool g1, g2, g3, g4;
    if ((rc = ensure(h, h->Xrow, (size_t)NP * d * 8))) return rc;      // room for the rows gpk_fit_append may add
    if ((rc = ensure(h, h->Xt, (size_t)d * NP * 8))) return rc;
    if ((rc = ensure(h, h->y, (size_t)NP * 8))) return rc;
    if ((rc = ensure(h, h->Kbuf, (size_t)(NP + BM) * NP * 8, &g1))) return rc;
    if ((rc = ensure(h, h->P, (size_t)NP * NP * 8, &g2))) return rc;
    if ((rc = ensure(h, h->Q, (size_t)NP * NP * 8, &g3))) return rc;
    if ((rc = ensure(h, h->W, (size_t)NP * NP * 8, &g4))) return rc;
    if ((rc = ensure(h, h->logdet_part, (size_t)(NP / BM) * 8))) return rc;
    const bool relayout = (h->layout_NP != NP) || g1 || g2 || g3 || g4;
    h->n = n; h->d = d; h->NP = (int)NP; h->nb = (int)(NP / BM);
    if (relayout || h->jobs_nb != (int)(NP / BM)) drop_fit_graph(h);       // the graph holds buffer / job-table addresses
    if (relayout) {
        CK(cudaMemsetAsync(h->Kbuf.p, 0, (size_t)(NP + BM) * NP * 8, h->stream));
        CK(cudaMemsetAsync(h->P.p, 0, (size_t)NP * NP * 8, h->stream));
        CK(cudaMemsetAsync(h->Q.p, 0, (size_t)NP * NP * 8, h->stream));
        CK(cudaMemsetAsync(h->W.p, 0, (size_t)NP * NP * 8, h->stream));
        h->layout_NP = (int)NP;
        h->maps_ok = false;
    }
    CK(cudaMemcpyAsync(h->Xrow.p, X, (size_t)n * d * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemsetAsync(h->y.p, 0, (size_t)NP * 8, h->stream));
    CK(cudaMemcpyAsync(h->y.p, y, (size_t)n * 8, cudaMemcpyHostToDevice, h->stream));
    {
        long total = (long)d * NP;
        gpk_transpose_kernel<<<(unsigned)((total + 255) / 256), 256, 0, h->stream>>>(ptr<double>(h->Xrow), n, d, nullptr,
                                                                                    nullptr, ptr<double>(h->Xt), NP);
        CKL();
    }
    CK(cudaStreamSynchronize(h->stream));     // host buffers are caller-owned: done with them
    if ((rc = build_job_tables(h))) return rc;
    if (!h->maps_ok && (rc = rebuild_maps(h))) return rc;
    h->has_data = true;
    h->fitted = false;
    h->linv_ready = false;
    h->alpha_ready = false;
    return GPK_OK;
}

int gpk_set_input_bounds(gpk_handle* h, const double* lower, const double* upper, int d) {
    if (!h) return GPK_BAD_ARG;
    CK(cudaSetDevice(h->device));
    if (!lower || !upper) { h->has_bounds = false; return GPK_OK; }
    if (d <= 0 || d > GPK_MAX_TERMS) BAD("gpk_set_input_bounds: bad d");
    int rc;
    if ((rc = ensure(h, h->lower, (size_t)d * 8))) return rc;
    if ((rc = ensure(h, h->upper, (size_t)d * 8))) return rc;
    CK(cudaMemcpyAsync(h->lower.p, lower, (size_t)d * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->upper.p, upper, (size_t)d * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->has_bounds = true;
    return GPK_OK;
}

int gpk_set_output_transform(gpk_handle* h, int enabled, double y_mean, double y_std) {
    if (!h) return GPK_BAD_ARG;
    h->norm_out = enabled ? 1 : 0;
    h->y_mean = y_mean;
    h->y_std = y_std;
    return GPK_OK;
}

int gpk_set_kernel(gpk_handle* h, int family, double log_amp, int n_terms, const int* axis, const int* group,
                   const double* log_metric) {
    if (!h) return GPK_BAD_ARG;
    if (family < GPK_MATERN52 || family > GPK_MATERN32) BAD("gpk_set_kernel: unknown family %d", family);
    if (n_terms <= 0 || n_terms > GPK_MAX_TERMS || !axis || !group || !log_metric)
        BAD("gpk_set_kernel: need 1..%d terms", GPK_MAX_TERMS);
    KSpec s;
    memset(&s, 0, sizeof(s));
    s.family = family;
    s.n_terms = n_terms;
    s.amp = exp(log_amp);
    for (int t = 0; t < n_terms; ++t) {
        if (axis[t] < 0 || axis[t] >= GPK_MAX_TERMS) BAD("gpk_set_kernel: axis out of range");
        if (t > 0 && (group[t] < group[t - 1] || group[t] > group[t - 1] + 1)) BAD("gpk_set_kernel: groups must be contiguous");
        s.axis[t] = axis[t];
        s.inv_metric[t] = 1.0 / exp(log_metric[t]);
        s.scale[t] = sqrt((family == GPK_MATERN52 ? 5.0 : family == GPK_MATERN32 ? 3.0 : 0.5) * s.inv_metric[t]);
        s.last[t] = (t == n_terms - 1) || (group[t + 1] != group[t]);
    }
    if (group[0] != 0) BAD("gpk_set_kernel: groups must start at 0");
    h->spec = s;
    h->log_amp = log_amp;
    h->log_metric.assign(log_metric, log_metric + n_terms);
    h->has_spec = true;
    h->fitted = false;
    h->linv_ready = false;
    h->alpha_ready = false;
    return GPK_OK;
}

int gpk_fit_begin(gpk_handle* h, double diag_add, double mean) {
    int rc = require(h, true, true, false);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    for (int t = 0; t < h->spec.n_terms; ++t)
        if (h->spec.axis[t] >= h->d) BAD("gpk_fit: kernel axis %d >= d = %d", h->spec.axis[t], h->d);
    const long NP = h->NP;
    const int nb = h->nb;
    if (!h->maps_ok && (rc = rebuild_maps(h))) return rc;        // staging mode changed after gpk_set_data
    h->fitted = false;
    h->linv_ready = false;
    h->alpha_ready = false;
    h->mean = mean;
    h->diag_add = diag_add;
    double* K = ptr<double>(h->Kbuf);

    CK(cudaEventRecord(h->ev[0], h->stream));
    {
        if (cov_tma(h)) {               // the pre-scaled operand depends on the hyper-parameters: rebuilt per fit (n_terms x NP)
            if ((rc = ensure(h, h->Xts, (size_t)GPK_MAX_TERMS * NP * 8))) return rc;
            if ((rc = build_cov_operand(h, h->stream, ptr<double>(h->Xrow), h->n, h->d, nullptr, nullptr, ptr<double>(h->Xts), NP)))
                return rc;
        }
        if ((rc = launch_cov_tiles(h, h->stream, train_operand(h), NP, h->n, ptr<double>(h->Xrow), h->d, (long)h->n, NP,
                                   nullptr, nullptr, K, NP, 1, false)))
            return rc;
        gpk_kfix_kernel<<<(unsigned)((NP + 255) / 256), 256, 0, h->stream>>>(K, NP, h->n, (int)NP, diag_add,
                                                                            ptr<double>(h->y), mean);
        CKL();
    }
    CK(cudaMemsetAsync(h->status.p, 0, 4, h->stream));
    CK(cudaEventRecord(h->ev[1], h->stream));
    while ((int)h->ev_panel.size() < nb) {
        cudaEvent_t e1, e2;
        CK(cudaEventCreateWithFlags(&e1, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&e2, cudaEventDisableTiming));
        h->ev_panel.push_back(e1);
        h->ev_rest.push_back(e2);
    }
    std::vector<char> rest_recorded(nb, 0);
    const bool fuse = h->fusechain && h->smalltile == 1 && h->lookahead;
    if (fuse) {
        if ((rc = ensure(h, h->chain_cnt, (size_t)nb * 4))) return rc;
        CK(cudaMemsetAsync(h->chain_cnt.p, 0, (size_t)nb * 4, h->stream));
    }
    // ---- split chain (default): only block row k+1 of step k stays between diag(k) and diag(k+1) ----------------
    // Step k of the right-looking factorisation used to put diag(k) -> panel solve (all rows) -> update of block column
    // k+1 (all rows) on the critical chain.  diag(k+1) only needs A[k+1,k+1] -= L[k+1,k] L[k+1,k]^T with
    // L[k+1,k] = A[k+1,k] inv(L_kk)^T: one launch of gpk_chain_step_kernel on the four 32-row tiles of block row k+1
    // ("X(k)").  The rows below go to a second high-priority stream and overlap diag(k+1); the trailing update is cut
    // in two (block column k+2 first) so that the chain waits for one column, not for the whole update (look-ahead 2).
    // Every tile still receives its panels in increasing order: the factor is bit-identical to the other schedules.
    //   C (h->stream)     diag(k) . X(k) . diag(k+1) ...
    //   P (panel_stream)  solve'(k) [rows > k+1] . update'(k) [block column k+1, rows > k+1]
    //   R (side_stream)   rest_a(k) [block column k+2] . rest_b(k) [block columns >= k+3]
    const bool split = h->chainsplit && h->smalltile == 1 && h->lookahead && !fuse && h->diag_kernel >= 3 &&
                       h->loader != LOADER_CPASYNC && nb >= 3;
    if (split) {
        if ((rc = ensure(h, h->chain_cnt, (size_t)nb * 4))) return rc;
        while ((int)h->ev_cs.size() < 5 * nb + 3) {
            cudaEvent_t e;
            CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            h->ev_cs.push_back(e);
        }
        auto evD = [&](int k) { return h->ev_cs[5 * k]; };
        auto evX = [&](int k) { return h->ev_cs[5 * k + 1]; };
        auto evT = [&](int k) { return h->ev_cs[5 * k + 2]; };
        auto evPU = [&](int k) { return h->ev_cs[5 * k + 3]; };
        auto evRA = [&](int k) { return h->ev_cs[5 * k + 4]; };
        cudaStream_t C = h->stream, Pst = h->panel_stream, R = h->side_stream;
        cudaEvent_t evFork = h->ev_cs[5 * nb], evJoinP = h->ev_cs[5 * nb + 1], evJoinR = h->ev_cs[5 * nb + 2];
        // the whole schedule of one factorisation (about 6 launches, 5 event records and 7 stream waits per step);
        // depends on the buffers and job tables only, so it is captured ONCE into a CUDA graph and replayed per fit
        auto enqueue = [&]() -> int {
        std::vector<char> haveX(nb, 0), havePU(nb, 0), haveRA(nb, 0);
        CK(cudaMemsetAsync(h->chain_cnt.p, 0, (size_t)nb * 4, C));
        CK(cudaEventRecord(evFork, C));                            // K is built: the other streams may start
        CK(cudaStreamWaitEvent(Pst, evFork, 0));
        CK(cudaStreamWaitEvent(R, evFork, 0));
        gpk_diag_prezero_kernel<<<nb, 256, 0, C>>>(K, (long)NP, ptr<double>(h->P), (long)NP);
        CKL();
        for (int k = 0; k < nb; ++k) {
            long long* dprof = h->diag_prof ? ptr<long long>(h->dprof) : nullptr;
            // ---- C: diag(k)
            if (h->diag_kernel == 4)
                gpk_potrf_diag_dmma_kernel<<<1, 256, DIAG4_SMEM, C>>>(K, NP, k, ptr<double>(h->P), ptr<double>(h->Q), NP,
                                                                     ptr<int>(h->status), ptr<double>(h->logdet_part), dprof);
            else
                gpk_potrf_diag_blocked_kernel<<<1, 256, DIAG3_SMEM, C>>>(K, NP, k, ptr<double>(h->P), ptr<double>(h->Q), NP,
                                                                        ptr<int>(h->status), ptr<double>(h->logdet_part), dprof);
            CKL();
            CK(cudaEventRecord(evD(k), C));
            const int nsolve = h->trsm32_r[k].cnt, nupd = h->pu32_r[k].cnt;
            const bool hasX = (k + 1 < nb);                              // block row k+1 exists: 4 solve + 4 update tiles
            // ---- C: X(k)
            if (hasX) {
                if (k >= 1 && havePU[k - 1]) CK(cudaStreamWaitEvent(C, evPU(k - 1), 0));     // A[k+1,k] carries panel k-1
                if (k >= 1 && haveRA[k - 1]) CK(cudaStreamWaitEvent(C, evRA(k - 1), 0));     // A[k+1,k+1] carries panel k-1
                ChainArgs c;
                c.K = K; c.ld = NP; c.P = ptr<double>(h->P); c.ldp = NP;
                c.solve_jobs = ptr<GemmJob>(h->jobs) + h->trsm32_r[k].off;
                c.update_jobs = ptr<GemmJob>(h->jobs) + h->pu32_r[k].off;
                c.counter = ptr<int>(h->chain_cnt) + k;
                c.status = ptr<int>(h->status);
                gpk_chain_step_kernel<<<4, GEMM_THREADS, CH_SMEM, C>>>(c);
                CKL();
                CK(cudaEventRecord(evX(k), C));
                haveX[k] = 1;
            }
            // ---- P: the rest of the panel (rows below block row k+1, and the right-hand-side row)
            const int skip = hasX ? 4 : 0;
            GemmArgs a;
            memset(&a, 0, sizeof(a));
            a.A = K; a.lda = NP; a.B = ptr<double>(h->P); a.ldb = NP; a.C = K; a.ldc = NP;
            a.alpha = 1.0; a.beta = 0; a.job_mode = JOBS_TABLE; a.status = ptr<int>(h->status);
            a.jobs = ptr<GemmJob>(h->jobs) + h->trsm32_r[k].off + skip;
            CK(cudaStreamWaitEvent(Pst, evD(k), 0));
            if (nsolve - skip > 0) {
                if ((rc = launch_gemm<EPI_STORE, 2>(h, h->mapK32, h->mapP, a, nsolve - skip, Pst))) return rc;
            }
            CK(cudaEventRecord(evT(k), Pst));
            if (hasX && nupd - 4 > 0) {
                GemmArgs u;
                memset(&u, 0, sizeof(u));
                u.A = K; u.lda = NP; u.B = K; u.ldb = NP; u.C = K; u.ldc = NP;
                u.alpha = -1.0; u.beta = 1; u.job_mode = JOBS_TABLE; u.status = ptr<int>(h->status);
                u.jobs = ptr<GemmJob>(h->jobs) + h->pu32_r[k].off + 4;
                CK(cudaStreamWaitEvent(Pst, evX(k), 0));                                       // L[k+1,k] is the B operand
                if (k >= 1 && haveRA[k - 1]) CK(cudaStreamWaitEvent(Pst, evRA(k - 1), 0));    // column k+1 carries panel k-1
                if ((rc = launch_gemm<EPI_STORE, 2>(h, h->mapK32, h->mapK, u, nupd - 4, Pst))) return rc;
                CK(cudaEventRecord(evPU(k), Pst));
                havePU[k] = 1;
            }
            // ---- R: trailing update beyond block column k+1: column k+2 first (what step k+1 waits for), then the rest
            const int off = h->syrk_r[k].off, cnt = h->syrk_r[k].cnt, npu = nb - k;       // first npu jobs: block column k+1
            if (cnt > npu) {
                const int na = nb - k - 1;                                                // block column k+2: rows k+2 .. nb
                GemmArgs s2;
                memset(&s2, 0, sizeof(s2));
                s2.A = K; s2.lda = NP; s2.B = K; s2.ldb = NP; s2.C = K; s2.ldc = NP;
                s2.alpha = -1.0; s2.beta = 1; s2.job_mode = JOBS_TABLE; s2.status = ptr<int>(h->status);
                CK(cudaStreamWaitEvent(R, evT(k), 0));
                if (hasX) CK(cudaStreamWaitEvent(R, evX(k), 0));
                s2.jobs = ptr<GemmJob>(h->jobs) + off + npu;
                if ((rc = launch_gemm<EPI_STORE>(h, h->mapK, h->mapK, s2, std::min(na, cnt - npu), R))) return rc;
                CK(cudaEventRecord(evRA(k), R));
                haveRA[k] = 1;
                if (cnt - npu - na > 0) {
                    s2.jobs = ptr<GemmJob>(h->jobs) + off + npu + na;
                    if ((rc = launch_gemm<EPI_STORE>(h, h->mapK, h->mapK, s2, cnt - npu - na, R))) return rc;
                }
            }
        }
        // join: everything the factor consists of is complete once P and R have drained
        CK(cudaEventRecord(evJoinP, Pst));
        CK(cudaStreamWaitEvent(C, evJoinP, 0));
        CK(cudaEventRecord(evJoinR, R));
        CK(cudaStreamWaitEvent(C, evJoinR, 0));
        gpk_diag_qfill_kernel<<<nb, 256, 0, C>>>(ptr<double>(h->P), ptr<double>(h->Q), (long)NP, ptr<int>(h->status));
        CKL();
        return GPK_OK;
        };
        const bool want_graph = h->use_graph && !h->diag_prof;
        if (want_graph && h->fit_graph == nullptr) {
            // capture (thread-local mode: other threads' CUDA calls are unaffected); P and R join the capture through
            // evFork and are joined back before the end.  A failed capture falls back to direct enqueueing.
            const double launches_before = h->launches_total;
            cudaGraph_t graph = nullptr;
            if (cudaStreamBeginCapture(C, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
                const int erc = enqueue();
                const cudaError_t ce = cudaStreamEndCapture(C, &graph);
                if (erc == GPK_OK && ce == cudaSuccess && graph != nullptr &&
                    cudaGraphInstantiate(&h->fit_graph, graph, 0) == cudaSuccess) {
                    h->fit_graph_launches = h->launches_total - launches_before;
                } else {
                    h->fit_graph = nullptr;
                    h->use_graph = 0;                               // do not try again on this handle
                }
                if (graph) cudaGraphDestroy(graph);
                cudaGetLastError();
                h->launches_total = launches_before;
            } else {
                cudaGetLastError();
                h->use_graph = 0;
            }
        }
        if (want_graph && h->fit_graph != nullptr) {
            CK(cudaGraphLaunch(h->fit_graph, C));
            h->launches_total += h->fit_graph_launches;
        } else if ((rc = enqueue())) {
            return rc;
        }
    }
    if (!split && h->diag_kernel >= 3) {
        gpk_diag_prezero_kernel<<<nb, 256, 0, h->stream>>>(K, (long)NP, ptr<double>(h->P), (long)NP);
        CKL();
    }
    for (int k = 0; k < nb && !split; ++k) {
        long long* dprof = h->diag_prof ? ptr<long long>(h->dprof) : nullptr;
        if (h->diag_kernel == 4 && h->pdl && k > 0)
            CK(launch_pdl(gpk_potrf_diag_dmma_kernel, dim3(1), dim3(256), (size_t)DIAG4_SMEM, h->stream, K, (long)NP, k,
                          ptr<double>(h->P), ptr<double>(h->Q), (long)NP, ptr<int>(h->status), ptr<double>(h->logdet_part), dprof));
        else if (h->diag_kernel == 4)
            gpk_potrf_diag_dmma_kernel<<<1, 256, DIAG4_SMEM, h->stream>>>(K, NP, k, ptr<double>(h->P), ptr<double>(h->Q), NP,
                                                                          ptr<int>(h->status), ptr<double>(h->logdet_part), dprof);
        else if (h->diag_kernel == 3 && h->pdl && k > 0)
            CK(launch_pdl(gpk_potrf_diag_blocked_kernel, dim3(1), dim3(256), (size_t)DIAG3_SMEM, h->stream, K, (long)NP, k,
                          ptr<double>(h->P), ptr<double>(h->Q), (long)NP, ptr<int>(h->status), ptr<double>(h->logdet_part), dprof));
        else if (h->diag_kernel == 3)
            gpk_potrf_diag_blocked_kernel<<<1, 256, DIAG3_SMEM, h->stream>>>(K, NP, k, ptr<double>(h->P), ptr<double>(h->Q), NP,
                                                                             ptr<int>(h->status), ptr<double>(h->logdet_part), dprof);
        else if (h->diag_kernel == 2 && h->pdl && k > 0)
            CK(launch_pdl(gpk_potrf_diag_fused_kernel, dim3(1), dim3(256), (size_t)DIAG2_SMEM, h->stream, K, (long)NP, k,
                          ptr<double>(h->P), ptr<double>(h->Q), (long)NP, ptr<int>(h->status), ptr<double>(h->logdet_part)));
        else if (h->diag_kernel == 2)
            gpk_potrf_diag_fused_kernel<<<1, 256, DIAG2_SMEM, h->stream>>>(K, NP, k, ptr<double>(h->P), ptr<double>(h->Q), NP,
                                                                           ptr<int>(h->status), ptr<double>(h->logdet_part));
        else
            gpk_potrf_diag_kernel<<<1, 256, DIAG_SMEM, h->stream>>>(K, NP, k, ptr<double>(h->P), ptr<double>(h->Q), NP,
                                                                    ptr<int>(h->status), ptr<double>(h->logdet_part));
        CKL();
        if (fuse) {
            // one launch for panel solve + next-panel update (gpk_chain.cuh).  Its second pass writes block column
            // k+1, which the rest of step k-1 (side stream) also updates: wait for that first.
            const int npu = nb - k;
            if (k >= 1 && rest_recorded[k - 1]) CK(cudaStreamWaitEvent(h->stream, h->ev_rest[k - 1], 0));
            ChainArgs c;
            c.K = K; c.ld = NP; c.P = ptr<double>(h->P); c.ldp = NP;
            c.solve_jobs = ptr<GemmJob>(h->jobs) + h->trsm32_r[k].off;
            c.update_jobs = h->pu32_r[k].cnt > 0 ? ptr<GemmJob>(h->jobs) + h->pu32_r[k].off : nullptr;
            c.counter = ptr<int>(h->chain_cnt) + k;
            c.status = ptr<int>(h->status);
            if (h->pdl)
                CK(launch_pdl(gpk_chain_step_kernel, dim3((unsigned)h->trsm32_r[k].cnt), dim3(GEMM_THREADS), (size_t)CH_SMEM,
                              h->stream, c));
            else
                gpk_chain_step_kernel<<<(unsigned)h->trsm32_r[k].cnt, GEMM_THREADS, CH_SMEM, h->stream>>>(c);
            CKL();
            h->launches_total += 1;
            const int off = h->syrk_r[k].off, cnt = h->syrk_r[k].cnt;
            if (cnt > npu) {
                CK(cudaEventRecord(h->ev_panel[k], h->stream));
                CK(cudaStreamWaitEvent(h->side_stream, h->ev_panel[k], 0));
                GemmArgs s2;
                memset(&s2, 0, sizeof(s2));
                s2.A = K; s2.lda = NP; s2.B = K; s2.ldb = NP; s2.C = K; s2.ldc = NP;
                s2.alpha = -1.0; s2.beta = 1; s2.job_mode = JOBS_TABLE; s2.status = ptr<int>(h->status);
                s2.jobs = ptr<GemmJob>(h->jobs) + off + npu;
                if ((rc = launch_gemm<EPI_STORE>(h, h->mapK, h->mapK, s2, cnt - npu, h->side_stream))) return rc;
                CK(cudaEventRecord(h->ev_rest[k], h->side_stream));
                rest_recorded[k] = 1;
            }
            continue;
        }
        GemmArgs a;
        memset(&a, 0, sizeof(a));
        a.A = K; a.lda = NP;
        a.B = ptr<double>(h->P); a.ldb = NP;
        a.C = K; a.ldc = NP;
        a.alpha = 1.0; a.beta = 0;
        a.job_mode = JOBS_TABLE;
        a.status = ptr<int>(h->status);
        if (h->smalltile == 2) {
            a.jobs = ptr<GemmJob>(h->jobs) + h->trsm16_r[k].off;
            if ((rc = launch_gemm<EPI_STORE, 1>(h, h->mapK16, h->mapP, a, h->trsm16_r[k].cnt, nullptr, true))) return rc;
        } else if (h->smalltile) {
            a.jobs = ptr<GemmJob>(h->jobs) + h->trsm32_r[k].off;
            if ((rc = launch_gemm<EPI_STORE, 2>(h, h->mapK32, h->mapP, a, h->trsm32_r[k].cnt, nullptr, true))) return rc;
        } else {
            a.jobs = ptr<GemmJob>(h->jobs) + h->trsm_r[k].off;
            if ((rc = launch_gemm<EPI_STORE>(h, h->mapK, h->mapP, a, h->trsm_r[k].cnt))) return rc;
        }
        GemmArgs s;
        memset(&s, 0, sizeof(s));
        s.A = K; s.lda = NP;
        s.B = K; s.ldb = NP;
        s.C = K; s.ldc = NP;
        s.alpha = -1.0; s.beta = 1;
        s.job_mode = JOBS_TABLE;
        s.status = ptr<int>(h->status);
        const int off = h->syrk_r[k].off, cnt = h->syrk_r[k].cnt;
        if (!h->lookahead) {
            s.jobs = ptr<GemmJob>(h->jobs) + off;
            if ((rc = launch_gemm<EPI_STORE>(h, h->mapK, h->mapK, s, cnt))) return rc;
        } else if (cnt > 0) {
            // Look-ahead: the first nb-k jobs update column block k+1 (what the next diagonal block
            // and panel solve need) and stay on the critical stream; the rest of the trailing update
            // runs on the low-priority side stream, overlapped with diag(k+1) / panel(k+1).
            const int npu = nb - k;
            CK(cudaEventRecord(h->ev_panel[k], h->stream));                       // panel k solved
            if (k >= 1 && rest_recorded[k - 1]) CK(cudaStreamWaitEvent(h->stream, h->ev_rest[k - 1], 0));
            if (h->smalltile == 2) {
                s.jobs = ptr<GemmJob>(h->jobs) + h->pu16_r[k].off;
                if ((rc = launch_gemm<EPI_STORE, 1>(h, h->mapK16, h->mapK, s, h->pu16_r[k].cnt, nullptr, true))) return rc;
            } else if (h->smalltile) {
                s.jobs = ptr<GemmJob>(h->jobs) + h->pu32_r[k].off;
                if ((rc = launch_gemm<EPI_STORE, 2>(h, h->mapK32, h->mapK, s, h->pu32_r[k].cnt, nullptr, true))) return rc;
            } else {
                s.jobs = ptr<GemmJob>(h->jobs) + off;
                if ((rc = launch_gemm<EPI_STORE>(h, h->mapK, h->mapK, s, npu))) return rc;
            }
            const bool d2 = h->smalltile && (h->depth2 == 1 || (h->depth2 == 2 && nb >= 48));
            if (cnt > npu && !d2) {
                CK(cudaStreamWaitEvent(h->side_stream, h->ev_panel[k], 0));
                s.jobs = ptr<GemmJob>(h->jobs) + off + npu;
                if ((rc = launch_gemm<EPI_STORE>(h, h->mapK, h->mapK, s, cnt - npu, h->side_stream))) return rc;
                CK(cudaEventRecord(h->ev_rest[k], h->side_stream));
                rest_recorded[k] = 1;
            } else if (cnt > npu) {
                // depth 2: even steps update block column k+2 only (what step k+1 needs) and defer the columns behind it;
                // odd steps apply panels k-1 and k together to every column >= k+2 in one K = 256 contraction (twice the
                // work per tile: the 128-long updates run at 45 % of the DMMA peak, mostly pipeline fill and tile I/O)
                CK(cudaStreamWaitEvent(h->side_stream, h->ev_panel[k], 0));
                if ((k & 1) == 0) {
                    s.jobs = ptr<GemmJob>(h->jobs) + off + npu;
                    if ((rc = launch_gemm<EPI_STORE>(h, h->mapK, h->mapK, s, std::min(nb - k - 1, cnt - npu), h->side_stream))) return rc;
                } else {
                    s.jobs = ptr<GemmJob>(h->jobs) + h->syrk2_r[k].off;
                    if ((rc = launch_gemm<EPI_STORE>(h, h->mapK, h->mapK, s, h->syrk2_r[k].cnt, h->side_stream))) return rc;
                }
                CK(cudaEventRecord(h->ev_rest[k], h->side_stream));
                rest_recorded[k] = 1;
            }
        }
    }
    if (!split && h->diag_kernel >= 3) {
        gpk_diag_qfill_kernel<<<nb, 256, 0, h->stream>>>(ptr<double>(h->P), ptr<double>(h->Q), (long)NP, ptr<int>(h->status));
        CKL();
    }
    CK(cudaEventRecord(h->ev[2], h->stream));
    gpk_fit_reduce_kernel<<<1, 256, 0, h->stream>>>(K + NP * NP, h->n, ptr<double>(h->logdet_part), nb,
                                                    ptr<double>(h->scal));
    CKL();
    CK(cudaEventRecord(h->ev[3], h->stream));
    CK(cudaMemcpyAsync(h->pin, h->scal.p, 16, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(h->pin + 2, h->status.p, 4, cudaMemcpyDeviceToHost, h->stream));
    h->fit_pending = true;
    return GPK_OK;
}

int gpk_fit_end(gpk_handle* h, double* logdet, double* loglik) {
    if (!h) return GPK_BAD_ARG;
    if (!h->fit_pending) BAD("gpk_fit_end without gpk_fit_begin");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    h->fit_pending = false;
    const double* sc = h->pin;
    int st = 0;
    memcpy(&st, h->pin + 2, 4);
    h->fit_timed = true;
    if (st != 0) {
        set_err(h, "matrix is not positive definite: pivot %d <= 0", st - 1);
        return GPK_NOT_PD;
    }
    const double ld = sc[1];
    const double ll = -0.5 * sc[0] - 0.5 * ld - 0.5 * (double)h->n * log(2.0 * M_PI);
    if (logdet) *logdet = ld;
    if (loglik) *loglik = ll;
    h->fitted = true;
    return GPK_OK;
}

int gpk_fit(gpk_handle* h, double diag_add, double mean, double* logdet, double* loglik) {
    int rc = gpk_fit_begin(h, diag_add, mean);
    if (rc) return rc;
    return gpk_fit_end(h, logdet, loglik);
}

// ---------------------------------------------------------------------------------------
// Incremental refit (SURVEY.md 8f-4: BaseModel.update / train(do_optimize=False) with frozen hyper-parameters).
// The rows appended since the last fit live in the last 128-row block b of the padded layout, so the leading factor
// L11 (N1 = 128 b rows), its inverse P11 and every earlier block of K are unchanged.  With L11^-1 explicit:
//   L_row = K[b, 0:N1] P11^T                      (one launch, 32-row tiles)
//   S     = K[b, b] - L_row L_row^T               (b partial Gram tiles + fixed-order sum)
//   L_bb, P_bb = chol / inverse of S              (the diagonal-block kernel)
//   P[b, 0:N1] = -P_bb (L_row P11)                (two launches; transposes kept in Q)
//   z = P (y - mean),  log|K| = 2 sum log diag    (y and the mean change with every new observation)
// O(N^2) work instead of the O(N^3) factorisation + inversion.  Returns GPK_NOT_APPLICABLE (nothing touched) when
// the preconditions do not hold; the caller then runs gpk_set_data + gpk_fit.
// ---------------------------------------------------------------------------------------
int gpk_fit_append(gpk_handle* h, const double* X, const double* y, int n, int d, double diag_add, double mean,
                   double* logdet, double* loglik) {
    if (!h) return GPK_BAD_ARG;
    if (!X || !y || n <= 0 || d <= 0) BAD("gpk_fit_append: need X, y, n > 0, d > 0");
    const long NP = h->NP;
    const int nb = h->nb, b = nb - 1, N1 = b * BM;
    if (!h->has_data || !h->has_spec || !h->fitted || !h->linv_ready || h->fit_pending || d != h->d || nb < 2 ||
        round_up(n, BM) != NP || n <= h->n || h->n <= N1 || diag_add != h->diag_add) {
        set_err(h, "gpk_fit_append: not applicable (needs a fitted model with L^-1 built, the same kernel / "
                   "diagonal term, new rows inside the last 128-row block)");
        return GPK_NOT_APPLICABLE;
    }
    CK(cudaSetDevice(h->device));
    int rc;
    if (!h->maps_ok && (rc = rebuild_maps(h))) return rc;
    double* K = ptr<double>(h->Kbuf);
    double* P = ptr<double>(h->P);
    double* Q = ptr<double>(h->Q);
    double* W = ptr<double>(h->W);
    if ((rc = ensure(h, h->tmp1, (size_t)NP * 8))) return rc;
    CK(cudaEventRecord(h->ev[0], h->stream));
    // inputs (everything is re-uploaded: 8 n (d + 1) bytes; the first h->n rows of X must be the ones already fitted)
    if ((rc = ensure(h, h->Xrow, (size_t)NP * d * 8))) return rc;      // no-op: gpk_set_data sized it for NP rows
    CK(cudaMemcpyAsync(h->Xrow.p, X, (size_t)n * d * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemsetAsync(h->y.p, 0, (size_t)NP * 8, h->stream));
    CK(cudaMemcpyAsync(h->y.p, y, (size_t)n * 8, cudaMemcpyHostToDevice, h->stream));
    {
        long total = (long)d * NP;
        gpk_transpose_kernel<<<(unsigned)((total + 255) / 256), 256, 0, h->stream>>>(ptr<double>(h->Xrow), n, d, nullptr,
                                                                                    nullptr, ptr<double>(h->Xt), NP);
        CKL();
    }
    // block row b of K (all columns), diagonal term, padding rows
    {
        if (cov_tma(h)) {
            if ((rc = ensure(h, h->Xts, (size_t)GPK_MAX_TERMS * NP * 8))) return rc;
            if ((rc = build_cov_operand(h, h->stream, ptr<double>(h->Xrow), n, d, nullptr, nullptr, ptr<double>(h->Xts), NP)))
                return rc;
        }
        if ((rc = launch_cov_tiles(h, h->stream, train_operand(h), NP, n, ptr<double>(h->Xrow) + (long)N1 * d, d,
                                   (long)(n - N1), BM, nullptr, nullptr, K + (long)N1 * NP, NP, 0, false)))
            return rc;
        gpk_kfix_rows_kernel<<<1, 128, 0, h->stream>>>(K, NP, n, (int)NP, diag_add, N1);
        CKL();
    }
    CK(cudaMemsetAsync(h->status.p, 0, 4, h->stream));
    CK(cudaEventRecord(h->ev[1], h->stream));
    GemmArgs a;
    // L_row = K[b, 0:N1] P11^T -> W[b, 0:N1]: split-K partial tiles into the free tiles W(c, j), then a fixed-order sum
    memset(&a, 0, sizeof(a));
    a.A = K; a.lda = NP; a.B = P; a.ldb = NP; a.C = W; a.ldc = NP;
    a.alpha = 1.0; a.beta = 0; a.job_mode = JOBS_TABLE;
    a.jobs = ptr<GemmJob>(h->jobs) + h->app_row2_r.off;
    if ((rc = launch_gemm<EPI_STORE>(h, h->mapK, h->mapP, a, h->app_row2_r.cnt))) return rc;
    gpk_append_reduce_kernel<<<dim3(b, 64), 256, 0, h->stream>>>(W, NP, b, 0, W + (long)N1 * NP, NP, nullptr, 0, 0);
    CKL();
    // partial Gram tiles, then the Schur complement of the last block
    memset(&a, 0, sizeof(a));
    a.A = W; a.lda = NP; a.B = W; a.ldb = NP; a.C = W; a.ldc = NP;
    a.alpha = 1.0; a.beta = 0; a.job_mode = JOBS_TABLE;
    a.jobs = ptr<GemmJob>(h->jobs) + h->app_syrk_r.off;
    if ((rc = launch_gemm<EPI_STORE>(h, h->mapW, h->mapW, a, h->app_syrk_r.cnt))) return rc;
    gpk_append_schur_kernel<<<64, 256, 0, h->stream>>>(K, W, NP, N1, b);
    CKL();
    // L_row to its final place (rows N1.. of K, columns 0..N1)
    CK(cudaMemcpy2DAsync(K + (long)N1 * NP, (size_t)NP * 8, W + (long)N1 * NP, (size_t)NP * 8, (size_t)N1 * 8, BM,
                         cudaMemcpyDeviceToDevice, h->stream));
    // factor + invert the last diagonal block
    if (h->diag_kernel >= 3) {
        gpk_diag_prezero_kernel<<<1, 256, 0, h->stream>>>(K + (long)N1 * NP + N1, (long)NP, P + (long)N1 * NP + N1, (long)NP);
        CKL();
        if (h->diag_kernel == 4)
            gpk_potrf_diag_dmma_kernel<<<1, 256, DIAG4_SMEM, h->stream>>>(K, NP, b, P, Q, NP, ptr<int>(h->status),
                                                                          ptr<double>(h->logdet_part), nullptr);
        else
            gpk_potrf_diag_blocked_kernel<<<1, 256, DIAG3_SMEM, h->stream>>>(K, NP, b, P, Q, NP, ptr<int>(h->status),
                                                                             ptr<double>(h->logdet_part), nullptr);
        CKL();
        gpk_diag_qfill_kernel<<<1, 256, 0, h->stream>>>(P + (long)N1 * NP + N1, Q + (long)N1 * NP + N1, (long)NP,
                                                         ptr<int>(h->status));
    } else if (h->diag_kernel == 2) {
        gpk_potrf_diag_fused_kernel<<<1, 256, DIAG2_SMEM, h->stream>>>(K, NP, b, P, Q, NP, ptr<int>(h->status),
                                                                       ptr<double>(h->logdet_part));
    } else {
        gpk_potrf_diag_kernel<<<1, 256, DIAG_SMEM, h->stream>>>(K, NP, b, P, Q, NP, ptr<int>(h->status),
                                                                ptr<double>(h->logdet_part));
    }
    CKL();
    // T = L_row P11 -> P[b, 0:N1], T^T -> Q[0:N1, b]   (split-K like L_row; the Gram partials in W(s, b) are consumed)
    memset(&a, 0, sizeof(a));
    a.A = K; a.lda = NP; a.B = Q; a.ldb = NP; a.C = W; a.ldc = NP;
    a.alpha = 1.0; a.beta = 0; a.job_mode = JOBS_TABLE; a.status = ptr<int>(h->status);
    a.jobs = ptr<GemmJob>(h->jobs) + h->app_t2_r.off;
    if ((rc = launch_gemm<EPI_STORE>(h, h->mapK, h->mapQ, a, h->app_t2_r.cnt))) return rc;
    gpk_append_reduce_kernel<<<dim3(b, 64), 256, 0, h->stream>>>(W, NP, b, 1, P + (long)N1 * NP, NP, Q, NP, N1);
    CKL();
    // P[b, 0:N1] = -P_bb T (and its transpose into Q)
    memset(&a, 0, sizeof(a));
    a.A = P; a.lda = NP; a.B = Q; a.ldb = NP; a.C = P; a.ldc = NP; a.Ct = Q; a.ldct = NP;
    a.alpha = -1.0; a.beta = 0; a.job_mode = JOBS_TABLE; a.status = ptr<int>(h->status);
    a.jobs = ptr<GemmJob>(h->jobs) + h->app_p_r.off;
    if ((rc = launch_gemm<EPI_STORE>(h, h->mapP, h->mapQ, a, h->app_p_r.cnt))) return rc;
    // z = P (y - mean) into row NP of K, then z^T z and the log-determinant
    gpk_resid_kernel<<<(unsigned)((NP + 255) / 256), 256, 0, h->stream>>>(ptr<double>(h->y), mean, n, (int)NP,
                                                                          ptr<double>(h->tmp1));
    CKL();
    gpk_rowdot_kernel<<<(unsigned)((NP + 7) / 8), 256, 0, h->stream>>>(P, NP, NP, (int)NP, 0, ptr<double>(h->tmp1),
                                                                       K + NP * NP);
    CKL();
    CK(cudaEventRecord(h->ev[2], h->stream));
    gpk_fit_reduce_kernel<<<1, 256, 0, h->stream>>>(K + NP * NP, n, ptr<double>(h->logdet_part), nb, ptr<double>(h->scal));
    CKL();
    CK(cudaEventRecord(h->ev[3], h->stream));
    CK(cudaMemcpyAsync(h->pin, h->scal.p, 16, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(h->pin + 2, h->status.p, 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->launches_total += 12;
    h->fit_timed = true;
    int st = 0;
    memcpy(&st, h->pin + 2, 4);
    if (st != 0) {                      // the block row of K / P is half updated: the model has to be refitted
        h->fitted = false;
        h->linv_ready = false;
        h->alpha_ready = false;
        h->n = n;
        set_err(h, "matrix is not positive definite: pivot %d <= 0", st - 1);
        return GPK_NOT_PD;
    }
    h->n = n;
    h->mean = mean;
    h->alpha_ready = false;
    h->linv_serial += 1;                 // L^-1 changed in place: slices / alpha derived from it are stale
    const double ld2 = h->pin[1];
    const double ll = -0.5 * h->pin[0] - 0.5 * ld2 - 0.5 * (double)n * log(2.0 * M_PI);
    if (logdet) *logdet = ld2;
    if (loglik) *loglik = ll;
    return GPK_OK;
}

int gpk_acq_dev(gpk_handle* h, const void* d_Xs, long m, int kind, double eta, double par, void* d_out, void* d_mu,
                void* d_var, void* d_best) {
    int rc = require(h, true, true, true);
    if (rc) return rc;
    if (!d_Xs || m <= 0) BAD("gpk_acq_dev: need candidates");
    if (kind < GPK_ACQ_NONE || kind > GPK_ACQ_LCB) BAD("gpk_acq_dev: unknown acquisition %d", kind);
    CK(cudaSetDevice(h->device));
    return score_dev(h, (const double*)d_Xs, m, kind, eta, par, (double*)d_out, (double*)d_mu, (double*)d_var,
                     (BestPair*)d_best, nullptr);
}

// Pageable host memory reaches the device at 1-2 GB/s through cudaMemcpyAsync (the driver stages it synchronously in
// small pieces): a 2^20 x 8 candidate batch (67 MB, config C3) took 40 ms to copy for 3 ms of scoring.  Large pageable
// batches are therefore copied by the host into two pinned staging buffers and go out by DMA while the next piece is
// being staged.  Pinned / registered caller buffers are used in place.
static bool host_is_pinned(const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
}

static int ensure_stage(gpk_handle* h, size_t bytes) {
    if (bytes <= h->stage_cap) return GPK_OK;
    for (int i = 0; i < 2; ++i) {
        if (h->stage[i]) CK(cudaFreeHost(h->stage[i]));
        h->stage[i] = nullptr;
    }
    h->stage_cap = 0;
    for (int i = 0; i < 2; ++i) CK(cudaHostAlloc((void**)&h->stage[i], bytes, cudaHostAllocDefault));
    h->stage_cap = bytes;
    return GPK_OK;
}

namespace {
// rows of a host batch -> h->cand, piece by piece on the copy stream; pageable memory goes through two pinned staging
// buffers filled by the host while the previous piece is in flight
struct HostFeeder : Feeder {
    gpk_handle* h;
    const double* Xs;          // first row of the (super-)batch being scored
    long rows, piece;
    bool staged;
    long next = 0;             // rows already enqueued
    int npieces = 0;
    int ready(long lo, long hi, cudaStream_t st) override {
        (void)lo;
        const long d = h->d;
        while (next < hi && next < rows) {
            const int i = npieces;
            const long mc = std::min(piece, rows - next);
            while ((int)h->ev_copied.size() <= i) {
                cudaEvent_t e1;
                CK(cudaEventCreateWithFlags(&e1, cudaEventDisableTiming));
                h->ev_copied.push_back(e1);
            }
            const double* src = Xs + next * d;
            if (staged) {
                if (i >= 2) CK(cudaEventSynchronize(h->ev_copied[i - 2]));   // the DMA out of this staging buffer is done
                memcpy(h->stage[i & 1], src, (size_t)mc * d * 8);
                src = h->stage[i & 1];
            }
            CK(cudaMemcpyAsync(ptr<double>(h->cand) + next * d, src, (size_t)mc * d * 8, cudaMemcpyHostToDevice, h->copy_stream));
            CK(cudaEventRecord(h->ev_copied[i], h->copy_stream));
            next += mc;
            ++npieces;
        }
        if (npieces > 0) CK(cudaStreamWaitEvent(st, h->ev_copied[npieces - 1], 0));
        return GPK_OK;
    }
};
}  // namespace

int gpk_acq(gpk_handle* h, const double* Xs, long m, int kind, double eta, double par, double* out, double* mu,
            double* var, double* best_val, long* best_idx, long* n_negative) {
    int rc = require(h, true, true, true);
    if (rc) return rc;
    if (!Xs || m <= 0) BAD("gpk_acq: need candidates");
    if (kind < GPK_ACQ_NONE || kind > GPK_ACQ_LCB) BAD("gpk_acq: unknown acquisition %d", kind);
    CK(cudaSetDevice(h->device));
    const long d = h->d;
    // the device copy of the batch: whole batches up to 1 GiB, larger ones in super-batches of that size
    const long super = std::max<long>(BM, (((long)1 << 30) / (d * 8)) / BM * BM);
    if ((rc = ensure(h, h->cand, (size_t)std::min<long>(m, super) * d * 8))) return rc;
    if (out && (rc = ensure(h, h->out_acq, (size_t)m * 8))) return rc;
    if (mu && (rc = ensure(h, h->out_mu, (size_t)m * 8))) return rc;
    if (var && (rc = ensure(h, h->out_var, (size_t)m * 8))) return rc;
    CK(cudaEventRecord(h->ev[14], h->stream));
    const long piece = std::min<long>(chunk_rows(h), round_up(m, BM));       // one H2D piece per scoring chunk
    const bool small = (size_t)m * d * 8 <= ((size_t)1 << 20);
    const bool staged = !small && !host_is_pinned(Xs);
    if (staged && (rc = ensure_stage(h, (size_t)piece * d * 8))) return rc;
    if (small) {
        CK(cudaMemcpyAsync(h->cand.p, Xs, (size_t)m * d * 8, cudaMemcpyHostToDevice, h->stream));
        rc = score_dev(h, ptr<double>(h->cand), m, kind, eta, par, out ? ptr<double>(h->out_acq) : nullptr,
                       mu ? ptr<double>(h->out_mu) : nullptr, var ? ptr<double>(h->out_var) : nullptr, nullptr, nullptr);
        if (rc) return rc;
    } else {
        for (long base = 0; base < m; base += super) {
            const long rows = std::min(super, m - base);
            // the copy stream starts after everything already queued on the scoring stream (earlier users of h->cand)
            CK(cudaEventRecord(h->ev_order, h->stream));
            CK(cudaStreamWaitEvent(h->copy_stream, h->ev_order, 0));
            if (base > 0) CK(cudaStreamSynchronize(h->copy_stream));     // staging buffers and h->cand are reused
            HostFeeder feeder;
            feeder.h = h; feeder.Xs = Xs + base * d; feeder.rows = rows; feeder.piece = piece; feeder.staged = staged;
            rc = score_dev(h, ptr<double>(h->cand), rows, kind, eta, par, out ? ptr<double>(h->out_acq) : nullptr,
                           mu ? ptr<double>(h->out_mu) : nullptr, var ? ptr<double>(h->out_var) : nullptr, nullptr, nullptr,
                           base, base == 0, 0, &feeder);
            if (rc) return rc;
        }
    }
    if (out) CK(cudaMemcpyAsync(out, h->out_acq.p, (size_t)m * 8, cudaMemcpyDeviceToHost, h->stream));
    if (mu) CK(cudaMemcpyAsync(mu, h->out_mu.p, (size_t)m * 8, cudaMemcpyDeviceToHost, h->stream));
    if (var) CK(cudaMemcpyAsync(var, h->out_var.p, (size_t)m * 8, cudaMemcpyDeviceToHost, h->stream));
    BestPair bp;
    unsigned long long nn = 0;
    CK(cudaMemcpyAsync(&bp, h->best.p, sizeof(bp), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(&nn, h->nneg.p, 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaEventRecord(h->ev[15], h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (best_val) *best_val = bp.val;
    if (best_idx) *best_idx = (long)bp.idx;
    if (n_negative) *n_negative = (long)nn;
    return GPK_OK;
}

// candidates [first, first+count) of the device generator into h->cand (device, count x d)
static int generate_candidates(gpk_handle* h, unsigned long long seed, long first, long count, long n_uniform, int d,
                               const double* lower, const double* upper, const double* incumbent, double scale) {
    int rc;
    if ((rc = ensure(h, h->cand, (size_t)count * d * 8))) return rc;
    if ((rc = ensure(h, h->tmp1, (size_t)3 * d * 8))) return rc;
    double* dl = ptr<double>(h->tmp1);
    CK(cudaMemcpyAsync(dl, lower, (size_t)d * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(dl + d, upper, (size_t)d * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(dl + 2 * d, incumbent, (size_t)d * 8, cudaMemcpyHostToDevice, h->stream));
    const long total = count * ((d + 1) / 2);
    gpk_candidates_kernel<<<(unsigned)((total + 255) / 256), 256, 0, h->stream>>>(seed, first, count, n_uniform, d, dl, dl + d,
                                                                              dl + 2 * d, scale, ptr<double>(h->cand));
    CKL();
    return GPK_OK;
}

int gpk_generate_candidates(gpk_handle* h, unsigned long long seed, long first, long count, long n_uniform, int d,
                            const double* lower, const double* upper, const double* incumbent, double scale,
                            double* out) {
    if (!h) return GPK_BAD_ARG;
    if (!lower || !upper || !incumbent || !out || count <= 0 || d <= 0 || d > GPK_MAX_TERMS || first < 0)
        BAD("gpk_generate_candidates: bad arguments");
    CK(cudaSetDevice(h->device));
    int rc = generate_candidates(h, seed, first, count, n_uniform, d, lower, upper, incumbent, scale);
    if (rc) return rc;
    CK(cudaMemcpyAsync(out, h->cand.p, (size_t)count * d * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return GPK_OK;
}

int gpk_maximize_random(gpk_handle* h, unsigned long long seed, long first, long count, long n_uniform,
                        const double* lower, const double* upper, const double* incumbent, double scale, int kind,
                        double eta, double par, double* best_x, double* best_val, long* best_idx) {
    int rc = require(h, true, true, true);
    if (rc) return rc;
    if (!lower || !upper || !incumbent || count <= 0 || first < 0) BAD("gpk_maximize_random: bad arguments");
    if (kind < GPK_ACQ_EI || kind > GPK_ACQ_LCB) BAD("gpk_maximize_random: unknown acquisition %d", kind);
    CK(cudaSetDevice(h->device));
    if ((rc = generate_candidates(h, seed, first, count, n_uniform, h->d, lower, upper, incumbent, scale))) return rc;
    if ((rc = score_dev(h, ptr<double>(h->cand), count, kind, eta, par, nullptr, nullptr, nullptr, nullptr, nullptr)))
        return rc;
    BestPair bp;
    CK(cudaMemcpyAsync(&bp, h->best.p, sizeof(bp), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (bp.idx >= 0 && best_x)
        CK(cudaMemcpy(best_x, ptr<double>(h->cand) + bp.idx * h->d, (size_t)h->d * 8, cudaMemcpyDeviceToHost));
    if (best_val) *best_val = bp.val;
    if (best_idx) *best_idx = bp.idx >= 0 ? (long)(first + bp.idx) : -1;
    return GPK_OK;
}

int gpk_predict(gpk_handle* h, const double* Xs, long m, double* mu, double* var) {
    return gpk_acq(h, Xs, m, GPK_ACQ_NONE, 0.0, 0.0, nullptr, mu, var, nullptr, nullptr, nullptr);
}

static int predict_cov_impl(gpk_handle* h, const double* Xs, long m, double* mu, double* cov, int clip) {
    int rc = require(h, true, true, true);
    if (rc) return rc;
    if (!Xs || m <= 0 || !mu || !cov) BAD("gpk_predict_cov: need Xs, mu, cov");
    if (m > 16384) BAD("gpk_predict_cov: m = %ld too large for a dense m x m covariance", m);
    CK(cudaSetDevice(h->device));
    if ((rc = build_linv(h))) return rc;
    const long NP = h->NP, mp = round_up(m, BM);
    const int nb = h->nb, mb = (int)(mp / BM);
    if ((rc = ensure(h, h->cand, (size_t)m * h->d * 8))) return rc;
    if ((rc = ensure_score_scratch(h, mp))) return rc;
    bool grew = false;
    if ((rc = ensure(h, h->Vt, (size_t)mp * NP * 8, &grew))) return rc;
    if (grew || h->mapVt_rows != mp) {
        if (h->loader != LOADER_CPASYNC && (rc = make_map(h, &h->mapVt, h->Vt.p, mp, NP, NP))) return rc;
        h->mapVt_rows = mp;
    }
    if ((rc = ensure(h, h->cov, (size_t)mp * mp * 8))) return rc;
    if ((rc = ensure(h, h->XsT, cov_operand_rows(h, h->d) * mp * 8))) return rc;
    if ((rc = ensure(h, h->out_mu, (size_t)mp * 8))) return rc;
    CK(cudaMemcpyAsync(h->cand.p, Xs, (size_t)m * h->d * 8, cudaMemcpyHostToDevice, h->stream));
    const double* lo = h->has_bounds ? ptr<double>(h->lower) : nullptr;
    const double* up = h->has_bounds ? ptr<double>(h->upper) : nullptr;
    // K* (mp x NP)
    if ((rc = launch_cov_tiles(h, h->stream, train_operand(h), NP, h->n, ptr<double>(h->cand), h->d, m, mp, lo, up,
                               ptr<double>(h->Kstar), NP, 0, false)))
        return rc;
    // K** (mp x mp): candidates against the (scaled, transposed) candidates
    if ((rc = build_cov_operand(h, h->stream, ptr<double>(h->cand), m, h->d, lo, up, ptr<double>(h->XsT), mp))) return rc;
    if ((rc = launch_cov_tiles(h, h->stream, ptr<double>(h->XsT), mp, (int)m, ptr<double>(h->cand), h->d, m, mp, lo, up,
                               ptr<double>(h->cov), mp, 0, false)))
        return rc;
    // V^T = (L^-1 K*^T)^T  ->  Vt[cand][i]
    std::vector<GemmJob> jobs;
    for (int ib = nb - 1; ib >= 0; --ib)
        for (int cb = 0; cb < mb; ++cb) jobs.push_back({ib * BM, cb * BM, 0, (ib + 1) * BM, ib * BM, cb * BM, 0, 0});
    const size_t n1 = jobs.size();
    for (int a = 0; a < mb; ++a)
        for (int b = 0; b < mb; ++b) jobs.push_back({a * BM, b * BM, 0, (int)NP, a * BM, b * BM, 0, 0});
    if ((rc = ensure(h, h->tmpjobs, jobs.size() * sizeof(GemmJob)))) return rc;
    CK(cudaMemcpyAsync(h->tmpjobs.p, jobs.data(), jobs.size() * sizeof(GemmJob), cudaMemcpyHostToDevice, h->stream));
    {
        GemmArgs a;
        memset(&a, 0, sizeof(a));
        a.A = ptr<double>(h->P); a.lda = NP;
        a.B = ptr<double>(h->Kstar); a.ldb = NP;
        a.Ct = ptr<double>(h->Vt); a.ldct = NP;
        a.alpha = 1.0;
        a.jobs = ptr<GemmJob>(h->tmpjobs);
        a.job_mode = JOBS_TABLE;
        if ((rc = launch_gemm<EPI_STORE>(h, h->mapP, h->mapKs, a, (int)n1))) return rc;
    }
    // mu = Vt z ; cov = K** - Vt Vt^T
    gpk_rowdot_kernel<<<(unsigned)((mp + 7) / 8), 256, 0, h->stream>>>(ptr<double>(h->Vt), NP, m, (int)NP, 0,
                                                                        ptr<double>(h->Kbuf) + NP * NP,
                                                                        ptr<double>(h->out_mu));
    CKL();
    gpk_mu_finish_kernel<<<(unsigned)((m + 255) / 256), 256, 0, h->stream>>>(ptr<double>(h->out_mu), m, h->mean,
                                                                            h->norm_out, h->y_mean, h->y_std);
    CKL();
    {
        GemmArgs a;
        memset(&a, 0, sizeof(a));
        a.A = ptr<double>(h->Vt); a.lda = NP;
        a.B = ptr<double>(h->Vt); a.ldb = NP;
        a.C = ptr<double>(h->cov); a.ldc = mp;
        a.alpha = -1.0; a.beta = 1;
        a.jobs = ptr<GemmJob>(h->tmpjobs) + n1;
        a.job_mode = JOBS_TABLE;
        if ((rc = launch_gemm<EPI_STORE>(h, h->mapVt, h->mapVt, a, (int)(jobs.size() - n1)))) return rc;
    }
    gpk_cov_finish_kernel<<<(unsigned)((m * m + 255) / 256), 256, 0, h->stream>>>(ptr<double>(h->cov), mp, m,
                                                                                 h->norm_out, h->y_std, clip);
    CKL();
    CK(cudaMemcpyAsync(mu, h->out_mu.p, (size_t)m * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpy2DAsync(cov, (size_t)m * 8, h->cov.p, (size_t)mp * 8, (size_t)m * 8, (size_t)m, cudaMemcpyDeviceToHost,
                         h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return GPK_OK;
}

int gpk_predict_cov(gpk_handle* h, const double* Xs, long m, double* mu, double* cov) {
    return predict_cov_impl(h, Xs, m, mu, cov, 1);
}

int gpk_posterior_cov(gpk_handle* h, const double* Xs, long m, double* mu, double* cov) {
    return predict_cov_impl(h, Xs, m, mu, cov, 0);
}

int gpk_predict_grad(gpk_handle* h, const double* Xs, long m, int kind, double eta, double par, double* mu, double* var,
                     double* dmu, double* dvar, double* f, double* df) {
    int rc = require(h, true, true, true);
    if (rc) return rc;
    if (!Xs || m <= 0 || !mu || !var || !dmu || !dvar) BAD("gpk_predict_grad: need Xs, mu, var, dmu, dvar");
    if (m > 16384) BAD("gpk_predict_grad: m = %ld too large", m);
    if (kind != GPK_ACQ_NONE && (kind == GPK_ACQ_LOG_EI || kind < GPK_ACQ_NONE || kind > GPK_ACQ_LCB || !f || !df))
        BAD("gpk_predict_grad: acquisition gradients exist for EI, PI, LCB and need f, df");
    CK(cudaSetDevice(h->device));
    if ((rc = build_linv(h))) return rc;
    const long NP = h->NP, mp = round_up(m, BM);
    const int nb = h->nb, mb = (int)(mp / BM), d = h->d;
    if ((rc = ensure(h, h->cand, (size_t)m * d * 8))) return rc;
    if ((rc = ensure_score_scratch(h, mp))) return rc;
    bool grew = false;
    if ((rc = ensure(h, h->Vt, (size_t)mp * NP * 8, &grew))) return rc;
    if (grew || h->mapVt_rows != mp) {
        if (h->loader != LOADER_CPASYNC && (rc = make_map(h, &h->mapVt, h->Vt.p, mp, NP, NP))) return rc;
        h->mapVt_rows = mp;
    }
    if ((rc = ensure(h, h->cov, (size_t)mp * NP * 8))) return rc;            // Wt = (K^-1 K*^T)^T
    if ((rc = ensure(h, h->alpha, (size_t)NP * 8))) return rc;
    if ((rc = ensure(h, h->out_mu, (size_t)mp * 8))) return rc;
    if ((rc = ensure(h, h->out_var, (size_t)mp * 8))) return rc;
    if ((rc = ensure(h, h->tmp1, (size_t)m * d * 8 * 2))) return rc;
    if ((rc = ensure(h, h->tmp2, (size_t)m * (d + 1) * 8))) return rc;
    CK(cudaMemcpyAsync(h->cand.p, Xs, (size_t)m * d * 8, cudaMemcpyHostToDevice, h->stream));
    // moments through the regular scoring path (same numbers as gpk_predict)
    if ((rc = score_dev(h, ptr<double>(h->cand), m, GPK_ACQ_NONE, 0.0, 0.0, nullptr, ptr<double>(h->out_mu),
                        ptr<double>(h->out_var), nullptr, nullptr)))
        return rc;
    const double* lo = h->has_bounds ? ptr<double>(h->lower) : nullptr;
    const double* up = h->has_bounds ? ptr<double>(h->upper) : nullptr;
    if ((rc = ensure_score_scratch(h, mp))) return rc;       // score_dev may have sized the K* map for a smaller chunk
    // K* again into the first buffer (score_dev may have used either), then Vt = (L^-1 K*^T)^T, Wt = (L^-T V)^T
    if ((rc = launch_cov_tiles(h, h->stream, train_operand(h), NP, h->n, ptr<double>(h->cand), d, m, mp, lo, up,
                               ptr<double>(h->Kstar), NP, 0, false)))
        return rc;
    std::vector<GemmJob> jobs;
    for (int ib = nb - 1; ib >= 0; --ib)
        for (int cb = 0; cb < mb; ++cb) jobs.push_back({ib * BM, cb * BM, 0, (ib + 1) * BM, ib * BM, cb * BM, 0, 0});
    const size_t n1 = jobs.size();
    for (int jb = 0; jb < nb; ++jb)
        for (int cb = 0; cb < mb; ++cb) jobs.push_back({cb * BM, jb * BM, jb * BM, (int)NP, cb * BM, jb * BM, 0, 0});
    if ((rc = ensure(h, h->tmpjobs, jobs.size() * sizeof(GemmJob)))) return rc;
    CK(cudaMemcpyAsync(h->tmpjobs.p, jobs.data(), jobs.size() * sizeof(GemmJob), cudaMemcpyHostToDevice, h->stream));
    {
        GemmArgs a;
        memset(&a, 0, sizeof(a));
        a.A = ptr<double>(h->P); a.lda = NP;
        a.B = ptr<double>(h->Kstar); a.ldb = NP;
        a.Ct = ptr<double>(h->Vt); a.ldct = NP;
        a.alpha = 1.0;
        a.jobs = ptr<GemmJob>(h->tmpjobs);
        a.job_mode = JOBS_TABLE;
        if ((rc = launch_gemm<EPI_STORE>(h, h->mapP, h->mapKs, a, (int)n1))) return rc;
        GemmArgs b;
        memset(&b, 0, sizeof(b));
        b.A = ptr<double>(h->Vt); b.lda = NP;                // Wt[c][j] = sum_{i >= j} Vt[c][i] Q[j][i]
        b.B = ptr<double>(h->Q); b.ldb = NP;
        b.C = ptr<double>(h->cov); b.ldc = NP;
        b.alpha = 1.0;
        b.jobs = ptr<GemmJob>(h->tmpjobs) + n1;
        b.job_mode = JOBS_TABLE;
        if ((rc = launch_gemm<EPI_STORE>(h, h->mapVt, h->mapQ, b, (int)(jobs.size() - n1)))) return rc;
    }
    gpk_rowdot_kernel<<<(unsigned)((NP + 7) / 8), 256, 0, h->stream>>>(ptr<double>(h->Q), NP, NP, (int)NP, 1,
                                                                       ptr<double>(h->Kbuf) + NP * NP,
                                                                       ptr<double>(h->alpha));
    CKL();
    double* d_dmu = ptr<double>(h->tmp1);
    double* d_dvar = d_dmu + m * d;
    gpk_predict_grad_kernel<<<(unsigned)m, 256, 0, h->stream>>>(h->spec, ptr<double>(h->Xt), NP, h->n, ptr<double>(h->cand), d,
                                                              lo, up, ptr<double>(h->alpha), ptr<double>(h->cov), NP,
                                                              h->norm_out, h->y_std, d_dmu, d_dvar);
    CKL();
    CK(cudaMemcpyAsync(mu, h->out_mu.p, (size_t)m * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(var, h->out_var.p, (size_t)m * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(dmu, d_dmu, (size_t)m * d * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(dvar, d_dvar, (size_t)m * d * 8, cudaMemcpyDeviceToHost, h->stream));
    if (kind != GPK_ACQ_NONE) {
        double* d_f = ptr<double>(h->tmp2);
        double* d_df = d_f + m;
        gpk_acq_grad_kernel<<<(unsigned)((m * d + 255) / 256), 256, 0, h->stream>>>(
            ptr<double>(h->out_mu), ptr<double>(h->out_var), d_dmu, d_dvar, m, d, kind, eta, par, d_f, d_df);
        CKL();
        CK(cudaMemcpyAsync(f, d_f, (size_t)m * 8, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemcpyAsync(df, d_df, (size_t)m * d * 8, cudaMemcpyDeviceToHost, h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    return GPK_OK;
}

int gpk_acq_moments(gpk_handle* h, const double* mu, const double* var, long m, int kind, double eta, double par,
                    double* out, long* n_negative) {
    if (!h) return GPK_BAD_ARG;
    if (!mu || !var || !out || m <= 0) BAD("gpk_acq_moments: need mu, var, out");
    if (kind < GPK_ACQ_EI || kind > GPK_ACQ_LCB) BAD("gpk_acq_moments: unknown acquisition %d", kind);
    CK(cudaSetDevice(h->device));
    int rc;
    if ((rc = ensure(h, h->tmp1, (size_t)m * 8))) return rc;
    if ((rc = ensure(h, h->tmp2, (size_t)m * 8))) return rc;
    if ((rc = ensure(h, h->tmp3, (size_t)m * 8))) return rc;
    if ((rc = ensure(h, h->nneg, 8))) return rc;
    CK(cudaMemcpyAsync(h->tmp1.p, mu, (size_t)m * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->tmp2.p, var, (size_t)m * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemsetAsync(h->nneg.p, 0, 8, h->stream));
    gpk_acq_moments_kernel<<<(unsigned)((m + 255) / 256), 256, 0, h->stream>>>(
        ptr<double>(h->tmp1), ptr<double>(h->tmp2), m, kind, eta, par, ptr<double>(h->tmp3),
        ptr<unsigned long long>(h->nneg));
    CKL();
    unsigned long long nn = 0;
    CK(cudaMemcpyAsync(out, h->tmp3.p, (size_t)m * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(&nn, h->nneg.p, 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (n_negative) *n_negative = (long)nn;
    return GPK_OK;
}

int gpk_reduce_models(gpk_handle* h, const double* A, const double* B, int n_models, long m, int mode, double* out1,
                      double* out2) {
    if (!h) return GPK_BAD_ARG;
    if (!A || !out1 || n_models <= 0 || m <= 0 || (mode != 0 && mode != 1)) BAD("gpk_reduce_models: bad arguments");
    if (mode == 1 && (!B || !out2)) BAD("gpk_reduce_models: mode 1 needs B and out2");
    CK(cudaSetDevice(h->device));
    int rc;
    const size_t bytes = (size_t)n_models * m * 8;
    if ((rc = ensure(h, h->tmp1, bytes))) return rc;
    if ((rc = ensure(h, h->tmp2, mode == 1 ? bytes : 8))) return rc;
    if ((rc = ensure(h, h->tmp3, (size_t)m * 16))) return rc;
    CK(cudaMemcpyAsync(h->tmp1.p, A, bytes, cudaMemcpyHostToDevice, h->stream));
    if (mode == 1) CK(cudaMemcpyAsync(h->tmp2.p, B, bytes, cudaMemcpyHostToDevice, h->stream));
    double* o1 = ptr<double>(h->tmp3);
    double* o2 = o1 + m;
    gpk_reduce_models_kernel<<<(unsigned)((m + 255) / 256), 256, 0, h->stream>>>(
        ptr<double>(h->tmp1), mode == 1 ? ptr<double>(h->tmp2) : nullptr, n_models, m, mode, o1, o2);
    CKL();
    CK(cudaMemcpyAsync(out1, o1, (size_t)m * 8, cudaMemcpyDeviceToHost, h->stream));
    if (mode == 1) CK(cudaMemcpyAsync(out2, o2, (size_t)m * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return GPK_OK;
}

int gpk_kernel_matrix(gpk_handle* h, const double* X1, long n1, const double* X2, long n2, int d, double* out) {
    int rc = require(h, false, true, false);
    if (rc) return rc;
    if (!X1 || !X2 || !out || n1 <= 0 || n2 <= 0 || d <= 0 || d > GPK_MAX_TERMS) BAD("gpk_kernel_matrix: bad arguments");
    for (int t = 0; t < h->spec.n_terms; ++t)
        if (h->spec.axis[t] >= d) BAD("gpk_kernel_matrix: kernel axis %d >= d = %d", h->spec.axis[t], d);
    CK(cudaSetDevice(h->device));
    const long n1p = round_up(n1, 32), n2p = round_up(n2, 128);
    if ((rc = ensure(h, h->tmp1, (size_t)n1 * d * 8))) return rc;
    const long x2off = round_up(n2 * d, 16);                 // keeps the operand 128-byte aligned (TMA source)
    if ((rc = ensure(h, h->tmp2, (size_t)(x2off + (long)cov_operand_rows(h, d) * n2p) * 8))) return rc;
    if ((rc = ensure(h, h->tmp3, (size_t)n1p * n2p * 8))) return rc;
    double* X2row = ptr<double>(h->tmp2);
    double* X2t = X2row + x2off;
    CK(cudaMemcpyAsync(h->tmp1.p, X1, (size_t)n1 * d * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(X2row, X2, (size_t)n2 * d * 8, cudaMemcpyHostToDevice, h->stream));
    if ((rc = build_cov_operand(h, h->stream, X2row, n2, d, nullptr, nullptr, X2t, n2p))) return rc;
    if ((rc = launch_cov_tiles(h, h->stream, X2t, n2p, (int)n2, ptr<double>(h->tmp1), d, n1, n1p, nullptr, nullptr,
                               ptr<double>(h->tmp3), n2p, 0, false)))
        return rc;
    CK(cudaMemcpy2DAsync(out, (size_t)n2 * 8, h->tmp3.p, (size_t)n2p * 8, (size_t)n2 * 8, (size_t)n1,
                         cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return GPK_OK;
}

int gpk_nll_grad(gpk_handle* h, double noise_var, double* grad) {
    int rc = require(h, true, true, true);
    if (rc) return rc;
    if (!grad) BAD("gpk_nll_grad: null output");
    CK(cudaSetDevice(h->device));
    if ((rc = build_linv(h))) return rc;
    const long NP = h->NP;
    const int nv = h->spec.n_terms + 2;
    // alpha = L^-T z
    if ((rc = ensure(h, h->alpha, (size_t)NP * 8))) return rc;
    gpk_rowdot_kernel<<<(unsigned)((NP + 7) / 8), 256, 0, h->stream>>>(ptr<double>(h->Q), NP, NP, (int)NP, 1,
                                                                       ptr<double>(h->Kbuf) + NP * NP,
                                                                       ptr<double>(h->alpha));
    CKL();
    // K^-1 (lower tiles) into W
    {
        GemmArgs a;
        memset(&a, 0, sizeof(a));
        a.A = ptr<double>(h->Q); a.lda = NP;
        a.B = ptr<double>(h->Q); a.ldb = NP;
        a.C = ptr<double>(h->W); a.ldc = NP;
        a.alpha = 1.0; a.beta = 0;
        a.jobs = ptr<GemmJob>(h->jobs) + h->kinv_r.off;
        a.job_mode = JOBS_TABLE;
        if ((rc = launch_gemm<EPI_STORE>(h, h->mapQ, h->mapQ, a, h->kinv_r.cnt))) return rc;
    }
    dim3 tg((unsigned)(NP / 128), (unsigned)(NP / 32));
    const long nblocks = (long)tg.x * tg.y;
    if ((rc = ensure(h, h->tmp1, (size_t)nblocks * nv * 8))) return rc;
    if ((rc = ensure(h, h->tmp2, (size_t)nv * 8))) return rc;
    gpk_grad_trace_kernel<<<tg, 256, 0, h->stream>>>(h->spec, ptr<double>(h->Xt), NP, h->n, ptr<double>(h->Xrow), h->d,
                                                     ptr<double>(h->W), NP, ptr<double>(h->alpha), ptr<double>(h->tmp1));
    CKL();
    gpk_grad_final_kernel<<<nv, 256, 0, h->stream>>>(ptr<double>(h->tmp1), nblocks, nv, noise_var, ptr<double>(h->tmp2));
    CKL();
    CK(cudaMemcpyAsync(grad, h->tmp2.p, (size_t)nv * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return GPK_OK;
}

int gpk_measure_fp64_peaks(gpk_handle* h, double* dmma_tflops, double* dfma_tflops) {
    if (!h) return GPK_BAD_ARG;
    CK(cudaSetDevice(h->device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, h->device));
    const int blocks = prop.multiProcessorCount, warps = 16, threads = warps * 32, iters = 8000;
    int rc;
    if ((rc = ensure(h, h->tmp1, 64))) return rc;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    double best_mma = 0.0, best_fma = 0.0;
    for (int rep = 0; rep < 3; ++rep) {
        float ms = 0.f;
        CK(cudaEventRecord(e0, h->stream));
        gpk_peak_dmma_kernel<<<blocks, threads, 0, h->stream>>>(ptr<double>(h->tmp1), iters);
        CKL();
        CK(cudaEventRecord(e1, h->stream));
        CK(cudaEventSynchronize(e1));
        CK(cudaEventElapsedTime(&ms, e0, e1));
        best_mma = std::max(best_mma, 2.0 * 256 * 16 * (double)iters * warps * blocks / (ms * 1e-3) / 1e12);
        CK(cudaEventRecord(e0, h->stream));
        gpk_peak_dfma_kernel<<<blocks, threads, 0, h->stream>>>(ptr<double>(h->tmp1), iters);
        CKL();
        CK(cudaEventRecord(e1, h->stream));
        CK(cudaEventSynchronize(e1));
        CK(cudaEventElapsedTime(&ms, e0, e1));
        best_fma = std::max(best_fma, 2.0 * 8 * (double)iters * threads * blocks / (ms * 1e-3) / 1e12);
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (dmma_tflops) *dmma_tflops = best_mma;
    if (dfma_tflops) *dfma_tflops = best_fma;
    return GPK_OK;
}

int gpk_measure_int8_peak(gpk_handle* h, double* tops) {
    if (!h || !tops) return GPK_BAD_ARG;
    CK(cudaSetDevice(h->device));
    const int blocks = std::max(h->n_sm, 1), iters = 4000, smem = 2 * 8192 + 1024 + 64;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    double best = 0.0;
    for (int rep = 0; rep < 3; ++rep) {
        float ms = 0.f;
        CK(cudaEventRecord(e0, h->stream));
        gpk_peak_i8_kernel<<<blocks, 128, smem, h->stream>>>(iters, 0);
        CKL();
        CK(cudaEventRecord(e1, h->stream));
        CK(cudaEventSynchronize(e1));
        CK(cudaEventElapsedTime(&ms, e0, e1));
        best = std::max(best, 2.0 * 128 * 128 * 32 * 2.0 * iters * blocks / (ms * 1e-3) / 1e12);
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *tops = best;
    return GPK_OK;
}

int gpk_measure_int8_peak_sustained(gpk_handle* h, double seconds, int random_operands, double* tops) {
    if (!h || !tops || !(seconds > 0.0) || seconds > 10.0) return GPK_BAD_ARG;
    CK(cudaSetDevice(h->device));
    // back-to-back launches of the issue-rate kernel for `seconds`; the rate of the SECOND half is reported: by then the
    // SM clock has settled where the board's power limit puts it (the int8 pipe at full rate runs into sw_power_cap)
    const int blocks = std::max(h->n_sm, 1), iters = 8000, smem = 2 * 8192 + 1024 + 64;
    const double ops = 2.0 * 128 * 128 * 32 * 2.0 * iters * blocks;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    float ms1 = 0.f;
    CK(cudaEventRecord(e0, h->stream));
    gpk_peak_i8_kernel<<<blocks, 128, smem, h->stream>>>(iters, random_operands);
    CKL();
    CK(cudaEventRecord(e1, h->stream));
    CK(cudaEventSynchronize(e1));
    CK(cudaEventElapsedTime(&ms1, e0, e1));
    const int n_half = std::max(1, (int)(0.5 * seconds * 1e3 / std::max(ms1, 1e-3f)));
    for (int i = 0; i < n_half; ++i) gpk_peak_i8_kernel<<<blocks, 128, smem, h->stream>>>(iters, random_operands);
    CK(cudaEventRecord(e0, h->stream));
    for (int i = 0; i < n_half; ++i) gpk_peak_i8_kernel<<<blocks, 128, smem, h->stream>>>(iters, random_operands);
    CKL();
    CK(cudaEventRecord(e1, h->stream));
    CK(cudaEventSynchronize(e1));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *tops = ops * n_half / (ms * 1e-3) / 1e12;
    return GPK_OK;
}

int gpk_get_factor(gpk_handle* h, double* L) {
    int rc = require(h, true, true, true);
    if (rc) return rc;
    if (!L) BAD("gpk_get_factor: null output");
    CK(cudaSetDevice(h->device));
    const long n = h->n, NP = h->NP;
    CK(cudaMemcpy2DAsync(L, (size_t)n * 8, h->Kbuf.p, (size_t)NP * 8, (size_t)n * 8, (size_t)n, cudaMemcpyDeviceToHost,
                         h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (long i = 0; i < n; ++i)
        for (long j = i + 1; j < n; ++j) L[i * n + j] = 0.0;
    return GPK_OK;
}

int gpk_get_linv(gpk_handle* h, double* Linv) {
    int rc = require(h, true, true, true);
    if (rc) return rc;
    if (!Linv) BAD("gpk_get_linv: null output");
    CK(cudaSetDevice(h->device));
    if ((rc = build_linv(h))) return rc;
    const long n = h->n, NP = h->NP;
    CK(cudaMemcpy2DAsync(Linv, (size_t)n * 8, h->P.p, (size_t)NP * 8, (size_t)n * 8, (size_t)n, cudaMemcpyDeviceToHost,
                         h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return GPK_OK;
}

int gpk_get_z(gpk_handle* h, double* z) {
    int rc = require(h, true, true, true);
    if (rc) return rc;
    if (!z) BAD("gpk_get_z: null output");
    CK(cudaSetDevice(h->device));
    CK(cudaMemcpyAsync(z, ptr<double>(h->Kbuf) + (long)h->NP * h->NP, (size_t)h->n * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return GPK_OK;
}

int gpk_get_oz_profile(gpk_handle* h, long long* out, int max_ctas, int* n_ctas) {
    if (!h || !out || !n_ctas) return GPK_BAD_ARG;
    CK(cudaSetDevice(h->device));
    const int n = std::min(h->oz_prof_ctas, max_ctas);
    *n_ctas = n;
    if (n > 0) {
        CK(cudaStreamSynchronize(h->stream));
        CK(cudaMemcpy(out, h->oz_profbuf.p, (size_t)n * 64, cudaMemcpyDeviceToHost));
    }
    return GPK_OK;
}

int gpk_get_diag_profile(gpk_handle* h, long long* out34) {      // 64 entries
    if (!h || !out34) return GPK_BAD_ARG;
    if (!h->diag_prof || !h->dprof.p) BAD("gpk_get_diag_profile: set option diagprof = 1 first");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(out34, h->dprof.p, 64 * 8, cudaMemcpyDeviceToHost));
    return GPK_OK;
}

int gpk_get_timings(gpk_handle* h, double* out /* 16 */) {
    if (!h || !out) return GPK_BAD_ARG;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < 16; ++i) out[i] = 0.0;
    float ms = 0.f;
    if (h->fit_timed) {
        if (cudaEventElapsedTime(&ms, h->ev[0], h->ev[3]) == cudaSuccess) out[0] = ms;
        if (cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]) == cudaSuccess) out[1] = ms;
        if (cudaEventElapsedTime(&ms, h->ev[1], h->ev[2]) == cudaSuccess) out[2] = ms;
    }
    if (h->linv_ready && cudaEventElapsedTime(&ms, h->ev[4], h->ev[5]) == cudaSuccess) out[3] = ms;
    if (h->score_timed) {
        if (cudaEventElapsedTime(&ms, h->ev[6], h->ev[7]) == cudaSuccess) out[4] = ms;
        if (cudaEventElapsedTime(&ms, h->ev[8], h->ev[10]) == cudaSuccess) out[5] = ms;    // K* of the last chunk
        // variance GEMM: mean over the FULL-SIZE chunk launches of the last scoring call (the last chunk
        // is included only when it is the only one)
        double sum = 0.0;
        int cnt = 0;
        const int nfull = h->last_nchunks > 1 ? h->last_nchunks - 1 : h->last_nchunks;
        for (int i = 0; i < nfull && i < (int)h->ev_g0.size(); ++i)
            if (cudaEventElapsedTime(&ms, h->ev_g0[i], h->ev_g1[i]) == cudaSuccess) { sum += ms; ++cnt; }
        if (cnt > 0) out[6] = sum / cnt;
        if (cudaEventElapsedTime(&ms, h->ev[11], h->ev[12]) == cudaSuccess) out[7] = ms;   // epilogue, last chunk
    }
    cudaGetLastError();
    out[8] = h->launches_var;
    out[9] = h->launches_total;
    out[10] = h->oz_launches;
    out[11] = (double)h->oz_emax_host;
    out[12] = (double)h->persist;
    out[13] = (double)OZ_PAIRS;
    out[14] = (double)h->oz_last_variant;
    return GPK_OK;
}

}  // extern "C"

#include "gpk_multi.inl"
#include "gpk_es.cuh"
