// gpk_es.cuh — included at the end of gpk_api.cu: entropy search (robo/acquisition_functions/information_gain.py and
// information_gain_per_unit_cost.py) on the device.
//
//   gpk_es_ep_kernel      expectation propagation of robo/util/epmgp.py (min_faktor / lt_factor / log_relative_gauss and
//                         the log Z + derivative formulas), one CTA per representer point k, V resident in shared memory
//   gpk_es_renorm_kernel  the renormalisation of logP and of the three derivative arrays (epmgp.py:54-81)
//   gpk_es_pack_kernel    [A_i ; G_i] folded into one packed-symmetric operand F (2 NB8 x TP) for the quadratic forms
//   gpk_es_gemm_kernel    fp64 DMMA (mma.sync m8n8k4) products: B^T = (L^-1 k(X, zb))^T L^-1 per update, and the
//                         cross-covariance S = k(zb, X*) - B^T k(X, X*)^T per candidate chunk
//   gpk_es_score_kernel   per 32-candidate tile: s = max(S y_std^2, eps), F . vech(s s^T) on DMMA with vech(s s^T)
//                         generated in shared memory, then one warp per candidate for the Np x Nb log-sum-exp
//
// Shapes: Nb representer points (2 <= Nb <= 128), T = Nb (Nb + 1) / 2 lower-triangle entries in row-major order (the
// layout of both dVdx[np.triu(ones).T] at information_gain.py:177 and rot90(., 2)[triu_indices][::-1] at epmgp.py:168).

namespace {

constexpr int ES_MAX_NB = 128;
constexpr int ES_THREADS = 256;
constexpr int ES_TN = 32;                              // candidates per score tile
constexpr int ES_KB = 32;                              // k block of the DMMA products
constexpr double ES_SQ2 = 1.4142135623730951;          // np.sqrt(2)
constexpr double ES_EPS32 = 1.1920928955078125e-07;    // np.finfo(np.float32).eps (epmgp.py:7)
constexpr double ES_L2P = 1.8378770664093453;          // np.log(2) + np.log(np.pi)
constexpr double ES_DBL_MAX = 1.7976931348623157e308;

inline int es_nb8(int nb) { return (nb + 7) / 8 * 8; }
inline int es_tp(int nb) { return (nb * (nb + 1) / 2 + ES_KB - 1) / ES_KB * ES_KB; }

// np.max([a, b]): NaN propagates
__device__ __forceinline__ double es_npmax(double a, double b) {
    if (isnan(a) || isnan(b)) return a + b;
    return a > b ? a : b;
}

__device__ __forceinline__ void es_dmma(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};\n"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// In-place lower Cholesky of the n x n matrix in shared memory (row stride n).  Returns false on a pivot that is not
// > 0 (numpy.linalg.cholesky raises LinAlgError there).
__device__ bool es_chol_smem(double* A, int n, int* flag) {
    if (threadIdx.x == 0) *flag = 0;
    __syncthreads();
    for (int c = 0; c < n; ++c) {
        if (threadIdx.x == 0) {
            const double piv = A[c * n + c];
            if (!(piv > 0.0)) *flag = 1;
            A[c * n + c] = sqrt(piv);
        }
        __syncthreads();
        if (*flag) return false;
        const double dc = A[c * n + c];
        for (int r = c + 1 + threadIdx.x; r < n; r += blockDim.x) A[r * n + c] /= dc;
        __syncthreads();
        const int rem = n - c - 1;
        for (int idx = threadIdx.x; idx < rem * rem; idx += blockDim.x) {
            const int r = c + 1 + idx / rem, q = c + 1 + idx % rem;
            if (q <= r) A[r * n + q] -= A[r * n + c] * A[q * n + c];
        }
        __syncthreads();
    }
    return true;
}

// One CTA per representer point k.  Outputs (un-normalised, epmgp.py:43-52): logZ[k], dMu[k][D], dSig[k][T],
// dMuMu[k][D][D]; sweeps[k] = EP sweeps run (the reference's count + 1); status |= 1 when an update produced a NaN
// variance (epmgp.py:204-207 raises), |= 2 when I + R^T Sigma R is not positive definite even with jitter 1e-6.
// scr: (D-1)^2 doubles per k.  Dynamic shared memory: (D*D + 10*D) doubles.
__global__ void __launch_bounds__(ES_THREADS) gpk_es_ep_kernel(const double* __restrict__ mu, const double* __restrict__ Sig,
                                                               long lds, int D, double* __restrict__ logZ,
                                                               double* __restrict__ dMu, double* __restrict__ dSig,
                                                               double* __restrict__ dMuMu, int* __restrict__ sweeps,
                                                               int* __restrict__ status, double* __restrict__ scr)
{
    extern __shared__ double es_sm[];
    const int k = blockIdx.x, tid = threadIdx.x, D1 = D - 1, T = D * (D + 1) / 2;
    double* V = es_sm;
    double* M = V + D * D;
    double* Vc = M + D;
    double* P = Vc + D;
    double* MP = P + D;
    double* LS = MP + D;
    double* sc = LS + D;          // 4 scalars of the current factor update
    double* v1 = sc + D;          // work vectors
    double* v2 = v1 + D;
    double* v3 = v2 + D;
    __shared__ int s_bad, s_flag;
    __shared__ double s_red[8];
    for (int i = tid; i < D * D; i += blockDim.x) V[i] = Sig[(long)(i / D) * lds + i % D];
    for (int i = tid; i < D; i += blockDim.x) { M[i] = mu[i]; P[i] = 0.0; MP[i] = 0.0; LS[i] = 0.0; }
    if (tid == 0) s_bad = 0;
    __syncthreads();

    // ---- EP sweeps (min_faktor, epmgp.py:96-114) ------------------------------------------------------------
    bool nan_exit = false;
    int count = 0;
    for (; count < 50; ++count) {
        double diff = 0.0, d = 0.0;
        for (int i = 0; i < D1; ++i) {
            const int l = i < k ? i : i + 1;
            for (int t = tid; t < D; t += blockDim.x) Vc[t] = (V[t * D + l] - V[t * D + k]) / ES_SQ2;
            if (tid == 0) {
                // lt_factor (epmgp.py:172-233), s = k
                const double p = P[i], mp = MP[i];
                const double cVc = (V[l * D + l] - 2.0 * V[k * D + l] + V[k * D + k]) / 2.0;
                const double cM = (M[l] - M[k]) / ES_SQ2;
                const double cVnic = es_npmax(cVc / (1.0 - p * cVc), 0.0);
                const double cmni = cM + cVnic * (p * cM - mp);
                double z = cmni / sqrt(cVnic + 1e-25);
                if (isnan(z)) z = -INFINITY;
                double dd, tV = 0.0, tM = 0.0, upd = 0.0;
                if (z < -6.0) {                                  // log_relative_gauss exit -1
                    dd = NAN;
                } else if (z > 6.0) {                            // exit 1: remove the message
                    const double dp = -p, dmp = -mp;
                    dd = dmp > dp ? dmp : dp;                    // builtin max([dmp, dp])
                    tV = dp / (1.0 + dp * cVc);
                    tM = (dmp - cM * dp) / (1.0 + dp * cVc);
                    P[i] = 0.0; MP[i] = 0.0; LS[i] = 0.0;
                    upd = 1.0;
                } else {
                    const double logphi = -0.5 * (z * z + ES_L2P);
                    const double logPhi = log(0.5 * erfc(-z / ES_SQ2));
                    const double e = exp(logphi - logPhi);
                    const double alpha = e / sqrt(cVnic);
                    const double beta = alpha * (alpha * cVnic + cmni);
                    const double r = beta / (1.0 - beta);
                    double pnew = r / cVnic;
                    double mpnew = r * (alpha + cmni / cVnic) + alpha;
                    const double dp = es_npmax(-p + ES_EPS32, pnew - p);
                    const double dmp = es_npmax(-mp + ES_EPS32, mpnew - mp);
                    dd = es_npmax(dmp, dp);
                    pnew = p + dp;
                    mpnew = mp + dmp;
                    tV = dp / (1.0 + dp * cVc);
                    tM = (dmp - cM * dp) / (1.0 + dp * cVc);
                    LS[i] = logPhi - 0.5 * (log(beta) - log(pnew) - log(cVnic)) + (alpha * alpha) / (2.0 * beta) * cVnic;
                    P[i] = pnew; MP[i] = mpnew;
                    upd = 1.0;
                }
                sc[0] = tV; sc[1] = tM; sc[2] = upd; sc[3] = dd;
            }
            __syncthreads();
            const double tV = sc[0], tM = sc[1];
            d = sc[3];
            if (sc[2] != 0.0) {
                // V - t * outer(Vc, Vc) and M + u * Vc, rounded like numpy (no fused multiply-add)
                for (int idx = tid; idx < D * D; idx += blockDim.x) {
                    const double nv = __dsub_rn(V[idx], __dmul_rn(tV, __dmul_rn(Vc[idx / D], Vc[idx % D])));
                    if (isnan(nv)) s_bad = 1;
                    V[idx] = nv;
                }
                for (int t = tid; t < D; t += blockDim.x) M[t] = __dadd_rn(M[t], __dmul_rn(tM, Vc[t]));
            }
            __syncthreads();
            if (isnan(d)) break;
            diff += fabs(d);
        }
        if (isnan(d)) { nan_exit = true; break; }
        if (fabs(diff) < 0.001) break;
    }
    if (tid == 0) {
        sweeps[k] = count < 50 ? count + 1 : 50;
        if (s_bad) atomicOr(status, 1);
    }
    const long T64 = T;
    if (nan_exit) {                                      // epmgp.py:115-126
        if (tid == 0) logZ[k] = -INFINITY;
        for (int i = tid; i < D; i += blockDim.x) dMu[(long)k * D + i] = 0.0;
        for (long i = tid; i < T64; i += blockDim.x) dSig[(long)k * T64 + i] = 0.0;
        for (long i = tid; i < (long)D * D; i += blockDim.x) dMuMu[(long)k * D * D + i] = 0.0;
        return;
    }

    // ---- log Z and its derivatives (epmgp.py:128-169) --------------------------------------------------------
    // R = sqrt(P) * C: column j has rho_j = sqrt(P_j) / sqrt(2) in row l_j and -rho_j in row k
    double* rho = Vc;
    for (int j = tid; j < D1; j += blockDim.x) rho[j] = sqrt(P[j]) * (1.0 / ES_SQ2);
    __syncthreads();
    double* C = V;                                       // I + R^T Sigma R, (D-1) x (D-1), then its Cholesky factor
    const double skk = Sig[(long)k * lds + k];
    double jitter = 0.0;
    bool ok = false;
    for (int attempt = 0; attempt < 3 && !ok; ++attempt) {
        for (int idx = tid; idx < D1 * D1; idx += blockDim.x) {
            const int i = idx / D1, j = idx % D1;
            const int li = i < k ? i : i + 1, lj = j < k ? j : j + 1;
            const double q = Sig[(long)li * lds + lj] - Sig[(long)li * lds + k] - Sig[(long)k * lds + lj] + skk;
            C[idx] = (i == j ? 1.0 : 0.0) + rho[i] * rho[j] * q + (i == j ? jitter : 0.0);
        }
        __syncthreads();
        ok = es_chol_smem(C, D1, &s_flag);
        jitter = attempt == 0 ? 1e-10 : 1e-6;            // numpy retries with + 1e-10 I, then + 1e-6 I
    }
    if (!ok) {
        if (tid == 0) { atomicOr(status, 2); logZ[k] = NAN; }
        return;
    }
    // G = (I + R^T Sigma R)^-1, one column per thread (forward then backward substitution), column-major in scr
    double* G = scr + (long)k * D1 * D1;
    for (int j = tid; j < D1; j += blockDim.x) {
        double* g = G + (long)j * D1;
        for (int i = 0; i < j; ++i) g[i] = 0.0;
        for (int i = j; i < D1; ++i) {
            double acc = (i == j) ? 1.0 : 0.0;
            for (int q = j; q < i; ++q) acc -= C[i * D1 + q] * g[q];
            g[i] = acc / C[i * D1 + i];
        }
        for (int i = D1 - 1; i >= 0; --i) {
            double acc = g[i];
            for (int q = i + 1; q < D1; ++q) acc -= C[q * D1 + i] * g[q];
            g[i] = acc / C[i * D1 + i];
        }
    }
    if (tid == 0) {                                       // dts = 2 sum log diag(chol)
        double s = 0.0;
        for (int i = 0; i < D1; ++i) s += log(C[i * D1 + i]);
        s_red[0] = 2.0 * s;
    }
    __syncthreads();
    // gr_i = sum_j G_ij rho_j, rg_j = sum_i rho_i G_ij (G[i][j] = G[j * D1 + i])
    for (int i = tid; i < D1; i += blockDim.x) {
        double a = 0.0, b = 0.0;
        for (int j = 0; j < D1; ++j) { a += G[(long)j * D1 + i] * rho[j]; b += rho[j] * G[(long)i * D1 + j]; }
        v1[i] = a; v2[i] = b;
    }
    __syncthreads();
    if (tid == 0) {
        double s = 0.0;
        for (int i = 0; i < D1; ++i) s += rho[i] * v1[i];
        s_red[1] = s;
    }
    __syncthreads();
    // A = R G R^T, symmetrised (epmgp.py:142-144), into shared memory (the factor is no longer needed)
    double* A = V;
    const double grr = s_red[1];
    for (int idx = tid; idx < D * D; idx += blockDim.x) {
        const int a = idx / D, b = idx % D;
        const int ia = a < k ? a : a - 1, ib = b < k ? b : b - 1;
        double ab, ba;
        if (a != k && b != k) {
            ab = rho[ia] * G[(long)ib * D1 + ia] * rho[ib];
            ba = rho[ib] * G[(long)ia * D1 + ib] * rho[ia];
        } else if (a != k) {
            ab = -rho[ia] * v1[ia];
            ba = -rho[ia] * v2[ia];
        } else if (b != k) {
            ab = -rho[ib] * v2[ib];
            ba = -rho[ib] * v1[ib];
        } else {
            ab = ba = grr;
        }
        A[idx] = 0.5 * (ba + ab);
    }
    __syncthreads();
    // r = C MP, b = Mu + Sigma r, Ab = A b
    double* r = v1;
    double* bb = v2;
    double* Ab = v3;
    if (tid == 0) {
        double rk = 0.0;
        for (int j = 0; j < D1; ++j) rk += MP[j] * (-1.0 / ES_SQ2);
        r[k] = rk;
    }
    for (int j = tid; j < D1; j += blockDim.x) r[j < k ? j : j + 1] = MP[j] * (1.0 / ES_SQ2);
    __syncthreads();
    for (int a = tid; a < D; a += blockDim.x) {
        double s = 0.0;
        for (int b = 0; b < D; ++b) s += Sig[(long)a * lds + b] * r[b];
        bb[a] = mu[a] + s;
        Vc[a] = s;                                        // Sigma r (rho is no longer needed)
    }
    __syncthreads();
    for (int a = tid; a < D; a += blockDim.x) {
        double s = 0.0;
        for (int b = 0; b < D; ++b) s += A[a * D + b] * bb[b];
        Ab[a] = s;
    }
    __syncthreads();
    if (tid == 0) {
        double mpm = 0.0, sls = 0.0, rSr = 0.0, bAb = 0.0, Mur = 0.0;
        for (int j = 0; j < D1; ++j) {
            if (MP[j] != 0.0) mpm += MP[j] * MP[j] / P[j];
            sls += LS[j];
        }
        for (int a = 0; a < D; ++a) { rSr += Vc[a] * r[a]; bAb += bb[a] * Ab[a]; Mur += mu[a] * r[a]; }
        logZ[k] = 0.5 * (rSr - bAb - s_red[0]) + Mur + sls - 0.5 * mpm;
    }
    for (int a = tid; a < D; a += blockDim.x) dMu[(long)k * D + a] = r[a] - Ab[a];
    for (long idx = tid; idx < (long)D * D; idx += blockDim.x) dMuMu[(long)k * D * D + idx] = -A[idx];
    // dlogZdSigma = sym(-A - 2 r Ab^T + r r^T + Ab Ab^T) with the diagonal halved, lower triangle row-major
    for (long t = tid; t < T64; t += blockDim.x) {
        int a = (int)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
        while ((long)a * (a + 1) / 2 > t) --a;
        while ((long)(a + 1) * (a + 2) / 2 <= t) ++a;
        const int b = (int)(t - (long)a * (a + 1) / 2);
        const double eab = -A[a * D + b] - 2.0 * (r[a] * Ab[b]) + r[a] * r[b] + Ab[a] * Ab[b];
        const double eba = -A[b * D + a] - 2.0 * (r[b] * Ab[a]) + r[b] * r[a] + Ab[b] * Ab[a];
        dSig[(long)k * T64 + t] = a == b ? 0.5 * (eab + eba - eab) : 0.5 * (eab + eba);
    }
}

// Renormalisation (epmgp.py:54-81): logP[isinf] = -500, logP -= logsumexp, and the derivative corrections
// Zm, Zs, gg.  adds[i][j] = -gg[i][j] + Zm[j]^2 (Zm.T * Zm of a 1-D array is element-wise).
__global__ void gpk_es_renorm_kernel(int D, const double* __restrict__ rlogZ, const double* __restrict__ rdMu,
                                     const double* __restrict__ rdSig, const double* __restrict__ rdMuMu,
                                     double* __restrict__ logP, double* __restrict__ dMu, double* __restrict__ dSig,
                                     double* __restrict__ dMuMu)
{
    const long T = (long)D * (D + 1) / 2;
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    const long DD = (long)D * D;
    if (idx > DD + T) return;
    double Z = 0.0, mx = -INFINITY;
    for (int k = 0; k < D; ++k) {
        const double lp = isinf(rlogZ[k]) ? -500.0 : rlogZ[k];
        Z += exp(lp);
        mx = es_npmax(mx, lp);
    }
    if (idx == DD + T) {
        double se = 0.0;
        for (int k = 0; k < D; ++k) se += exp((isinf(rlogZ[k]) ? -500.0 : rlogZ[k]) - mx);
        double s = mx + log(se);
        if (isinf(s)) s = mx;
        for (int k = 0; k < D; ++k) logP[k] = (isinf(rlogZ[k]) ? -500.0 : rlogZ[k]) - s;
        return;
    }
    if (idx < DD) {
        const int i = (int)(idx / D), j = (int)(idx % D);
        double zm = 0.0, gg = 0.0;
        for (int k = 0; k < D; ++k) {
            const double e = exp(isinf(rlogZ[k]) ? -500.0 : rlogZ[k]);
            zm += e * rdMu[(long)k * D + j];
            gg += (rdMuMu[(long)k * DD + idx] + rdMu[(long)k * D + i] * rdMu[(long)k * D + j]) * e;
        }
        zm /= Z;
        gg /= Z;
        const double add = -gg + zm * zm;
        for (int k = 0; k < D; ++k) dMuMu[(long)k * DD + idx] = rdMuMu[(long)k * DD + idx] + add;
        if (i == 0)
            for (int k = 0; k < D; ++k) dMu[(long)k * D + j] = rdMu[(long)k * D + j] - zm;
        return;
    }
    const long t = idx - DD;
    double zs = 0.0;
    for (int k = 0; k < D; ++k) zs += exp(isinf(rlogZ[k]) ? -500.0 : rlogZ[k]) * rdSig[(long)k * T + t];
    zs /= Z;
    for (int k = 0; k < D; ++k) dSig[(long)k * T + t] = rdSig[(long)k * T + t] - zs;
}

// F (2 NB8 x TP, row-major): row i < nb: s^T dMuMu[i] s as a packed form (diagonal, and A_jl + A_lj below it);
// row NB8 + i: dlogPdSigma[i] as stored (s^T G_i s with the off-diagonal halved = dSig[i] . vech(s s^T)).
__global__ void gpk_es_pack_kernel(int nb, const double* __restrict__ dSig, const double* __restrict__ dMuMu,
                                   const int2* __restrict__ jl, double* __restrict__ F)
{
    const int nb8 = (nb + 7) / 8 * 8, TP = (nb * (nb + 1) / 2 + ES_KB - 1) / ES_KB * ES_KB, T = nb * (nb + 1) / 2;
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= 2L * nb8 * TP) return;
    const int row = (int)(idx / TP), t = (int)(idx % TP);
    const int i = row % nb8;
    double v = 0.0;
    if (t < T && i < nb) {
        if (row < nb8) {
            const int2 p = jl[t];
            const double* Ai = dMuMu + (long)i * nb * nb;
            v = p.x == p.y ? Ai[p.x * nb + p.x] : Ai[p.x * nb + p.y] + Ai[p.y * nb + p.x];
        } else {
            v = dSig[(long)i * T + t];
        }
    }
    F[idx] = v;
}

// The Np quantiles of the hallucinated values: W = norm.ppf(linspace(1/(Np+1), 1 - 1/(Np+1), Np))
__global__ void gpk_es_grid_kernel(int np_grid, double* __restrict__ W) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= np_grid) return;
    const double start = 1.0 / (np_grid + 1), stop = 1.0 - 1.0 / (np_grid + 1);
    double q = start;
    if (np_grid > 1) {
        const double step = (stop - start) / (double)(np_grid - 1);
        q = p == np_grid - 1 ? stop : __dadd_rn(__dmul_rn((double)p, step), start);
    }
    W[p] = normcdfinv(q);
}

// C (M x N) = A (M x K) . op(B), op(B)[k][j] = BT ? B[j][k] : B[k][j]; with E: C[i][j] = E[j][i] - (A op(B))[i][j].
// 32 x 64 tile per CTA, 8 warps of 8 x 32, DMMA m8n8k4 from shared memory.
template <bool BT>
__global__ void __launch_bounds__(256) gpk_es_gemm_kernel(int Mr, long N, int K, const double* __restrict__ A, long lda,
                                                          const double* __restrict__ B, long ldb, double* __restrict__ Cm,
                                                          long ldc, const double* __restrict__ E, long lde)
{
    __shared__ double As[32][ES_KB + 1];
    __shared__ double Bs[64][ES_KB + 1];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t4 = lane & 3;
    const int i0 = blockIdx.y * 32;
    const long j0 = (long)blockIdx.x * 64;
    const int mt = warp & 3, nt0 = (warp >> 2) * 4;
    double acc[4][2];
#pragma unroll
    for (int q = 0; q < 4; ++q) acc[q][0] = acc[q][1] = 0.0;
    for (int k0 = 0; k0 < K; k0 += ES_KB) {
        for (int idx = threadIdx.x; idx < 32 * ES_KB; idx += 256) {
            const int r = idx / ES_KB, q = idx % ES_KB;
            As[r][q] = (i0 + r < Mr && k0 + q < K) ? A[(long)(i0 + r) * lda + k0 + q] : 0.0;
        }
        for (int idx = threadIdx.x; idx < 64 * ES_KB; idx += 256) {
            int n, q;
            if (BT) { n = idx / ES_KB; q = idx % ES_KB; } else { q = idx / 64; n = idx % 64; }
            const long j = j0 + n;
            Bs[n][q] = (j < N && k0 + q < K) ? (BT ? B[j * ldb + k0 + q] : B[(long)(k0 + q) * ldb + j]) : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int ks = 0; ks < ES_KB; ks += 4) {
            const double a = As[mt * 8 + g][ks + t4];
#pragma unroll
            for (int q = 0; q < 4; ++q) es_dmma(acc[q][0], acc[q][1], a, Bs[(nt0 + q) * 8 + g][ks + t4]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int i = i0 + mt * 8 + g;
            const long j = j0 + (nt0 + q) * 8 + 2 * t4 + e;
            if (i < Mr && j < N) Cm[(long)i * ldc + j] = E ? E[j * lde + i] - acc[q][e] : acc[q][e];
        }
}

struct EsScoreArgs {
    const double* S; long lds;            // cross-covariance chunk, nb rows (normalised units, unclipped)
    const double* var;                    // predictive variance of the chunk (un-normalised, clipped)
    const double* cand; int d;            // raw candidate inputs (bounds rule)
    const double* lo; const double* up;   // acquisition bounds, NULL: no rule
    long mc;
    int nb, nb8, T, TP;
    int norm_out; double ystd2; double sn2;
    const double* F; const int2* jl;
    const double* U; const double* logP; const double* lmb; const double* W; int np_grid; double H;
    double* out;                          // chunk values (NULL: none)
    BestPair* bb; long base;              // per-CTA arg-max; base = global index of the chunk's first candidate
};

inline size_t es_score_smem(int nb) {
    const int nb8 = es_nb8(nb);
    return (size_t)(nb8 * ES_TN + ES_KB * ES_TN + 2 * nb8 * ES_TN + 2 * 8 * nb8 + nb8 + ES_TN) * 8;
}

__global__ void __launch_bounds__(256) gpk_es_score_kernel(EsScoreArgs a) {
    extern __shared__ double es_sm[];
    const int nb = a.nb, nb8 = a.nb8;
    double* sS = es_sm;                          // [nb8][ES_TN]
    double* sB = sS + nb8 * ES_TN;               // [ES_KB][ES_TN]
    double* sQ = sB + ES_KB * ES_TN;             // [2 nb8][ES_TN]
    double* sab = sQ + 2 * nb8 * ES_TN;          // per warp: a[nb8], b[nb8]
    double* slmb = sab + 2 * 8 * nb8;
    double* sval = slmb + nb8;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t4 = lane & 3;
    const long c0 = (long)blockIdx.x * ES_TN;
    const int nc = (int)min((long)ES_TN, a.mc - c0);
    for (int idx = threadIdx.x; idx < nb8 * ES_TN; idx += blockDim.x) {
        const int j = idx / ES_TN, c = idx % ES_TN;
        double x = 0.0;
        if (j < nb && c < nc) {
            x = a.S[(long)j * a.lds + c0 + c];
            if (a.norm_out) x *= a.ystd2;
            if (x < GPK_EPS) x = GPK_EPS;        // predict(full_cov=True) clips every entry (gaussian_process.py:290-294)
        }
        sS[idx] = x;
    }
    for (int i = threadIdx.x; i < nb8; i += blockDim.x) slmb[i] = i < nb ? a.lmb[i] : 0.0;
    __syncthreads();

    // Q = F . vech(s s^T): warp w owns m-tiles w, w + 8, ... (2 nb8 / 8 <= 32 of them) and all 4 n-tiles
    const int MT = 2 * nb8 / 8;
    double acc[4][4][2];
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int n = 0; n < 4; ++n) acc[q][n][0] = acc[q][n][1] = 0.0;
    for (int k0 = 0; k0 < a.TP; k0 += ES_KB) {
        for (int idx = threadIdx.x; idx < ES_KB * ES_TN; idx += blockDim.x) {
            const int q = idx / ES_TN, c = idx % ES_TN;
            const int t = k0 + q;
            double v = 0.0;
            if (t < a.T) {
                const int2 p = a.jl[t];
                v = sS[p.x * ES_TN + c] * sS[p.y * ES_TN + c];
            }
            sB[idx] = v;
        }
        __syncthreads();
#pragma unroll
        for (int ks = 0; ks < ES_KB; ks += 4) {
            double bf[4];
#pragma unroll
            for (int n = 0; n < 4; ++n) bf[n] = sB[(ks + t4) * ES_TN + n * 8 + g];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int mt = warp + 8 * q;
                if (mt < MT) {
                    const double af = __ldg(a.F + (long)(mt * 8 + g) * a.TP + k0 + ks + t4);
#pragma unroll
                    for (int n = 0; n < 4; ++n) es_dmma(acc[q][n][0], acc[q][n][1], af, bf[n]);
                }
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int mt = warp + 8 * q;
        if (mt < MT)
#pragma unroll
            for (int n = 0; n < 4; ++n) {
                sQ[(mt * 8 + g) * ES_TN + n * 8 + 2 * t4] = acc[q][n][0];
                sQ[(mt * 8 + g) * ES_TN + n * 8 + 2 * t4 + 1] = acc[q][n][1];
            }
    }
    __syncthreads();

    // one warp per candidate: a_i, b_i, then the Np x Nb log-sum-exp with one exp per (i, p)
    double* wa = sab + warp * 2 * nb8;
    double* wb = wa + nb8;
    for (int c = warp; c < nc; c += 8) {
        const double v = a.var[c0 + c];
        const double v_ = v - a.sn2;                    // sn2 in normalised units, v un-normalised (reference quirk)
        const double inv = 1.0 / v_;
        const double sq = sqrt(v + 1e-10);
        const double cs = inv * sq;
        for (int i = lane; i < nb; i += 32) {
            double us = 0.0;
            const double* Ui = a.U + (long)i * nb;
            for (int j = 0; j < nb; ++j) us += Ui[j] * sS[j * ES_TN + c];
            const double qA = sQ[i * ES_TN + c], qG = sQ[(nb8 + i) * ES_TN + c];
            wa[i] = a.logP[i] + (-inv * qG + 0.5 * (cs * cs) * qA);
            wb[i] = cs * us;
        }
        __syncwarp();
        double accA = 0.0, accB = 0.0;
        bool anyinf = false;
        for (int p = lane; p < a.np_grid; p += 32) {
            const double w = a.W[p];
            double mx = -INFINITY;
            for (int i = 0; i < nb; ++i) {
                const double x = wa[i] + wb[i] * w;
                if (x > mx || isnan(x)) mx = isnan(mx) ? mx : x;
            }
            double Z = 0.0, T1 = 0.0;
            for (int i = 0; i < nb; ++i) {
                const double x = wa[i] + wb[i] * w;
                const double e = exp(x - mx);
                Z += e;
                T1 += e * (x + slmb[i]);
            }
            const double s = mx + log(Z);
            anyinf |= isinf(s);
            accA += T1 / Z - s;                         // sum_i exp(x_i - s) (x_i - s + lmb_i)
            accB += T1 - mx * Z;                        // the same with s = max (lselP when any column's s is inf)
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            accA += __shfl_xor_sync(0xffffffffu, accA, off);
            accB += __shfl_xor_sync(0xffffffffu, accB, off);
        }
        anyinf = __any_sync(0xffffffffu, anyinf);
        if (lane == 0) {
            double dH = (anyinf ? accB : accA) / (double)a.np_grid + a.H;
            if (isnan(dH) || dH == INFINITY) dH = -ES_DBL_MAX;      // information_gain.py:119-120
            if (a.lo) {
                const double* x = a.cand + (c0 + c) * a.d;
                for (int q = 0; q < a.d; ++q)
                    if (x[q] < a.lo[q] || x[q] > a.up[q]) { dH = GPK_EPS; break; }   // np.spacing(1), :219-222
            }
            sval[c] = dH;
            if (a.out) a.out[c0 + c] = dH;
        }
        __syncwarp();
    }
    __syncthreads();
    if (warp == 0) {
        double val = 0.0;
        long long idx = -1;
        for (int c = lane; c < nc; c += 32)
            if (gpk_better(sval[c], a.base + c0 + c, val, idx)) { val = sval[c]; idx = a.base + c0 + c; }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, val, off);
            const long long oi = __shfl_xor_sync(0xffffffffu, idx, off);
            if (gpk_better(ov, oi, val, idx)) { val = ov; idx = oi; }
        }
        if (lane == 0) { a.bb[blockIdx.x].val = val; a.bb[blockIdx.x].idx = idx; }
    }
}

inline long es_T(int nb) { return (long)nb * (nb + 1) / 2; }

// EP on moments already on the device (mu: nb, V: nb x nb with row stride ldv): writes es_logP / es_dmu / es_dsig /
// es_dmumu / es_sweeps (+ status word at es_sweeps[nb]); asynchronous on the handle's stream.
int es_run_ep(gpk_handle* h, const double* d_mu, const double* d_V, long ldv, int nb) {
    const long T = es_T(nb), D = nb;
    int rc;
    if ((rc = ensure(h, h->es_raw, (size_t)(D + D * D + D * T + D * D * D) * 8))) return rc;
    if ((rc = ensure(h, h->es_scr, (size_t)D * (D - 1) * (D - 1) * 8))) return rc;
    if ((rc = ensure(h, h->es_logP, (size_t)D * 8))) return rc;
    if ((rc = ensure(h, h->es_dmu, (size_t)D * D * 8))) return rc;
    if ((rc = ensure(h, h->es_dsig, (size_t)D * T * 8))) return rc;
    if ((rc = ensure(h, h->es_dmumu, (size_t)D * D * D * 8))) return rc;
    if ((rc = ensure(h, h->es_sweeps, (size_t)(D + 1) * 4))) return rc;
    double* raw = ptr<double>(h->es_raw);
    double* rlogZ = raw;
    double* rdMu = rlogZ + D;
    double* rdSig = rdMu + D * D;
    double* rdMuMu = rdSig + D * T;
    int* sweeps = ptr<int>(h->es_sweeps);
    CK(cudaMemsetAsync(sweeps + D, 0, 4, h->stream));
    const size_t smem = (size_t)(D * D + 10 * D) * 8;
    CK(cudaFuncSetAttribute(gpk_es_ep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    gpk_es_ep_kernel<<<nb, ES_THREADS, smem, h->stream>>>(d_mu, d_V, ldv, nb, rlogZ, rdMu, rdSig, rdMuMu, sweeps,
                                                          sweeps + D, ptr<double>(h->es_scr));
    CKL();
    const long items = D * D + T + 1;
    gpk_es_renorm_kernel<<<(unsigned)((items + 255) / 256), 256, 0, h->stream>>>(
        nb, rlogZ, rdMu, rdSig, rdMuMu, ptr<double>(h->es_logP), ptr<double>(h->es_dmu), ptr<double>(h->es_dsig),
        ptr<double>(h->es_dmumu));
    CKL();
    return GPK_OK;
}

// status word of the last es_run_ep (after a synchronise)
int es_check_status(gpk_handle* h, int nb) {
    int st = 0;
    CK(cudaMemcpy(&st, ptr<int>(h->es_sweeps) + nb, 4, cudaMemcpyDeviceToHost));
    if (st & 2) { set_err(h, "entropy search: I + R^T Sigma R is not positive definite (epmgp.py:147-153)"); return GPK_NOT_PD; }
    if (st & 1) { set_err(h, "entropy search: expectation propagation produced a NaN variance (epmgp.py:204-207)"); return GPK_BAD_ARG; }
    return GPK_OK;
}

template <bool BT>
int es_gemm(gpk_handle* h, int Mr, long N, int K, const double* A, long lda, const double* B, long ldb, double* C, long ldc,
            const double* E, long lde) {
    dim3 grid((unsigned)((N + 63) / 64), (unsigned)((Mr + 31) / 32));
    gpk_es_gemm_kernel<BT><<<grid, 256, 0, h->stream>>>(Mr, N, K, A, lda, B, ldb, C, ldc, E, lde);
    CKL();
    return GPK_OK;
}

}  // namespace

extern "C" int gpk_es_joint_min(gpk_handle* h, const double* mu, const double* V, int nb, double* logP, double* dlogPdMu,
                                double* dlogPdSigma, double* dlogPdMudMu, int* sweeps) {
    if (!h) return GPK_BAD_ARG;
    if (!mu || !V) BAD("gpk_es_joint_min: need mu and V");
    if (nb < 2 || nb > ES_MAX_NB) BAD("gpk_es_joint_min: nb = %d outside 2..%d", nb, ES_MAX_NB);
    CK(cudaSetDevice(h->device));
    h->es_ready = false;                       // the EP buffers of the handle's entropy-search state are reused
    int rc;
    if ((rc = ensure(h, h->es_KZ, (size_t)(nb + nb * nb) * 8))) return rc;
    double* d = ptr<double>(h->es_KZ);
    CK(cudaMemcpyAsync(d, mu, (size_t)nb * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(d + nb, V, (size_t)nb * nb * 8, cudaMemcpyHostToDevice, h->stream));
    if ((rc = es_run_ep(h, d, d + nb, nb, nb))) return rc;
    h->es_nb = nb;
    CK(cudaStreamSynchronize(h->stream));
    if ((rc = es_check_status(h, nb))) return rc;
    return gpk_es_get_state(h, logP, dlogPdMu, dlogPdSigma, dlogPdMudMu, sweeps);
}

extern "C" int gpk_es_get_state(gpk_handle* h, double* logP, double* dlogPdMu, double* dlogPdSigma, double* dlogPdMudMu,
                                int* sweeps) {
    if (!h) return GPK_BAD_ARG;
    const int nb = h->es_nb;
    if (nb < 2) BAD("gpk_es_get_state: no entropy-search state (gpk_es_update)");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    if (logP) CK(cudaMemcpy(logP, h->es_logP.p, (size_t)nb * 8, cudaMemcpyDeviceToHost));
    if (dlogPdMu) CK(cudaMemcpy(dlogPdMu, h->es_dmu.p, (size_t)nb * nb * 8, cudaMemcpyDeviceToHost));
    if (dlogPdSigma) CK(cudaMemcpy(dlogPdSigma, h->es_dsig.p, (size_t)nb * es_T(nb) * 8, cudaMemcpyDeviceToHost));
    if (dlogPdMudMu) CK(cudaMemcpy(dlogPdMudMu, h->es_dmumu.p, (size_t)nb * nb * nb * 8, cudaMemcpyDeviceToHost));
    if (sweeps) CK(cudaMemcpy(sweeps, h->es_sweeps.p, (size_t)nb * 4, cudaMemcpyDeviceToHost));
    return GPK_OK;
}

extern "C" int gpk_es_update(gpk_handle* h, const double* zb, int nb, const double* lmb, int np_grid, double sn2,
                             double* logP_out) {
    int rc = require(h, true, true, true);
    if (rc) return rc;
    if (!zb || !lmb) BAD("gpk_es_update: need zb and lmb");
    if (nb < 2 || nb > ES_MAX_NB) BAD("gpk_es_update: nb = %d outside 2..%d", nb, ES_MAX_NB);
    if (np_grid < 1) BAD("gpk_es_update: np_grid = %d < 1", np_grid);
    for (int i = 0; i < nb; ++i)
        if (!std::isfinite(lmb[i])) BAD("gpk_es_update: lmb should not be infinite (information_gain.py:207-211)");
    CK(cudaSetDevice(h->device));
    h->es_ready = false;
    const int d = h->d, nb8 = es_nb8(nb), TP = es_tp(nb);
    const long NP = h->NP, T = es_T(nb);
    // Mb, Vb = predict(zb, full_cov=True), clipped at eps: leaves mu in out_mu, the covariance in cov (row stride 128)
    // and (L^-1 k(X, zb))^T in Vt, all on the device
    std::vector<double> hmu(nb), hcov((size_t)nb * nb);
    if ((rc = predict_cov_impl(h, zb, nb, hmu.data(), hcov.data(), 1))) return rc;
    const long mp = round_up(nb, BM);
    if ((rc = es_run_ep(h, ptr<double>(h->out_mu), ptr<double>(h->cov), mp, nb))) return rc;
    h->es_nb = nb;
    // packed quadratic-form operand
    std::vector<int2> jl(TP, make_int2(0, 0));
    for (int j = 0, t = 0; j < nb; ++j)
        for (int l = 0; l <= j; ++l, ++t) jl[t] = make_int2(j, l);
    if ((rc = ensure(h, h->es_jl, (size_t)TP * sizeof(int2)))) return rc;
    CK(cudaMemcpyAsync(h->es_jl.p, jl.data(), (size_t)TP * sizeof(int2), cudaMemcpyHostToDevice, h->stream));
    if ((rc = ensure(h, h->es_F, (size_t)2 * nb8 * TP * 8))) return rc;
    gpk_es_pack_kernel<<<(unsigned)((2L * nb8 * TP + 255) / 256), 256, 0, h->stream>>>(
        nb, ptr<double>(h->es_dsig), ptr<double>(h->es_dmumu), ptr<int2>(h->es_jl), ptr<double>(h->es_F));
    CKL();
    // B^T = (K^-1 k(X, zb))^T = Vt L^-1 (nb x NP); rows nb..nb8 stay zero
    if ((rc = ensure(h, h->es_Bt, (size_t)nb8 * NP * 8))) return rc;
    CK(cudaMemsetAsync(h->es_Bt.p, 0, (size_t)nb8 * NP * 8, h->stream));
    if ((rc = es_gemm<false>(h, nb, NP, (int)NP, ptr<double>(h->Vt), NP, ptr<double>(h->P), NP, ptr<double>(h->es_Bt), NP,
                             nullptr, 0)))
        return rc;
    // operand of the k(X*, zb) builder
    if ((rc = ensure(h, h->es_zb, (size_t)nb * d * 8))) return rc;
    CK(cudaMemcpyAsync(h->es_zb.p, zb, (size_t)nb * d * 8, cudaMemcpyHostToDevice, h->stream));
    if ((rc = ensure(h, h->es_zbop, cov_operand_rows(h, d) * BM * 8))) return rc;
    const double* lo = h->has_bounds ? ptr<double>(h->lower) : nullptr;
    const double* up = h->has_bounds ? ptr<double>(h->upper) : nullptr;
    if ((rc = build_cov_operand(h, h->stream, ptr<double>(h->es_zb), nb, d, lo, up, ptr<double>(h->es_zbop), BM))) return rc;
    if ((rc = ensure(h, h->es_W, (size_t)np_grid * 8))) return rc;
    gpk_es_grid_kernel<<<(unsigned)((np_grid + 255) / 256), 256, 0, h->stream>>>(np_grid, ptr<double>(h->es_W));
    CKL();
    if ((rc = ensure(h, h->es_lmb, (size_t)nb * 8))) return rc;
    CK(cudaMemcpyAsync(h->es_lmb.p, lmb, (size_t)nb * 8, cudaMemcpyHostToDevice, h->stream));
    std::vector<double> lp(nb);
    CK(cudaMemcpyAsync(lp.data(), h->es_logP.p, (size_t)nb * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if ((rc = es_check_status(h, nb))) return rc;
    // H = -sum exp(logP) (logP + lmb), the current entropy (information_gain.py:82)
    double H = 0.0;
    for (int i = 0; i < nb; ++i) H += std::exp(lp[i]) * (lp[i] + lmb[i]);
    h->es_H = -H;
    h->es_np = np_grid;
    h->es_sn2 = sn2;
    h->es_linv_serial = h->linv_serial;
    h->es_ready = true;
    if (logP_out) memcpy(logP_out, lp.data(), (size_t)nb * 8);
    return GPK_OK;
}

extern "C" int gpk_es_compute(gpk_handle* h, const double* Xs, long m, const double* lower, const double* upper, double* out,
                              double* best_val, long* best_idx) {
    int rc = require(h, true, true, true);
    if (rc) return rc;
    if (!h->es_ready) BAD("gpk_es_compute: no entropy-search state; call gpk_es_update first");
    if (!Xs || m <= 0) BAD("gpk_es_compute: need Xs and m >= 1");
    if (!h->linv_ready || h->linv_serial != h->es_linv_serial) {
        set_err(h, "gpk_es_compute: the model was refitted after gpk_es_update");
        return GPK_NOT_FITTED;
    }
    CK(cudaSetDevice(h->device));
    const int d = h->d, nb = h->es_nb, nb8 = es_nb8(nb);
    const long NP = h->NP;
    const long cap = std::min<long>(chunk_rows(h), round_up(m, BM));
    if ((rc = ensure(h, h->es_cand, (size_t)cap * d * 8))) return rc;
    if ((rc = ensure(h, h->es_var, (size_t)cap * 8))) return rc;
    if ((rc = ensure(h, h->es_KZ, (size_t)cap * BM * 8))) return rc;
    if ((rc = ensure(h, h->es_S, (size_t)nb8 * cap * 8))) return rc;
    if ((rc = ensure(h, h->es_bb, (size_t)(cap / ES_TN + 1) * sizeof(BestPair)))) return rc;
    if ((rc = ensure(h, h->es_best, sizeof(BestPair)))) return rc;
    if (out && (rc = ensure(h, h->out_acq, (size_t)cap * 8))) return rc;
    const bool rule = lower && upper;
    if (rule) {
        if ((rc = ensure(h, h->es_lo, (size_t)d * 8))) return rc;
        if ((rc = ensure(h, h->es_up, (size_t)d * 8))) return rc;
        CK(cudaMemcpyAsync(h->es_lo.p, lower, (size_t)d * 8, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(h->es_up.p, upper, (size_t)d * 8, cudaMemcpyHostToDevice, h->stream));
    }
    CK(cudaMemsetAsync(h->es_best.p, 0xFF, sizeof(BestPair), h->stream));
    const size_t smem = es_score_smem(nb);
    CK(cudaFuncSetAttribute(gpk_es_score_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const double* lo = h->has_bounds ? ptr<double>(h->lower) : nullptr;
    const double* up = h->has_bounds ? ptr<double>(h->upper) : nullptr;
    for (long base = 0; base < m; base += cap) {
        const long mc = std::min(cap, m - base), mcp = round_up(mc, BM);
        double* dX = ptr<double>(h->es_cand);
        CK(cudaMemcpyAsync(dX, Xs + base * d, (size_t)mc * d * 8, cudaMemcpyHostToDevice, h->stream));
        // v: the existing scoring pass (int8 or fp64 variance contraction), un-normalised and clipped
        if ((rc = score_dev(h, dX, mc, GPK_ACQ_NONE, 0.0, 0.0, nullptr, nullptr, ptr<double>(h->es_var), nullptr, nullptr)))
            return rc;
        // fp64 K* of the chunk and k(X*, zb)
        if ((rc = ensure_score_scratch(h, mcp))) return rc;
        if ((rc = launch_cov_tiles(h, h->stream, train_operand(h), NP, h->n, dX, d, mc, mcp, lo, up, ptr<double>(h->Kstar),
                                   NP, 0, false)))
            return rc;
        if ((rc = launch_cov_tiles(h, h->stream, ptr<double>(h->es_zbop), BM, nb, dX, d, mc, mcp, lo, up,
                                   ptr<double>(h->es_KZ), BM, 0, false)))
            return rc;
        // S = k(zb, X*) - B^T K*^T  (nb x mc)
        if ((rc = es_gemm<true>(h, nb, mc, (int)NP, ptr<double>(h->es_Bt), NP, ptr<double>(h->Kstar), NP,
                                ptr<double>(h->es_S), cap, ptr<double>(h->es_KZ), BM)))
            return rc;
        EsScoreArgs a;
        a.S = ptr<double>(h->es_S); a.lds = cap;
        a.var = ptr<double>(h->es_var);
        a.cand = dX; a.d = d;
        a.lo = rule ? ptr<double>(h->es_lo) : nullptr; a.up = rule ? ptr<double>(h->es_up) : nullptr;
        a.mc = mc;
        a.nb = nb; a.nb8 = nb8; a.T = (int)es_T(nb); a.TP = es_tp(nb);
        a.norm_out = h->norm_out; a.ystd2 = h->y_std * h->y_std; a.sn2 = h->es_sn2;
        a.F = ptr<double>(h->es_F); a.jl = ptr<int2>(h->es_jl);
        a.U = ptr<double>(h->es_dmu); a.logP = ptr<double>(h->es_logP); a.lmb = ptr<double>(h->es_lmb);
        a.W = ptr<double>(h->es_W); a.np_grid = h->es_np; a.H = h->es_H;
        a.out = out ? ptr<double>(h->out_acq) : nullptr;
        a.bb = ptr<BestPair>(h->es_bb); a.base = base;
        const int nblk = (int)((mc + ES_TN - 1) / ES_TN);
        gpk_es_score_kernel<<<nblk, 256, smem, h->stream>>>(a);
        CKL();
        gpk_argmax_final_kernel<<<1, 256, 0, h->stream>>>(ptr<BestPair>(h->es_bb), nblk, ptr<BestPair>(h->es_best));
        CKL();
        if (out) CK(cudaMemcpyAsync(out + base, h->out_acq.p, (size_t)mc * 8, cudaMemcpyDeviceToHost, h->stream));
    }
    BestPair bp;
    CK(cudaMemcpyAsync(&bp, h->es_best.p, sizeof(BestPair), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (best_val) *best_val = bp.val;
    if (best_idx) *best_idx = (long)bp.idx;
    return GPK_OK;
}
