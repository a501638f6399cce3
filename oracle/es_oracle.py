"""Entropy search restated in numpy (CHECKER ONLY, never imported by the product): expectation propagation for the
probability of each representer point being the minimum (Cunningham, Hennig & Lacoste-Julien 2011, as RoBO runs it in
robo/util/epmgp.py) and the information gain of InformationGain (robo/acquisition_functions/information_gain.py),
vectorised over candidates.

Conventions the reference fixes and this restatement keeps:
  * vech(M) lists the lower triangle in row-major order: (0,0), (1,0), (1,1), (2,0), ...
  * the EP message update rounds like the reference (no fused multiply-add); sweeps stop when the summed |d| of a
    sweep is < 1e-3, after at most 50 sweeps; a NaN d ends EP with log Z = -inf and zero derivatives
  * logP = -inf becomes -500 before the renormalisation; the second-derivative correction adds Zm[j]^2 (an
    element-wise square, as the reference's Zm.T * Zm of a 1-D array does)
  * v (noisy variance, un-normalised) minus sn2 (noise in normalised units); cross-covariances clipped at eps
"""
import numpy as np
from scipy import special

SQ2 = np.sqrt(2)
EPS32 = np.finfo(np.float32).eps
L2P = np.log(2) + np.log(np.pi)


def vech_index(D):
    """(rows, cols) of vech for a D x D matrix."""
    r, c = np.tril_indices(D)
    return r, c


def _np_max(a, b):
    return np.max([a, b])


def _ep_point(mu, S, k):
    """EP for 'point k is the minimum' -> (logZ, dMu (D,), dSig vech (T,), dMuMu (D, D), sweeps)."""
    D = mu.shape[0]
    P, MP, LS = np.zeros(D - 1), np.zeros(D - 1), np.zeros(D - 1)
    M, V = mu.copy(), S.copy()
    d = 0.0
    sweeps = 50
    for sweep in range(50):
        diff = 0.0
        for i in range(D - 1):
            l = i if i < k else i + 1
            p, mp = P[i], MP[i]
            cVc = (V[l, l] - 2 * V[k, l] + V[k, k]) / 2.0
            Vc = (V[:, l] - V[:, k]) / SQ2
            cM = (M[l] - M[k]) / SQ2
            cVnic = _np_max(cVc / (1 - p * cVc), 0)
            cmni = cM + cVnic * (p * cM - mp)
            z = cmni / np.sqrt(cVnic + 1e-25)
            if np.isnan(z):
                z = -np.inf
            if z < -6:
                d = np.nan
            else:
                if z > 6:
                    dp, dmp = -p, -mp
                    d = max([dmp, dp])
                    P[i], MP[i], LS[i] = 0.0, 0.0, 0.0
                else:
                    logPhi = np.log(0.5 * special.erfc(-z / SQ2))
                    e = np.exp(-0.5 * (z * z + L2P) - logPhi)
                    alpha = e / np.sqrt(cVnic)
                    beta = alpha * (alpha * cVnic + cmni)
                    r = beta / (1 - beta)
                    dp = _np_max(-p + EPS32, r / cVnic - p)
                    dmp = _np_max(-mp + EPS32, r * (alpha + cmni / cVnic) + alpha - mp)
                    d = _np_max(dmp, dp)
                    P[i], MP[i] = p + dp, mp + dmp
                    LS[i] = logPhi - 0.5 * (np.log(beta) - np.log(P[i]) - np.log(cVnic)) + (alpha * alpha) / (2 * beta) * cVnic
                t = dp / (1 + dp * cVc)
                V = V - t * np.outer(Vc, Vc)
                M = M + (dmp - cM * dp) / (1 + dp * cVc) * Vc
                if np.any(np.isnan(V)):
                    raise ValueError("EP variance contains NaN")
            if np.isnan(d):
                break
            diff += np.abs(d)
        if np.isnan(d) or np.abs(diff) < 0.001:
            sweeps = sweep + 1
            break
    T = D * (D + 1) // 2
    if np.isnan(d):
        return -np.inf, np.zeros(D), np.zeros(T), np.zeros((D, D)), sweeps
    # columns j of R: rho_j in row l_j, -rho_j in row k
    ls = np.array([j if j < k else j + 1 for j in range(D - 1)])
    R = np.zeros((D, D - 1))
    rho = np.sqrt(P) / SQ2
    R[ls, np.arange(D - 1)] = rho
    R[k, :] = -rho
    r = np.zeros(D)
    r[ls] = MP / SQ2
    r[k] = -np.sum(MP) / SQ2
    nz = MP != 0
    mpm = np.sum(MP[nz] ** 2 / P[nz])
    IRSR = np.eye(D - 1) + R.T @ S @ R
    A = R @ np.linalg.solve(IRSR, R.T)
    A = 0.5 * (A + A.T)
    b = mu + S @ r
    Ab = A @ b
    for jit in (0.0, 1e-10, 1e-6):
        try:
            L = np.linalg.cholesky(IRSR + jit * np.eye(D - 1))
            break
        except np.linalg.LinAlgError:
            if jit == 1e-6:
                raise
    logZ = 0.5 * (r @ S @ r - b @ Ab - 2 * np.sum(np.log(np.diag(L)))) + mu @ r + np.sum(LS) - 0.5 * mpm
    E = -A - 2 * np.outer(r, Ab) + np.outer(r, r) + np.outer(Ab, Ab)
    E = 0.5 * (E + E.T - np.diag(np.diag(E)))
    return logZ, r - Ab, E[vech_index(D)], -A, sweeps


def joint_min(mu, S):
    """-> logP (D,), dlogPdMu (D, D), dlogPdSigma (D, T), dlogPdMudMu (D, D, D), sweeps (D,)."""
    mu, S = np.asarray(mu, dtype=np.float64).ravel(), np.asarray(S, dtype=np.float64)
    D = mu.shape[0]
    parts = [_ep_point(mu, S, k) for k in range(D)]
    logZ = np.array([p[0] for p in parts])
    dMu = np.array([p[1] for p in parts])
    dSig = np.array([p[2] for p in parts])
    dMuMu = np.array([p[3] for p in parts])
    sweeps = np.array([p[4] for p in parts])
    logZ[np.isinf(logZ)] = -500
    e = np.exp(logZ)
    Z = np.sum(e)
    mx = np.max(logZ)
    s = mx + np.log(np.sum(np.exp(logZ - mx)))
    s = mx if np.isinf(s) else s
    Zm = e @ dMu / Z
    Zs = e @ dSig / Z
    gg = np.einsum("kij,k->ij", dMuMu + np.einsum("ki,kj->kij", dMu, dMu), e) / Z
    return logZ - s, dMu - Zm, dSig - Zs, dMuMu + (-gg + Zm * Zm)[None], sweeps


def grid(Np):
    """W: Np standard-normal quantiles."""
    from scipy.stats import norm
    return norm.ppf(np.linspace(1. / (Np + 1), 1 - 1. / (Np + 1), Np))


def information_gain(state, s, v, X=None, lower=None, upper=None):
    """dH per candidate.  state: dict(logP, dlogPdMu, dlogPdSigma, dlogPdMudMu, lmb, W, sn2); s (M, Nb) clipped
    cross-covariances with the representer points; v (M,) predictive variances (both un-normalised)."""
    logP = np.asarray(state["logP"]).ravel()
    lmb = np.asarray(state["lmb"]).ravel()
    W = np.asarray(state["W"]).ravel()
    U, Gs, A = state["dlogPdMu"], state["dlogPdSigma"], state["dlogPdMudMu"]
    Nb = logP.size
    r, c = vech_index(Nb)
    v_ = v - state["sn2"]
    inv = 1.0 / v_
    sq = np.sqrt(v + 1e-10)
    dm = s * (inv * sq)[:, None]                                    # (M, Nb)
    vss = s[:, r] * s[:, c]                                         # vech(s s^T), (M, T)
    det = -inv[:, None] * (vss @ Gs.T) + 0.5 * np.einsum("mj,ijl,ml->mi", dm, A, dm)
    a = logP[None, :] + det                                         # (M, Nb)
    b = dm @ U.T                                                    # (M, Nb)
    lP = a[:, :, None] + b[:, :, None] * W[None, None, :]           # (M, Nb, Np)
    with np.errstate(all="ignore"):
        mx = np.max(lP, axis=1)
        ssum = mx + np.log(np.sum(np.exp(lP - mx[:, None, :]), axis=1))
        anyinf = np.any(np.isinf(ssum), axis=1)
        L = np.where(anyinf[:, None], mx, ssum)
        lPn = lP - L[:, None, :]
        H = -np.sum(np.exp(logP) * (logP + lmb))
        dH = np.mean(np.sum(np.exp(lPn) * (lPn + lmb[None, :, None]), axis=1), axis=1) + H
    dH[np.isnan(dH) | (dH == np.inf)] = -np.finfo(np.float64).max
    if lower is not None:
        X = np.asarray(X)
        dH[np.any((X < lower) | (X > upper), axis=1)] = np.spacing(1)
    return dH


def gp_es_inputs(st, gp_predict, zb, X):
    """(mu_b, V_b, s (M, Nb), v (M,)) of a fitted oracle GP state: predict(zb, full_cov=True) clipped, the joint
    covariance of (zb, x) clipped (information_gain.py:263), v = predict(X) variance."""
    eps = np.finfo(np.float64).eps
    mu_b, V_b = gp_predict(st, zb, full_cov=True)
    Nb = zb.shape[0]
    _, Vj = gp_predict(st, np.concatenate([zb, X]), full_cov=True)
    s = np.clip(Vj[Nb:, :Nb], eps, np.inf)
    _, v = gp_predict(st, X)
    return mu_b, np.clip(V_b, eps, np.inf), s, v
