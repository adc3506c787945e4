"""CPU oracle of the emulator-based calibration (gladsgp_b200.calibration; DESIGN.md section 2 item 9).  TEST
INFRASTRUCTURE ONLY: NumPy / SciPy FP64.

* obs_terms: the per-sample Woodbury terms G, b, c0 of the observations;
* moments: predictive means / variances of the PC weights (sepia_oracle.w_pred's, addResidVar=False) at many points, one
  factorisation per (sample, PC) block (Emulator);
* loglik_dense: l_s from the dense n_o x n_o covariance with w_pred's moments (scipy.stats.multivariate_normal);
* loglik_woodbury: l_s from the Woodbury form; log_mean_exp: l from the l_s; loglik: both at given inputs;
* chain: random-walk Metropolis replaying given z / logu, with every decision's margin |logu - (l' - l)|;
* burnin_chol: the proposal factor after burn-in.
"""
from __future__ import annotations

import numpy as np
import scipy.linalg
from scipy import stats

from oracle import sepia_oracle as so


def obs_terms(K_O, r, tau, lamWOs):
    """K_O (pu, n_o), r, tau (n_o,), lamWOs (S,) -> G (S, pu, pu), b (S, pu), c0 (S,)."""
    K_O = np.asarray(K_O, dtype=np.float64)
    r = np.asarray(r, dtype=np.float64)
    D = 1.0 / np.asarray(lamWOs, dtype=np.float64).reshape(-1, 1) + np.asarray(tau, dtype=np.float64)[None, :] ** 2
    W = 1.0 / D
    G = np.einsum('pi,si,qi->spq', K_O, W, K_O)
    b = np.einsum('pi,si->sp', K_O, W * r[None, :])
    c0 = (W * r[None, :] ** 2).sum(1) + np.log(D).sum(1) + r.size * np.log(2.0 * np.pi)
    return G, b, c0


def standardized_obs(y_obs, obs_sd, ymean, ysd):
    """r, tau of native observations under the (scalar or per-output, already indexed) standardisation."""
    ysd = np.asarray(ysd, dtype=np.float64)
    r = (np.asarray(y_obs, dtype=np.float64) - np.asarray(ymean, dtype=np.float64)) / ysd
    tau = np.broadcast_to(np.asarray(obs_sd, dtype=np.float64), r.shape) / ysd
    return r, tau


class Emulator:
    """Cached factors of every (sample, PC) block of sepia_oracle.w_pred (S22 = block_cov)."""

    def __init__(self, num: so.OracleNum, samples):
        self.num = num
        d, pu, m = num.d, num.pu, num.m
        self.S = np.asarray(samples['lamWs']).reshape(-1, pu).shape[0]
        self.blocks = []
        for s in range(self.S):
            bU = np.asarray(samples['betaU'][s], dtype=np.float64).reshape((d, pu), order='F')
            lUz = np.asarray(samples['lamUz'][s], dtype=np.float64).reshape(-1)
            lWs = np.asarray(samples['lamWs'][s], dtype=np.float64).reshape(-1)
            lWOs = float(np.asarray(samples['lamWOs'][s]).reshape(-1)[0])
            for j in range(pu):
                cf = scipy.linalg.cho_factor(so.block_cov(num, bU[:, j], lUz[j], lWs[j], lWOs, j), lower=True)
                alpha = scipy.linalg.cho_solve(cf, num.wv[j * m:(j + 1) * m, 0])
                self.blocks.append((bU[:, j], lUz[j], 1.0 / lUz[j] + 1.0 / lWs[j], cf, alpha))

    def moments(self, t_trans):
        """t_trans (N, q) -> mu, var (S, pu, N)."""
        t_trans = np.asarray(t_trans, dtype=np.float64).reshape(-1, self.num.q)
        xp = np.concatenate([0.5 * np.ones((t_trans.shape[0], 1)), t_trans], axis=1)
        N, pu = xp.shape[0], self.num.pu
        mu = np.empty((self.S * pu, N))
        var = np.empty((self.S * pu, N))
        for k, (beta, lamz, s11, cf, alpha) in enumerate(self.blocks):
            S21 = so.cov_cross(self.num.zt, xp, beta, lamz)
            mu[k] = S21.T @ alpha
            var[k] = s11 - np.sum(S21 * scipy.linalg.cho_solve(cf, S21), axis=0)
        return mu.reshape(self.S, pu, N), var.reshape(self.S, pu, N)


def loglik_dense(num, t_trans, samples, K_O, r, tau):
    """l_s (S,) at one point t_trans (q,) from the dense covariance D_s + K_O^T diag(v_s) K_O, with w_pred's moments."""
    _, mus, Sigs = so.w_pred(num, np.asarray(t_trans, dtype=np.float64).reshape(1, -1), samples, draw=False)
    lamWOs = np.asarray(samples['lamWOs'], dtype=np.float64).reshape(-1)
    out = np.empty(mus.shape[0])
    for s in range(mus.shape[0]):
        v = np.maximum(np.diag(Sigs[s]), 0.0)
        cov = np.diag(1.0 / lamWOs[s] + tau ** 2) + K_O.T @ (v[:, None] * K_O)
        out[s] = stats.multivariate_normal.logpdf(r, mean=K_O.T @ mus[s], cov=cov)
    return out


def loglik_woodbury(mu, var, G, b, c0):
    """mu, var (S, pu, N), G (S, pu, pu), b (S, pu), c0 (S,) -> l_s (S, N)."""
    S, pu, N = mu.shape
    out = np.empty((S, N))
    for s in range(S):
        m_ = mu[s].T                                                   # (N, pu)
        sv = np.sqrt(np.maximum(var[s].T, 0.0))
        A = np.eye(pu)[None] + sv[:, :, None] * G[s][None] * sv[:, None, :]
        h = b[s][None, :] - m_ @ G[s]
        L = np.linalg.cholesky(A)
        y = sv * h
        z = np.empty_like(y)
        for k in range(pu):                                            # forward substitution L z = V^1/2 h
            z[:, k] = (y[:, k] - np.einsum('nj,nj->n', L[:, k, :k], z[:, :k])) / L[:, k, k]
        logdet = 2.0 * np.sum(np.log(np.diagonal(L, axis1=1, axis2=2)), axis=1)
        out[s] = -0.5 * (c0[s] - 2.0 * m_ @ b[s] + np.einsum('np,pq,nq->n', m_, G[s], m_) - np.sum(z * z, axis=1) + logdet)
    return out


def loglik(em, G, b, c0, t_trans):
    """l (N,) at transformed inputs t_trans (N, q) from an Emulator's moments."""
    return log_mean_exp(loglik_woodbury(*em.moments(t_trans), G, b, c0))


def log_mean_exp(ls):
    """log((1/S) sum_s exp l_s) over axis 0 with a max shift, summed over s in ascending order."""
    ls = np.asarray(ls, dtype=np.float64)
    mx = np.max(ls, axis=0)
    acc = np.zeros(ls.shape[1:])
    for s in range(ls.shape[0]):
        acc = acc + np.exp(ls[s] - mx)
    return mx + np.log(acc) - np.log(ls.shape[0])


def burnin_chol(states, step):
    """states (n, C, q) of the second half of burn-in -> chol((2.38^2 / q_free) Sigma) on the free inputs (step > 0), zero
    rows / columns for fixed ones; diag(step) when the Cholesky fails."""
    step = np.asarray(step, dtype=np.float64)
    q = step.size
    free = np.nonzero(step > 0)[0]
    if free.size == 0:
        return np.diag(step)
    X = np.asarray(states)[:, :, free].reshape(-1, free.size)
    if X.shape[0] < 2:
        return np.diag(step)
    Sig = np.atleast_2d(np.cov(X, rowvar=False, ddof=1)) * (2.38 ** 2 / free.size)
    try:
        Lf = np.linalg.cholesky(Sig)
    except np.linalg.LinAlgError:
        return np.diag(step)
    if not np.all(np.isfinite(Lf)):
        return np.diag(step)
    L = np.zeros((q, q))
    L[np.ix_(free, free)] = Lf
    return L


def propose(theta, L, z):
    """theta + L z per chain, summed over k ascending (the device's order)."""
    x = theta.copy()
    for i in range(theta.shape[1]):
        for k in range(i + 1):
            x[:, i] = x[:, i] + L[i, k] * z[:, k]
    return x


def chain(loglik, theta0, z, logu, lo, hi, step, n_burn):
    """Random-walk Metropolis of C chains replaying z (T, C, q) and logu (T, C); loglik(theta (C, q)) -> l (C,).  Burn-in
    proposes with diag(step); after n_burn steps with burnin_chol of the states n_burn // 2 ... n_burn - 1.
    Returns dict(theta (T, C, q), ll (T, C), accepted (T, C), margin (T, C): |logu - (l' - l)| of valid candidates, inf
    otherwise; L (q, q): the final proposal factor)."""
    T, C, q = z.shape
    L = np.diag(np.asarray(step, dtype=np.float64))
    theta = np.array(theta0, dtype=np.float64)
    ll = loglik(theta)
    out = dict(theta=np.empty((T, C, q)), ll=np.empty((T, C)), accepted=np.zeros((T, C), dtype=bool),
               margin=np.full((T, C), np.inf))
    cand = propose(theta, L, z[0])
    for t in range(T):
        valid = np.all((cand >= lo) & (cand <= hi), axis=1)
        lnew = np.full(C, np.nan)
        if valid.any():
            lnew[valid] = loglik(cand[valid])
        with np.errstate(invalid='ignore'):
            diff = lnew - ll
            acc = valid & (logu[t] < diff)
        out['margin'][t, valid] = np.abs(logu[t, valid] - diff[valid])
        theta[acc] = cand[acc]
        ll[acc] = lnew[acc]
        out['theta'][t], out['ll'][t], out['accepted'][t] = theta, ll, acc
        if t == n_burn - 1:
            L = burnin_chol(out['theta'][n_burn // 2:n_burn], step)
        if t + 1 < T:
            cand = propose(theta, L, z[t + 1])
    out['L'] = L
    return out
