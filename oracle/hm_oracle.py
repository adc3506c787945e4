"""CPU oracle of history matching (gladsgp_b200.history; DESIGN.md section 2 item 11).  TEST INFRASTRUCTURE ONLY: NumPy
FP64.

* mixture: the mean m (N, pu) and covariance M (N, pu, pu) of the PC weights over the samples (law of total variance);
* route_features: e and V as the products of the per-point feature rows [1, m], [M_jj, 2 M_jk (j < k); 1] with the
  per-output rows [r, -K], [K_j K_k; c] (the device's formulation);
* route_direct: e and V from each sample's output means K_O^T mu_s and variances sum_j K_ji^2 v_sj, then the mixture's
  mean and variance over the samples;
* history_match: impl, n_over, nroy, and each point's margins |impl[order-1] - cutoff| and min_i |I_i - cutoff|, with
  the moments of calib_oracle.Emulator.
"""
from __future__ import annotations

import numpy as np


def mixture(mu, var):
    """mu, var (S, pu, N) -> m (N, pu), M (N, pu, pu)."""
    mu = np.asarray(mu, dtype=np.float64)
    v = np.maximum(np.asarray(var, dtype=np.float64), 0.0)
    m = mu.mean(axis=0).T
    d = mu - m.T[None]
    M = np.einsum('sjn,skn->njk', d, d) / mu.shape[0]
    M[:, np.arange(mu.shape[1]), np.arange(mu.shape[1])] += v.mean(axis=0).T
    return m, M


def _pairs(pu):
    return [(j, k) for j in range(pu) for k in range(j, pu)]


def route_features(mu, var, K_O, r, c):
    """e, V (N, n_o) by the feature products."""
    m, M = mixture(mu, var)
    N, pu = m.shape
    pr = _pairs(pu)
    a_e = np.concatenate([np.ones((N, 1)), m], axis=1)
    a_v = np.stack([M[:, j, k] * (1.0 if j == k else 2.0) for j, k in pr] + [np.ones(N)], axis=1)
    b_e = np.concatenate([np.asarray(r, dtype=np.float64)[:, None], -K_O.T], axis=1)
    b_v = np.stack([K_O[j] * K_O[k] for j, k in pr] + [np.asarray(c, dtype=np.float64)], axis=1)
    return a_e @ b_e.T, a_v @ b_v.T


def route_direct(mu, var, K_O, r, c):
    """e, V (N, n_o): per-sample output moments, then the mixture's mean and variance over the samples."""
    mu = np.asarray(mu, dtype=np.float64)
    v = np.maximum(np.asarray(var, dtype=np.float64), 0.0)
    ys = np.einsum('ji,sjn->sni', K_O, mu)                     # (S, N, n_o)
    vs = np.einsum('ji,sjn->sni', K_O * K_O, v)
    Ey = ys.mean(axis=0)
    Vy = vs.mean(axis=0) + ((ys - Ey[None]) ** 2).mean(axis=0)
    return np.asarray(r)[None, :] - Ey, Vy + np.asarray(c)[None, :]


def implausibility(e, V):
    with np.errstate(divide='ignore', invalid='ignore'):
        I = np.abs(e) / np.sqrt(V)
    return np.where(np.isnan(I), np.inf, I)


def reduce(I, order, cutoff):
    """I (N, n_o) -> dict(impl (N, order) descending, n_over, nroy, margin, edge)."""
    impl = -np.sort(-I, axis=1)[:, :order]
    return dict(impl=impl, n_over=np.sum(I > cutoff, axis=1), nroy=impl[:, order - 1] <= cutoff,
                margin=np.abs(impl[:, order - 1] - cutoff), edge=np.min(np.abs(I - cutoff), axis=1))


def scale(mu, var, K_O, r, c):
    """Per point, max_i of (|r_i| + sum_j |K_ji m_j|) / sqrt(V_i) + I_i (sum_j sqrt(M_jj) |K_ji|)^2 / V_i: the size of the
    terms whose rounding enters I_i (e's terms over sqrt(V), and V's terms, bounded by Cauchy-Schwarz, times dI/dV)."""
    m, M = mixture(mu, var)
    e, V = route_features(mu, var, K_O, r, c)
    I = implausibility(e, V)
    te = np.abs(np.asarray(r))[None, :] + np.abs(m) @ np.abs(K_O)
    sv = np.sqrt(np.maximum(np.diagonal(M, axis1=1, axis2=2), 0.0)) @ np.abs(K_O)
    with np.errstate(divide='ignore', invalid='ignore'):
        s = te / np.sqrt(V) + I * sv * sv / V
    return np.max(np.where(np.isfinite(s), s, 0.0), axis=1)


def history_match(em, t_trans, K_O, r, c, order, cutoff, route='features'):
    """With an oracle Emulator (calib_oracle.Emulator) at transformed inputs t_trans (N, q): dict of reduce() plus I,
    scale."""
    mu, var = em.moments(t_trans)
    K_O = np.asarray(K_O, dtype=np.float64)
    e, V = (route_features if route == 'features' else route_direct)(mu, var, K_O, r, c)
    I = implausibility(e, V)
    out = reduce(I, order, cutoff)
    out.update(I=I, scale=scale(mu, var, K_O, r, c))
    return out
