"""FP64 reference of the MCMC convergence diagnostics (DESIGN.md section 2, "Chain diagnostics").

Rank-normalized split R-hat, bulk ESS and tail ESS of Vehtari, Gelman, Simpson, Carpenter and Buerkner (2021), the
statistics ArviZ computes as rhat(method="rank"), ess(method="bulk") and ess(method="tail"), restated in NumPy / SciPy:
ranks with scipy.stats.rankdata(method="average"), the normal quantile with scipy.special.ndtri, and the autocovariance as
a direct sum (ArviZ uses an FFT, which differs only by rounding).  Lags are computed in blocks as Geyer's sequence asks for
them, so a fast-mixing series costs a few lags.

x of one element: (C, n) float64, chain-major.
"""
import numpy as np
from scipy.special import ndtri
from scipy.stats import rankdata

LAG_BLOCK = 64


def split_chains(a):
    """(C, n) -> (2C, n // 2): first halves of every chain, then second halves (the middle draw of odd n is dropped)."""
    h = a.shape[1] // 2
    return np.concatenate([a[:, :h], a[:, a.shape[1] - h:]], axis=0)


def z_scale(a):
    """Rank-normalize over all values of a, pooled over chains; -0.0 and +0.0 rank as one value."""
    r = rankdata(a + 0.0, method='average').reshape(a.shape)
    return ndtri((r - 0.375) / (a.size + 0.25))


def rhat_raw(a):
    """R-hat of a (k chains, h draws); NaN when the within-chain variance is 0."""
    h = a.shape[1]
    B = h * np.var(a.mean(axis=1), ddof=1)
    W = np.mean(np.var(a, axis=1, ddof=1))
    if W == 0:
        return np.nan
    return float(np.sqrt((B / W + h - 1) / h))


class _Acov:
    """Mean over chains of acov_c[t] = (1/h) sum_{i < h-t} (a_ci - mean_c)(a_c,i+t - mean_c), by blocks of lags."""

    def __init__(self, a):
        self.d = a - a.mean(axis=1, keepdims=True)
        self.h = a.shape[1]
        self.vals = np.empty(0)

    def __getitem__(self, t):
        while t >= self.vals.size:
            t0 = self.vals.size
            lags = range(t0, min(t0 + LAG_BLOCK, self.h))
            blk = [np.mean(np.sum(self.d[:, :self.h - u] * self.d[:, u:], axis=1) / self.h) for u in lags]
            self.vals = np.concatenate([self.vals, blk])
        return self.vals[t]


def ess_raw(a, margins=None, info=None):
    """ESS of a (k chains, h draws), ArviZ's _ess loops as written.  margins (a list) receives the smallest |even + odd|
    Geyer's loop tested (and |even| of the improvement step) and the smallest gap of the monotone comparisons (inf when a
    test never ran).  info (a dict) receives max_t, the last lag of the initial positive sequence."""
    k, h = a.shape
    if np.max(a) == np.min(a):
        if margins is not None:
            margins += [np.inf, np.inf]
        return float(k * h)
    acov = _Acov(a)
    chain_mean = a.mean(axis=1)
    mean_var = acov[0] * h / (h - 1.0)
    var_plus = mean_var * (h - 1.0) / h + np.var(chain_mean, ddof=1)

    def rho_hat(t):
        return 1.0 - (mean_var - acov[t]) / var_plus
    rho = np.zeros(h)
    even = 1.0
    rho[0] = even
    odd = rho_hat(1)
    rho[1] = odd
    m_geyer = m_mono = np.inf
    t = 1
    while t < h - 3:
        m_geyer = min(m_geyer, abs(even + odd))
        if not even + odd > 0.0:
            break
        even = rho_hat(t + 1)
        odd = rho_hat(t + 2)
        m_geyer = min(m_geyer, abs(even + odd))
        if even + odd >= 0:
            rho[t + 1] = even
            rho[t + 2] = odd
        t += 2
    max_t = t - 2
    m_geyer = min(m_geyer, abs(even))
    if even > 0:
        rho[max_t + 1] = even
    t = 1
    while t <= max_t - 2:
        lhs, rhs = rho[t + 1] + rho[t + 2], rho[t - 1] + rho[t]
        m_mono = min(m_mono, abs(lhs - rhs))
        if lhs > rhs:
            rho[t + 1] = rhs / 2.0
            rho[t + 2] = rho[t + 1]
        t += 2
    tau = -1.0 + 2.0 * np.sum(rho[:max_t + 1]) + np.sum(rho[max_t + 1:max_t + 2])
    tau = max(tau, 1.0 / np.log10(k * h))
    if margins is not None:
        margins += [m_geyer, m_mono]
    if info is not None:
        info['max_t'] = max_t
    return float(k * h / tau)


def diagnose(x, margins=None):
    """One element, x (C, n) -> (rhat, ess_bulk, ess_tail).  margins (a list) receives, per ESS series (bulk, q05
    indicator, q95 indicator), the pair of decision margins of ess_raw."""
    x = np.asarray(x, dtype=np.float64)
    if x.ndim != 2 or x.shape[1] < 4:
        raise ValueError('x must be (n_chains, n_draws) with n_draws >= 4')
    if not np.all(np.isfinite(x)):
        return np.nan, np.nan, np.nan
    s = split_chains(x)
    zb = z_scale(s)
    bulk = rhat_raw(zb)
    folded = rhat_raw(z_scale(np.abs(s - np.median(s))))
    rhat = max(bulk, folded)
    ess_bulk = ess_raw(zb, margins)
    q05, q95 = np.quantile(x, (0.05, 0.95))
    e05 = ess_raw(split_chains((x <= q05).astype(np.float64)), margins)
    e95 = ess_raw(split_chains((x <= q95).astype(np.float64)), margins)
    return rhat, ess_bulk, min(e05, e95)


def diagnose_all(x):
    """x (n, C, E) -> three (E,) arrays, the smallest Geyer margin and the smallest monotone gap over all elements and
    series.  Only the Geyer tests can move the ESS by more than rounding when they flip (they decide where the sequence
    ends and whether the improvement step adds a lag).  The initial monotone sequence is a running minimum of pair sums,
    continuous in rho: a flip at a near-tie moves tau by at most the gap, and indicator series tie exactly (gap 0) often."""
    x = np.asarray(x, dtype=np.float64)
    n, C, E = x.shape
    out = np.empty((3, E))
    margins = []
    for e in range(E):
        out[:, e] = diagnose(x[:, :, e].T, margins)
    return out[0], out[1], out[2], min(margins[0::2], default=np.inf), min(margins[1::2], default=np.inf)
