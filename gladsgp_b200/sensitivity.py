"""Sobol' / Saltelli sensitivity indices of the emulator with bootstrap confidence limits (SURVEY 8f rank 3).

Mirror of /root/reference/src/utils.py:27-125 (`saltelli_sensitivity_indices`) and :128-256
(`PCA_saltelli_sensitivity_indices`): same names, arguments, return tuples and the same consumption of randomness (an
unseeded scrambled `scipy.stats.qmc.Sobol(d=2*n_dim)`, one draw of `n_resamples x N` resampling indices per statistic from
the global `np.random` state, in the reference's order), so `experiments/synthetic/analysis/sensitivity_indices.py:96,214`
run unchanged with `from gladsgp_b200 import sensitivity as utils`.  What differs is where the work happens: the reference
hands a Python closure to `scipy.stats.bootstrap`, which evaluates it 9999 times per statistic plus N times for the BCa
jackknife; here the statistic of every index set is computed by one CUDA kernel launch (`ggp_sobol_stats_f64`) and only the
BCa arithmetic on the resulting distributions (normal quantiles, `scipy.stats.quantile`) stays on the host, restated from
scipy's `_bca_interval`.  There is no CPU fallback.

`emulator_mean_function(model, samples)` builds the `func` of sensitivity_indices.py:73-91 on the cached-factor device
predictor: posterior-sample average of the emulator's PC weights at N designs per call.

`gp_sensitivity_indices(model, samples, option, pcvar, ngrid)` computes the indices of that function (and of each
posterior sample's mean function) exactly instead: the mean is a sum of product squared-exponential kernels, so every
Sobol' integral over uniform inputs is a closed form in erf and exp (csrc/ggp_gp_sens.cu).
"""
from collections import namedtuple
from dataclasses import dataclass

import numpy as np
from scipy import special, stats
from scipy._lib._util import check_random_state, rng_integers

from . import ops

ConfidenceInterval = namedtuple('ConfidenceInterval', ['low', 'high'])


@dataclass
class BootstrapResult:
    """Same attributes as scipy.stats._resampling.BootstrapResult."""
    confidence_interval: ConfidenceInterval
    bootstrap_distribution: np.ndarray
    standard_error: np.ndarray


def _evaluate_blocks(func, n_dim, m, AB=None):
    """f_A, f_B, f_AB in the reference's call order (src/utils.py:66-80)."""
    if AB is None:
        AB = stats.qmc.Sobol(d=2 * n_dim).random_base2(m=int(m))
    AB = np.asarray(AB)
    base_a, base_b = AB[:, n_dim:], AB[:, :n_dim]                       # src/utils.py:68-69
    f_A = np.asarray(func(base_a), dtype=np.float64)
    f_B = np.asarray(func(base_b), dtype=np.float64)
    f_AB = np.empty((n_dim,) + f_A.shape)
    for i in range(n_dim):                                              # B with column i taken from A (:76-80)
        f_AB[i] = func(np.where((np.arange(n_dim) == i)[None, :], base_a, base_b))
    return f_A, f_B, f_AB


class _Estimator:
    """Function values resident on the device; statistics of index sets through ggp_sobol_stats_f64."""

    def __init__(self, f_A, f_B, f_AB):
        self.N, self.p = f_A.shape
        self.n_dim = f_AB.shape[0]
        self.dev = ops.sobol_upload(f_A, f_B, f_AB)
        self._jack = None

    def stats(self, idx=None, clamp=True):
        """(first, total), each (R, p, n_dim) float64 on the host; idx (R, n) integer index sets or None = full sample."""
        return ops.sobol_stats(self.dev, self.N, self.p, self.n_dim, idx=idx, clamp=clamp)

    def jackknife(self):
        if self._jack is None:
            N = self.N
            j = np.ones((N, N), dtype=bool)
            np.fill_diagonal(j, False)
            idx = np.broadcast_to(np.arange(N), (N, N))[j].reshape(N, N - 1)
            self._jack = (self.stats(None, clamp=True), self.stats(idx, clamp=True))
        return self._jack


def _select(first_total, kind, pcvar):
    """(R, p, n_dim) pair -> the statistic's values with the resample axis last, as scipy lays them out."""
    arr = first_total[0] if 'first' in kind else first_total[1]
    if kind.startswith('general'):
        arr = np.sum(arr * np.asarray(pcvar, dtype=np.float64)[None, :, None], axis=1)       # (R, n_dim)
    return np.moveaxis(arr, 0, -1)


def _bootstrap(est, kind, pcvar=None, n_resamples=9999, confidence_level=0.95, rng=None):
    """scipy.stats.bootstrap([arange(N)], statistic, n_resamples=..., method='BCa') with the statistic on the device."""
    N = est.N
    rng = check_random_state(rng)
    i = rng_integers(rng, 0, N, (n_resamples, N))                       # scipy _bootstrap_resample: one draw per call
    theta_hat_b = _select(est.stats(i, clamp=True), kind, pcvar)        # (..., n_resamples)
    full, jack = est.jackknife()
    theta_hat = _select(full, kind, pcvar)                              # (..., 1)
    theta_hat_i = _select(jack, kind, pcvar)                            # (..., N)
    # scipy _bca_interval
    B = theta_hat_b.shape[-1]
    percentile = (np.count_nonzero(theta_hat_b < theta_hat, axis=-1)
                  + np.count_nonzero(theta_hat_b <= theta_hat, axis=-1)).astype(np.float64) / (2 * B)
    z0_hat = special.ndtri(percentile)
    n = float(N)
    theta_dot = np.mean(theta_hat_i, axis=-1, keepdims=True)
    U = (n - 1) * (theta_dot - theta_hat_i)
    with np.errstate(invalid='ignore', divide='ignore'):
        a_hat = 1 / 6 * (np.sum(U ** 3, axis=-1) / n ** 3) / (np.sum(U ** 2, axis=-1) / n ** 2) ** (3 / 2)
        alpha = (1 - confidence_level) / 2
        z_alpha = float(special.ndtri(alpha))
        num1 = z0_hat + z_alpha
        alpha_1 = special.ndtr(z0_hat + num1 / (1 - a_hat * num1))
        num2 = z0_hat - z_alpha
        alpha_2 = special.ndtr(z0_hat + num2 / (1 - a_hat * num2))
    interval = np.stack((alpha_1, alpha_2), axis=-1)
    ci = stats.quantile(theta_hat_b, interval, axis=-1)
    se = np.std(theta_hat_b, ddof=1, axis=-1)
    return BootstrapResult(ConfidenceInterval(ci[..., 0], ci[..., 1]), theta_hat_b, se)


def saltelli_sensitivity_indices(func, n_dim, m, bootstrap=True, AB=None, n_resamples=9999, rng=None):
    """first_order (p, n_dim), total_index (p, n_dim), res {'first_order', 'total_index'} (src/utils.py:27-125).
    func(x: (N, n_dim)) -> (N, p) with N = 2**m.  AB / n_resamples / rng pin what the reference draws at random."""
    f_A, f_B, f_AB = _evaluate_blocks(func, n_dim, m, AB)
    est = _Estimator(f_A, f_B, f_AB)
    first, total = est.stats(None, clamp=False)
    res = None
    if bootstrap:
        res = {k: _bootstrap(est, k, n_resamples=n_resamples, rng=rng) for k in ('first_order', 'total_index')}
    return first[0], total[0], res


def PCA_saltelli_sensitivity_indices(func, n_dim, m, pcvar, bootstrap=True, AB=None, n_resamples=9999, rng=None):
    """first_order, total_index (p, n_dim), general first / total (n_dim,) weighted by the PCs' explained variance, res with
    the four bootstrap results (src/utils.py:128-256)."""
    pcvar = np.asarray(pcvar, dtype=np.float64)
    f_A, f_B, f_AB = _evaluate_blocks(func, n_dim, m, AB)
    est = _Estimator(f_A, f_B, f_AB)
    first, total = est.stats(None, clamp=False)
    first, total = first[0], total[0]
    res = None
    if bootstrap:
        res = {k: _bootstrap(est, k, pcvar=pcvar, n_resamples=n_resamples, rng=rng)
               for k in ('first_order', 'total_index', 'general_first_order', 'general_total_index')}
    gen_first = np.sum(first.T * pcvar, axis=1)
    gen_total = np.sum(total.T * pcvar, axis=1)
    return first, total, gen_first, gen_total, res


def emulator_mean_function(model, samples):
    """func(x: (N, q)) -> (N, pu): average over the posterior samples of the emulator's predictive mean of the PC weights.
    The reference's func (sensitivity_indices.py:73-91) averages realisations `pred.w`; their Monte-Carlo noise around
    this mean only inflates the estimated variance.  The nsamp*pu covariance factors are built once and reused by every
    call (the (n_dim + 2) design blocks of the Saltelli scheme)."""
    from .sepia.SepiaPredict import SepiaEmulatorPrediction
    q = model.num.q
    proto = SepiaEmulatorPrediction(t_pred=np.full((1, q), 0.5), samples=samples, model=model, do_call=False)
    ns, beta, lamz, dadd, s11, W = proto._blocks()
    pred = ops.Predictor(model.num.zt, W, beta, lamz, dadd, s11)
    pu = model.num.pu

    def func(x):
        xp = SepiaEmulatorPrediction(t_pred=np.asarray(x), samples=samples, model=model, do_call=False).xpredt
        mean, _ = pred.predict(xp)
        return mean.reshape(ns, pu, xp.shape[0]).mean(dim=0).T.contiguous().cpu().numpy()
    return func


def emulator_expansion(model, samples):
    """The emulator's predictive mean of PC j under posterior sample s as a sum of product kernels over the inputs,
    mu_sj(x) = sum_i a_sji prod_k exp(-beta_sjk (x_k - z_ik)^2),  a_sj = S22_sj^-1 w_j / lamUz_sj.
    The inputs are the columns of model.num.zt except a dummy x (prediction puts x = 0.5 there, as in every training
    row, so its kernel factor is 1).  S22^-1 w comes from the factors SepiaEmulatorPrediction caches with the model (built
    and cached here if absent): (S22^-1 w)_i = z_i . u with z_i = L^-1 e_i.
    Returns (Z (m, q), beta (ns*pu, q), a (ns*pu, m), ns), float64 device tensors, block b = s*pu + j."""
    from .sepia.SepiaPredict import SepiaEmulatorPrediction
    num = model.num
    dummy = bool(model.data.dummy_x)
    cols = np.arange(1 if dummy else 0, num.p + num.q)
    if cols.size == 0:
        raise ValueError('the model has no inputs to analyse (q = 0)')
    x_pred = None if dummy else np.full((1, num.p), 0.5)
    t_pred = np.full((1, num.q), 0.5) if num.q else None
    proto = SepiaEmulatorPrediction(x_pred=x_pred, t_pred=t_pred, samples=samples, model=model, do_call=False)
    ns = proto._predictor()
    pred = proto._pred
    alpha, _ = pred.xval_solve(np.arange(num.m))
    a = alpha / pred.lamz[:, None]
    c = pred.torch.as_tensor(cols, device='cuda')
    return pred.X[:, c].contiguous(), pred.beta[:, c].contiguous(), a, ns


def gp_sensitivity_indices(model, samples, option='samples', pcvar=None, ngrid=21):
    """Exact first-order and total Sobol' indices and main-effect curves of the emulator's predictive mean, inputs
    independent and uniform on [0, 1] in the transformed scale (csrc/ggp_gp_sens.cu; no sampling, no bootstrap).

    option='samples': f = mu_sj for every posterior sample s and PC j: first, total (ns, pu, q); variance, mean (ns, pu);
    the spread over s is the index's posterior uncertainty.  option='mean': f_j = mean_s mu_sj, the function
    emulator_mean_function(model, samples) evaluates: first, total (pu, q); variance, mean (pu,).
    An input with beta = 0 (for every sample, in 'mean') does not enter f: its indices are exactly 0.
    pcvar (pu,): also general_first / general_total = sum_j pcvar_j S_jk, as PCA_saltelli_sensitivity_indices weights them.
    grid = linspace(0, 1, ngrid); main_effect (..., q, ngrid) = E[f | x_k = grid] in PC-weight units; for a scalar-output
    model also main_effect_native = main_effect * sd + mean.  Returns a dict of NumPy arrays."""
    if option not in ('samples', 'mean'):
        raise ValueError("option must be 'samples' or 'mean'")
    ngrid = int(ngrid)
    if ngrid < 1:
        raise ValueError('ngrid must be at least 1')
    pu = model.num.pu
    if pcvar is not None:
        pcvar = np.asarray(pcvar, dtype=np.float64).reshape(-1)
        if pcvar.size != pu:
            raise ValueError('pcvar must have one entry per PC (%d)' % pu)
    Z, beta, a, ns = emulator_expansion(model, samples)
    q = Z.shape[1]
    mode = 0 if option == 'samples' else 1
    if mode == 1:
        a = a / ns
    M, E0 = ops.gp_sens(Z, beta, a, ns, pu, mode)
    grid = np.linspace(0.0, 1.0, ngrid)
    me = ops.main_effects(Z, beta, a, ns, pu, grid, mode)
    lead = (ns, pu) if mode == 0 else (pu,)
    M = M.cpu().numpy().reshape(lead + (2 * q + 1,))
    E0 = E0.cpu().numpy().reshape(lead)
    zero = (beta == 0).cpu().numpy().reshape(ns, pu, q)
    if mode == 1:
        zero = np.all(zero, axis=0)
    e2 = (E0 * E0)[..., None]
    V = M[..., 2 * q] - E0 * E0
    first = np.where(zero, 0.0, (M[..., :q] - e2) / V[..., None])
    total = np.where(zero, 0.0, 1.0 - (M[..., q:2 * q] - e2) / V[..., None])
    out = dict(first=first, total=total, variance=V, mean=E0, grid=grid,
               main_effect=me.cpu().numpy().reshape(lead + (q, ngrid)))
    if pcvar is not None:
        out['general_first'] = np.einsum('...jk,j->...k', first, pcvar)
        out['general_total'] = np.einsum('...jk,j->...k', total, pcvar)
    if model.data.scalar_out:
        sd = model.data.sim_data
        out['main_effect_native'] = (out['main_effect'] * float(np.asarray(sd.orig_y_sd).reshape(-1)[0]) +
                                     float(np.asarray(sd.orig_y_mean).reshape(-1)[0]))
    return out
