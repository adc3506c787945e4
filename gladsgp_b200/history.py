"""History matching: the simulator inputs that observed outputs rule out, by the implausibility of the emulator's
prediction at each output (DESIGN.md section 2 item 11; Vernon, Goldstein and Bower 2010).

For a point t the emulator's posterior-predictive mixture over the samples gives each observed output i a mean and a
variance; with the observation and model-discrepancy variances added,
    I_i(t) = |y_obs,i - E y_i(t)| / sqrt(Var y_i(t) + obs_sd_i^2 + disc_sd_i^2),
and t is ruled out when the `order`-th largest I_i exceeds the cutoff (order 1: the maximum over the outputs; 2 or 3
tolerate that many outliers).  Unlike calibration, no independence between outputs is assumed, so the observations may
be a whole field.  The points not ruled out (nroy) are the candidates of the next wave, e.g. for design.next_runs.

The predictive moments come from ggp_predict_f64 on the prediction factors cached with the model (model._pred_cache,
shared with calibration and design); the (point, output) products run on the FP64 tensor cores and are never stored
(csrc/ggp_hm.cu).
"""
import numpy as np

from . import _lib, ops
from .calibration import _check_model, _designs, _obs, _predictor, _to_trans
from .design import _points

POINT_CHUNK_BYTES = 1 << 30   # predictive moments of about 1 GiB of points at a time
MAX_ORDER = 8                 # largest `order` of csrc/ggp_hm.cu


def _sd(v, name, n_o):
    """A scalar or (n_o,) native-unit standard deviation, finite and >= 0 -> (n_o,) float64."""
    v = np.asarray(v, dtype=np.float64).reshape(-1)
    if v.size not in (1, n_o):
        raise ValueError('%s must be a scalar or have one value per observed output (%d), got %d' % (name, n_o, v.size))
    if not np.all(np.isfinite(v)) or np.any(v < 0):
        raise ValueError('%s must be finite and >= 0' % name)
    return np.broadcast_to(v, (n_o,))


def history_match(model, samples, y_obs, t, obs_index=None, obs_sd=0.0, disc_sd=0.0, order=1, cutoff=3.0):
    """Implausibility of the native-unit inputs t (N, q) against y_obs (n_o,) native units at the outputs obs_index
    (default: every output).  obs_sd and disc_sd (observation and model-discrepancy standard deviations, native units):
    scalars or (n_o,).  order: an integer in [1, min(8, n_o)]; cutoff: finite and > 0.

    Returns dict(impl (N, order) float64: each point's `order` largest I_i in descending order, n_over (N,) int64: the
    number of outputs with I_i > cutoff, nroy (N,) bool: impl[:, order - 1] <= cutoff (not ruled out), nroy_fraction,
    order, cutoff)."""
    q, pu = _check_model(model)
    O, r, tau = _obs(model, y_obs, obs_index, obs_sd)
    n_o = O.size
    _sd(obs_sd, 'obs_sd', n_o)
    disc = _sd(disc_sd, 'disc_sd', n_o)
    if isinstance(order, (bool, np.bool_)) or int(order) != order or not 1 <= int(order) <= min(MAX_ORDER, n_o):
        raise ValueError('order must be an integer in [1, min(%d, n_o)] = [1, %d]' % (MAX_ORDER, min(MAX_ORDER, n_o)))
    order = int(order)
    cutoff = float(cutoff)
    if not np.isfinite(cutoff) or cutoff <= 0:
        raise ValueError('cutoff must be finite and > 0')
    t = _points(t, 't', q)
    torch = _lib.require_cuda()
    sd = model.data.sim_data
    ysd = np.asarray(sd.orig_y_sd, dtype=np.float64).reshape(-1)
    ysd = np.broadcast_to(ysd, (n_o,)) if ysd.size == 1 else ysd[O]
    delta = disc / ysd
    lamWOs = np.asarray(samples['lamWOs'], dtype=np.float64).reshape(-1)
    rho = float(np.mean(1.0 / lamWOs))
    c = rho + tau * tau + delta * delta
    if model.data.scalar_out:
        K_O = torch.ones((1, 1), dtype=torch.float64, device='cuda')
    else:
        K = sd.K_device() if np.asarray(sd.K).dtype == np.float32 else torch.as_tensor(np.asarray(sd.K), device='cuda')
        K_O = K[:, torch.as_tensor(O, device='cuda')].to(torch.float64).contiguous()
    rd = torch.as_tensor(np.ascontiguousarray(r), device='cuda')
    cd = torch.as_tensor(np.ascontiguousarray(c), device='cuda')
    pred, S = _predictor(model, samples)
    tt = torch.as_tensor(_to_trans(model, t), device='cuda')
    N = tt.shape[0]
    chunk = max(1, POINT_CHUNK_BYTES // (16 * S * pu))
    impl = np.empty((N, order))
    n_over = np.empty(N, dtype=np.int64)
    for i0 in range(0, N, chunk):
        i1 = min(N, i0 + chunk)
        mean, var = pred.predict(_designs(tt[i0:i1]))
        im, no = ops.hm_impl(mean, var, K_O, rd, cd, order, cutoff)
        impl[i0:i1] = im.cpu().numpy()
        n_over[i0:i1] = no.cpu().numpy()
    nroy = impl[:, order - 1] <= cutoff
    return dict(impl=impl, n_over=n_over, nroy=nroy, nroy_fraction=float(nroy.mean()), order=order, cutoff=cutoff)
