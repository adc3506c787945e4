"""Emulator Jacobians: the gradient of the emulator's prediction at given simulator inputs, with its posterior
uncertainty (DESIGN.md section 2 item 13).

For a (sample, PC) block the gradient of the predictive mean, the joint posterior covariance of the value and its
gradient, and the gradient of the predictive variance (d v / d t_k = 2 Cov(f, d_k f)) come from one triangular solve
with q + 1 right-hand sides per design on the prediction factors cached with the model (model._pred_cache, shared with
SepiaEmulatorPrediction, calibration, history matching and design; csrc/ggp_jacobian.cu).  This replaces 2q + 1
prediction calls of central differences, without their step-size error, and gives the gradient an uncertainty.

Every result is in native input units: a transformed-scale derivative is divided by the input's native span
(orig_t_max - orig_t_min, 1 for an untransformed column), a covariance on both sides.
"""
import numpy as np

from . import _lib
from .calibration import _check_t_model, _designs, _predictor, _to_trans
from .design import _points
from .sensitivity import _input_span

POINT_CHUNK_BYTES = 1 << 30     # Jacobian-kernel output of about 1 GiB of points at a time
OUTPUT_CHUNK_BYTES = 1 << 30    # field products: about 1 GiB of (sample, point, input, output) values at a time
FIELD_SAMPLES_BYTES = 1 << 34   # largest per-sample field Jacobian (S, N, n_O, q) returned by option='samples'
MAX_Q = 31                      # differentiated inputs of csrc/ggp_jacobian.cu: q + 1 rows fit one warp's 32


def _outputs(model, outputs):
    """Validated output indices (host int64 array) or None for every output, and their number."""
    ny = 1 if model.data.scalar_out else int(np.asarray(model.data.sim_data.K).shape[1])
    if outputs is None:
        return None, ny
    O = np.atleast_1d(np.asarray(outputs))
    if O.ndim != 1 or O.size == 0 or O.dtype.kind not in 'iu' or O.min() < 0 or O.max() >= ny:
        raise ValueError('outputs must be a non-empty list of output indices in [0, %d)' % ny)
    return O.astype(np.int64), O.size


def _coef(model, O):
    """(pu, n_O) = K_O diag(orig_y_sd_O) and orig_y_mean_O, float64 on the device (K = [[1]] for a scalar-output
    model); O None: every output."""
    torch = _lib.require_cuda()
    sd = model.data.sim_data
    K = np.ones((1, 1)) if model.data.scalar_out else np.asarray(sd.K)
    ny = K.shape[1]
    ysd = np.broadcast_to(np.asarray(sd.orig_y_sd, dtype=np.float64).reshape(-1), (ny,))
    ymu = np.broadcast_to(np.asarray(sd.orig_y_mean, dtype=np.float64).reshape(-1), (ny,))
    if O is not None:
        K, ysd, ymu = K[:, O], ysd[O], ymu[O]
    Kd = torch.as_tensor(np.ascontiguousarray(K), device='cuda').to(torch.float64)
    return (Kd * torch.as_tensor(np.ascontiguousarray(ysd), device='cuda')[None, :],
            torch.as_tensor(np.ascontiguousarray(ymu), device='cuda'))


def _mixture(mean, var, grad, grad_var, gcov):
    """Law of total (co)variance over the sample axis 0; gcov: (S, ..., q, q) or the diagonal (S, ..., q)."""
    S = mean.shape[0]
    m, g = mean.mean(0), grad.mean(0)
    dm, dg = mean - m, grad - g
    out = dict(mean=m, grad=g, var=var.mean(0) + (dm * dm).mean(0),
               grad_var=grad_var.mean(0) + (2.0 / S) * (dm.unsqueeze(-1) * dg).sum(0))
    if gcov.dim() == grad.dim() + 1:
        out['grad_cov'] = gcov.mean(0) + (dg.unsqueeze(-1) * dg.unsqueeze(-2)).sum(0) / S
    else:
        out['grad_sd2'] = gcov.mean(0) + (dg * dg).mean(0)
    return out


def emulator_jacobian(model, samples, t, target='pc', outputs=None, option='samples', full=True, device=False):
    """Gradient of the emulator's prediction with respect to the native inputs t (N, q) of a model without x_sim,
    q <= 31, at the posterior samples `samples` (the prediction of SepiaEmulatorPrediction with addResidVar=False).

    target='pc', option='samples': per (sample, point, PC) mean, var (S, N, pu); grad (S, N, pu, q) = d mu / d t;
    grad_var (S, N, pu, q) = d v / d t; with full, grad_cov (S, N, pu, q, q), the posterior covariance of the gradient
    of f, else grad_sd (S, N, pu, q), its marginal sds.  option='mean': the posterior mixture over the samples,
    mean = E_s mu_s, var = E_s v_s + Var_s mu_s, grad = E_s grad mu_s, grad_var = E_s d v_s + (2/S) sum_s (mu_s - mean)
    (grad mu_s - grad), grad_cov = E_s Sigma_s + Cov_s(grad mu_s) (or grad_sd), each without the S axis.
    target=c, an array (pu,): the same for the linear quantity sum_j c_j f_j (the PC axis dropped).
    target='field': the native-unit outputs `outputs` (default: all) y_c = sum_j K_jc orig_y_sd_c f_j + orig_y_mean_c:
    mean (S, N, n_O) or (N, n_O), jacobian dy/dt (S, N, n_O, q) or (N, n_O, q), and grad_sd of the same shape, the
    marginal posterior sd of every dy_c/dt_k (for 'mean' the mixture sd).  The PC-truncation residual (precision lamWOs)
    is white noise: it has no derivative and does not enter grad_sd.  `full` does not apply to 'field'.
    var and every sd are clamped at 0.  Returns a dict of NumPy arrays, or of CUDA tensors with device=True."""
    _check_t_model(model, 'emulator_jacobian', 'differentiate')
    num = model.num
    q, pu = num.q, num.pu
    if q > MAX_Q:
        raise ValueError('emulator_jacobian supports q <= %d inputs (got q = %d)' % (MAX_Q, q))
    if option not in ('samples', 'mean'):
        raise ValueError("option must be 'samples' or 'mean'")
    c = None
    if isinstance(target, str):
        if target not in ('pc', 'field'):
            raise ValueError("target must be 'pc', 'field' or an array of pu coefficients")
    else:
        c = np.asarray(target, dtype=np.float64).reshape(-1)
        if c.size != pu or not np.all(np.isfinite(c)):
            raise ValueError('target coefficients must be %d finite values (one per PC)' % pu)
        target = 'linear'
    if outputs is not None and target != 'field':
        raise ValueError("outputs applies to target='field' only")
    t = _points(t, 't', q)
    N = t.shape[0]
    S = np.asarray(samples['lamUz']).reshape(-1, pu).shape[0]
    if target == 'field':
        O, n_O = _outputs(model, outputs)
        if option == 'samples' and S * N * n_O * q * 8 > FIELD_SAMPLES_BYTES:
            raise ValueError("target='field' with option='samples' would return %d x %d x %d x %d values (%.3g GB > "
                             "%.3g GB): use option='mean', fewer points or fewer outputs"
                             % (S, N, n_O, q, S * N * n_O * q * 8e-9, FIELD_SAMPLES_BYTES * 1e-9))
        full = False
    torch = _lib.require_cuda()
    coef = ymu = None
    if target == 'field':
        coef, ymu = _coef(model, O)
    pred, S = _predictor(model, samples)
    span = torch.as_tensor(_input_span(model), device='cuda')
    cd = None if c is None else torch.as_tensor(c, device='cuda')
    tt = torch.as_tensor(_to_trans(model, t), device='cuda')
    per_pt = 8 * S * pu * ((q + 1) + ((q + 1) ** 2 if full else 2 * q + 1))
    chunk = max(1, POINT_CHUNK_BYTES // per_pt)
    parts = []
    for i0 in range(0, N, chunk):
        i1 = min(N, i0 + chunk)
        n = i1 - i0
        mv, cv = pred.jacobian(_designs(tt[i0:i1]), 1, full=full)
        mv = mv.reshape(S, pu, n, q + 1).transpose(1, 2)                      # (S, n, pu, q+1)
        mean, grad = mv[..., 0], mv[..., 1:] / span
        if full:
            cv = cv.reshape(S, pu, n, q + 1, q + 1).transpose(1, 2)
            var, grad_var = cv[..., 0, 0], 2.0 * cv[..., 1:, 0] / span
            gcov = cv[..., 1:, 1:] / (span[:, None] * span[None, :])
        else:
            cv = cv.reshape(S, pu, n, 2 * q + 1).transpose(1, 2)
            var, grad_var = cv[..., 0], 2.0 * cv[..., 1:q + 1] / span
            gcov = cv[..., q + 1:] / (span * span)                            # the diagonal only
        if target == 'field':
            parts.append(_field_part(mean, grad, gcov, coef, ymu, option))
            continue
        if target == 'linear':
            c2 = cd * cd
            mean, var = mean @ cd, var @ c2
            grad = torch.einsum('snjk,j->snk', grad, cd)
            grad_var = torch.einsum('snjk,j->snk', grad_var, c2)
            gcov = torch.einsum('snjkl,j->snkl', gcov, c2) if full else torch.einsum('snjk,j->snk', gcov, c2)
        if option == 'mean':
            r = _mixture(mean, var, grad, grad_var, gcov)
        else:
            r = dict(mean=mean, var=var, grad=grad, grad_var=grad_var)
            r['grad_cov' if full else 'grad_sd2'] = gcov
        r['var'] = torch.clamp(r['var'], min=0.0)
        if 'grad_sd2' in r:
            r['grad_sd'] = torch.sqrt(torch.clamp(r.pop('grad_sd2'), min=0.0))
        parts.append({k: v.contiguous() for k, v in r.items()})
    axis = 1 if option == 'samples' else 0
    out = {k: torch.cat([p[k] for p in parts], dim=axis) for k in parts[0]}
    if device:
        return out
    return {k: v.cpu().numpy() for k, v in out.items()}


def _field_part(mean, grad, gd2, coef, ymu, option):
    """Native-output mean, Jacobian and its marginal sd at one chunk of points, in chunks of outputs; grad (S, n, pu, q),
    gd2 (S, n, pu, q) the variances of the gradient entries (native input units), coef (pu, n_O)."""
    torch = _lib.require_cuda()
    S, n, pu, q = grad.shape
    n_O = coef.shape[1]
    oc = max(1, OUTPUT_CHUNK_BYTES // (8 * S * n * q))
    gT = grad.transpose(2, 3)                                                  # (S, n, q, pu)
    vT = gd2.transpose(2, 3)
    if option == 'mean':
        gm = gT.mean(0)
        dT = gT - gm
    ys, Js, sds = [], [], []
    for o0 in range(0, n_O, oc):
        cf = coef[:, o0:o0 + oc]
        y = mean @ cf + ymu[o0:o0 + oc]                                        # (S, n, n_Oc)
        V = vT @ (cf * cf)                                                     # (S, n, q, n_Oc)
        if option == 'samples':
            J = gT @ cf
        else:
            y = y.mean(0)
            J = gm @ cf
            B = dT @ cf                                                        # between-sample deviations
            V = V.mean(0) + (B * B).mean(0)
            del B
        ys.append(y)
        Js.append(J.transpose(-1, -2))
        sds.append(torch.sqrt(torch.clamp(V, min=0.0)).transpose(-1, -2))
        del V
    return dict(mean=torch.cat(ys, -1).contiguous(), jacobian=torch.cat(Js, -2).contiguous(),
                grad_sd=torch.cat(sds, -2).contiguous())
