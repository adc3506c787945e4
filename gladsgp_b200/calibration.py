"""Emulator-based calibration: the posterior of a simulator's inputs theta given observed outputs, with a fitted PC
emulator standing in for the simulator (DESIGN.md section 2 item 9).

The emulator's hyper-parameters stay at the posterior samples the user already has; theta has a uniform prior on a box.
The likelihood of the observed outputs O of y_obs under sample s combines the emulator's predictive error, the
PC-truncation residual (precision lamWOs per output, the sim-only model's own assumption) and the observation error:
    l_s(theta) = log N(r; K_O^T mu_s(theta), D_s + K_O^T diag(v_s(theta)) K_O),   D_s = diag(1/lamWOs_s + tau^2),
in standardized units, and l(theta) = log mean_s exp l_s(theta).  The n_o x n_o covariance is never formed: its
per-sample Woodbury terms G, b, c0 are computed once (_obs_terms), so a likelihood evaluation costs what the predictive
moments of pu PCs cost.  Many chains step together on the GPU: one ggp_predict_f64 launch for every chain's candidate
and one ggp_calib_step_f64 launch that evaluates l, decides and proposes the next candidate (csrc/ggp_calib.cu).

This is not SEPIA's Kennedy-O'Hagan calibration (no discrepancy, no lamOs); it claims no parity with it.  Treating the
truncation residual as independent over many correlated outputs (a whole field) makes the posterior overconfident; the
choice of obs_index and obs_sd is the user's.
"""
import math

import numpy as np

from . import _lib, diagnostics, ops

OBS_CHUNK_BYTES = 1 << 30     # scratch of _obs_terms: about 1 GiB of weighted basis columns at a time
POINT_CHUNK_BYTES = 1 << 30   # log_likelihood: predictive moments of about 1 GiB of points at a time
STEP_CHUNK = 256              # steps whose proposal and acceptance draws are generated together
MAX_DIM = 32                  # pu and q limit of csrc/ggp_calib.cu


def _check_t_model(model, what='calibration', verb='calibrate'):
    """A model whose inputs are all in t (no x_sim) and that has at least one (shared with gladsgp_b200.design)."""
    if not model.data.dummy_x:
        raise ValueError('%s needs a model without x_sim (its inputs are all in t)' % what)
    if model.num.q == 0:
        raise ValueError('the model has no inputs to %s (q = 0)' % verb)


def _check_model(model):
    num = model.num
    _check_t_model(model)
    if num.pu > MAX_DIM or num.q > MAX_DIM:
        raise ValueError('calibration supports pu <= %d and q <= %d (got pu = %d, q = %d)' % (MAX_DIM, MAX_DIM, num.pu, num.q))
    return num.q, num.pu


def _n_outputs(model):
    return 1 if model.data.scalar_out else int(np.asarray(model.data.sim_data.K).shape[1])


def _obs(model, y_obs, obs_index, obs_sd):
    """Validated observations -> (O (n_o,) int64, r (n_o,), tau (n_o,)) in standardized units (host float64)."""
    n_y = _n_outputs(model)
    y = np.asarray(y_obs, dtype=np.float64).reshape(-1)
    if obs_index is None:
        O = np.arange(n_y, dtype=np.int64)
    else:
        O = np.atleast_1d(np.asarray(obs_index))
        if O.ndim != 1 or O.size == 0 or O.dtype.kind not in 'iu':
            raise ValueError('obs_index must be a non-empty 1-D array of integer output indices')
        if O.min() < 0 or O.max() >= n_y:
            raise ValueError('obs_index out of range [0, %d)' % n_y)
        if np.unique(O).size != O.size:
            raise ValueError('obs_index holds an output twice')
        O = O.astype(np.int64)
    if y.size != O.size:
        raise ValueError('y_obs has %d values for %d observed outputs' % (y.size, O.size))
    sd_o = np.asarray(obs_sd, dtype=np.float64).reshape(-1)
    if sd_o.size not in (1, O.size):
        raise ValueError('obs_sd must be a scalar or have one value per observed output (%d), got %d' % (O.size, sd_o.size))
    if not np.all(sd_o >= 0):
        raise ValueError('obs_sd must be >= 0')
    sd = model.data.sim_data

    def at(v):
        v = np.asarray(v, dtype=np.float64).reshape(-1)
        return np.broadcast_to(v, (O.size,)) if v.size == 1 else v[O]
    ysd = at(sd.orig_y_sd)
    r = (y - at(sd.orig_y_mean)) / ysd
    tau = np.broadcast_to(sd_o, (O.size,)) / ysd
    return O, r, tau


def _obs_terms(model, samples, y_obs, obs_index, obs_sd):
    """Per-sample Woodbury terms of the observations, FP64 on the device:
    G (S, pu, pu) = K_O D_s^-1 K_O^T (made exactly symmetric), b (S, pu) = K_O D_s^-1 r,
    c0 (S,) = r^T D_s^-1 r + sum log D_s,ii + n_o log 2 pi, with D_s,ii = 1/lamWOs_s + tau_i^2.
    The outputs are taken in chunks of about OBS_CHUNK_BYTES of scratch (a full field has n_o = n_y)."""
    torch = _lib.require_cuda()
    O, r, tau = _obs(model, y_obs, obs_index, obs_sd)
    pu = model.num.pu
    sd = model.data.sim_data
    if model.data.scalar_out:
        K = torch.ones((1, 1), dtype=torch.float64, device='cuda')
    elif np.asarray(sd.K).dtype == np.float32:
        K = sd.K_device()
    else:
        K = torch.as_tensor(np.asarray(sd.K), device='cuda')
    lamWOs = torch.as_tensor(np.asarray(samples['lamWOs'], dtype=np.float64).reshape(-1), device='cuda')
    S = lamWOs.numel()
    G = torch.zeros((S, pu, pu), dtype=torch.float64, device='cuda')
    b = torch.zeros((S, pu), dtype=torch.float64, device='cuda')
    c0 = torch.zeros(S, dtype=torch.float64, device='cuda')
    Od = torch.as_tensor(O, device='cuda')
    rd = torch.as_tensor(np.ascontiguousarray(r), device='cuda')
    td = torch.as_tensor(np.ascontiguousarray(tau), device='cuda')
    chunk = max(1, OBS_CHUNK_BYTES // (8 * S * (pu + 3)))
    for i0 in range(0, O.size, chunk):
        i1 = min(O.size, i0 + chunk)
        Kc = K[:, Od[i0:i1]].to(torch.float64)                          # (pu, nc)
        D = 1.0 / lamWOs[:, None] + (td[i0:i1] ** 2)[None, :]              # (S, nc)
        W = 1.0 / D
        KW = Kc[None, :, :] * W[:, None, :]                                # (S, pu, nc)
        G += KW @ Kc.T
        b += KW @ rd[i0:i1]
        c0 += (W * rd[i0:i1][None, :] ** 2).sum(1) + torch.log(D).sum(1)
        del KW, W, D
    c0 += O.size * math.log(2.0 * math.pi)
    G = 0.5 * (G + G.transpose(1, 2))
    return G, b, c0


def _predictor(model, samples):
    """The cached-factor predictor of these samples (shared with SepiaEmulatorPrediction through model._pred_cache)."""
    from .sepia.SepiaPredict import SepiaEmulatorPrediction
    proto = SepiaEmulatorPrediction(t_pred=np.full((1, model.num.q), 0.5), samples=samples, model=model, do_call=False)
    ns = proto._predictor()
    return proto._pred, ns


def _to_trans(model, t):
    return np.asarray(model.data.transform_xt(t=np.asarray(t, dtype=np.float64))[1], dtype=np.float64)


def _designs(theta_trans):
    """(N, q) transformed inputs -> (N, 1 + q) prediction designs [0.5 (dummy x), theta]."""
    torch = _lib.require_cuda()
    X = torch.full((theta_trans.shape[0], theta_trans.shape[1] + 1), 0.5, dtype=torch.float64, device='cuda')
    X[:, 1:] = theta_trans
    return X


def log_likelihood(model, samples, y_obs, obs_index=None, obs_sd=0.0, t=None, per_sample=False):
    """l(theta) at the native-unit inputs t (N, q) for profile and grid plots.  y_obs (n_o,) native units at the outputs
    obs_index (default: every output); obs_sd scalar or (n_o,), native units.  Returns l (N,) [, l_s (S, N)] as NumPy
    float64 arrays."""
    q, pu = _check_model(model)
    _obs(model, y_obs, obs_index, obs_sd)
    if t is None:
        raise TypeError('t is required')
    t = np.asarray(t, dtype=np.float64)
    t = t.reshape(1, -1) if t.ndim == 1 else t
    if t.ndim != 2 or t.shape[1] != q:
        raise ValueError('t must be (N, %d)' % q)
    torch = _lib.require_cuda()
    G, b, c0 = _obs_terms(model, samples, y_obs, obs_index, obs_sd)
    pred, S = _predictor(model, samples)
    tt = torch.as_tensor(_to_trans(model, t), device='cuda')
    N = tt.shape[0]
    chunk = max(1, POINT_CHUNK_BYTES // (16 * S * pu))
    ll = np.empty(N)
    ll_s = np.empty((S, N)) if per_sample else None
    for i0 in range(0, N, chunk):
        i1 = min(N, i0 + chunk)
        mean, var = pred.predict(_designs(tt[i0:i1]))
        out = ops.calib_loglik(mean, var, G, b, c0, want_per_sample=per_sample)
        if per_sample:
            ll[i0:i1] = out[0].cpu().numpy()
            ll_s[:, i0:i1] = out[1].cpu().numpy()
        else:
            ll[i0:i1] = out.cpu().numpy()
    return (ll, ll_s) if per_sample else ll


def _bounds(model, bounds):
    """-> (lo, hi) native (q,), (lo, hi) transformed (q,); default: the training design's column min / max."""
    q = model.num.q
    if bounds is None:
        tn = np.asarray(model.data.sim_data.t, dtype=np.float64)
        lo, hi = tn.min(axis=0), tn.max(axis=0)
    else:
        bd = np.asarray(bounds, dtype=np.float64)
        if bd.shape != (2, q):
            raise ValueError('bounds must be (2, %d): lower and upper native values of every input' % q)
        lo, hi = bd[0], bd[1]
    if not np.all(lo < hi):
        raise ValueError('bounds: every lower bound must be below its upper bound')
    return lo, hi, _to_trans(model, lo[None])[0], _to_trans(model, hi[None])[0]


def burnin_proposal(states, step):
    """Proposal factor after burn-in: chol((2.38^2 / q_free) Sigma) on the free inputs (step > 0), Sigma the covariance
    (ddof 1) of the states (n, C, q) of every chain; zero rows and columns for fixed inputs.  Falls back to diag(step)
    when the Cholesky fails.  states: float64 CUDA tensor; returns a (q, q) float64 CUDA tensor."""
    torch = _lib.require_cuda()
    step = np.asarray(step, dtype=np.float64)
    q = step.size
    free = np.nonzero(step > 0)[0]
    L = torch.diag(torch.as_tensor(step, device='cuda'))
    if free.size == 0:
        return L
    X = states[:, :, torch.as_tensor(free, device='cuda')].reshape(-1, free.size)
    if X.shape[0] < 2:
        return L
    Xc = X - X.mean(dim=0)
    Sig = (Xc.T @ Xc) / (X.shape[0] - 1) * (2.38 ** 2 / free.size)
    Lf, info = torch.linalg.cholesky_ex(Sig)
    if int(info) != 0 or not bool(torch.isfinite(Lf).all()):
        return L
    L = torch.zeros((q, q), dtype=torch.float64, device='cuda')
    fi = torch.as_tensor(free, device='cuda')
    L[fi[:, None], fi[None, :]] = Lf
    return L


def calibrate(model, samples, y_obs, obs_index=None, obs_sd=0.0, bounds=None, n_chains=1024, n_burn=1000, n_steps=1000,
              step=0.1, theta0=None, seed=None, replay=None, device=False):
    """Posterior of the inputs theta given y_obs (native units) at the outputs obs_index, with a uniform prior on the box
    `bounds` ((2, q) native; default: the training design's range), sampled by n_chains random-walk Metropolis chains.

    Burn-in (n_burn steps) proposes theta + diag(step) z in transformed units (step scalar or (q,); 0 fixes an input at
    its initial value).  At its end the proposal becomes chol((2.38^2 / q_free) Sigma), Sigma the covariance of all
    chains' states over the second half of burn-in on the free inputs (diag(step) if that Cholesky fails).  Initial
    states: theta0 (native, (q,) or (n_chains, q)) or uniform in the box.  The initial states, then the normal z (T, C, q)
    and log-uniform (T, C) draws of the T = n_burn + n_steps steps, in chunks of STEP_CHUNK steps, come from one device
    torch.Generator seeded with `seed`; replay=dict(z=, logu=[, theta0=]) supplies them instead.

    Returns dict(theta (n_steps, C, q) native, theta_trans, loglik (n_steps, C), accepted (n_steps, C), accept_rate (C,),
    proposal_chol (q, q), bounds (2, q) native, diagnostics = diagnostics.chain_diagnostics(theta_trans, loglik)); the
    arrays are NumPy unless device=True (then theta, theta_trans, loglik, accepted are CUDA tensors)."""
    q, pu = _check_model(model)
    _obs(model, y_obs, obs_index, obs_sd)
    lo_n, hi_n, lo_t, hi_t = _bounds(model, bounds)
    C, n_burn, n_steps = int(n_chains), int(n_burn), int(n_steps)
    if C < 1 or n_burn < 0 or n_steps < 1:
        raise ValueError('need n_chains >= 1, n_burn >= 0 and n_steps >= 1')
    step = np.broadcast_to(np.asarray(step, dtype=np.float64).reshape(-1), (q,)).copy()
    if not np.all(step >= 0):
        raise ValueError('step must be >= 0')
    T = n_burn + n_steps
    if theta0 is None and replay is not None:
        theta0 = replay.get('theta0')
    th0 = None
    if theta0 is not None:
        th0 = _to_trans(model, np.broadcast_to(np.asarray(theta0, dtype=np.float64), (C, q)))
        if not np.all((th0 >= lo_t) & (th0 <= hi_t)):
            raise ValueError('theta0 lies outside the bounds')
    if replay is not None:
        zr = np.asarray(replay['z'], dtype=np.float64)
        ur = np.asarray(replay['logu'], dtype=np.float64)
        if zr.shape != (T, C, q) or ur.shape != (T, C):
            raise ValueError('replay z must be (%d, %d, %d) and logu (%d, %d)' % (T, C, q, T, C))
    torch = _lib.require_cuda()
    dev = 'cuda'
    G, b, c0 = _obs_terms(model, samples, y_obs, obs_index, obs_sd)
    pred, S = _predictor(model, samples)
    lo = torch.as_tensor(lo_t, device=dev)
    hi = torch.as_tensor(hi_t, device=dev)
    gen = None
    if replay is None:
        gen = torch.Generator(device=dev)
        if seed is None:
            gen.seed()
        else:
            gen.manual_seed(int(seed))
    if th0 is not None:
        theta = torch.as_tensor(np.ascontiguousarray(th0), device=dev)
    else:
        theta = lo + (hi - lo) * torch.rand((C, q), generator=gen, dtype=torch.float64, device=dev)
    if replay is not None:
        zr = torch.as_tensor(zr, device=dev)
        ur = torch.as_tensor(ur, device=dev)
    draws = {}

    def z_logu(t):
        """Draws of step t; the generator fills a chunk of STEP_CHUNK steps at a time, z before logu."""
        if replay is not None:
            return zr[t], ur[t]
        c = t // STEP_CHUNK
        if c not in draws:
            draws.clear()
            k = min(STEP_CHUNK, T - c * STEP_CHUNK)
            z = torch.randn((k, C, q), generator=gen, dtype=torch.float64, device=dev)
            u = torch.log(torch.rand((k, C), generator=gen, dtype=torch.float64, device=dev))
            draws[c] = (z, u)
        z, u = draws[c]
        return z[t - c * STEP_CHUNK], u[t - c * STEP_CHUNK]

    L = torch.diag(torch.as_tensor(step, device=dev))
    Xp = _designs(theta)
    mean, var = pred.predict(Xp)
    ll = ops.calib_loglik(mean, var, G, b, c0)
    rec_theta = torch.empty((T, C, q), dtype=torch.float64, device=dev)
    rec_ll = torch.empty((T, C), dtype=torch.float64, device=dev)
    rec_acc = torch.empty((T, C), dtype=torch.uint8, device=dev)
    Xp[:, 1:] = theta + z_logu(0)[0] @ L.T
    for t in range(T):
        logu = z_logu(t)[1]
        adapt = t == n_burn - 1
        z_next = z_logu(t + 1)[0] if t + 1 < T and not adapt else None
        mean, var = pred.predict(Xp)
        ops.calib_step(mean, var, G, b, c0, Xp, lo, hi, L, z_next, logu, theta, ll, rec_theta[t], rec_ll[t], rec_acc[t])
        if adapt:
            L = burnin_proposal(rec_theta[n_burn // 2:n_burn], step).contiguous()
            if t + 1 < T:
                Xp[:, 1:] = theta + z_logu(t + 1)[0] @ L.T
    tt = rec_theta[n_burn:]
    lp = rec_ll[n_burn:]
    acc = rec_acc[n_burn:].to(torch.bool)
    diag = diagnostics.chain_diagnostics(tt, lp)
    span = torch.as_tensor(model.data.sim_data.orig_t_max - model.data.sim_data.orig_t_min, device=dev).reshape(-1)
    tmin = torch.as_tensor(model.data.sim_data.orig_t_min, device=dev).reshape(-1)
    th_native = tt * span + tmin
    out = dict(theta=th_native, theta_trans=tt, loglik=lp, accepted=acc,
               accept_rate=acc.to(torch.float64).mean(dim=0).cpu().numpy(), proposal_chol=L.cpu().numpy(),
               bounds=np.stack([lo_n, hi_n]), diagnostics=diag)
    if not device:
        for k in ('theta', 'theta_trans', 'loglik', 'accepted'):
            out[k] = out[k].cpu().numpy()
    return out
