"""SepiaEmulatorPrediction mirror (SURVEY.md 8a rows a7-a8, A.7; 8b).

Callers (always t_pred= / samples= / model= keywords):
/root/reference/experiments/synthetic/analysis/assess_all_models.py:489-492,510-513;
plot_test_error.py:77-80; time_predictions.py:76-79; sensitivity_indices.py:85-88;
fit_scalar_models.py:481-483; include_trunc_error.py:86-88.

Differences from the reference implementation, all behind the same results:
* every (sample, PC) covariance is factored ONCE per prediction object (SEPIA re-solves S22 for
  every call) and test designs are pushed through the cached factor on the GPU;
* the factors are kept with the model and re-used by later prediction objects built from the same samples
  (the reference's callers build one object per batch of test designs, assess_all_models.py:476-492);
* the multivariate-normal realisation uses a Cholesky factor of each per-PC covariance block (positive
  definite: Sigma >= I / lamWs) instead of one SVD of the block-diagonal matrix: same distribution, and
  the same np.random.normal draws are consumed, but a realisation is not bit-comparable with SEPIA's
  (SVD sign ambiguity, SURVEY 7.2); parity is asserted on mu / Sigma (storeMuSigma=True).
"""
import warnings

import numpy as np

from .. import ops, _lib

CHOL_DRAW_MAX_N = 16384   # ggp_chol_draw_f64 keeps an n-vector and n/8 offsets in shared memory
MAX_JOINT = 1024      # above this many designs per call the joint covariance is not formed unless joint=True is passed
FIELD_CHUNK_BYTES = 1 << 30   # get_y_error_stats beyond the fused kernels: mean / limit fields of at most ~1 GiB at a time


def _samples_key(samples, model, add_resid):
    """Identity of a (model, posterior samples) pair: the callers of the reference construct one prediction object per
    batch of test designs with the same samples (assess_all_models.py:476-492), so the nsamp x pu factorisations are kept
    with the model and re-used while the sample arrays are unchanged (same objects, same shapes, same checksums)."""
    parts = [id(model), bool(add_resid)]
    for k in ('betaU', 'lamUz', 'lamWs', 'lamWOs'):
        a = np.asarray(samples[k])
        parts += [k, a.shape, a.dtype.str, float(np.sum(a, dtype=np.float64)), float(np.sum(np.square(a, dtype=np.float64)))]
    return tuple(parts)


def _pinned(owner, name, numel):
    """Cached page-locked float64 staging buffer kept with the predictor (page-locking per call costs more than the copy)."""
    import torch
    pool = owner.__dict__.setdefault('_pin', {})
    buf = pool.get(name)
    if buf is None or buf.numel() < numel:
        buf = torch.empty(max(int(numel), 1), dtype=torch.float64).pin_memory()
        pool[name] = buf
    return buf[:numel]


class SepiaPrediction:
    def __init__(self, x_pred=None, samples=None, model=None, t_pred=None, addResidVar=False,
                 storeRlz=True, storeMuSigma=False):
        if samples is None or model is None:
            raise TypeError('samples and model are required')
        if x_pred is None and t_pred is None:
            raise TypeError('at least one of x_pred, t_pred is required')
        data = model.data
        sd = data.sim_data
        if t_pred is not None:
            t_pred = np.asarray(t_pred)
            if t_pred.ndim == 1:
                t_pred = t_pred[None, :]
        npred = (t_pred if t_pred is not None else np.asarray(x_pred)).shape[0]
        if x_pred is None:
            if not data.dummy_x:
                raise TypeError('x_pred is required for a model built with x_sim')
            x_pred = 0.5 * np.ones((npred, 1))
        x_pred = np.asarray(x_pred)
        if x_pred.ndim == 1:
            x_pred = x_pred[:, None]
        if x_pred.shape[1] != model.num.p or (t_pred is not None and t_pred.shape[1] != model.num.q):
            raise ValueError('x_pred / t_pred have the wrong number of columns')
        if (t_pred is None) != (model.num.q == 0):
            raise ValueError('t_pred must be given iff the model has t inputs')
        self.model = model
        self.xpred, self.t_pred = x_pred, t_pred
        xt, tt = data.transform_xt(x=x_pred, t=t_pred)
        if data.dummy_x:
            xt = 0.5 * np.ones((npred, 1))
        cols = [np.asarray(xt, dtype=np.float64)]
        if tt is not None:
            cols.append(np.asarray(tt, dtype=np.float64))
        self.xpredt = np.ascontiguousarray(np.concatenate(cols, axis=1))
        self.samples = samples
        self.addResidVar = addResidVar
        self.storeRlz = storeRlz
        self.storeMuSigma = storeMuSigma
        self.w = None
        self.mu = None
        self.sigma = None


class SepiaEmulatorPrediction(SepiaPrediction):
    def __init__(self, x_pred=None, samples=None, model=None, t_pred=None, addResidVar=False,
                 storeRlz=True, storeMuSigma=False, do_call=True, joint=None):
        super().__init__(x_pred=x_pred, samples=samples, model=model, t_pred=t_pred, addResidVar=addResidVar,
                         storeRlz=storeRlz, storeMuSigma=storeMuSigma)
        self.joint = joint
        if do_call:
            self._w_pred()

    # ------------------------------------------------------------------ wPred
    def _blocks(self):
        num = self.model.num
        d, pu, m = num.p + num.q, num.pu, num.m
        s = self.samples
        lamUz = np.asarray(s['lamUz'], dtype=np.float64).reshape(-1, pu)
        lamWs = np.asarray(s['lamWs'], dtype=np.float64).reshape(-1, pu)
        lamWOs = np.asarray(s['lamWOs'], dtype=np.float64).reshape(-1, 1)
        ns = lamUz.shape[0]
        bU = np.asarray(s['betaU'], dtype=np.float64).reshape(ns, -1)
        if bU.shape[1] != d * pu:
            raise ValueError('samples["betaU"] must be flat (n, %d); got %s' % (d * pu, np.asarray(s['betaU']).shape))
        beta = bU.reshape(ns, pu, d).reshape(ns * pu, d)          # row (s, j) = betaU[:, j] (Fortran flat)
        lamz = lamUz.reshape(-1)
        dadd = (1.0 / (num.LamSim[None, :] * lamWOs) + 1.0 / lamWs).reshape(-1)
        s11 = (1.0 / lamUz + 1.0 / lamWs)
        if self.addResidVar:
            s11 = s11 + 1.0 / (num.LamSim[None, :] * lamWOs)
        W = np.broadcast_to(self.model._w_pcs[None], (ns, pu, m)).reshape(ns * pu, m)
        return ns, beta, lamz, dadd, s11.reshape(-1), np.ascontiguousarray(W)

    def _predictor(self):
        """self._pred: the factored (sample, PC) blocks of these samples, from the model's cache or built and cached.
        Returns the number of samples."""
        num = self.model.num
        key = _samples_key(self.samples, self.model, self.addResidVar)
        cached = getattr(self.model, '_pred_cache', None)
        if cached is not None and cached[0] == key:
            self._pred, ns = cached[1], cached[2]
        else:
            ns, beta, lamz, dadd, s11, W = self._blocks()
            self._pred = ops.Predictor(num.zt, W, beta, lamz, dadd, s11)
            bad = int((self._pred.info != 0).sum().item())
            if bad:
                raise np.linalg.LinAlgError('%d of %d (sample, PC) covariance matrices are not positive definite' %
                                            (bad, ns * num.pu))
            self.model._pred_cache = (key, self._pred, ns)
        return ns

    def _w_pred(self):
        torch = _lib.require_cuda()
        num = self.model.num
        pu = num.pu
        npred = self.xpredt.shape[0]
        ns = self._predictor()
        if self.joint is None and npred > MAX_JOINT:
            # SEPIA draws one joint realisation over all designs of a call; above MAX_JOINT designs the npred x npred blocks
            # (nsamp*pu of them) are not formed unless asked for: say so instead of changing the distribution silently
            if self.storeMuSigma:
                raise ValueError('storeMuSigma with %d > %d designs per call needs the joint covariance: pass joint=True '
                                 '(memory: nsamp*pu*npred^2 doubles) or joint=False for marginal variances' % (npred, MAX_JOINT))
            warnings.warn('SepiaEmulatorPrediction: %d designs in one call (> %d): realisations are drawn from the marginal '
                          'predictive distributions (no cross-design covariance); pass joint=True for SEPIA\'s joint draw or '
                          'split the designs into smaller calls' % (npred, MAX_JOINT), RuntimeWarning, stacklevel=3)
        joint = self.joint if self.joint is not None else (npred <= MAX_JOINT)
        # the designs go up once, through a page-locked buffer: a pageable copy issued between the two launches below would
        # hold the host until the first kernel has finished, and the np.random draws further down would start that much later
        xh = np.ascontiguousarray(self.xpredt, dtype=np.float64)
        xst = _pinned(self._pred, 'xp', xh.size)
        xst.copy_(torch.from_numpy(xh.reshape(-1)))
        xpd = xst.to('cuda', non_blocking=True).reshape(xh.shape)
        if joint and npred > 1:
            mean, var, V = self._pred.predict(xpd, want_V=True)
            Sig = self._pred.pred_cov(xpd, V)                         # (B, n, n)
            del V
        else:
            mean, var = self._pred.predict(xpd)
            Sig = None
        self.launches = 2 + (1 if Sig is not None else 0)
        mean = mean.reshape(ns, pu, npred)
        if self.storeMuSigma:
            self.mu = mean.reshape(ns, pu * npred).cpu().numpy()
            self.sigma = np.zeros((ns, pu * npred, pu * npred))
            blk = (Sig.reshape(ns, pu, npred, npred).cpu().numpy() if Sig is not None
                   else np.einsum('spt,tu->sptu', var.reshape(ns, pu, npred).cpu().numpy(), np.eye(npred)))
            for j in range(pu):
                sl = slice(j * npred, (j + 1) * npred)
                self.sigma[:, sl, sl] = blk[:, j]
        if self.storeRlz:
            # SEPIA's rmultnormsvd consumes one np.random.normal(size=npred*pu) per sample, in sample order: the legacy
            # stream is the same for one call of ns*npred*pu values (tests/test_host_cpu.py)
            z = np.random.normal(size=ns * npred * pu)
            eng = self._pred
            stage = _pinned(eng, 'z', z.size)
            stage.copy_(torch.from_numpy(z))
            zd = stage.to('cuda', non_blocking=True).reshape(ns, pu, npred)
            if Sig is not None:
                # realisation = mean + F z with F F^T = Sigma.  Sigma >= I / lamWs is positive definite, so the factor is a
                # Cholesky factor (SEPIA uses U sqrt(s) of an SVD: the same distribution; neither is bit-comparable across
                # implementations, SURVEY 7.2); the eigen-factor stays as the fall-back when a block is rejected (info != 0)
                if npred <= CHOL_DRAW_MAX_N:
                    dev, info = ops.chol_draw(Sig, zd.reshape(ns * pu, npred))
                    dev = dev.reshape(ns, pu, npred)
                    self.launches += 1
                else:                         # beyond the kernel's shared-memory limit (explicit joint=True on a very large call)
                    L, info = torch.linalg.cholesky_ex(Sig.reshape(ns, pu, npred, npred))
                    dev = torch.matmul(L, zd.unsqueeze(-1)).squeeze(-1)
                bad = _pinned(eng, 'bad', 1)
                bad.copy_((info != 0).any().to(torch.float64).reshape(1), non_blocking=True)
            else:
                dev = torch.sqrt(torch.clamp(var.reshape(ns, pu, npred), min=0.0)) * zd
                bad = None
            w = (mean + dev).permute(0, 2, 1).contiguous()           # (ns, npred, pu)
            out = _pinned(eng, 'w', w.numel())
            out.copy_(w.reshape(-1), non_blocking=True)
            torch.cuda.current_stream().synchronize()
            if bad is not None and float(bad[0]) != 0.0:
                lam, Qm = torch.linalg.eigh(Sig.reshape(ns, pu, npred, npred))
                dev = torch.einsum('spij,spj->spi', Qm, torch.sqrt(torch.clamp(lam, min=0.0)) * zd)
                out.copy_((mean + dev).permute(0, 2, 1).contiguous().reshape(-1))
                torch.cuda.current_stream().synchronize()
            self.w = out.numpy().reshape(ns, npred, pu).copy()
        else:
            torch.cuda.current_stream().synchronize()                # the staging buffers are reused by the next call

    # ------------------------------------------------------------------ outputs
    def get_w(self):
        return self.w

    def get_mu_sigma(self):
        return self.mu, self.sigma

    def get_y(self, std=False, device=False):
        """(nsamp, npred, n_y) in native units (std=False); dtype follows self.w (callers cast w to
        float32 first, assess_all_models.py:491).  device=True returns the torch CUDA tensor."""
        torch = _lib.require_cuda()
        sd = self.model.data.sim_data
        w = np.asarray(self.w)
        ns, npred, pu = w.shape
        ysd = 1.0 if std else sd.orig_y_sd
        ymu = 0.0 if std else sd.orig_y_mean
        if self.model.data.scalar_out:
            dt = torch.float32 if w.dtype == np.float32 else torch.float64
            y = torch.as_tensor(w, device='cuda').to(dt) * torch.as_tensor(np.asarray(ysd), device='cuda').to(dt) \
                + torch.as_tensor(np.asarray(ymu), device='cuda').to(dt)
            y = y.reshape(ns, npred, -1)
        elif w.dtype == np.float32:
            Kd, (sdd, mud) = self._basis_device(), ((1.0, 0.0) if std else sd.stats_device())
            y = ops.reconstruct(w.reshape(ns * npred, pu), Kd, sdd, mud).reshape(ns, npred, -1)
        else:
            Kd = torch.as_tensor(np.asarray(sd.K), device='cuda').double()
            y = torch.as_tensor(w, device='cuda').double().reshape(ns * npred, pu) @ Kd
            y = y * torch.as_tensor(np.asarray(ysd), device='cuda').double() + \
                torch.as_tensor(np.asarray(ymu), device='cuda').double()
            y = y.reshape(ns, npred, -1)
        return y if device else y.cpu().numpy()

    def _basis_device(self):
        """K on the device (cached in sim_data when it is float32: 58 MB at cfg3, re-used by every get_y call)."""
        sd = self.model.data.sim_data
        return sd.K_device() if np.asarray(sd.K).dtype == np.float32 else sd.K

    def _stats_inputs(self):
        """float32 w and the device basis, sd and mean of the statistics kernels; a scalar-output model is the unit 1 x 1
        basis (get_y: y = w sd + mean)."""
        torch = _lib.require_cuda()
        sd = self.model.data.sim_data
        K = torch.ones((1, 1), dtype=torch.float32, device='cuda') if self.model.data.scalar_out else self._basis_device()
        sdd, mud = sd.stats_device()
        return np.asarray(self.w, dtype=np.float32), K, sdd, mud

    @staticmethod
    def _fused_serves(w, quantile):
        """The fused (q, 1-q) kernels run wherever they support the call -- every call that worked before keeps its bits --
        and for an out-of-range quantile, which they reject; everything else goes through reconstruct_quantiles."""
        ns, npred, pu = w.shape
        return not (0.0 < quantile < 0.5) or (npred <= 65535 and ops.stats_supported(ns, pu, quantile))

    def get_y_quantiles(self, quantiles=(0.025, 0.5, 0.975), noise=None, device=False):
        """Extension (SURVEY 8f rank 1): mean over samples of get_y() and np.quantile(get_y() + sd_y * noise[s, t], q, axis=0)
        for every q in `quantiles` (1-32 values in [0, 1]; NumPy's 'linear' method on the float32 values, bit for bit), for
        up to 16 384 samples -- the per-sample fields are never materialised.  `noise` as in get_y_stats.
        Returns dict(mean (npred, n_y), quantiles (nq, npred, n_y), q (nq,)), float32 fields."""
        w, K, sdd, mud = self._stats_inputs()
        q = np.atleast_1d(np.asarray(quantiles, dtype=np.float64)).reshape(-1)
        m_, yq = ops.reconstruct_quantiles(w, K, sdd, mud, q, noise=noise)
        if device:
            return dict(mean=m_, quantiles=yq, q=q)
        return dict(mean=m_.cpu().numpy(), quantiles=yq.cpu().numpy(), q=q)

    def get_y_stats(self, quantile=0.025, noise=None, device=False):
        """Extension (SURVEY 8f rank 1): mean over samples of get_y() and the (quantile, 1-quantile) quantiles of
        get_y() + sd_y * noise[s, t], fused on the GPU -- the per-sample fields are never materialised.  This is
        the post-processing of assess_all_models.py:493-500 / plot_test_error.py:81-87 (`noise[s, t]` there is
        np.random.normal(scale=1/sqrt(lamWOs[s]))).  Returns dict(mean, lq, uq), each (npred, n_y) float32."""
        w, K, sdd, mud = self._stats_inputs()
        if self._fused_serves(w, quantile):
            m_, lo, hi = ops.reconstruct_stats(w, K, sdd, mud, q=quantile, noise=noise)
        else:
            m_, yq = ops.reconstruct_quantiles(w, K, sdd, mud, (quantile, 1.0 - quantile), noise=noise)
            lo, hi = yq[0], yq[1]
        if device:
            return dict(mean=m_, lq=lo, uq=hi)
        return dict(mean=m_.cpu().numpy(), lq=lo.cpu().numpy(), uq=hi.cpu().numpy())

    def get_y_error_stats(self, y_test, quantile=0.025, noise=None, mape_floor=None, fields=False):
        """Extension (SURVEY 8f rank 1): the test-error table of assess_all_models.py:523-552 for this object's designs in one
        streaming pass -- reconstruction, mean / quantiles over samples and the comparison with the test fields are fused, so
        neither the per-sample fields nor (unless `fields`) the mean / limit fields are written to memory.
        y_test (npred, n_y) in native units; `noise` as in get_y_stats; `mape_floor`: outputs below it are left out of the
        MAPE (the reference uses the 10 % quantile of its whole test matrix; default: that quantile of `y_test`).
        Returns dict(rmse, mape, lq, uq, frac_covered (each (npred,)), integrated_ci, mape_floor[, mean, lq_field, uq_field])."""
        torch = _lib.require_cuda()
        yt = y_test if torch.is_tensor(y_test) else torch.as_tensor(np.ascontiguousarray(np.asarray(y_test, dtype=np.float32)))
        yt = yt.to(device='cuda', dtype=torch.float32)
        if mape_floor is None:
            # np.quantile(y_test, 0.1): linear interpolation between the two neighbouring order statistics
            flat = yt.reshape(-1)
            pos = 0.1 * (flat.numel() - 1)
            k0 = int(np.floor(pos))
            lo_v = torch.kthvalue(flat, k0 + 1).values
            hi_v = torch.kthvalue(flat, min(k0 + 2, flat.numel())).values
            mape_floor = float(lo_v + (hi_v - lo_v) * (pos - k0))
        w, K, sdd, mud = self._stats_inputs()
        yt = yt.reshape(w.shape[1], K.shape[1])
        if self._fused_serves(w, quantile):
            err, fl = ops.reconstruct_errstats(w, K, sdd, mud, yt, mape_floor, q=quantile, noise=noise, want_fields=fields)
        else:
            err, fl = self._fields_error_stats(w, K, sdd, mud, yt, mape_floor, quantile, noise, fields)
        n_y = yt.shape[1]
        out = dict(rmse=np.sqrt(err[:, 0] / n_y), mape=err[:, 1] / err[:, 2], lq=err[:, 4] / n_y, uq=err[:, 5] / n_y,
                   frac_covered=err[:, 3] / n_y, integrated_ci=float(np.mean((err[:, 5] - err[:, 4]) / n_y)),
                   mape_floor=mape_floor)
        if fields:
            out.update(mean=fl[0], lq_field=fl[1], uq_field=fl[2])
        return out

    @staticmethod
    def _fields_error_stats(w, K, sdd, mud, yt, mape_floor, quantile, noise, fields):
        """get_y_error_stats where the fused kernels do not serve the call: mean and (q, 1-q) quantile fields of a chunk of
        designs (about FIELD_CHUNK_BYTES of them; all at once when the fields are returned), then their error sums."""
        ns, npred, _ = w.shape
        n_y = K.shape[1]
        nz = None if noise is None else ops._f32(noise).reshape(ns, npred)
        chunk = npred if fields else max(1, min(npred, FIELD_CHUNK_BYTES // (3 * 4 * n_y)))
        err, fl = [], []
        for t0 in range(0, npred, chunk):
            t1 = min(npred, t0 + chunk)
            m_, yq = ops.reconstruct_quantiles(w[:, t0:t1], K, sdd, mud, (quantile, 1.0 - quantile),
                                               noise=None if nz is None else nz[:, t0:t1])
            err.append(ops.fields_errstats(m_, yq[0], yq[1], yt[t0:t1], mape_floor))
            if fields:
                fl = (m_, yq[0], yq[1])
            del m_, yq
        return np.concatenate(err, axis=0), (fl if fields else None)


def _check_folds(folds, m):
    """leave_out_inds -> list of int64 index arrays; ValueError for anything SEPIA's per-fold refit could not run."""
    try:
        folds = list(folds)
    except TypeError:
        raise ValueError('leave_out_inds must be a list of arrays of training-row indices') from None
    if not folds:
        raise ValueError('leave_out_inds has no folds')
    out = []
    for k, f in enumerate(folds):
        a = np.atleast_1d(np.asarray(f))
        if a.ndim != 1 or a.size == 0:
            raise ValueError('fold %d of leave_out_inds is empty or not one-dimensional' % k)
        if a.dtype.kind not in 'iu':
            raise ValueError('fold %d of leave_out_inds: indices must be integers, got %s' % (k, a.dtype))
        if a.min() < 0 or a.max() >= m:
            raise ValueError('fold %d of leave_out_inds: index out of range [0, %d)' % (k, m))
        if np.unique(a).size != a.size:
            raise ValueError('fold %d of leave_out_inds holds a row twice' % k)
        if a.size == m:
            raise ValueError('fold %d of leave_out_inds holds all %d training rows: nothing is left to predict from' % (k, m))
        out.append(a.astype(np.int64))
    return out


class SepiaXvalEmulatorPrediction(SepiaEmulatorPrediction):
    """Cross-validated emulator predictions (SEPIA's emulator check; imported by assess_all_models.py:31-32): the training
    rows of every fold are predicted from the other simulations with the same posterior samples, so an emulator can be
    validated without a test ensemble.

    SEPIA builds a sub-model per fold and runs wPred at its held-out rows.  Here the factors of the full S22 -- shared with
    SepiaEmulatorPrediction through the model's cache -- give the same moments in closed form (ops.Predictor.xval).
    leave_out_inds: list of folds (arrays of training-row indices; folds may overlap); default leave-one-out
    [[0], [1], ..., [m-1]].  Outputs:
    * .w (nsamp, sum |F|, pu): fold-major, in the given order within a fold; get_y / get_y_stats / get_y_error_stats work
      on it as on any prediction (y_test = the held-out rows of y_sim);
    * .xpred / .t_pred: the held-out rows of x_trans / t_trans; .leave_out_inds: the folds (int64 arrays);
    * storeMuSigma: .mu / .sigma are lists with one entry per fold, (nsamp, pu |F|) / (nsamp, pu |F|, pu |F|), PC-major.
    Realisations consume one np.random.normal value per (fold, sample, PC, row), in that order, as SEPIA's per-fold wPred
    calls do; a one-row fold is drawn as sqrt(var) z, a larger one through a Cholesky factor of each per-PC block."""

    def __init__(self, samples=None, model=None, leave_out_inds=None, addResidVar=False, storeRlz=True,
                 storeMuSigma=False):
        if samples is None or model is None:
            raise TypeError('samples and model are required')
        m = model.num.m
        self.leave_out_inds = _check_folds([[i] for i in range(m)] if leave_out_inds is None else leave_out_inds, m)
        rows = np.concatenate(self.leave_out_inds)
        sd = model.data.sim_data
        self.model = model
        self.samples = samples
        self.addResidVar = addResidVar
        self.storeRlz = storeRlz
        self.storeMuSigma = storeMuSigma
        self.joint = None
        self.xpred = np.asarray(sd.x_trans)[rows]
        self.t_pred = None if sd.t_trans is None else np.asarray(sd.t_trans)[rows]
        self.xpredt = model.num.zt[rows]
        self.w = None
        self.mu = None
        self.sigma = None
        self._xval()

    def _xval(self):
        torch = _lib.require_cuda()
        num = self.model.num
        pu = num.pu
        ns = self._predictor()
        folds = self.leave_out_inds
        sizes = np.array([f.size for f in folds])
        offs = np.concatenate([[0], np.cumsum(sizes)])
        N = int(offs[-1])
        lamWOs = np.asarray(self.samples['lamWOs'], dtype=np.float64).reshape(-1, 1)
        # SEPIA's predictive variance of a held-out row leaves out the 1/(LamSim lamWOs) part of S22's nugget unless
        # addResidVar (then it is S22's own diagonal, as the s11 of SepiaEmulatorPrediction)
        sub = np.zeros((ns, pu)) if self.addResidVar else 1.0 / (num.LamSim[None, :] * lamWOs)
        mu, var, Sig = self._pred.xval(folds, sub.reshape(-1))
        mu = mu.reshape(ns, pu, N)
        var = var.reshape(ns, pu, N)
        if self.storeMuSigma:
            muh, varh = mu.cpu().numpy(), var.cpu().numpy()
            self.mu, self.sigma = [], []
            for k, s in enumerate(sizes):
                sl = slice(offs[k], offs[k + 1])
                self.mu.append(muh[:, :, sl].reshape(ns, pu * s))
                blk = Sig[k].reshape(ns, pu, s, s).cpu().numpy() if s > 1 else varh[:, :, sl, None]
                sig = np.zeros((ns, pu * s, pu * s))
                for j in range(pu):
                    sig[:, j * s:(j + 1) * s, j * s:(j + 1) * s] = blk[:, j]
                self.sigma.append(sig)
        if self.storeRlz:
            # fold k takes the ns * pu * |F_k| values from ns * pu * offs[k] on, ordered (sample, PC, row)
            zd = torch.as_tensor(np.random.normal(size=ns * pu * N), device='cuda')
            B = ns * pu
            dev = torch.empty((ns, pu, N), dtype=torch.float64, device='cuda')
            one = offs[:-1][sizes == 1]
            if one.size:
                cols = torch.as_tensor(one, device='cuda')
                zi = cols[None, :] * B + torch.arange(B, device='cuda')[:, None]
                dev[:, :, cols] = torch.sqrt(torch.clamp(var[:, :, cols], min=0.0)) * zd[zi].reshape(ns, pu, -1)
            for s in sorted(set(sizes[sizes > 1].tolist())):
                ks = np.nonzero(sizes == s)[0]
                S = torch.stack([Sig[k] for k in ks]).reshape(-1, s, s)
                zz = torch.stack([zd[B * offs[k]:B * offs[k + 1]] for k in ks]).reshape(-1, s)
                d_, info = ops.chol_draw(S, zz)
                if bool(info.any()):                  # a block rejected by the Cholesky draw: eigen-factor, as wPred falls back
                    lam, Qm = torch.linalg.eigh(S)
                    d_ = torch.einsum('bij,bj->bi', Qm, torch.sqrt(torch.clamp(lam, min=0.0)) * zz)
                d_ = d_.reshape(len(ks), ns, pu, s)
                for t, k in enumerate(ks):
                    dev[:, :, offs[k]:offs[k + 1]] = d_[t]
            self.w = (mu + dev).permute(0, 2, 1).contiguous().cpu().numpy()      # (ns, N, pu)
        else:
            torch.cuda.current_stream().synchronize()
