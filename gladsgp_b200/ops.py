"""Thin Python wrappers over the C ABI (device tensors in, device tensors out).

Each function cites the reference-side routine it stands in for; see include/gladsgp_b200.h.
No function here has a CPU path.
"""
import ctypes as C
import numpy as np

from . import _lib
from ._lib import ptr, stream_ptr, check, McmcArgs


def _f64(t, torch, dev):
    return torch.as_tensor(np.ascontiguousarray(t, dtype=np.float64) if not torch.is_tensor(t) else t,
                           dtype=torch.float64, device=dev).contiguous()


def cov_build(X, beta, lamz, diag_add):
    """SepiaDistCov.compute_cov_mat type 1 + nugget diagonal (SURVEY A.10 cov_self).  -> (B, m, m)."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    dev = 'cuda'
    X = _f64(X, torch, dev); beta = _f64(beta, torch, dev).reshape(-1, X.shape[1])
    lamz = _f64(lamz, torch, dev).reshape(-1); diag_add = _f64(diag_add, torch, dev).reshape(-1)
    B, (m, d) = beta.shape[0], X.shape
    out = torch.empty((B, m, m), dtype=torch.float64, device=dev)
    check(lib.ggp_cov_build_f64(ptr(X), m, d, ptr(beta), ptr(lamz), ptr(diag_add), B, ptr(out), stream_ptr()),
          'ggp_cov_build_f64')
    return out


def cross_cov(X, Xp, beta, lamz):
    """SepiaDistCov type 2 (SURVEY A.10 cov_cross).  -> (B, m, n)."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    dev = 'cuda'
    X = _f64(X, torch, dev); Xp = _f64(Xp, torch, dev)
    beta = _f64(beta, torch, dev).reshape(-1, X.shape[1]); lamz = _f64(lamz, torch, dev).reshape(-1)
    B, (m, d), n = beta.shape[0], X.shape, Xp.shape[0]
    out = torch.empty((B, m, n), dtype=torch.float64, device=dev)
    check(lib.ggp_cross_cov_f64(ptr(X), m, ptr(Xp), n, d, ptr(beta), ptr(lamz), B, ptr(out), stream_ptr()),
          'ggp_cross_cov_f64')
    return out


def loglik_batched(X, W, beta, lamz, diag_add, want_factor=False, want_u=False, factor_ws=None):
    """doLogLik over a batch (SURVEY A.10 do_loglik).  W: (B, m).  Returns dict(loglik, info[, factor, u])."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    dev = 'cuda'
    X = _f64(X, torch, dev); W = _f64(W, torch, dev)
    beta = _f64(beta, torch, dev).reshape(-1, X.shape[1])
    lamz = _f64(lamz, torch, dev).reshape(-1); diag_add = _f64(diag_add, torch, dev).reshape(-1)
    B, (m, d) = beta.shape[0], X.shape
    assert W.shape == (B, m)
    fd = lib.ggp_factor_doubles(m)
    Mp = lib.ggp_padded_m(m)
    if factor_ws is None:
        factor_ws = torch.empty((B, fd), dtype=torch.float64, device=dev)
    u = torch.empty((B, Mp), dtype=torch.float64, device=dev) if want_u else None
    ll = torch.empty(B, dtype=torch.float64, device=dev)
    info = torch.empty(B, dtype=torch.int32, device=dev)
    check(lib.ggp_loglik_batched_f64(ptr(X), m, d, ptr(W), W.stride(0), ptr(beta), ptr(lamz), ptr(diag_add), B,
                                     ptr(factor_ws), ptr(u), ptr(ll), ptr(info), stream_ptr()),
          'ggp_loglik_batched_f64')
    out = dict(loglik=ll, info=info)
    if want_factor:
        out['factor'] = factor_ws
    if want_u:
        out['u'] = u
    return out


def factor_unpack(factor_ws, m):
    torch = _lib.require_cuda()
    lib = _lib.load()
    B = factor_ws.shape[0]
    out = torch.empty((B, m, m), dtype=torch.float64, device=factor_ws.device)
    check(lib.ggp_factor_unpack_f64(ptr(factor_ws), m, B, ptr(out), stream_ptr()), 'ggp_factor_unpack_f64')
    return out


PRIOR_KIND = {'Uniform': 0, 'Gamma': 1, 'Beta': 2, 'Normal': 3}
PROP_KIND = {'Uniform': 0, 'BetaRho': 1, 'PropMH': 2}
FIXED_NEUTRAL = 3


def mark_neutral_sites(X, fixed, pu):
    """The fixed table with every sampled betaU element (k, j) whose column k of X (m, d) is constant marked
    FIXED_NEUTRAL.  Such a column adds beta * (x_ik - x_jk)^2 = 0 to every covariance entry whatever beta is, so the PC's
    log-likelihood does not change under a betaU[k, j] proposal: the sampler decides it from the prior ratio alone
    (include/gladsgp_b200.h).  betaU comes first in the table, in Fortran order (element k + j d)."""
    X = np.asarray(X, dtype=np.float64)
    d = X.shape[1]
    const = np.all(X == X[:1], axis=0) & np.all(np.isfinite(X), axis=0)
    fx = np.array(fixed, dtype=np.uint8).reshape(-1)
    beta = fx[:d * pu].reshape(pu, d)                   # view: row j = PC j
    beta[(beta == 0) & const[None, :]] = FIXED_NEUTRAL
    return fx


class McmcEngine:
    """Owns the device-side model + tables of one sim-only SEPIA model and runs chains on it.

    X (m,d) = zt, W (pu,m) PC weights, lamsim (pu,).  tables: dict of length-P numpy arrays
    (prior_kind, prior_a, prior_b, lo, hi, prop_kind, fixed) in SEPIA sampling order.  The betaU elements of constant
    columns of X are marked in the device's fixed table (mark_neutral_sites): decided without an evaluation.
    per_chain=True: chain c is its own model on the shared design -- W (n_chains,pu,m), lamsim (n_chains,pu),
    tables['prior_a'] / ['prior_b'] (n_chains,P); the other tables are shared.
    """

    def __init__(self, X, W, lamsim, tables, n_chains=1, per_chain=False):
        torch = _lib.require_cuda()
        self.torch = torch
        self.lib = _lib.load()
        dev = 'cuda'
        self.per_chain = bool(per_chain)
        self.X = _f64(X, torch, dev); self.W = _f64(W, torch, dev); self.lamsim = _f64(lamsim, torch, dev)
        self.m, self.d = self.X.shape
        self.n_chains = int(n_chains)
        if self.per_chain:
            if self.W.dim() != 3 or self.W.shape[0] != self.n_chains or self.W.shape[2] != self.m:
                raise ValueError('per_chain: W must be (n_chains, pu, m)')
            self.pu = self.W.shape[1]
            if tuple(self.lamsim.shape) != (self.n_chains, self.pu):
                raise ValueError('per_chain: lamsim must be (n_chains, pu)')
        else:
            self.pu = self.W.shape[0]
        self.P = self.d * self.pu + 2 * self.pu + 1
        self.X_host = self.X.cpu().numpy()
        self.set_tables(tables)
        nb = self.lib.ggp_mcmc_workspace_bytes(self.m, self.d, self.pu, self.n_chains)
        self.ws = torch.empty(nb, dtype=torch.uint8, device=dev)
        self._pin = {}
        self._h2d_done = None
        self.theta = torch.zeros((self.n_chains, self.P), dtype=torch.float64, device=dev)
        self.sigwl = torch.zeros((self.n_chains, self.pu), dtype=torch.float64, device=dev)
        self.upos = torch.zeros(self.n_chains, dtype=torch.int64, device=dev)
        self.launches_per_step = 1          # one fused step kernel per mcmc_step (+ one plan kernel per run)

    def set_tables(self, tb):
        torch, dev = self.torch, 'cuda'
        P = self.P
        self.t_prior_kind = torch.as_tensor(np.asarray(tb['prior_kind'], dtype=np.int32).reshape(P), device=dev)
        pshape = (self.n_chains, P) if self.per_chain else (P,)
        self.t_prior_a = _f64(np.asarray(tb['prior_a']).reshape(pshape), torch, dev)
        self.t_prior_b = _f64(np.asarray(tb['prior_b']).reshape(pshape), torch, dev)
        self.t_lo = _f64(np.asarray(tb['lo']).reshape(P), torch, dev)
        self.t_hi = _f64(np.asarray(tb['hi']).reshape(P), torch, dev)
        self.t_prop_kind = torch.as_tensor(np.asarray(tb['prop_kind'], dtype=np.int32).reshape(P), device=dev)
        fixed = mark_neutral_sites(self.X_host, np.asarray(tb['fixed'], dtype=np.uint8).reshape(P), self.pu)
        self.t_fixed = torch.as_tensor(fixed, device=dev)

    def set_state(self, theta):
        th = _f64(np.asarray(theta, dtype=np.float64).reshape(-1, self.P), self.torch, 'cuda')
        if th.shape[0] == 1 and self.n_chains > 1:
            th = th.expand(self.n_chains, self.P)
        self.theta.copy_(th)

    def _build_args(self, n_steps, step, uniforms, replay, do_propMH, init_sigwl, record, record_accept):
        """ggp_mcmc_args for a run of n_steps (SEPIA tables, state, random stream or replay tables, output buffers)."""
        torch, dev = self.torch, 'cuda'
        a = McmcArgs()
        a.m, a.d, a.pu, a.n_chains, a.n_steps = self.m, self.d, self.pu, self.n_chains, int(n_steps)
        a.do_propMH, a.init_sigwl = int(bool(do_propMH)), int(bool(init_sigwl))
        a.per_chain_data = int(self.per_chain)
        keep = []
        step = _f64(step, torch, dev); keep.append(step)
        if step.dim() == 1:
            a.step_stride_t, a.step_stride_c = 0, 0
        elif step.shape[0] == n_steps and step.dim() == 2:
            a.step_stride_t, a.step_stride_c = self.P, 0
        elif step.dim() == 3 and step.shape[0] == 1:          # (1, n_chains, P): per-chain sizes, constant in time
            a.step_stride_t, a.step_stride_c = 0, self.P
        elif step.dim() == 3:
            a.step_stride_t, a.step_stride_c = self.n_chains * self.P, self.P
        else:
            raise ValueError('step must be (P,), (n_steps,P) or (n_steps,n_chains,P)')
        a.X, a.W, a.lamsim = self.X.data_ptr(), self.W.data_ptr(), self.lamsim.data_ptr()
        a.prior_kind, a.prior_a, a.prior_b = self.t_prior_kind.data_ptr(), self.t_prior_a.data_ptr(), self.t_prior_b.data_ptr()
        a.lo, a.hi = self.t_lo.data_ptr(), self.t_hi.data_ptr()
        a.prop_kind, a.fixed = self.t_prop_kind.data_ptr(), self.t_fixed.data_ptr()
        a.step = step.data_ptr()
        a.theta, a.sigwl = self.theta.data_ptr(), self.sigwl.data_ptr()
        if replay is not None:
            a.replay = 1
            sh = (n_steps, self.n_chains, self.P)
            rc = _f64(np.asarray(replay['cand']).reshape(sh), torch, dev)
            ra = _f64(np.asarray(replay['logacorr']).reshape(sh), torch, dev)
            ru = _f64(np.asarray(replay['logu']).reshape(sh), torch, dev)
            rv = torch.as_tensor(np.asarray(replay['valid'], dtype=np.uint8).reshape(sh), device=dev)
            keep += [rc, ra, ru, rv]
            a.r_cand, a.r_logacorr, a.r_logu, a.r_valid = rc.data_ptr(), ra.data_ptr(), ru.data_ptr(), rv.data_ptr()
        else:
            a.replay = 0
            if not torch.is_tensor(uniforms):
                uniforms = torch.as_tensor(np.ascontiguousarray(uniforms, dtype=np.float64))
            uniforms = uniforms.reshape(self.n_chains, -1)
            if uniforms.device.type != 'cuda':
                # host -> device through a cached page-locked staging buffer (page-locking per call costs more than
                # the copy and its cost varies a lot between hosts)
                if self._h2d_done is not None:
                    self._h2d_done.synchronize()           # the previous upload has left the staging buffer
                stage = self._pinned('uniforms', uniforms.numel(), torch.float64)
                stage.copy_(uniforms.reshape(-1))
                uniforms = stage.to(dev, non_blocking=True).reshape(self.n_chains, -1)
                self._h2d_done = torch.cuda.Event()
                self._h2d_done.record()
            keep.append(uniforms)
            a.uniforms, a.n_uniform = uniforms.data_ptr(), uniforms.shape[1]
            self.upos.zero_()
            a.upos = self.upos.data_ptr()
        draws = lp = acc = None
        if record:
            draws = torch.empty((n_steps, self.n_chains, self.P), dtype=torch.float64, device=dev)
            lp = torch.empty((n_steps, self.n_chains), dtype=torch.float64, device=dev)
            a.draws, a.lp_draws = draws.data_ptr(), lp.data_ptr()
        if record_accept:
            acc = torch.empty((n_steps, self.n_chains, self.P), dtype=torch.uint8, device=dev)
            a.accepted = acc.data_ptr()
        a.workspace, a.workspace_bytes = self.ws.data_ptr(), self.ws.numel()
        return a, keep, draws, lp, acc

    def run(self, n_steps, step, uniforms=None, replay=None, do_propMH=True, init_sigwl=True,
            record=True, record_accept=False, time_kernels=False):
        """step: (P,) or (n_steps,P) or (n_chains,P) [see step_axes] numpy/tensor of step sizes.
        uniforms: (n_chains, n_uniform) U[0,1) stream, or replay = dict(cand, logacorr, logu, valid)
        each (n_steps, n_chains, P).  Returns dict(draws, lp, accepted, consumed)."""
        torch, dev = self.torch, 'cuda'
        a, keep, draws, lp, acc = self._build_args(n_steps, step, uniforms, replay, do_propMH, init_sigwl, record, record_accept)
        kms = (C.c_double * 2)(0.0, 0.0)
        cnt = None
        if time_kernels:
            a.kernel_ms = C.cast(kms, C.c_void_p)
            cnt = torch.zeros(2, dtype=torch.int64, device=dev)
            a.eval_count = cnt.data_ptr()
        check(self.lib.ggp_mcmc_run_f64(C.byref(a), stream_ptr()), 'ggp_mcmc_run_f64')
        self._keep = keep
        return dict(draws=draws, lp=lp, accepted=acc, consumed=self.upos,
                    kernel_ms=(kms[0], kms[1]) if time_kernels else None,
                    eval_count=cnt.cpu().numpy() if cnt is not None else None)

    def run_by_pc(self, n_steps, step, uniforms=None, replay=None, do_propMH=True, init_sigwl=True,
                  record=True, record_accept=False, shards=None, gather=None):
        """The same chain(s) with the PCs of every step spread over shards (SURVEY 8e ii; north_star "by independent PC
        component"): a shard sweeps the betaU / lamUz / lamWs sites and the lamWOs term of its own PCs, the per-PC result
        rows are exchanged, and every shard closes the step identically (lamWOs decision, record, next candidates).

        shards: list of (pc_begin, pc_count) this process sweeps one after the other (default: all PCs as one shard; a
        list of several emulates several ranks on one GPU).  gather(xchg): called after this process's shards have written
        their rows of xchg (pu_padded, n_chains, 2d+6) and before the close -- under torch.distributed it all_gathers the
        other ranks' rows in place (gladsgp_b200.dist.mcmc_by_pc).  Results are bit-identical to run()."""
        torch, dev = self.torch, 'cuda'
        a, keep, draws, lp, acc = self._build_args(n_steps, step, uniforms, replay, do_propMH, init_sigwl, record, record_accept)
        if shards is None:
            shards = [(0, self.pu)]
        rows = self.pu if gather is None else gather.padded_pcs
        xchg = torch.zeros((rows, self.n_chains, 2 * self.d + 6), dtype=torch.float64, device=dev)
        a.xchg = xchg.data_ptr()
        total_steps = int(n_steps)
        a.n_steps = 1
        sp = stream_ptr
        a.pc_begin, a.pc_count = 0, 0
        check(self.lib.ggp_mcmc_plan_f64(C.byref(a), 0, sp()), 'ggp_mcmc_plan_f64')
        for t in range(total_steps):
            a.step_index = t
            first = True
            for (b, cnt) in shards:
                if cnt <= 0:
                    continue
                a.pc_begin, a.pc_count = int(b), int(cnt)
                a.init_sigwl = int(bool(init_sigwl) and t == 0 and first)
                first = False
                check(self.lib.ggp_mcmc_run_f64(C.byref(a), sp()), 'ggp_mcmc_run_f64 (PC shard)')
            if gather is not None:
                gather(xchg)
            a.pc_begin, a.pc_count = 0, 0
            check(self.lib.ggp_mcmc_close_f64(C.byref(a), t, int(t + 1 < total_steps), sp()), 'ggp_mcmc_close_f64')
        self._keep = keep + [xchg]
        return dict(draws=draws, lp=lp, accepted=acc, consumed=self.upos, kernel_ms=None, eval_count=None)

    def _pinned(self, name, numel, dtype):
        """Cached page-locked host buffer (grown on demand) -> view of `numel` elements."""
        buf = self._pin.get(name)
        if buf is None or buf.numel() < numel or buf.dtype != dtype:
            buf = self.torch.empty(max(int(numel), 1), dtype=dtype).pin_memory()
            self._pin[name] = buf
        return buf[:numel]

    def to_host(self, t, name):
        """Device tensor -> NumPy copy through a cached page-locked buffer."""
        stage = self._pinned(name, t.numel(), t.dtype)
        stage.copy_(t.reshape(-1), non_blocking=True)
        self.torch.cuda.current_stream().synchronize()
        return stage.numpy().reshape(tuple(t.shape)).copy()


class Predictor:
    """Cached-factor predictor for a set of B = nsamp*pu (sample, PC) hyper-parameter blocks.

    Factors every S22 once (the reference re-solves it for every call, SURVEY 3.2), then pushes
    blocks of test designs through ggp_predict_f64.
    """

    def __init__(self, X, W, beta, lamz, diag_add, s11_diag):
        torch = _lib.require_cuda()
        self.torch, self.lib = torch, _lib.load()
        dev = 'cuda'
        self.X = _f64(X, torch, dev)
        self.m, self.d = self.X.shape
        self.beta = _f64(beta, torch, dev).reshape(-1, self.d)
        self.B = self.beta.shape[0]
        self.lamz = _f64(lamz, torch, dev).reshape(-1)
        self.s11 = _f64(s11_diag, torch, dev).reshape(-1)
        self.W = _f64(W, torch, dev).reshape(self.B, self.m)          # training weights: the means of cross-validation
        self.dadd = _f64(diag_add, torch, dev).reshape(-1)              # the S22 nugget (sequential design's Schur complement)
        out = loglik_batched(self.X, self.W, self.beta, self.lamz, diag_add, want_factor=True, want_u=True)
        self.factor, self.u, self.loglik, self.info = out['factor'], out['u'], out['loglik'], out['info']
        self.Mp = self.u.shape[1]
        self._ws = None
        self._xws = None

    def predict(self, Xp, want_V=False, b0=0, nb=None):
        """Xp (n,d) -> mean (nb,n), var (nb,n)[, V (nb,n,Mp)] of blocks [b0, b0+nb) (default: all B)."""
        torch, lib, dev = self.torch, self.lib, 'cuda'
        Xp = _f64(Xp, torch, dev)
        n = Xp.shape[0]
        nb = self.B - b0 if nb is None else nb
        need = lib.ggp_predict_workspace_bytes(self.m, n, nb)
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=dev)
        mean = torch.empty((nb, n), dtype=torch.float64, device=dev)
        var = torch.empty((nb, n), dtype=torch.float64, device=dev)
        V = torch.empty((nb, n, self.Mp), dtype=torch.float64, device=dev) if want_V else None
        check(lib.ggp_predict_f64(ptr(self.X), self.m, self.d, ptr(self.factor[b0:]), ptr(self.u[b0:]), ptr(self.beta[b0:]),
                                  ptr(self.lamz[b0:]), ptr(self.s11[b0:]), ptr(Xp), n, nb, ptr(mean), ptr(var), ptr(V),
                                  ptr(self._ws), self._ws.numel(), stream_ptr()), 'ggp_predict_f64')
        return (mean, var, V) if want_V else (mean, var)

    def jacobian(self, Xp, col0, full=True, b0=0, nb=None):
        """Gradients of the predictive moments at Xp (n,d) with respect to inputs col0 .. d-1 (q = d - col0 in [1, 31]) on
        blocks [b0, b0+nb) (csrc/ggp_jacobian.cu).  Returns (mean (nb,n,q+1) = [mu, grad mu], cov): with full, cov
        (nb,n,q+1,q+1) is the joint posterior covariance of [f, grad f]; otherwise (nb,n,2q+1) = [v, Cov(f, d_k f),
        Var(d_k f)].  mu and v equal predict's bit for bit; nothing is clamped."""
        torch, lib, dev = self.torch, self.lib, 'cuda'
        Xp = _f64(Xp, torch, dev)
        n = Xp.shape[0]
        nb = self.B - b0 if nb is None else nb
        q = self.d - int(col0)
        need = lib.ggp_jacobian_workspace_bytes(self.m, self.d, int(col0), n, nb)
        if need < 0:
            raise ValueError('jacobian needs 1 <= q = d - col0 <= 31 differentiated inputs and m <= 8192 (got q=%d, m=%d)'
                             % (q, self.m))
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=dev)
        mean = torch.empty((nb, n, q + 1), dtype=torch.float64, device=dev)
        cov = torch.empty((nb, n, q + 1, q + 1) if full else (nb, n, 2 * q + 1), dtype=torch.float64, device=dev)
        check(lib.ggp_jacobian_f64(ptr(self.X), self.m, self.d, ptr(self.factor[b0:]), ptr(self.u[b0:]),
                                   ptr(self.beta[b0:]), ptr(self.lamz[b0:]), ptr(self.s11[b0:]), ptr(Xp), n, nb, int(col0),
                                   1 if full else 0, ptr(mean), ptr(cov), ptr(self._ws), self._ws.numel(), stream_ptr()),
              'ggp_jacobian_f64')
        return mean, cov

    def pred_cov(self, Xp, V):
        """Joint covariance Sigma (B,n,n) = S11 - V V^T."""
        torch, lib, dev = self.torch, self.lib, 'cuda'
        Xp = _f64(Xp, torch, dev)
        n = Xp.shape[0]
        Sig = torch.empty((self.B, n, n), dtype=torch.float64, device=dev)
        check(lib.ggp_pred_cov_f64(ptr(Xp), n, self.d, ptr(self.beta), ptr(self.lamz), ptr(self.s11), ptr(V),
                                   self.m, self.B, ptr(Sig), stream_ptr()), 'ggp_pred_cov_f64')
        return Sig

    def xval_solve(self, idx, want_Z=False, b0=0, nb=None):
        """ggp_xval_solve_f64 on blocks [b0, b0+nb): training rows idx (n,) -> alpha (nb,n) = z.u, p (nb,n) = z.z
        [, Z (nb,n,Mp)] with z = L^-1 e_idx."""
        torch, lib, dev = self.torch, self.lib, 'cuda'
        nb = self.B - b0 if nb is None else nb
        idx = torch.as_tensor(np.asarray(idx) if not torch.is_tensor(idx) else idx, device=dev).to(torch.int32).contiguous()
        n = idx.numel()
        need = lib.ggp_xval_workspace_bytes(self.m, n, nb)
        if self._xws is None or self._xws.numel() < need:
            self._xws = torch.empty(need, dtype=torch.uint8, device=dev)
        alpha = torch.empty((nb, n), dtype=torch.float64, device=dev)
        p = torch.empty((nb, n), dtype=torch.float64, device=dev)
        Z = torch.empty((nb, n, self.Mp), dtype=torch.float64, device=dev) if want_Z else None
        check(lib.ggp_xval_solve_f64(ptr(self.factor[b0:]), ptr(self.u[b0:]), self.m, nb, ptr(idx), n, ptr(alpha), ptr(p),
                                     ptr(Z), ptr(self._xws), self._xws.numel(), stream_ptr()), 'ggp_xval_solve_f64')
        return (alpha, p, Z) if want_Z else (alpha, p)

    def xval(self, folds, sub_diag):
        """Cross-validated moments of held-out training rows from the factors of the full S22 (SEPIA refits a sub-model
        per fold; the Schur complement gives the same moments): for a fold F, with G = (S22^-1)_FF and a = (S22^-1 w)_F,
          mu_F = w_F - G^-1 a,   Sig_F = G^-1 - sub_diag I.
        folds: sequence of 1-D arrays of distinct rows in [0, m) (checked by the caller).  sub_diag (B,): the part of the
        S22 nugget a prediction leaves out (1 / (LamSim lamWOs), or 0 with addResidVar).
        Returns (mu, var, Sig): mu, var (B, N), N = sum |F|, fold-major and in the given order within a fold; Sig has one
        entry per fold, (B, |F|, |F|) for |F| > 1 and None for a one-row fold (its variance is var)."""
        torch, dev = self.torch, 'cuda'
        folds = [np.asarray(f, dtype=np.int64).reshape(-1) for f in folds]
        sizes = np.array([f.size for f in folds])
        offs = np.concatenate([[0], np.cumsum(sizes)])
        flat = np.concatenate(folds)
        idx = np.unique(flat)                                  # ascending: each row skips the panels above it
        pos = np.searchsorted(idx, flat)                       # flat[k] = idx[pos[k]]
        N, n = flat.size, idx.size
        sub = _f64(sub_diag, torch, dev).reshape(self.B, 1)
        w = self.W[:, torch.as_tensor(idx, device=dev)]
        mu = torch.empty((self.B, N), dtype=torch.float64, device=dev)
        var = torch.empty((self.B, N), dtype=torch.float64, device=dev)
        Sig = [None] * len(folds)
        groups = {}                                            # fold size > 1 -> fold numbers
        for k, s in enumerate(sizes):
            if s > 1:
                groups.setdefault(int(s), []).append(k)
        if groups:
            # the rows z_i go through the Gram products in chunks of blocks, at most XVAL_Z_BYTES of them at a time
            per = n * self.Mp * 8
            chunk = max(1, min(self.B, XVAL_Z_BYTES // per))
            alpha = torch.empty((self.B, n), dtype=torch.float64, device=dev)
            p = torch.empty((self.B, n), dtype=torch.float64, device=dev)
            gsig = {s: torch.empty((self.B, len(ks), s, s), dtype=torch.float64, device=dev) for s, ks in groups.items()}
            for b0 in range(0, self.B, chunk):
                nb = min(chunk, self.B - b0)
                a_c, p_c, Z = self.xval_solve(idx, want_Z=True, b0=b0, nb=nb)
                alpha[b0:b0 + nb] = a_c
                p[b0:b0 + nb] = p_c
                for s, ks in groups.items():
                    rows = torch.as_tensor(np.concatenate([pos[offs[k]:offs[k + 1]] for k in ks]), device=dev)
                    cols = torch.as_tensor(np.concatenate([np.arange(offs[k], offs[k + 1]) for k in ks]), device=dev)
                    Zg = Z[:, rows].reshape(nb, len(ks), s, self.Mp)
                    L, info = torch.linalg.cholesky_ex(Zg @ Zg.transpose(-1, -2))
                    if bool(info.any()):
                        raise np.linalg.LinAlgError('cross-validation: a held-out block of S22^-1 is not positive definite')
                    Gi = torch.cholesky_inverse(L)
                    a = a_c[:, rows].reshape(nb, len(ks), s, 1)
                    mu[b0:b0 + nb, cols] = (w[b0:b0 + nb, rows].reshape(nb, len(ks), s) -
                                            (Gi @ a).squeeze(-1)).reshape(nb, -1)
                    Sg = Gi - sub[b0:b0 + nb, :, None, None] * torch.eye(s, dtype=torch.float64, device=dev)
                    gsig[s][b0:b0 + nb] = Sg
                    var[b0:b0 + nb, cols] = torch.diagonal(Sg, dim1=-2, dim2=-1).reshape(nb, -1)
                del Z
            for s, ks in groups.items():
                for t, k in enumerate(ks):
                    Sig[k] = gsig[s][:, t]
        else:
            alpha, p = self.xval_solve(idx)
        one = np.nonzero(sizes == 1)[0]
        if one.size:
            cols = torch.as_tensor(offs[one], device=dev)
            r = torch.as_tensor(pos[offs[one]], device=dev)
            pr = p[:, r]
            mu[:, cols] = w[:, r] - alpha[:, r] / pr
            var[:, cols] = 1.0 / pr - sub
        return mu, var, Sig


CHOL_DRAW_WS_BYTES = 1 << 30         # scratch factors of chol_draw: at most 1 GiB, more blocks go in several launches
XVAL_Z_BYTES = 1 << 30               # rows z_i of Predictor.xval's multi-row folds: at most 1 GiB, more blocks in several launches


def chol_draw(Sigma, z):
    """One multivariate-normal deviate per block: Sigma (B,n,n) f64 symmetric, z (B,n) -> (L z (B,n), info (B,) int32) with
    Sigma = L L^T (the draw step of SEPIA's wPred; info[b] != 0: block b is not positive definite, its row is undefined)."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    B, n = int(Sigma.shape[0]), int(Sigma.shape[-1])
    assert Sigma.is_cuda and Sigma.dtype == torch.float64 and Sigma.is_contiguous() and tuple(Sigma.shape) == (B, n, n)
    z = z.to(device='cuda', dtype=torch.float64).contiguous().reshape(B, n)
    out = torch.empty((B, n), dtype=torch.float64, device='cuda')
    info = torch.empty((B,), dtype=torch.int32, device='cuda')
    need = int(lib.ggp_chol_draw_workspace_bytes(n, B))
    one = int(lib.ggp_chol_draw_workspace_bytes(n, 1))
    nbytes = max(one, min(need, CHOL_DRAW_WS_BYTES))
    ws = torch.empty((nbytes // 8,), dtype=torch.float64, device='cuda')
    check(lib.ggp_chol_draw_f64(ptr(Sigma), n, B, ptr(z), ptr(out), ptr(info), ptr(ws), nbytes, stream_ptr()), 'ggp_chol_draw_f64')
    return out, info


def reconstruct(w, K, sd, mean, out=None):
    """get_y: w (R,pu) f32, K (pu,n_y) f32, sd/mean scalar or (n_y,) -> y (R,n_y) f32 on the device."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    dev = 'cuda'

    def f32(t):
        if not torch.is_tensor(t):
            t = torch.as_tensor(np.ascontiguousarray(np.asarray(t, dtype=np.float32)))
        return t.to(device=dev, dtype=torch.float32).contiguous()
    w = f32(w); K = f32(K); sd = f32(sd).reshape(-1); mean = f32(mean).reshape(-1)
    R, pu = w.shape
    n_y = K.shape[1]
    if out is None:
        out = torch.empty((R, n_y), dtype=torch.float32, device=dev)
    check(lib.ggp_reconstruct_f32(ptr(w), ptr(K), ptr(sd), sd.numel(), ptr(mean), mean.numel(), R, pu, n_y,
                                  ptr(out), stream_ptr()), 'ggp_reconstruct_f32')
    return out


def reconstruct_stats(w, K, sd, mean, q=0.025, noise=None):
    """Fused get_y + mean / (q, 1-q) quantiles over samples (SURVEY 8f rank 1).
    w (nsamp,npred,pu) f32, noise (nsamp,npred) f32 or None -> (ymean, ylo, yhi), each (npred, n_y) f32 on the device."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    dev = 'cuda'

    def f32(t):
        if not torch.is_tensor(t):
            t = torch.as_tensor(np.ascontiguousarray(np.asarray(t, dtype=np.float32)))
        return t.to(device=dev, dtype=torch.float32).contiguous()
    w = f32(w); K = f32(K); sd = f32(sd).reshape(-1); mean = f32(mean).reshape(-1)
    nsamp, npred, pu = w.shape
    n_y = K.shape[1]
    nz = None if noise is None else f32(noise).reshape(nsamp, npred)
    outs = [torch.empty((npred, n_y), dtype=torch.float32, device=dev) for _ in range(3)]
    check(lib.ggp_reconstruct_stats_f32(ptr(w), ptr(K), ptr(sd), sd.numel(), ptr(mean), mean.numel(), ptr(nz), nsamp,
                                        npred, pu, n_y, float(q), ptr(outs[0]), ptr(outs[1]), ptr(outs[2]), stream_ptr()),
          'ggp_reconstruct_stats_f32')
    return tuple(outs)


# ------------------------------------------------------------------ ensemble ingest (SURVEY 8f rank 2)
def _ens_dims(Y, transposed):
    if Y.dim() != 2 or Y.stride(1) != 1 or Y.dtype != _lib.require_cuda().float32:
        raise ValueError('ensemble must be a 2-D float32 device tensor with unit column stride')
    m, n = (Y.shape[1], Y.shape[0]) if transposed else Y.shape
    return m, n, Y.stride(0)


def colstats(Y, transposed=False, ddof=1, sd_floor=0.0):
    """Column mean and standard deviation of the ensemble (src/model.py:60-64).  Y: device float32 (m, n), or (n, m)
    with transposed=True (the file layout); a row-sliced view (y[:m] / yt[:, :m]) is used in place.
    Returns (mean, sd), float32 device vectors of length n."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    m, n, ld = _ens_dims(Y, transposed)
    mean = torch.empty(n, dtype=torch.float32, device='cuda')
    sd = torch.empty(n, dtype=torch.float32, device='cuda')
    check(lib.ggp_colstats_f32(ptr(Y), ld, m, n, int(bool(transposed)), int(ddof), float(sd_floor), ptr(mean), ptr(sd),
                               stream_ptr()), 'ggp_colstats_f32')
    return mean, sd


def standardize(Y, mean, sd, transposed=False, out=None):
    """(Y - mean) / sd in float32 -> (m, n) device tensor (SepiaData.standardize_y; src/model.py:71-72)."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    m, n, ld = _ens_dims(Y, transposed)
    if out is None:
        out = torch.empty((m, n), dtype=torch.float32, device='cuda')
    check(lib.ggp_standardize_f32(ptr(Y), ld, m, n, int(bool(transposed)), ptr(mean), mean.numel(), ptr(sd), sd.numel(),
                                  ptr(out), stream_ptr()), 'ggp_standardize_f32')
    return out


def project(X, Kt):
    """P (m, pu+2) float64 = [X @ Kt.T, X.sum(1), (X*X).sum(1)] accumulated in FP64 (src/model.py:219-223)."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    m, n = X.shape
    pu = Kt.shape[0]
    if Kt.shape[1] != n:
        raise ValueError('Kt must be (pu, n)')
    nb = lib.ggp_project_workspace_bytes(m, pu)
    if nb < 0:
        raise ValueError('project: pu must be in [1, 32]')
    ws = torch.empty(nb, dtype=torch.uint8, device='cuda')
    P = torch.empty((m, pu + 2), dtype=torch.float64, device='cuda')
    check(lib.ggp_project_f32(ptr(X), m, n, ptr(Kt), pu, ptr(P), ptr(ws), ws.numel(), stream_ptr()), 'ggp_project_f32')
    return P


def rsvd_sketch_tc(X, omegaT, ws=None):
    """Y = X @ omega on the tcgen05 tensor cores (3xTF32 split, FP32-level accuracy); any m."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    m, n = X.shape
    r = omegaT.shape[0]
    need = lib.ggp_rsvd_tc_workspace_bytes(m)
    if ws is None or ws.numel() < need:
        ws = torch.empty(need, dtype=torch.uint8, device='cuda')
    Y = torch.empty((m, r), dtype=torch.float32, device='cuda')
    check(lib.ggp_rsvd_sketch_tc_f32(ptr(X), m, n, ptr(omegaT), r, ptr(Y), ptr(ws), ws.numel(), stream_ptr()),
          'ggp_rsvd_sketch_tc_f32')
    return Y


def rsvd_xty_tc(X, Y):
    """Bt (r,n) = Y^T X on the tcgen05 tensor cores (3xTF32 split); any m."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    m, n = X.shape
    r = Y.shape[1]
    Bt = torch.empty((r, n), dtype=torch.float32, device='cuda')
    check(lib.ggp_rsvd_xty_tc_f32(ptr(X), m, n, ptr(Y.contiguous()), r, ptr(Bt), stream_ptr()), 'ggp_rsvd_xty_tc_f32')
    return Bt


def sobol_upload(f_A, f_B, f_AB):
    """Function values of the Saltelli scheme -> device (f_A, f_B (N,p); f_AB (n_dim,N,p)), float64."""
    torch = _lib.require_cuda()
    return tuple(torch.as_tensor(np.ascontiguousarray(np.asarray(a, dtype=np.float64)), device='cuda') for a in (f_A, f_B, f_AB))


def sobol_stats(dev, N, p, n_dim, idx=None, clamp=True):
    """First-order / total Saltelli statistics of R index sets (SURVEY 8f rank 3; src/utils.py:97-118): two (R,p,n_dim) host arrays.
    idx (R,n) integers in [0,N) or None (one set: the full sample)."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    fA, fB, fAB = dev
    if idx is None:
        R, n, it = 1, N, None
    else:
        idx = np.asarray(idx)
        if idx.ndim != 2 or idx.size == 0 or idx.min() < 0 or idx.max() >= N:
            raise ValueError('idx must be a non-empty (R, n) array of indices in [0, N)')
        R, n = idx.shape
        it = torch.as_tensor(np.ascontiguousarray(idx.astype(np.int32)), device='cuda')
    first = torch.empty((R, p, n_dim), dtype=torch.float64, device='cuda')
    total = torch.empty((R, p, n_dim), dtype=torch.float64, device='cuda')
    check(lib.ggp_sobol_stats_f64(ptr(fA), ptr(fB), ptr(fAB), N, p, n_dim, ptr(it), n, n, R, 1 if clamp else 0,
                                  ptr(first), ptr(total), stream_ptr()), 'ggp_sobol_stats_f64')
    return first.cpu().numpy(), total.cpu().numpy()


def reconstruct_errstats(w, K, sd, mean, y_test, mape_floor, q=0.025, noise=None, want_fields=False):
    """reconstruct_stats with the test-error sums of assess_all_models.py:523-538 fused in (SURVEY 8f rank 1).
    y_test (npred, n_y) f32 (device tensor or array).  Returns (err (npred, 6) float64 host array, fields or None):
    err columns = sum resid^2, sum |resid / y_test| over y_test >= mape_floor, count of those, covered count, sum lq, sum uq."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    dev = 'cuda'

    def f32(t):
        if not torch.is_tensor(t):
            t = torch.as_tensor(np.ascontiguousarray(np.asarray(t, dtype=np.float32)))
        return t.to(device=dev, dtype=torch.float32).contiguous()
    w = f32(w); K = f32(K); sd = f32(sd).reshape(-1); mean = f32(mean).reshape(-1)
    nsamp, npred, pu = w.shape
    n_y = K.shape[1]
    yt = f32(y_test).reshape(npred, n_y)
    nz = None if noise is None else f32(noise).reshape(nsamp, npred)
    outs = [torch.empty((npred, n_y), dtype=torch.float32, device=dev) for _ in range(3)] if want_fields else [None] * 3
    need = lib.ggp_errstats_workspace_bytes(npred, n_y)
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    err = torch.empty((npred, 6), dtype=torch.float64, device=dev)
    check(lib.ggp_reconstruct_errstats_f32(ptr(w), ptr(K), ptr(sd), sd.numel(), ptr(mean), mean.numel(), ptr(nz), nsamp,
                                           npred, pu, n_y, float(q), ptr(yt), float(mape_floor), ptr(outs[0]), ptr(outs[1]),
                                           ptr(outs[2]), ptr(err), ptr(ws), need, stream_ptr()),
          'ggp_reconstruct_errstats_f32')
    return err.cpu().numpy(), (tuple(outs) if want_fields else None)


def _f32(t):
    torch = _lib.require_cuda()
    if not torch.is_tensor(t):
        t = torch.as_tensor(np.ascontiguousarray(np.asarray(t, dtype=np.float32)))
    return t.to(device='cuda', dtype=torch.float32).contiguous()


def stats_supported(nsamp, pu, q):
    """True if reconstruct_stats / reconstruct_errstats serve (nsamp, pu, q) (ggp_reconstruct_stats_supported)."""
    return bool(_lib.load().ggp_reconstruct_stats_supported(int(nsamp), int(pu), float(q)))


def reconstruct_quantiles(w, K, sd, mean, quantiles, noise=None):
    """Mean over samples of get_y and exact np.quantile fields of get_y + sd * noise[s, t] (float32, method 'linear'), any
    sample count up to 16 384, 1-32 quantiles in [0, 1], pu <= 32.  w (nsamp,npred,pu) f32, noise (nsamp,npred) f32 or None
    -> (ymean (npred, n_y), yq (nq, npred, n_y)) f32 on the device."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    w = _f32(w); K = _f32(K); sd = _f32(sd).reshape(-1); mean = _f32(mean).reshape(-1)
    nsamp, npred, pu = w.shape
    n_y = K.shape[1]
    nz = None if noise is None else _f32(noise).reshape(nsamp, npred)
    q = np.ascontiguousarray(np.atleast_1d(np.asarray(quantiles, dtype=np.float64)).reshape(-1))
    ymean = torch.empty((npred, n_y), dtype=torch.float32, device='cuda')
    yq = torch.empty((q.size, npred, n_y), dtype=torch.float32, device='cuda')
    check(lib.ggp_reconstruct_quantiles_f32(ptr(w), ptr(K), ptr(sd), sd.numel(), ptr(mean), mean.numel(), ptr(nz), nsamp,
                                            npred, pu, n_y, q.ctypes.data_as(C.POINTER(C.c_double)), q.size, ptr(ymean),
                                            ptr(yq), stream_ptr()),
          'ggp_reconstruct_quantiles_f32')
    return ymean, yq


def fields_errstats(ymean, ylo, yhi, y_test, mape_floor):
    """The six per-design error sums of reconstruct_errstats from stored fields, each (npred, n_y) f32 (device tensors or
    arrays) -> err (npred, 6) float64 host array (same columns, same summation order)."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    ymean = _f32(ymean)
    npred, n_y = ymean.shape
    ylo, yhi, yt = (_f32(a).reshape(npred, n_y) for a in (ylo, yhi, y_test))
    need = lib.ggp_errstats_workspace_bytes(npred, n_y)
    ws = torch.empty(need, dtype=torch.uint8, device='cuda')
    err = torch.empty((npred, 6), dtype=torch.float64, device='cuda')
    check(lib.ggp_fields_errstats_f32(ptr(ymean), ptr(ylo), ptr(yhi), ptr(yt), npred, n_y, float(mape_floor), ptr(err),
                                      ptr(ws), need, stream_ptr()),
          'ggp_fields_errstats_f32')
    return err.cpu().numpy()


CHAIN_DIAG_WS_BYTES = 8 << 30        # workspace of chain_diagnostics: at most 8 GiB, more elements go in several launches


def chain_diagnostics(x):
    """Rank-normalized split R-hat, bulk ESS and tail ESS per element (csrc/ggp_chain_diag.cu; DESIGN.md section 2).
    x: CUDA float64 tensor (n_draws, n_chains, n_elem), any strides.  Returns (rhat, ess_bulk, ess_tail), three (n_elem,)
    float64 device tensors.  Elements are processed CHAIN_DIAG_WS_BYTES of workspace at a time; the results do not depend
    on how they are grouped."""
    torch = _lib.require_cuda()
    lib = _lib.load()
    if not torch.is_tensor(x) or not x.is_cuda or x.dtype != torch.float64 or x.dim() != 3:
        raise ValueError('x must be a CUDA float64 tensor (n_draws, n_chains, n_elem)')
    n, C, E = x.shape
    per = lib.ggp_chain_diag_workspace_bytes(n, C, 1)
    if per < 0:
        raise ValueError('chain_diagnostics needs n_draws >= 4, n_chains >= 1 and n_chains * n_draws < 2^31 (got %d x %d)'
                         % (n, C))
    out = [torch.empty(E, dtype=torch.float64, device=x.device) for _ in range(3)]
    if E == 0:
        return tuple(out)
    chunk = max(1, min(E, CHAIN_DIAG_WS_BYTES // per))
    ws = torch.empty(chunk * per, dtype=torch.uint8, device=x.device)
    sd, sc, se = x.stride()
    for e0 in range(0, E, chunk):
        ne = min(chunk, E - e0)
        check(lib.ggp_chain_diag_f64(ptr(x[:, :, e0]), n, C, ne, sd, sc, se, ptr(out[0][e0:]), ptr(out[1][e0:]),
                                     ptr(out[2][e0:]), ptr(ws), ws.numel(), stream_ptr()), 'ggp_chain_diag_f64')
    return tuple(out)


def _gp_sens_args(Z, beta, a, S, pu, mode):
    torch = _lib.require_cuda()
    Z = _f64(Z, torch, 'cuda')
    if Z.dim() != 2:
        raise ValueError('Z must be (m, q)')
    m, q = Z.shape
    beta = _f64(beta, torch, 'cuda').reshape(-1)
    a = _f64(a, torch, 'cuda').reshape(-1)
    if beta.numel() != S * pu * q or a.numel() != S * pu * m:
        raise ValueError('beta must hold (S * pu, q) and a (S * pu, m) values')
    if mode not in (0, 1):
        raise ValueError("mode must be 0 ('samples') or 1 ('mean')")
    nb = _lib.load().ggp_gp_sens_workspace_bytes(m, q, S, pu, mode)
    if nb < 0:
        raise ValueError('gp_sens needs m, S, pu >= 1 and 1 <= q <= 32 (got m=%d, q=%d, S=%d, pu=%d)' % (m, q, S, pu))
    return torch, Z, beta, a, m, q, torch.empty(nb, dtype=torch.uint8, device='cuda')


def gp_sens(Z, beta, a, S, pu, mode=0):
    """Exact Sobol' moments of f = sum_n a_n prod_k exp(-beta_nk (x_k - z_nk)^2) on [0,1]^q (csrc/ggp_gp_sens.cu).
    Z (m, q) training inputs, beta (S*pu, q) and a (S*pu, m) per block b = s*pu + j.  mode 0: one function per block;
    mode 1: one per PC over every sample's terms (the weights as given).  Returns (M (F, 2q+1), E0 (F,)) float64 device
    tensors: M[:, k] = M({k}), M[:, q+k] = M(all\\k), M[:, 2q] = M(all)."""
    torch, Z, beta, a, m, q, ws = _gp_sens_args(Z, beta, a, S, pu, mode)
    F = S * pu if mode == 0 else pu
    M = torch.empty((F, 2 * q + 1), dtype=torch.float64, device='cuda')
    E0 = torch.empty(F, dtype=torch.float64, device='cuda')
    check(_lib.load().ggp_gp_sens_f64(ptr(Z), m, q, ptr(beta), ptr(a), S, pu, mode, ptr(M), ptr(E0), ptr(ws), ws.numel(),
                                      stream_ptr()), 'ggp_gp_sens_f64')
    return M, E0


def main_effects(Z, beta, a, S, pu, grid, mode=0):
    """Main-effect curves E[f | x_k = g] of the functions of gp_sens at the values of grid -> (F, q, ngrid) device tensor."""
    torch, Z, beta, a, m, q, ws = _gp_sens_args(Z, beta, a, S, pu, mode)
    g = _f64(grid, torch, 'cuda').reshape(-1)
    F = S * pu if mode == 0 else pu
    out = torch.empty((F, q, g.numel()), dtype=torch.float64, device='cuda')
    check(_lib.load().ggp_main_effects_f64(ptr(Z), m, q, ptr(beta), ptr(a), S, pu, mode, ptr(g), g.numel(), ptr(out),
                                           ptr(ws), ws.numel(), stream_ptr()), 'ggp_main_effects_f64')
    return out


def grad_sens(Z, beta, a, S, pu, mode, omega=None):
    """Gradient outer-product matrices C = E[grad g grad g^T] on [0,1]^q (csrc/ggp_grad_sens.cu) of the functions
    g = sum over terms of a_n Omega-weighted products of squared-exponential kernels.  Z (m, q), beta (S*pu, q), a (S*pu, m)
    per block b = s*pu + j, as gp_sens takes them.  mode 0: one function per block; 1: one per PC over every sample's
    terms; 2: one per sample over every PC's terms, weighted by omega (pu, pu); 3: one function over every block, omega.
    The weights are used as given (scale by 1/S for the posterior mean).  Returns C (F, q, q), a float64 device tensor."""
    torch = _lib.require_cuda()
    Z = _f64(Z, torch, 'cuda')
    if Z.dim() != 2:
        raise ValueError('Z must be (m, q)')
    m, q = Z.shape
    beta = _f64(beta, torch, 'cuda').reshape(-1)
    a = _f64(a, torch, 'cuda').reshape(-1)
    if beta.numel() != S * pu * q or a.numel() != S * pu * m:
        raise ValueError('beta must hold (S * pu, q) and a (S * pu, m) values')
    if mode not in (0, 1, 2, 3):
        raise ValueError('mode must be 0 (per block), 1 (per PC), 2 (per sample) or 3 (one function)')
    if mode < 2:
        omega = None
    else:
        if omega is None:
            raise ValueError('modes 2 and 3 need omega (pu, pu)')
        omega = _f64(omega, torch, 'cuda')
        if tuple(omega.shape) != (pu, pu):
            raise ValueError('omega must be (pu, pu) = (%d, %d)' % (pu, pu))
    nb = _lib.load().ggp_grad_sens_workspace_bytes(m, q, S, pu, mode)
    if nb < 0:
        raise ValueError('grad_sens needs m, S, pu >= 1, 1 <= q <= 32 and fewer than 2^31 terms per function '
                         '(got m=%d, q=%d, S=%d, pu=%d, mode=%d)' % (m, q, S, pu, mode))
    ws = torch.empty(nb, dtype=torch.uint8, device='cuda')
    F = (S * pu, pu, S, 1)[mode]
    out = torch.empty((F, q, q), dtype=torch.float64, device='cuda')
    check(_lib.load().ggp_grad_sens_f64(ptr(Z), m, q, ptr(beta), ptr(a), S, pu, mode,
                                        None if omega is None else ptr(omega), ptr(out), ptr(ws), ws.numel(),
                                        stream_ptr()), 'ggp_grad_sens_f64')
    return out


def calib_loglik(mean, var, G, b, c0, want_per_sample=False):
    """Calibration log-likelihood (csrc/ggp_calib.cu) at n points from the predictive moments mean, var (S*pu, n) of
    ggp_predict_f64 and the observation terms G (S, pu, pu), b (S, pu), c0 (S,).  Returns ll (n,) [, ll_s (S, n)], float64
    device tensors."""
    torch = _lib.require_cuda()
    mean = _f64(mean, torch, 'cuda'); var = _f64(var, torch, 'cuda')
    G = _f64(G, torch, 'cuda'); b = _f64(b, torch, 'cuda'); c0 = _f64(c0, torch, 'cuda').reshape(-1)
    S, pu = c0.numel(), G.shape[-1]
    n = mean.shape[-1]
    if G.numel() != S * pu * pu or b.numel() != S * pu:
        raise ValueError('G, b, c0 must be (S, pu, pu), (S, pu), (S,)')
    if tuple(mean.shape) != (S * pu, n) or tuple(var.shape) != (S * pu, n):
        raise ValueError('mean and var must be (S * pu, n)')
    ll = torch.empty(n, dtype=torch.float64, device='cuda')
    ll_s = torch.empty((S, n), dtype=torch.float64, device='cuda') if want_per_sample else None
    check(_lib.load().ggp_calib_loglik_f64(ptr(mean), ptr(var), S, pu, n, ptr(G), ptr(b), ptr(c0), ptr(ll), ptr(ll_s),
                                           stream_ptr()), 'ggp_calib_loglik_f64')
    return (ll, ll_s) if want_per_sample else ll


def calib_step(mean, var, G, b, c0, Xp, lo, hi, L_prop, z_next, logu, theta, ll, rec_theta, rec_ll, rec_acc):
    """One Metropolis step of C chains (csrc/ggp_calib.cu): the candidates are the last q columns of Xp (C, d), mean / var
    (S*pu, C) their predictive moments.  Updates theta (C, q), ll (C) and, unless z_next is None, writes the next
    candidates theta + L_prop z_next[c] into Xp; rec_theta (C, q), rec_ll (C), rec_acc (C) uint8 receive the step's record.
    Every tensor argument but G, b, c0 must already be a contiguous CUDA tensor of the right dtype (this runs every step)."""
    C, d = Xp.shape
    q = theta.shape[1]
    pu = G.shape[-1]
    S = c0.numel()
    check(_lib.load().ggp_calib_step_f64(ptr(mean), ptr(var), S, pu, C, ptr(G), ptr(b), ptr(c0), ptr(Xp), d, q, ptr(lo),
                                         ptr(hi), ptr(L_prop), ptr(z_next), ptr(logu), ptr(theta), ptr(ll), ptr(rec_theta),
                                         ptr(rec_ll), ptr(rec_acc), stream_ptr()), 'ggp_calib_step_f64')


def _design_blocks(pred, b0, nb):
    return (ptr(pred.beta[b0:]), ptr(pred.lamz[b0:]), ptr(pred.dadd[b0:]))


def design_score(pred, b0, XR, XC, V_R, V_C, A_R, A_C, t, wgt, score, imse, accumulate, ws=None):
    """ALC scores of greedy sequential design (csrc/ggp_design.cu) on blocks [b0, b0+nb) of a Predictor, nb = V_C.shape[0]:
    score (n_cand,) and imse (1,) receive (or, with accumulate, add in block order) sum_b wgt[b] sum_r Sigma_t(r, c)^2 /
    den_t(c) and sum_b wgt[b] sum_r v_t(r).  XR (n_ref, d), XC (n_cand, d) designs; V_R (nb, n_ref, Mp), V_C (nb, n_cand,
    Mp) from pred.predict(..., want_V=True, b0=b0, nb=nb); A_R (nb, n_ref, Kp), A_C (nb, n_cand, Kp) with t columns in use;
    wgt (nb,).  score may be None (imse only).  Every tensor must be a contiguous float64 CUDA tensor.  Returns the
    workspace (pass it back to reuse it)."""
    torch, lib = pred.torch, pred.lib
    nb, n_cand, _ = V_C.shape
    n_ref = V_R.shape[1]
    need = lib.ggp_design_workspace_bytes(n_cand, nb)
    if ws is None or ws.numel() < need:
        ws = torch.empty(max(need, 1), dtype=torch.uint8, device='cuda')
    be, lz, da = _design_blocks(pred, b0, nb)
    check(lib.ggp_design_score_f64(ptr(XR), n_ref, ptr(XC), n_cand, XC.shape[1], be, lz, da, ptr(pred.s11[b0:]), ptr(wgt),
                                   ptr(V_R), ptr(V_C), pred.m, ptr(A_R), ptr(A_C), A_C.shape[2], int(t), nb, int(accumulate),
                                   ptr(score), ptr(imse), ptr(ws), ws.numel(), stream_ptr()), 'ggp_design_score_f64')
    return ws


def design_condition(pred, b0, XR, XC, V_R, V_C, A_R, A_C, t, index):
    """Append column t of A_R and A_C (csrc/ggp_design.cu) after choosing candidate `index`, on the blocks of design_score.
    The same tensors for XR / XC, V_R / V_C and A_R / A_C mean the reference set is the candidate set."""
    lib = pred.lib
    nb, n_cand, _ = V_C.shape
    be, lz, da = _design_blocks(pred, b0, nb)
    check(lib.ggp_design_condition_f64(ptr(XR), V_R.shape[1], ptr(XC), n_cand, XC.shape[1], be, lz, da, ptr(V_R), ptr(V_C),
                                       pred.m, ptr(A_R), ptr(A_C), A_C.shape[2], int(t), nb, int(index), stream_ptr()),
          'ggp_design_condition_f64')


def hm_impl(mean, var, K_O, r, c, order, cutoff):
    """History-matching implausibility (csrc/ggp_hm.cu) at n points from the predictive moments mean, var (S*pu, n) of
    ggp_predict_f64 and the observed outputs' K_O (pu, n_o), r (n_o,) and c (n_o,) = rho + tau^2 + delta^2 (standardized
    units).  Returns impl (n, order) float64, the `order` largest I_i of each point in descending order, and n_over (n,)
    int32, the number of outputs with I_i > cutoff, as CUDA tensors."""
    torch = _lib.require_cuda()
    mean = _f64(mean, torch, 'cuda'); var = _f64(var, torch, 'cuda')
    K_O = _f64(K_O, torch, 'cuda'); r = _f64(r, torch, 'cuda').reshape(-1); c = _f64(c, torch, 'cuda').reshape(-1)
    if K_O.dim() != 2:
        raise ValueError('K_O must be (pu, n_o)')
    pu, n_o = K_O.shape
    if r.numel() != n_o or c.numel() != n_o:
        raise ValueError('r and c must be (n_o,) = (%d,)' % n_o)
    if mean.dim() != 2 or mean.shape[0] % pu != 0 or tuple(var.shape) != tuple(mean.shape):
        raise ValueError('mean and var must be (S * pu, n) with pu = %d' % pu)
    S, n = mean.shape[0] // pu, mean.shape[1]
    lib = _lib.load()
    need = lib.ggp_hm_workspace_bytes(n, n_o, pu, S)
    if need < 0:
        raise ValueError('hm_impl needs S, n, n_o >= 1 and 1 <= pu <= 32 (got S=%d, n=%d, n_o=%d, pu=%d)' % (S, n, n_o, pu))
    ws = torch.empty(need, dtype=torch.uint8, device='cuda')
    impl = torch.empty((n, int(order)), dtype=torch.float64, device='cuda')
    n_over = torch.empty(n, dtype=torch.int32, device='cuda')
    check(lib.ggp_hm_impl_f64(ptr(mean), ptr(var), S, pu, n, ptr(K_O), ptr(r), ptr(c), n_o, int(order), float(cutoff),
                              ptr(impl), ptr(n_over), ptr(ws), ws.numel(), stream_ptr()), 'ggp_hm_impl_f64')
    return impl, n_over
