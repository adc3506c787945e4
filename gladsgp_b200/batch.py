"""Several independent sim-only models fitted together (SURVEY 8f rank 4).

The reference fits its scalar quantity-of-interest emulators one after the other
(/root/reference/experiments/synthetic/analysis/fit_scalar_models.py:457-473: for every threshold a fresh
SepiaData / SepiaModel, `tune_step_sizes(100, 10)`, `do_mcmc(512)`).  Each of those chains keeps one 512 x 512
factorisation in flight at a time, which leaves a B200 almost idle.  `ModelBatch` runs the same sampler for all
models at once: model i becomes chain i of one batched launch sequence, with its own data vector, prior
parameters, step sizes and random stream.  Every model ends up in exactly the state it would reach on its own with
`np.random.seed(seeds[i])` before `tune_step_sizes` / `do_mcmc` (tests/test_gpu_api.py).
"""
import numpy as np

from . import ops


class ModelBatch:
    def __init__(self, models, seeds=None):
        if len(models) == 0:
            raise ValueError('no models')
        self.models = list(models)
        m0 = self.models[0]
        self.tables = [mm._tables() for mm in self.models]
        tb0 = self.tables[0]
        for mm, tb in zip(self.models, self.tables):
            if mm.num.zt.shape != m0.num.zt.shape or not np.array_equal(mm.num.zt, m0.num.zt):
                raise ValueError('all models of a batch must share the design matrix')
            if mm.num.pu != m0.num.pu:
                raise ValueError('all models of a batch must have the same number of PCs')
            for k in ('prior_kind', 'lo', 'hi', 'prop_kind', 'fixed'):
                if not np.array_equal(tb[k], tb0[k]):
                    raise ValueError('all models of a batch must share prior families, bounds and proposal types')
        n = len(self.models)
        self.rng = [np.random.RandomState(None if seeds is None else int(seeds[i])) for i in range(n)]
        tb = dict(tb0)
        tb['prior_a'] = np.stack([t['prior_a'] for t in self.tables])
        tb['prior_b'] = np.stack([t['prior_b'] for t in self.tables])
        W = np.stack([mm._w_pcs for mm in self.models])                       # (n, pu, m)
        lamsim = np.stack([np.asarray(mm.num.LamSim, dtype=np.float64).reshape(-1) for mm in self.models])
        self.engine = ops.McmcEngine(m0.num.zt, W, lamsim, tb, n_chains=n, per_chain=True)
        self.P = tb0['theta'].size

    # ------------------------------------------------------------------ internals
    def _state(self):
        return np.stack([mm._tables()['theta'] for mm in self.models])

    def _steps(self):
        return np.stack([mm._tables()['step'] for mm in self.models])

    def _run(self, nsteps, step, do_propMH, record_accept=False):
        eng, n, P = self.engine, len(self.models), self.P
        eng.set_state(self._state())
        states = [r.get_state() for r in self.rng]
        us = np.stack([r.random_sample(2 * P * nsteps) for r in self.rng])
        out = eng.run(nsteps, step, uniforms=us, do_propMH=do_propMH, init_sigwl=True, record=True,
                      record_accept=record_accept)
        used = eng.to_host(out['consumed'], 'consumed')
        for r, st, u in zip(self.rng, states, used):          # leave every stream where its own chain would
            r.set_state(st)
            r.random_sample(int(u))
        draws = eng.to_host(out['draws'], 'draws')
        lps = eng.to_host(out['lp'], 'lp')
        acc = eng.to_host(out['accepted'], 'accepted') if record_accept else None
        return draws, lps, acc

    # ------------------------------------------------------------------ public
    def do_mcmc(self, nsamp, do_propMH=True):
        """nsamp steps of every model; draws are appended to each model's own lists (get_samples, save_model_info)."""
        draws, lps, _ = self._run(int(nsamp), self._steps()[None], do_propMH)
        for i, mm in enumerate(self.models):
            mm._record(draws[:, i, :], lps[:, i])

    def tune_step_sizes(self, n_burn, n_levels, update_vals=True):
        """SepiaModel.tune_step_sizes for every model (same ladder, own acceptance counts and logit fits)."""
        from .sepia.SepiaModel import _logit_glm
        n, P = len(self.models), self.P
        n_burn, n_levels = int(n_burn), int(n_levels)
        base = self._steps()                                                        # (n, P)
        ex = np.linspace(-(n_levels - 1) / 2.0, (n_levels - 1) / 2.0, n_levels)
        ladder = base[None, :, :] * np.power(2.0, ex)[:, None, None]               # (n_levels, n, P)
        warm = 10
        nsteps = warm + n_burn * n_levels
        sched = np.empty((nsteps, n, P))
        sched[:warm] = base
        sched[warm:] = np.tile(ladder, (n_burn, 1, 1))
        saved = [[b.val.copy() for b in mm._blocks()[0]] for mm in self.models]
        saved_lp = [mm.params.lp.val for mm in self.models]
        draws, lps, acc = self._run(nsteps, sched, do_propMH=False, record_accept=True)
        target = np.log(1.0 / (np.exp(1.0) - 1.0))
        for i, mm in enumerate(self.models):
            tb = self.tables[i]
            a_i = acc[warm:, i, :].reshape(n_burn, n_levels, P).sum(axis=0)
            new_step = base[i].copy()
            for e in range(P):
                if tb['fixed'][e]:
                    continue
                coef = _logit_glm(np.log(ladder[:, i, e]), a_i[:, e].astype(np.float64), n_burn)
                if coef is not None and np.all(np.isfinite(coef)) and coef[1] < 0:
                    lg = (target - coef[0]) / coef[1]
                    if np.isfinite(lg) and abs(lg) < 600.0:
                        new_step[e] = np.exp(lg)
            mm._store_state(draws[-1, i, :])
            blocks = mm._blocks()[0]
            o = 0
            for b, v0 in zip(blocks, saved[i]):
                k = b.val.size
                b.mcmc.stepParam = new_step[o:o + k].reshape(b.val_shape, order='F').copy()
                if not update_vals:
                    b.val = v0
                o += k
            mm.params.lp.val = float(lps[-1, i]) if update_vals else saved_lp[i]

    def mcmc_diagnostics(self, nburn=0):
        """SepiaModel.mcmc_diagnostics of every model's recorded chain, in one device call: element (model i, parameter p)
        is one chain of the (n, models x (P + 1)) array of draws and logPost.  Returns one dict per model, equal bit for
        bit to that model's own mcmc_diagnostics()."""
        from . import diagnostics
        chains = [mm._recorded_chain() for mm in self.models]
        n = chains[0][0].shape[0]
        if n == 0 or any(d.shape[0] != n for d, _ in chains):
            raise ValueError('every model needs the same, non-zero number of recorded draws')
        x = np.stack([np.concatenate([d, l[:, None]], axis=1) for d, l in chains], axis=1)   # (n, models, P + 1)
        res = diagnostics.chain_diagnostics(x.reshape(n, 1, -1), nburn=nburn)
        Q = self.P + 1
        return [diagnostics.by_block(mm._blocks()[0], {k: v[i * Q:(i + 1) * Q] for k, v in res.items()})
                for i, mm in enumerate(self.models)]
