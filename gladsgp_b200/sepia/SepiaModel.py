"""SepiaModel mirror for the simulator-only emulator (SURVEY.md 8a rows a2, a5, a6; A.2-A.8).

Driven by the reference at /root/reference/src/model.py:106 (construction), :227-231 (parameter
override), :234-235 (tune_step_sizes, do_mcmc), :149/:238 (restore/save_model_info) and
experiments/synthetic/analysis/assess_all_models.py:469-471 (get_samples).

Host code here is set-up and bookkeeping only.  Every likelihood evaluation and the whole
Metropolis-within-Gibbs sweep run on the GPU (csrc/ggp_mcmc.cu); without the CUDA library or a
device the compute methods raise -- there is no NumPy fallback.
"""
import copy
import os
import pickle
import sys

import numpy as np

from .SepiaParam import SepiaParam
from .. import ops, ingest
from ..ops import PRIOR_KIND, PROP_KIND


class ModelContainer:
    """Numeric set-up (SepiaModel.num upstream)."""
    pass


class SepiaParamList:
    pass


def _progress(total, desc, enable):
    if not enable:
        return None
    try:
        from tqdm import tqdm
        return tqdm(total=total, desc=desc, file=sys.stderr)
    except Exception:
        return None


class SepiaModel:
    def __init__(self, data):
        if not getattr(data, 'sim_only', False):
            raise NotImplementedError('only simulator-only SepiaData is supported')
        sd = data.sim_data
        if sd.x_trans is None or (sd.t is not None and sd.t_trans is None):
            data.transform_xt()
        if not sd.has_y_std():
            data.standardize_y()
        if not data.scalar_out and sd.K is None:
            raise ValueError('create_K_basis must be called before SepiaModel for multivariate output')
        self.verbose = False
        self.data = data
        num = ModelContainer()
        self.num = num
        m = sd.x.shape[0]
        num.sim_only, num.scalar_out = True, data.scalar_out
        num.m, num.n = m, 0
        num.p = sd.x.shape[1]
        num.q = 0 if sd.t is None else sd.t.shape[1]
        num.pv = 0
        # zt is float64 because the dummy x is (SURVEY A.9 item 3)
        zt = [np.asarray(sd.x_trans, dtype=np.float64)]
        if sd.t is not None:
            zt.append(np.asarray(sd.t_trans, dtype=np.float64))
        num.zt = np.ascontiguousarray(np.concatenate(zt, axis=1))
        num.x0Dist = None
        if data.scalar_out:
            num.pu = 1
            w = np.asarray(sd.y_std, dtype=np.float64).reshape(m, 1)
            num.LamSim = np.ones(1)
            resid_ss = 0.0
            n_y = 1
        else:
            K = np.asarray(sd.K)
            num.pu = K.shape[0]
            n_y = K.shape[1]
        on_device = (not data.scalar_out and ingest.use_device(m * n_y) and K.dtype == np.float32 and
                     (sd._y_std_dev is not None or sd._y_std.dtype == np.float32))
        if on_device:
            # large ensemble: one streaming pass on the device (csrc/ggp_ingest.cu), FP64 accumulation
            if sd._proj is None:
                sd._proj = ingest.project_basis(sd.y_std_device(), sd.K_device())
            w = sd._proj['w']
            num.LamSim = np.diag(sd._proj['G']).copy()
            resid_ss = sd._proj['resid_ss']
        elif not data.scalar_out:
            # w = (pinv(K)^T y_std^T)^T  (src/model.py:219 restates it); K K^T is pu x pu
            K64 = K.astype(np.float64)
            G = K64 @ K64.T
            ys = np.asarray(sd.y_std)
            YK = np.asarray(ys @ K.T, dtype=np.float64) if ys.dtype == K.dtype else ys.astype(np.float64) @ K64.T
            w = np.linalg.solve(G, YK.T).T
            num.LamSim = np.diag(G).copy()
            # ||y_std - w K||^2 without forming the residual matrix
            ss_y = 0.0
            for c0 in range(0, n_y, 1 << 16):
                blk = ys[:, c0:c0 + (1 << 16)].astype(np.float64)
                ss_y += float(np.sum(blk * blk))
            resid_ss = max(ss_y - 2.0 * float(np.sum(w * YK)) + float(np.sum((w @ G) * w)), 0.0)
        num.w = w.reshape((-1, 1), order='F')           # PC-major stack (SURVEY A.2)
        self._w_pcs = np.ascontiguousarray(w.T)         # (pu, m)
        num.n_y = n_y
        self._set_params_sim_only(m, n_y, resid_ss)
        self._engine = None
        self._pred_cache = None          # (key, ops.Predictor, nsamp): factors of the last set of posterior samples predicted with
        self.launches = 0

    def __getstate__(self):              # device-side caches do not travel in pickles / deep copies
        st = dict(self.__dict__)
        st['_engine'] = None
        st['_pred_cache'] = None
        return st

    # ------------------------------------------------------------------ parameters (SURVEY A.3)
    def _set_params_sim_only(self, m, n_y, resid_ss):
        num = self.num
        d, pu = num.p + num.q, num.pu
        prm = SepiaParamList()
        prm.betaU = SepiaParam(val=0.1, name='betaU', val_shape=(d, pu), dist='Beta', params=[1., 0.1],
                               bounds=[0., np.inf], mcmcStepParam=0.1, mcmcStepType='BetaRho')
        prm.lamUz = SepiaParam(val=1., name='lamUz', val_shape=(1, pu), dist='Gamma', params=[5., 5.],
                               bounds=[0.3, np.inf], mcmcStepParam=5., mcmcStepType='PropMH')
        if num.scalar_out:
            a, b = 5.0, 5e-3
        else:
            a = 5.0 + 0.5 * m * (n_y - pu)
            b = 5e-3 + 0.5 * resid_ss
        prm.lamWOs = SepiaParam(val=max(100.0, a / b), name='lamWOs', val_shape=(1, 1), dist='Gamma',
                                params=[a, b], bounds=[60., 1e5], mcmcStepParam=100., mcmcStepType='PropMH')
        prm.lamWs = SepiaParam(val=1000., name='lamWs', val_shape=(1, pu), dist='Gamma', params=[3., 3e-3],
                               bounds=[60., 1e5], mcmcStepParam=100., mcmcStepType='PropMH')
        prm.mcmcList = [prm.betaU, prm.lamUz, prm.lamWs, prm.lamWOs]
        prm.lp = _LogPostRecorder()
        self.params = prm

    # ------------------------------------------------------------------ device tables
    def _blocks(self):
        """The four parameter blocks in the engine's fixed order, read from self.params (the reference
        re-assigns params.lamWOs and params.mcmcList, src/model.py:227-231)."""
        p = self.params
        blocks = [p.betaU, p.lamUz, p.lamWs, p.lamWOs]
        listed = [q.name for q in p.mcmcList]
        if listed != [b.name for b in blocks if b.name in listed] or \
                any(q is not b for q in p.mcmcList for b in blocks if b.name == q.name):
            raise NotImplementedError('mcmcList must hold the current betaU, lamUz, lamWs, lamWOs objects in that order')
        return blocks, listed

    def _tables(self):
        blocks, listed = self._blocks()
        tb = {k: [] for k in ('prior_kind', 'prior_a', 'prior_b', 'lo', 'hi', 'prop_kind', 'fixed', 'step', 'theta')}
        for b in blocks:
            n = b.val.size
            if b.prior.dist not in PRIOR_KIND:
                raise NotImplementedError('prior %s' % b.prior.dist)
            if b.mcmc.stepType not in PROP_KIND:
                raise NotImplementedError('%s proposals are not used on the GladsGP path' % b.mcmc.stepType)
            tb['prior_kind'] += [PRIOR_KIND[b.prior.dist]] * n
            tb['prior_a'] += list(b.prior.params[0].reshape(-1, order='F'))
            tb['prior_b'] += list(b.prior.params[1].reshape(-1, order='F'))
            tb['lo'] += [b.prior.bounds[0]] * n
            tb['hi'] += [b.prior.bounds[1]] * n
            tb['prop_kind'] += [PROP_KIND[b.mcmc.stepType]] * n
            fx = np.asarray(b.fixed, dtype=bool).reshape(b.val_shape).reshape(-1, order='F')
            fx = fx.astype(np.uint8)
            if b.name not in listed:
                fx[:] = 2                           # not in mcmcList: never visited, no RNG draw
            tb['fixed'] += list(fx)
            tb['step'] += list(np.asarray(b.mcmc.stepParam, dtype=np.float64).reshape(b.val_shape).reshape(-1, order='F'))
            tb['theta'] += list(np.asarray(b.val, dtype=np.float64).reshape(b.val_shape).reshape(-1, order='F'))
        return {k: np.asarray(v) for k, v in tb.items()}

    def _get_engine(self, n_chains=1):
        tb = self._tables()
        if self._engine is None or self._engine.n_chains != n_chains:
            num = self.num
            self._engine = ops.McmcEngine(num.zt, self._w_pcs, num.LamSim, tb, n_chains=n_chains)
        else:
            self._engine.set_tables(tb)
        self._engine.set_state(tb['theta'])
        return self._engine, tb

    def _store_state(self, theta):
        blocks, _ = self._blocks()
        o = 0
        for b in blocks:
            n = b.val.size
            b.val = np.asarray(theta[o:o + n], dtype=np.float64).reshape(b.val_shape, order='F').copy()
            o += n

    # ------------------------------------------------------------------ likelihood / posterior
    def logLik(self, cvar='all', cindex=None):
        """Sum over PCs of -sum log diag chol(C_j) - 1/2 ||L_j^-1 w_j||^2 (GPU, all PCs in one launch)."""
        num, p = self.num, self.params
        pu = num.pu
        beta = np.ascontiguousarray(p.betaU.val.T)                     # (pu, d)
        lamz = p.lamUz.val.reshape(-1)
        dadd = 1.0 / (num.LamSim * p.lamWOs.val[0, 0]) + 1.0 / p.lamWs.val.reshape(-1)
        out = ops.loglik_batched(num.zt, self._w_pcs, beta, lamz, dadd)
        self.launches += 1
        self.num.SigWl = out['loglik'].cpu().numpy()
        return float(np.sum(self.num.SigWl))

    def logPost(self, cvar='all', cindex=None):
        ll = self.logLik(cvar, cindex)
        lp = ll + sum(prm.prior.compute_log_prior() for prm in self.params.mcmcList)
        self.params.lp.val = lp
        return lp

    # ------------------------------------------------------------------ sampling
    def _run(self, nsteps, step, do_propMH, n_chains=1, record_accept=False, prog=None, chunk=None, device=False):
        """Run nsteps on the device, feeding the global np.random stream exactly as SEPIA would consume
        it: draw an upper bound of uniforms, then rewind and advance by the number actually used.
        device=True: draws and logPost stay the CUDA tensors the engine wrote."""
        eng, tb = self._get_engine(n_chains)
        P = tb['theta'].size
        draws, lps, accs = [], [], []
        done = 0
        init = True
        chunk = nsteps if not chunk else chunk
        step = np.asarray(step, dtype=np.float64)
        while done < nsteps:
            k = min(chunk, nsteps - done)
            state = np.random.get_state()
            us = np.random.random_sample(2 * P * k * n_chains).reshape(n_chains, -1)
            st = step if step.ndim in (1, 3) else step[done:done + k]      # (P,), (1, n_chains, P) or a per-step schedule
            out = eng.run(k, st, uniforms=us, do_propMH=do_propMH, init_sigwl=init, record=True,
                          record_accept=record_accept)
            used = eng.to_host(out['consumed'], 'consumed')
            if n_chains == 1:
                np.random.set_state(state)
                np.random.random_sample(int(used[0]))
            draws.append(out['draws'] if device else eng.to_host(out['draws'], 'draws'))
            lps.append(out['lp'] if device else eng.to_host(out['lp'], 'lp'))
            if record_accept:
                accs.append(eng.to_host(out['accepted'], 'accepted'))
            self.launches += (1 if init else 0) + 1 + k          # [initial per-PC terms] + plan + one step kernel per step
            init = False
            done += k
            if prog is not None:
                prog.update(k)
        if device:
            draws, lps = eng.torch.cat(draws, dim=0), eng.torch.cat(lps, dim=0)
        else:
            draws, lps = np.concatenate(draws, axis=0), np.concatenate(lps, axis=0)
        accs = np.concatenate(accs, axis=0) if record_accept else None
        return draws, lps, accs

    def _record(self, draws, lps):
        """Append (nsteps, P) draws of one chain to the per-parameter draw lists."""
        blocks, _ = self._blocks()
        o = 0
        for b in blocks:
            n = b.val.size
            arr = draws[:, o:o + n].reshape((draws.shape[0],) + b.val_shape[::-1]).transpose(0, 2, 1)
            b.mcmc.draws.extend(list(np.ascontiguousarray(arr)))
            o += n
        self.params.lp.mcmc.draws.extend(list(lps))
        self._store_state(draws[-1])
        self.params.lp.val = float(lps[-1])

    def do_mcmc(self, nsamp, prog=True, do_propMH=True, no_init=False, seed=None):
        """nsamp Metropolis-within-Gibbs steps (SEPIA order: betaU in Fortran order, lamUz, lamWs, lamWOs)."""
        if seed is not None:
            np.random.seed(seed)
        nsamp = int(nsamp)
        if nsamp <= 0:
            return
        _, tb = self._get_engine(1)
        bar = _progress(nsamp, 'MCMC sampling', prog)
        chunk = max(1, nsamp // 16) if bar is not None else None
        draws, lps, _ = self._run(nsamp, tb['step'], do_propMH, prog=bar, chunk=chunk)
        if bar is not None:
            bar.close()
        self._record(draws[:, 0, :], lps[:, 0])

    def mcmc_step(self, do_propMH=True):
        _, tb = self._get_engine(1)
        draws, lps, _ = self._run(1, tb['step'], do_propMH)
        self._record(draws[:, 0, :], lps[:, 0])

    def do_mcmc_chains(self, nsamp, n_chains, seed=None, do_propMH=True, device=False):
        """Extension: n_chains independent chains of this model in one batched run (chains x PCs CTAs).
        Returns draws (nsamp, n_chains, P) and logPost (nsamp, n_chains); the model's own draw lists
        are not touched.  Each chain gets its own slice of the np.random stream.
        device=True: the draws and logPost are returned as the CUDA tensors the sampler wrote, without a download, so
        that a large run can be diagnosed where it lives (mcmc_diagnostics)."""
        if seed is not None:
            np.random.seed(seed)
        _, tb = self._get_engine(n_chains)
        draws, lps, _ = self._run(int(nsamp), tb['step'], do_propMH, n_chains=n_chains, device=device)
        return draws, lps

    def _recorded_chain(self):
        """The recorded chain as (n, P) draws in the sampler's element order and (n,) logPost."""
        blocks, _ = self._blocks()
        cols = [np.asarray(b.mcmc.draws, dtype=np.float64).reshape((-1,) + b.val_shape).transpose(0, 2, 1)
                .reshape(-1, b.val.size) for b in blocks]
        return np.concatenate(cols, axis=1), np.asarray(self.params.lp.mcmc.draws, dtype=np.float64)

    def mcmc_diagnostics(self, draws=None, lps=None, nburn=0):
        """Rank-normalized split R-hat, bulk ESS and tail ESS per parameter element (DESIGN.md section 2), on the GPU.
        Without arguments: the model's recorded chain (one chain, split in two).  draws (n, C, P) and lps (n, C), NumPy
        arrays or CUDA tensors as do_mcmc_chains returns them: those chains.  The first nburn draws are left out.
        Returns {name: dict(rhat, ess_bulk, ess_tail)} for betaU, lamUz, lamWs, lamWOs (arrays in each block's val_shape)
        and logPost (scalars).  A fixed element, or one outside mcmcList, is constant: R-hat NaN, ESS = 2 C floor(n / 2)."""
        from .. import diagnostics
        if draws is None:
            if lps is not None:
                raise ValueError('lps without draws')
            d, l = self._recorded_chain()
            if d.shape[0] == 0:
                raise ValueError('no recorded draws')
            draws, lps = d[:, None, :], l[:, None]
        elif lps is None:
            raise ValueError('draws and lps go together')
        return diagnostics.by_block(self._blocks()[0], diagnostics.chain_diagnostics(draws, lps, nburn))

    # ------------------------------------------------------------------ step-size tuning (SURVEY A.6)
    def tune_step_sizes(self, n_burn, n_levels, prog=True, diagnostics=False, update_vals=True, verbose=False,
                        parallel=False):
        """SEPIA's step-size tuning (SURVEY A.6; src/model.py:234): one chain cycles through the ladder of trial sizes,
        n_burn visits per level, then a binomial-logit fit per element picks the size with acceptance 1/e.
        parallel=True (extension, SURVEY 8f rank 4): after the same 10 warm-up steps the n_levels trial sizes run as
        n_levels simultaneous chains of n_burn steps from the warmed-up state (one batched device run, n_levels times
        fewer sequential steps); the acceptance counts feed the same fit and the chain of the middle level hands its
        final state back.  Chain l is bit for bit the chain a single run with trial size l and its slice of the
        np.random stream would produce (tests/test_gpu_api.py)."""
        print('Starting tune_step_sizes...')
        print('Default step sizes:')
        for prm in self.params.mcmcList:
            print('%s' % prm.name)
            print(prm.mcmc.stepParam)
        blocks, _ = self._blocks()
        _, tb = self._get_engine(1)
        P = tb['theta'].size
        n_burn, n_levels = int(n_burn), int(n_levels)
        ex = np.linspace(-(n_levels - 1) / 2.0, (n_levels - 1) / 2.0, n_levels)
        ladder = tb['step'][None, :] * np.power(2.0, ex)[:, None]            # (n_levels, P)
        warm = 10
        saved = [b.val.copy() for b in blocks]
        saved_lp = self.params.lp.val
        bar = _progress(n_burn, 'Step size tuning', prog)
        if parallel:
            draws, lps, _ = self._run(warm, tb['step'], do_propMH=False)
            self._store_state(draws[-1, 0, :])
            draws, lps, acc = self._run(n_burn, ladder[None, :, :], do_propMH=False, n_chains=n_levels, record_accept=True)
            mid = n_levels // 2
            self._store_state(draws[-1, mid, :])
            final_lp = float(lps[-1, mid])
            acc = acc.astype(np.int64).sum(axis=0)                           # accepts per (level, element)
        else:
            nsteps = warm + n_burn * n_levels
            sched = np.empty((nsteps, P))
            sched[:warm] = tb['step']
            sched[warm:] = np.tile(ladder, (n_burn, 1))
            draws, lps, acc = self._run(nsteps, sched, do_propMH=False, record_accept=True)
            self._store_state(draws[-1, 0, :])          # SEPIA copies the tuning chain's final values back
            final_lp = float(lps[-1, 0])
            acc = acc[warm:, 0, :].reshape(n_burn, n_levels, P).sum(axis=0)      # accepts per (level, element)
        if bar is not None:
            bar.update(n_burn)
            bar.close()
        final_blocks = [b.val.copy() for b in blocks]
        target = np.log(1.0 / (np.exp(1.0) - 1.0))
        new_step = tb['step'].copy()
        for e in range(P):
            if tb['fixed'][e]:
                continue
            coef = _logit_glm(np.log(ladder[:, e]), acc[:, e].astype(np.float64), n_burn)
            if coef is not None and np.all(np.isfinite(coef)) and coef[1] < 0:
                lg = (target - coef[0]) / coef[1]
                if np.isfinite(lg) and abs(lg) < 600.0:
                    new_step[e] = np.exp(lg)
        o = 0
        for b, v0, v1 in zip(blocks, saved, final_blocks):
            n = b.val.size
            b.mcmc.stepParam = new_step[o:o + n].reshape(b.val_shape, order='F').copy()
            b.val = v1 if update_vals else v0
            o += n
        self.params.lp.val = final_lp if update_vals else saved_lp
        print('Done with tune_step_size.')
        print('Selected step sizes:')
        for prm in self.params.mcmcList:
            print('%s' % prm.name)
            print(prm.mcmc.stepParam)
        if diagnostics:
            return ladder, acc

    # ------------------------------------------------------------------ samples / persistence (SURVEY A.8)
    def get_num_samples(self):
        return self.params.lamWs.get_num_samples()

    def clear_samples(self):
        for prm in self.params.mcmcList:
            prm.mcmc.draws = []
        self.params.lp.mcmc.draws = []

    def get_samples(self, numsamples=False, nburn=0, sampleset=False, flat=True, includelogpost=True,
                    effectivesamples=False):
        total = self.get_num_samples()
        if total == 0:
            print('No samples to return')
            return None
        ss = np.arange(nburn, total)
        if numsamples is not False and numsamples is not None:
            if numsamples >= total:
                print('numsamples larger than number of draws; truncating to number of draws (%d).' % total)
            else:
                ss = np.array([int(ii) for ii in np.linspace(nburn, total - 1, numsamples)])
        if sampleset is not False and sampleset is not None:
            ss = np.asarray(sampleset, dtype=int)
        samples = {prm.name: prm.mcmc_to_array(sampleset=ss, flat=flat) for prm in self.params.mcmcList}
        if includelogpost:
            samples['logPost'] = np.array(self.params.lp.mcmc.draws, dtype=np.float64)[ss].reshape((-1, 1))
        return samples

    def save_model_info(self, file_name='saved_model', overwrite=True):
        path = file_name + '.pkl'
        if os.path.exists(path) and not overwrite:
            raise FileExistsError(path)
        info = {'samples': self.get_samples(flat=False) if self.get_num_samples() else {}, 'params': {}}
        for prm in self.params.mcmcList:
            info['params'][prm.name] = dict(val=prm.val.copy(), fixed=np.asarray(prm.fixed).copy(),
                                            prior_dist=prm.prior.dist, prior_params=[q.copy() for q in prm.prior.params],
                                            prior_bounds=list(prm.prior.bounds), mcmcStepParam=prm.mcmc.stepParam.copy(),
                                            mcmcStepType=prm.mcmc.stepType)
        with open(path, 'wb') as f:
            pickle.dump(info, f)

    def restore_model_info(self, file_name='saved_model'):
        with open(file_name + '.pkl', 'rb') as f:
            info = pickle.load(f)
        blocks = {b.name: b for b in self._blocks()[0]}
        for name, pi in info.get('params', {}).items():
            b = blocks[name]
            if tuple(pi['val'].shape) != b.val_shape:
                raise ValueError('saved %s has shape %s, model expects %s' % (name, pi['val'].shape, b.val_shape))
            if name == 'lamWOs' and (pi['prior_dist'] != b.prior.dist or pi['mcmcStepType'] != b.mcmc.stepType):
                nb = SepiaParam(val=pi['val'], name=name, val_shape=b.val_shape, dist=pi['prior_dist'],
                                params=pi['prior_params'], bounds=pi['prior_bounds'],
                                mcmcStepParam=pi['mcmcStepParam'], mcmcStepType=pi['mcmcStepType'])
                setattr(self.params, name, nb)
                self.params.mcmcList = [nb if q.name == name else q for q in self.params.mcmcList]
                b = nb
            b.val = pi['val'].copy()
            b.fixed = pi['fixed'].copy()
            b.mcmc.stepParam = pi['mcmcStepParam'].copy()
        samples = info.get('samples') or {}
        for b in self._blocks()[0]:
            if b.name in samples:
                b.mcmc.draws = list(np.asarray(samples[b.name], dtype=np.float64).reshape((-1,) + b.val_shape))
        if 'logPost' in samples:
            self.params.lp.mcmc.draws = list(np.asarray(samples['logPost'], dtype=np.float64).reshape(-1))

    # ------------------------------------------------------------------ printing
    def print_prior_info(self, pnames=None):
        for prm in self.params.mcmcList:
            if pnames is None or prm.name in pnames:
                print('%s prior distribution: %s' % (prm.name, prm.prior.dist))
                print('bounds: ')
                print(prm.prior.bounds)
                for i, q in enumerate(prm.prior.params):
                    print('prior param %d' % i)
                    print(q)

    def print_value_info(self, pnames=None):
        for prm in self.params.mcmcList:
            if pnames is None or prm.name in pnames:
                print('%s shape (%d, %d):' % ((prm.name,) + prm.val_shape))
                print('value:')
                print(prm.val)
                print('is fixed?:')
                print(prm.fixed)

    def print_mcmc_info(self, pnames=None):
        for prm in self.params.mcmcList:
            if pnames is None or prm.name in pnames:
                print('%s stepType: %s' % (prm.name, prm.mcmc.stepType))
                print('stepParam:')
                print(prm.mcmc.stepParam)


class _Rec:
    def __init__(self):
        self.draws = []


class _LogPostRecorder:
    """params.lp upstream: holds the current log posterior and its recorded draws."""

    def __init__(self):
        self.name = 'logPost'
        self.val = -np.inf
        self.mcmc = _Rec()

    def set_val(self, v):
        self.val = float(v)


def _logit_glm(x, k, n, iters=100, tol=1e-10):
    """Binomial-logit IRLS of k accepts out of n on [1, x]: stand-in for the statsmodels GLM that
    SEPIA uses (statsmodels==0.14.1, /root/reference/requirements-cc.txt:45; not installable here)."""
    X = np.stack([np.ones_like(x), x], axis=1)
    y = k / float(n)
    b = np.zeros(2)
    for _ in range(iters):
        eta = np.clip(X @ b, -30, 30)
        mu = 1.0 / (1.0 + np.exp(-eta))
        v = np.maximum(mu * (1.0 - mu), 1e-12)
        W = n * v
        z = eta + (y - mu) / v
        A = X.T @ (W[:, None] * X)
        try:
            bn = np.linalg.solve(A, X.T @ (W * z))
        except np.linalg.LinAlgError:
            return None
        if np.max(np.abs(bn - b)) < tol:
            return bn
        b = bn
    return b
