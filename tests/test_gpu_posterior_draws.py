"""The sampler and every posterior consumer at draws from a real posterior (tests/golden/posterior_cfg*.npz, made by
tests/golden/make_golden_posterior.py from the oracle sampler at default SEPIA priors), each against the FP64 oracle at
the tolerance its own suite uses.

The other consumer tests run at synthetic.posterior_samples, independent draws from fixed boxes.  The draws here come
from burned-in chains and reach where those never go:

                betaU              lamUz          lamWs          lamWOs         (64 draws each)
  synthetic     0.01 .. 5          0.45 .. 3.6    502 .. 4982    12 .. 196      (half outside the prior support [60, 1e5])
  cfg1          6.5e-4 .. 31       0.41 .. 1.45   126 .. 2899    60.01 .. 60.07 (m=100, q=8, pu=5)
  cfg2          4.2e-3 .. 13.5     0.31 .. 1.50   2418 .. 4172   2119 .. 3428   (m=1000, 1-D GP regression)
  cfg3          1.0e-4 .. 4.57     0.33 .. 3.59   60.06 .. 5477  60.02 .. 60.68 (m=512, q=8, pu=10)

with betaU spanning four decades inside one PC of one draw, and lamWOs at its lower prior bound: the smallest nugget a
chain returns.  Every item takes its draws from _draws(); replace its body by the commented line to rerun them all at
the synthetic draws.

Items: the sampler replaying a burned-in chain (every schedule), distinct chains over more than one wave of CTAs against
the same chains run alone and the oracle, the evaluator at every (draw, PC) block, prediction, cross-validation,
calibration, history matching, sequential design and GP sensitivity."""
import copy

import numpy as np
import pytest
import scipy.linalg

import posterior_helpers as ph
from helpers import so, synthetic, tables_from_oracle
from oracle import calib_oracle as co
from oracle import hm_oracle as ho
from oracle import xval_oracle as xo
from test_gpu_calib import LL_RTOL as CALIB_RTOL, _synthetic_obs
from test_gpu_core import LL_RTOL
from test_gpu_design import _check as _design_check, _oracle as _design_oracle, _points
from test_gpu_gp_sens import _check as _sens_check
from test_gpu_hm import _check as _hm_check
from test_gpu_predict import PRED_RTOL, _blocks

pytestmark = pytest.mark.gpu

_CACHE = {}


def _fixture(cfg):
    if cfg not in _CACHE:
        g = ph.load_posterior(cfg)
        pr = ph.fixture_problem(g)
        num = pr['num']
        _CACHE[cfg] = (g, pr, num.d, num.pu)
    return _CACHE[cfg]


def _draws(cfg):
    """(64, P) posterior draws in sampling order: the one place every item below takes its draws from."""
    g, _, d, pu = _fixture(cfg)
    return g['draws']
    # s = synthetic.posterior_samples(64, d, pu, f32=False); return np.concatenate([s[k] for k in ('betaU', 'lamUz', 'lamWs', 'lamWOs')], 1)


def _samples(cfg, idx=None):
    _, _, d, pu = _fixture(cfg)
    dr = _draws(cfg)
    return ph.split_draws(dr if idx is None else dr[idx], d, pu)


def _widest(cfg, n):
    """Indices of the n draws with the largest betaU, ascending: where a subset must do, the draws furthest out."""
    _, _, d, pu = _fixture(cfg)
    return np.sort(np.argsort(_draws(cfg)[:, :d * pu].max(1))[-n:])


def _model(cfg):
    """SepiaModel of the fixture's problem with the design left as it is (zt equal to the chain's)."""
    key = ('model', cfg)
    if key not in _CACHE:
        g, pr, _, _ = _fixture(cfg)
        _CACHE[key] = ph.sepia_model_of(pr, t_notrans=True) if str(g['kind']) == 'pca' else \
            ph.scalar_model_of(pr, t_notrans=True)
    return _CACHE[key]


def _emulator(cfg):
    key = ('em', cfg)
    if key not in _CACHE:
        _CACHE[key] = ph.emulator(_model(cfg), _samples(cfg))
    return _CACHE[key]


def _report(item, ratio):
    print('%s: largest error / tolerance %.3g' % (item, ratio))


# --------------------------------------------------------------------------------------------------------------------
# sampler
# --------------------------------------------------------------------------------------------------------------------
def _engine(cfg, n_chains):
    from gladsgp_b200 import ops
    g, pr, _, _ = _fixture(cfg)
    tb = {k[3:]: g[k] for k in g if k.startswith('tb_')}
    eng = ops.McmcEngine(pr['num'].zt, np.ascontiguousarray(g['w'].T), g['LamSim'], tb, n_chains=n_chains)
    return eng, tb


SCHEDULES = {'default': {}, 'cluster1': {'GGP_CLUSTER': '1'}, 'spec0': {'GGP_SPEC': '0'}, 'spec1': {'GGP_SPEC': '1'}}


@pytest.mark.parametrize('schedule', list(SCHEDULES))
@pytest.mark.parametrize('cfg', ['cfg1', 'cfg2', 'cfg3'])
def test_sampler_replays_the_burned_in_chain(cuda, monkeypatch, cfg, schedule):
    """From the chain's final state, the oracle's next n_replay steps (proposals and uniforms replayed): every decision
    and every draw bit-identical, lp within 1e-9 (as tests/test_gpu_chains.py from the prior defaults)."""
    for k, v in SCHEDULES[schedule].items():
        monkeypatch.setenv(k, v)
    g = _fixture(cfg)[0]
    eng, tb = _engine(cfg, 1)
    eng.set_state(g['state'])
    replay = {k[3:]: g[k] for k in g if k.startswith('rp_')}
    out = eng.run(int(g['n_steps']), tb['step'], replay=replay, record_accept=True)
    assert np.array_equal(out['accepted'].cpu().numpy(), g['chain_acc'])
    assert np.array_equal(out['draws'].cpu().numpy()[:, 0, :], g['chain_draws'])
    lp = out['lp'].cpu().numpy()[:, 0]
    np.testing.assert_allclose(lp, g['chain_lp'], rtol=1e-9)
    _report('replay %s %s (lp)' % (cfg, schedule), np.max(np.abs(lp - g['chain_lp']) / (1e-9 * np.abs(g['chain_lp']))))


class _Stream:
    """The uniform stream of a device chain as the oracle's rng."""

    def __init__(self, u):
        self.u, self.i = u, 0

    def random_sample(self):
        self.i += 1
        return self.u[self.i - 1]


def _oracle_stream_chain(cfg, state, us, steps):
    """The oracle chain on the fixture's model data and tables from `state`, fed the uniforms us."""
    g, pr, d, pu = _fixture(cfg)
    num = copy.copy(pr['num'])
    num.w = np.asarray(g['w'], dtype=np.float64)
    num.wv = num.w.reshape((-1, 1), order='F')
    num.LamSim = np.asarray(g['LamSim'], dtype=np.float64)
    mod = so.OracleModel(num)
    mod.lamWOs.params = [np.full((1, 1), g['tb_prior_a'][-1]), np.full((1, 1), g['tb_prior_b'][-1])]
    tb = tables_from_oracle(mod)
    for k in ('prior_kind', 'prior_a', 'prior_b', 'lo', 'hi', 'prop_kind', 'fixed', 'step'):
        assert np.array_equal(tb[k], g['tb_' + k]), k
    nb = d * pu
    mod.betaU.val = state[:nb].reshape((d, pu), order='F').copy()
    mod.lamUz.val = state[nb:nb + pu].reshape(1, pu).copy()
    mod.lamWs.val = state[nb + pu:nb + 2 * pu].reshape(1, pu).copy()
    mod.lamWOs.val = state[-1:].reshape(1, 1).copy()
    mod.trace = []
    rng = _Stream(us)
    mod.do_mcmc(steps, rng=rng)
    s = mod.get_samples()
    draws = np.concatenate([s['betaU'], s['lamUz'], s['lamWs'], s['lamWOs']], axis=1)
    acc = np.array([tr['accept'] for tr in mod.trace], dtype=np.uint8).reshape(steps, -1)
    return draws, acc, s['logPost'][:, 0], rng.i


def test_distinct_chains_over_more_than_one_wave(cuda):
    """cfg3, 160 chains in 160 states (the 64 draws under a fixed permutation, repeated), each with its own uniform stream:
    1600 matrices per evaluation round, more than the 592 one-CTA slots of a B200.  Four steps in stream mode; every chain
    equals, bit for bit, the same chain run alone, and 8 of them the oracle fed the same uniforms.

    Against the oracle the decisions and the uniforms consumed are compared exactly and the draws to 1e-12 relative, as in
    tests/test_gpu_core.py::test_mcmc_uniform_stream_matches_oracle: the betaU proposal -4 log(exp(-x/4) + step (u - 1/2))
    is formed with the device's exp and log, within an ulp of the host's."""
    g = _fixture('cfg3')[0]
    C, steps = 160, 4
    dr = _draws('cfg3')
    states = dr[np.resize(np.random.RandomState(17).permutation(dr.shape[0]), C)]
    P = states.shape[1]
    us = np.random.RandomState(23).random_sample((C, 2 * P * steps))
    eng, tb = _engine('cfg3', C)
    eng.set_state(states)
    out = eng.run(steps, tb['step'], uniforms=us, record_accept=True)
    draws, lp = out['draws'].cpu().numpy(), out['lp'].cpu().numpy()
    acc, used = out['accepted'].cpu().numpy(), out['consumed'].cpu().numpy().copy()
    assert np.all(np.isfinite(lp))
    assert np.any(draws[-1] != states)                        # the chains moved
    one, _ = _engine('cfg3', 1)
    for c in range(C):
        one.set_state(states[c])
        o = one.run(steps, tb['step'], uniforms=us[c:c + 1], record_accept=True)
        assert np.array_equal(o['draws'].cpu().numpy()[:, 0], draws[:, c]), c
        assert np.array_equal(o['lp'].cpu().numpy()[:, 0], lp[:, c]), c
        assert np.array_equal(o['accepted'].cpu().numpy()[:, 0], acc[:, c]), c
        assert int(o['consumed'].cpu().numpy()[0]) == used[c], c
    worst = 0.0
    for c in np.linspace(0, C - 1, 8).astype(int):
        rd, racc, rlp, rused = _oracle_stream_chain('cfg3', states[c], us[c], steps)
        assert np.array_equal(acc[:, c], racc), c
        assert int(used[c]) == rused, c
        np.testing.assert_allclose(draws[:, c], rd, rtol=1e-12, atol=0)
        np.testing.assert_allclose(lp[:, c], rlp, rtol=1e-9)
        worst = max(worst, float(np.max(np.abs(draws[:, c] - rd) / (1e-12 * np.abs(rd)))))
    _report('distinct chains vs oracle (draws)', worst)


# --------------------------------------------------------------------------------------------------------------------
# evaluator
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('cfg', ['cfg1', 'cfg3'])
def test_evaluator_at_every_draw_and_pc(cuda, monkeypatch, cfg):
    """loglik_batched at every (draw, PC) block (640 matrices at cfg3) under both schedules, bit for bit the same, and
    against so.do_loglik / np.linalg.cholesky at the bars of test_gpu_core.py::test_cov_and_loglik_match_oracle;
    cov_build against so.block_cov at 1e-13 on the blocks of the largest betaU."""
    import torch
    from gladsgp_b200 import _lib, ops
    _, pr, d, pu = _fixture(cfg)
    num = pr['num']
    m = num.m
    samples = _samples(cfg)
    beta, lamz, dadd, s11, W = _blocks(num, samples)
    B = beta.shape[0]
    # the packed factor workspace (csrc/ggp_common.cuh) holds the panels of L, the inverted diagonal blocks that the
    # prediction and cross-validation kernels read, and then Mp + 64 doubles of scratch that only the cluster schedule
    # uses (its running forward solve, u block and failure flag): everything before that scratch must agree
    lib = _lib.load()
    n_factor = lib.ggp_factor_doubles(m) - lib.ggp_padded_m(m) - 64
    res = {}
    for cl in ('1', '4'):
        monkeypatch.setenv('GGP_CLUSTER', cl)
        res[cl] = ops.loglik_batched(num.zt, W, beta, lamz, dadd, want_factor=True, want_u=True)
        res[cl]['factor'] = res[cl]['factor'][:, :n_factor]
    for k in ('loglik', 'info', 'factor', 'u'):
        assert torch.equal(res['1'][k], res['4'][k]), k
    out = res['4']
    assert not out['info'].any().item()
    ll = out['loglik'].cpu().numpy()
    ug = out['u'].cpu().numpy()[:, :m]
    lw = samples['lamWs']; lo = samples['lamWOs'][:, 0]; lz = samples['lamUz']
    r_ll = r_L = r_u = 0.0
    chunk = 64
    for b0 in range(0, B, chunk):
        Lg = ops.factor_unpack(out['factor'][b0:b0 + chunk], m).cpu().numpy()
        for b in range(b0, min(B, b0 + chunk)):
            s, j = divmod(b, pu)
            C = so.block_cov(num, beta[b], lz[s, j], lw[s, j], lo[s], j)
            ref = so.do_loglik(C, W[b])
            r_ll = max(r_ll, abs(ll[b] - ref) / (LL_RTOL * abs(ref)))
            L = np.linalg.cholesky(C)
            r_L = max(r_L, np.abs(Lg[b - b0] - L).max() / (1e-9 * np.abs(L).max()))
            u = scipy.linalg.solve_triangular(L, W[b], lower=True)
            r_u = max(r_u, np.abs(ug[b] - u).max() / (1e-8 * np.abs(u).max()))
    _report('evaluator %s: loglik / factor / u' % cfg, max(r_ll, r_L, r_u))
    print('  loglik %.3g  factor %.3g  u %.3g' % (r_ll, r_L, r_u))
    assert r_ll <= 1.0 and r_L <= 1.0 and r_u <= 1.0
    top = np.argsort(beta.max(1))[-(B if B <= 320 else 16):]
    Cg = ops.cov_build(num.zt, beta[top], lamz[top], dadd[top]).cpu().numpy()
    r_c = 0.0
    for i, b in enumerate(top):
        s, j = divmod(int(b), pu)
        C = so.block_cov(num, beta[b], lz[s, j], lw[s, j], lo[s], j)
        np.testing.assert_allclose(Cg[i], C, rtol=1e-13, atol=1e-300)
        r_c = max(r_c, float(np.max(np.abs(Cg[i] - C) / (1e-13 * np.abs(C) + 1e-300))))
    _report('cov_build %s (largest betaU %.3g)' % (cfg, beta[top].max()), r_c)


# --------------------------------------------------------------------------------------------------------------------
# prediction and cross-validation
# --------------------------------------------------------------------------------------------------------------------
def test_predictor_at_cfg3_draws(cuda):
    """Predictor.predict and pred_cov, the 16 draws of the largest betaU and 256 LHS designs, against so.w_pred at the
    bars of test_gpu_predict.py::test_predict_moments_match_oracle."""
    from gladsgp_b200 import ops
    _, pr, d, pu = _fixture('cfg3')
    num = pr['num']
    samples = _samples('cfg3', _widest('cfg3', 16))
    ns, npred = 16, 256
    tp = synthetic.test_design(npred, num.q)
    beta, lamz, dadd, s11, W = _blocks(num, samples)
    P = ops.Predictor(num.zt, W, beta, lamz, dadd, s11)
    assert not P.info.any().item()
    xp = np.concatenate([0.5 * np.ones((npred, 1)), tp.astype(np.float64)], axis=1)
    mean, var, V = P.predict(xp, want_V=True)
    Sg = P.pred_cov(xp, V).cpu().numpy()
    mean = mean.cpu().numpy(); var = var.cpu().numpy()
    refs = []
    for s in range(ns):                                      # one sample at a time: Sigma is (pu npred)^2 per sample
        one = {k: v[s:s + 1] for k, v in samples.items()}
        _, mu, Sig = so.w_pred(num, tp, one, draw=False)
        refs.append((mu[0], np.stack([Sig[0, j * npred:(j + 1) * npred, j * npred:(j + 1) * npred] for j in range(pu)])))
    scale = max(np.abs(r[0]).max() for r in refs)
    worst = 0.0
    for s, (mu, Sj) in enumerate(refs):
        for j in range(pu):
            b = s * pu + j
            sl = slice(j * npred, (j + 1) * npred)
            np.testing.assert_allclose(mean[b], mu[sl], rtol=PRED_RTOL, atol=PRED_RTOL * scale)
            np.testing.assert_allclose(var[b], np.diag(Sj[j]), rtol=PRED_RTOL)
            np.testing.assert_allclose(Sg[b], Sj[j], rtol=PRED_RTOL, atol=PRED_RTOL * np.abs(Sj[j]).max())
            worst = max(worst, np.max(np.abs(mean[b] - mu[sl]) / (PRED_RTOL * (np.abs(mu[sl]) + scale))),
                        np.max(np.abs(var[b] - np.diag(Sj[j])) / (PRED_RTOL * np.abs(np.diag(Sj[j])))))
    _report('Predictor cfg3 (mean / var)', worst)


def test_public_prediction_at_cfg1_draws(cuda):
    """SepiaEmulatorPrediction(storeMuSigma=True) at all 64 draws against so.w_pred on the model's own data."""
    from sepia.SepiaPredict import SepiaEmulatorPrediction
    model = _model('cfg1')
    samples = _samples('cfg1')
    tp = synthetic.test_design(40, model.num.q)
    np.random.seed(0)
    pe = SepiaEmulatorPrediction(t_pred=tp, samples=samples, model=model, storeRlz=False, storeMuSigma=True)
    _, mu, Sig = so.w_pred(ph.oracle_num(model), tp, samples, draw=False)
    np.testing.assert_allclose(pe.mu, mu, rtol=PRED_RTOL, atol=PRED_RTOL * np.abs(mu).max())
    np.testing.assert_allclose(pe.sigma, Sig, rtol=PRED_RTOL, atol=PRED_RTOL * np.abs(Sig).max())
    dg, rdg = np.diagonal(pe.sigma, axis1=1, axis2=2), np.diagonal(Sig, axis1=1, axis2=2)
    np.testing.assert_allclose(dg, rdg, rtol=PRED_RTOL)
    _report('SepiaEmulatorPrediction cfg1 (mean / var)',
            max(np.max(np.abs(pe.mu - mu) / (PRED_RTOL * (np.abs(mu) + np.abs(mu).max()))),
                np.max(np.abs(dg - rdg) / (PRED_RTOL * np.abs(rdg)))))


def test_xval_at_cfg1_draws(cuda):
    """SepiaXvalEmulatorPrediction, leave-one-out and a 5-fold split, all 64 draws, against oracle/xval_oracle.py at the
    bars of tests/test_gpu_xval.py.  lamWOs = 60 is the smallest nugget of the prior: there the closed form
    mu = w - alpha / p cancels most."""
    from sepia.SepiaPredict import SepiaXvalEmulatorPrediction
    model = _model('cfg1')
    samples = _samples('cfg1')
    num = ph.oracle_num(model)
    m, pu = num.m, num.pu
    ns = samples['lamWs'].shape[0]
    loo = SepiaXvalEmulatorPrediction(samples=samples, model=model, storeRlz=False, storeMuSigma=True)
    check = sorted({0, 1, 2, 7, 13, 20, 31, 32, 40, 49, 50, 63, 64, 71, 77, 85, 90, 96, 98, m - 1})
    _, ref_mu, ref_Sig = xo.xval_pred(num, samples, [[i] for i in check], draw=False)
    mu = np.stack([loo.mu[i] for i in check], axis=-1)                      # (ns, pu, n)
    var = np.stack([np.diagonal(loo.sigma[i], axis1=1, axis2=2) for i in check], axis=-1)
    rm = np.stack(ref_mu, axis=-1)
    rv = np.stack([np.diagonal(S, axis1=1, axis2=2) for S in ref_Sig], axis=-1)
    np.testing.assert_allclose(mu, rm, rtol=PRED_RTOL, atol=PRED_RTOL * np.abs(rm).max())
    np.testing.assert_allclose(var, rv, rtol=PRED_RTOL)
    worst = max(np.max(np.abs(mu - rm) / (PRED_RTOL * (np.abs(rm) + np.abs(rm).max()))),
                np.max(np.abs(var - rv) / (PRED_RTOL * np.abs(rv))))
    folds = [list(f) for f in np.array_split(np.random.RandomState(5).permutation(m), 5)]
    xv = SepiaXvalEmulatorPrediction(samples=samples, model=model, leave_out_inds=folds, storeRlz=False,
                                     storeMuSigma=True)
    _, ref_mu, ref_Sig = xo.xval_pred(num, samples, folds, draw=False)
    for k, f in enumerate(folds):
        n = len(f)
        np.testing.assert_allclose(xv.mu[k], ref_mu[k], rtol=PRED_RTOL, atol=PRED_RTOL * np.abs(ref_mu[k]).max())
        np.testing.assert_allclose(xv.sigma[k], ref_Sig[k], rtol=PRED_RTOL, atol=PRED_RTOL * np.abs(ref_Sig[k]).max())
        dg, rdg = np.diagonal(xv.sigma[k], axis1=1, axis2=2), np.diagonal(ref_Sig[k], axis1=1, axis2=2)
        np.testing.assert_allclose(dg, rdg, rtol=PRED_RTOL)
        assert xv.mu[k].shape == (ns, pu * n)
        worst = max(worst, np.max(np.abs(xv.mu[k] - ref_mu[k]) / (PRED_RTOL * (np.abs(ref_mu[k]) +
                                                                                 np.abs(ref_mu[k]).max()))),
                    np.max(np.abs(dg - rdg) / (PRED_RTOL * np.abs(rdg))))
    _report('cross-validation cfg1 (mean / var)', worst)


# --------------------------------------------------------------------------------------------------------------------
# consumers
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('cfg', ['cfg1', 'cfg2', 'cfg3'])
def test_calibration_loglik(cuda, cfg):
    """Per-sample and mixed calibration log-likelihoods at 64 inputs against calib_oracle, LL_RTOL of test_gpu_calib.py."""
    from gladsgp_b200 import calibration as cal
    model = _model(cfg)
    samples = _samples(cfg)
    em = _emulator(cfg)
    q, n_y = model.num.q, model.num.n_y
    rng = np.random.default_rng(int(cfg[-1]))
    if model.data.scalar_out:
        O, obs_sd, O_arg = np.array([0]), 0.02, None
    else:
        O = np.sort(rng.choice(n_y, size=min(30, n_y), replace=False))
        obs_sd, O_arg = rng.uniform(0.01, 0.1, O.size), O
    y = _synthetic_obs(model, em, O, rng.uniform(0.2, 0.8, q), obs_sd, seed=1)
    tt = rng.uniform(0, 1, (64, q))
    ll, ll_s = cal.log_likelihood(model, samples, y, obs_index=O_arg, obs_sd=obs_sd, t=ph.native(model, tt),
                                  per_sample=True)
    G, b, c0 = ph.calib_obs(model, O, y, obs_sd, samples)
    ref_s = co.loglik_woodbury(*em.moments(tt), G, b, c0)
    ref = co.log_mean_exp(ref_s)
    r_s = np.max(np.abs(ll_s - ref_s) / (CALIB_RTOL * (1 + np.abs(ref_s))))
    r = np.max(np.abs(ll - ref) / (CALIB_RTOL * (1 + np.abs(ref))))
    _report('calibration %s (per sample / mixed)' % cfg, max(r_s, r))
    assert r_s <= 1.0 and r <= 1.0, (r_s, r)


@pytest.mark.parametrize('cfg', ['cfg1', 'cfg3'])
def test_history_matching(cuda, cfg):
    """Implausibilities, counts and the region not ruled out at 300 inputs (100 at cfg3), third-largest implausibility, per-output
    observation and discrepancy sds, against hm_oracle with test_gpu_hm.py's _check."""
    from gladsgp_b200 import history
    model = _model(cfg)
    samples = _samples(cfg)
    em = _emulator(cfg)
    q, n_y = model.num.q, model.num.n_y
    rng = np.random.default_rng(10 + int(cfg[-1]))
    O = np.sort(rng.choice(n_y, size=100, replace=False))
    ysd = ph.at(model, model.data.sim_data.orig_y_sd, O)
    obs_sd = rng.uniform(0.01, 0.1, O.size) * ysd
    disc_sd = rng.uniform(0.0, 0.2, O.size) * ysd
    y = ph.mean_field(model, em, O, rng.uniform(0.2, 0.8, q)) + rng.standard_normal(O.size) * 0.05 * ysd
    tt = rng.uniform(0, 1, (300 if cfg == 'cfg1' else 100, q))
    out = history.history_match(model, samples, y, ph.native(model, tt), obs_index=O, obs_sd=obs_sd, disc_sd=disc_sd,
                                order=3, cutoff=3.0)
    K_O, r, c = ph.hm_obs(model, samples, O, y, obs_sd, disc_sd)
    ref = ho.history_match(em, tt, K_O, r, c, 3, 3.0)
    worst = _hm_check(out, ref, 3.0)
    _report('history matching %s (impl error / scale)' % cfg, worst / 1e-12)
    print('  nroy fraction %.3f' % out['nroy_fraction'])


@pytest.mark.parametrize('cfg', ['cfg1', 'cfg3'])
def test_design_next_runs(cuda, cfg):
    """Six greedy picks from 150 candidates over 100 reference inputs against design_oracle with test_gpu_design.py's
    _check (all 64 draws at cfg1, the 16 of the largest betaU at cfg3)."""
    from gladsgp_b200 import design
    model = _model(cfg)
    samples = _samples(cfg, None if cfg == 'cfg1' else _widest(cfg, 16))
    C = _points(model, 150, seed=1)
    R = _points(model, 100, seed=2)
    out = design.next_runs(model, samples, C, 6, reference=R)
    ref = _design_oracle(model, samples, C, R, 6, out['pc_weights'])
    n, worst = _design_check(out, ref, samples)
    assert n >= 3, (n, ref['margin'])
    _report('design %s (error / cancellation term, %d picks compared)' % (cfg, n), worst)


@pytest.mark.parametrize('option', ['samples', 'mean'])
@pytest.mark.parametrize('cfg', ['cfg1', 'cfg2', 'cfg3'])
def test_gp_sensitivity(cuda, cfg, option):
    """Moments, indices and main-effect curves of the emulator expansion of the draws (sensitivity.emulator_expansion)
    against gp_sens_oracle with test_gpu_gp_sens.py's _check.  The oracle's pair sums cost (S m)^2 per function in the mean
    mode: there it takes the draws of the largest betaU (8 at cfg1, 3 at cfg2, 2 at cfg3); the per-sample mode takes all
    64 draws.  At cfg3 the oracle checks the 8 blocks (per sample) or 3 PCs (mean) of the largest betaU."""
    from gladsgp_b200 import sensitivity
    model = _model(cfg)
    idx = None if option == 'samples' else _widest(cfg, {'cfg1': 8, 'cfg2': 3, 'cfg3': 2}[cfg])
    samples = _samples(cfg, idx)
    Z, beta, a, ns = sensitivity.emulator_expansion(model, samples)
    pu, m = model.num.pu, model.num.m
    Zin = Z.cpu().numpy()
    beta = beta.cpu().numpy().reshape(ns, pu, -1)
    a = a.cpu().numpy().reshape(ns, pu, m)
    which = None
    if cfg == 'cfg3':
        wide = beta.reshape(ns * pu, -1).max(1) if option == 'samples' else beta.max(axis=(0, 2))
        which = sorted(int(f) for f in np.argsort(wide)[-(8 if option == 'samples' else 3):])
    worst = _sens_check(Zin, beta, a, option, which=which)
    _report('gp_sens %s %s (indices; largest betaU %.3g)' % (cfg, option, beta.max()), worst)
