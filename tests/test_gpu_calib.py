"""GPU: emulator-based calibration (csrc/ggp_calib.cu, ops.calib_loglik / ops.calib_step, gladsgp_b200.calibration)
against the FP64 oracle (oracle/calib_oracle.py): the likelihood, replayed chains, the burn-in proposal, determinism, the
posterior of a two-input problem and a full-field precompute."""
import numpy as np
import pytest

from helpers import synthetic
from oracle import calib_oracle as co
from posterior_helpers import basis, at, calib_obs as _obs, emulator as _oracle, native as _native, \
    scalar_model as _scalar_model, sepia_model as _model

pytestmark = pytest.mark.gpu

LL_RTOL = 1e-9
TIE = 1e-6


def _synthetic_obs(model, em, O, theta_star, obs_sd, seed):
    """y_obs at outputs O: the oracle's posterior-mean prediction at theta_star (transformed) plus N(0, obs_sd^2)."""
    sd = model.data.sim_data
    mu, _ = em.moments(np.asarray(theta_star, dtype=np.float64)[None])
    ystd = mu[:, :, 0].mean(0) @ basis(model)[:, O]
    return ystd * at(model, sd.orig_y_sd, O) + at(model, sd.orig_y_mean, O) + \
        obs_sd * np.random.default_rng(seed).standard_normal(O.size)


@pytest.mark.parametrize('m,q,pu,S', [(64, 1, 1, 1), (100, 3, 2, 7), (64, 8, 10, 7), (100, 3, 32, 7), (512, 8, 10, 64),
                                      (64, 1, 2, 64)])
def test_loglik_matches_oracle(cuda, m, q, pu, S):
    from gladsgp_b200 import calibration as cal
    rng = np.random.default_rng(m + q + pu + S)
    K = None
    if pu > 25:                                              # beyond make_problem's 25 singular vectors
        K = (rng.standard_normal((pu, 200)) * 0.3).astype(np.float32)
    model = _model(m=m, q=q, pu=pu, K=K)
    samples = synthetic.posterior_samples(S, 1 + q, pu, seed=m + S)
    em = _oracle(model, samples)
    n_y = model.num.n_y
    O = np.sort(rng.choice(n_y, size=min(30, n_y), replace=False))
    obs_sd = rng.uniform(0.01, 0.1, O.size)
    y = _synthetic_obs(model, em, O, rng.uniform(0.2, 0.8, q), obs_sd, seed=1)
    tt = rng.uniform(0, 1, (64, q))
    ll, ll_s = cal.log_likelihood(model, samples, y, obs_index=O, obs_sd=obs_sd, t=_native(model, tt), per_sample=True)
    G, b, c0 = _obs(model, O, y, obs_sd, samples)
    ref_s = co.loglik_woodbury(*em.moments(tt), G, b, c0)
    ref = co.log_mean_exp(ref_s)
    assert np.all(np.abs(ll_s - ref_s) <= LL_RTOL * (1 + np.abs(ref_s))), np.max(np.abs(ll_s - ref_s))
    assert np.all(np.abs(ll - ref) <= LL_RTOL * (1 + np.abs(ref))), np.max(np.abs(ll - ref))
    # one call through the public entry point gives the same bits again
    np.testing.assert_array_equal(cal.log_likelihood(model, samples, y, obs_index=O, obs_sd=obs_sd, t=_native(model, tt)),
                                  ll)


def test_loglik_cfg2_scalar_problem(cuda):
    from gladsgp_b200 import calibration as cal
    model = _scalar_model()
    samples = synthetic.posterior_samples(7, 2, 1, seed=4)
    em = _oracle(model, samples)
    O = np.array([0])
    y = _synthetic_obs(model, em, O, [0.4], 0.02, seed=2)
    tt = np.random.default_rng(3).uniform(0, 1, (64, 1))
    ll, ll_s = cal.log_likelihood(model, samples, y, obs_sd=0.02, t=_native(model, tt), per_sample=True)
    G, b, c0 = _obs(model, O, y, 0.02, samples)
    ref_s = co.loglik_woodbury(*em.moments(tt), G, b, c0)
    assert np.all(np.abs(ll_s - ref_s) <= LL_RTOL * (1 + np.abs(ref_s)))
    ref = co.log_mean_exp(ref_s)
    assert np.all(np.abs(ll - ref) <= LL_RTOL * (1 + np.abs(ref)))


def _replay_problem(C, T, seed):
    model = _model(m=64, q=3, pu=2, seed=seed)
    samples = synthetic.posterior_samples(5, 4, 2, seed=seed)
    em = _oracle(model, samples)
    O = np.arange(3, model.num.n_y, 13)
    y = _synthetic_obs(model, em, O, [0.3, 0.5, 0.6], 0.2, seed=seed)
    G, b, c0 = _obs(model, O, y, 0.2, samples)
    rng = np.random.default_rng(seed)
    lo, hi = np.zeros(3), np.ones(3)
    step = np.array([0.25, 0.0, 0.4])                       # input 1 fixed; large steps leave the box often
    theta0 = rng.uniform(0.1, 0.9, (C, 3))
    z = rng.standard_normal((T, C, 3))
    logu = np.log(rng.uniform(size=(T, C)))
    return model, samples, em, O, y, (G, b, c0), (lo, hi, step, theta0, z, logu), rng


def _oracle_chain(em, obs, lo, hi, step, theta0, z, logu, n_burn, rng):
    """Oracle chain with every logu within TIE of its decision's margin re-drawn (the device's l differs in the last bits)."""
    G, b, c0 = obs
    for _ in range(50):
        out = co.chain(lambda th: co.loglik(em, G, b, c0, th), theta0, z, logu, lo, hi, step, n_burn)
        tie = out['margin'] < TIE
        if not tie.any():
            return out, logu
        logu = logu.copy()
        logu[tie] = np.log(rng.uniform(size=int(tie.sum())))
    raise AssertionError('could not avoid near-ties')


@pytest.mark.parametrize('C', [1, 3, 160])
def test_replay_matches_oracle_chain(cuda, C):
    from gladsgp_b200 import calibration as cal
    T, n_burn = 200, 100
    model, samples, em, O, y, obs, (lo, hi, step, theta0, z, logu), rng = _replay_problem(C, T, seed=C)
    ref, logu = _oracle_chain(em, obs, lo, hi, step, theta0, z, logu, n_burn, rng)
    out = cal.calibrate(model, samples, y, obs_index=O, obs_sd=0.2, bounds=_native(model, np.stack([lo, hi])),
                        n_chains=C, n_burn=n_burn, n_steps=T - n_burn, step=step,
                        replay=dict(z=z, logu=logu, theta0=_native(model, theta0)))
    np.testing.assert_array_equal(out['accepted'], ref['accepted'][n_burn:])
    assert np.max(np.abs(out['theta_trans'] - ref['theta'][n_burn:])) <= 1e-12
    np.testing.assert_allclose(out['loglik'], ref['ll'][n_burn:], rtol=LL_RTOL, atol=0)
    assert np.all(out['theta_trans'][:, :, 1] == out['theta_trans'][0, :, 1])          # the fixed input never moves
    cand = [co.propose(ref['theta'][t - 1], ref['L'], z[t]) for t in range(n_burn + 1, T)]
    assert sum(np.sum(~np.all((x >= lo) & (x <= hi), axis=1)) for x in cand) > 0       # rejected outside the box
    np.testing.assert_allclose(out['theta'], _native(model, out['theta_trans']), rtol=1e-15, atol=1e-15)
    np.testing.assert_allclose(out['accept_rate'], ref['accepted'][n_burn:].mean(0), rtol=1e-15)


def test_burnin_proposal_matches_oracle(cuda):
    from gladsgp_b200 import calibration as cal
    C, T, n_burn = 64, 64, 60
    model, samples, em, O, y, obs, (lo, hi, step, theta0, z, logu), rng = _replay_problem(C, T, seed=11)
    ref, logu = _oracle_chain(em, obs, lo, hi, step, theta0, z, logu, n_burn, rng)
    out = cal.calibrate(model, samples, y, obs_index=O, obs_sd=0.2, bounds=_native(model, np.stack([lo, hi])),
                        n_chains=C, n_burn=n_burn, n_steps=T - n_burn, step=step,
                        replay=dict(z=z, logu=logu, theta0=_native(model, theta0)))
    assert np.max(np.abs(out['proposal_chol'] - ref['L'])) <= 1e-12
    assert np.all(ref['L'][1] == 0) and np.all(ref['L'][:, 1] == 0) and ref['L'][2, 0] != 0


def test_same_seed_gives_identical_draws(cuda):
    from gladsgp_b200 import calibration as cal
    model = _model(m=64, q=3, pu=2)
    samples = synthetic.posterior_samples(4, 4, 2, seed=1)
    y = np.asarray(model.data.sim_data.y[7, ::11], dtype=np.float64)
    O = np.arange(0, model.num.n_y, 11)
    kw = dict(obs_index=O, obs_sd=0.1, n_chains=300, n_burn=300, n_steps=20, step=0.1)
    a = cal.calibrate(model, samples, y, seed=5, **kw)
    b = cal.calibrate(model, samples, y, seed=5, **kw)
    c = cal.calibrate(model, samples, y, seed=6, **kw)
    for k in ('theta', 'loglik', 'accepted', 'proposal_chol'):
        np.testing.assert_array_equal(a[k], b[k])
    assert not np.array_equal(a['theta'], c['theta'])


def test_posterior_matches_grid(cuda):
    from gladsgp_b200 import calibration as cal
    model = _model(m=64, q=2, pu=5)
    samples = synthetic.posterior_samples(4, 3, 5, seed=7)
    rr = np.random.default_rng(7)                            # smooth emulators: a unimodal posterior in the box below
    samples['betaU'] = np.exp(rr.uniform(np.log(0.5), np.log(3.0), samples['betaU'].shape)).astype(np.float32)
    samples['lamUz'] = rr.uniform(0.5, 1.5, samples['lamUz'].shape).astype(np.float32)
    em = _oracle(model, samples)
    O = np.arange(5, model.num.n_y, 10)
    y = _synthetic_obs(model, em, O, [0.35, 0.6], 0.05, seed=0)
    lo, hi = np.array([0.0, 0.35]), np.array([0.6, 0.85])
    G, b, c0 = _obs(model, O, y, 0.05, samples)
    g0, g1 = np.linspace(lo[0], hi[0], 201), np.linspace(lo[1], hi[1], 201)
    X0, X1 = np.meshgrid(g0, g1, indexing='ij')
    ll = co.loglik(em, G, b, c0, np.stack([X0.ravel(), X1.ravel()], 1)).reshape(201, 201)
    w = np.exp(ll - ll.max()) * np.outer(np.r_[0.5, np.ones(199), 0.5], np.r_[0.5, np.ones(199), 0.5])   # trapezoid
    w /= w.sum()
    gm = np.array([(w * X0).sum(), (w * X1).sum()])
    gsd = np.sqrt(np.array([(w * (X0 - gm[0]) ** 2).sum(), (w * (X1 - gm[1]) ** 2).sum()]))
    out = cal.calibrate(model, samples, y, obs_index=O, obs_sd=0.05, bounds=_native(model, np.stack([lo, hi])),
                        n_chains=512, n_burn=1000, n_steps=2000, step=0.05, seed=1)
    th = out['theta_trans']
    assert np.all(out['diagnostics']['rhat'] < 1.01), out['diagnostics']['rhat']
    ess = out['diagnostics']['ess_bulk'][:2]
    mean, sd = th.mean(axis=(0, 1)), th.std(axis=(0, 1))
    dev2 = (th - mean) ** 2
    se_mean = sd / np.sqrt(ess)
    se_sd = dev2.reshape(-1, 2).std(0) / np.sqrt(ess) / (2 * sd)
    assert np.all(np.abs(mean - gm) <= 4 * se_mean), (mean, gm, se_mean)
    assert np.all(np.abs(sd - gsd) <= 4 * se_sd), (sd, gsd, se_sd)
    assert 0.05 < float(out['accept_rate'].mean()) < 0.9


def test_full_field(cuda, monkeypatch):
    from gladsgp_b200 import calibration as cal
    model = _model(m=100, q=3, pu=4, n_x=64, n_t=40)
    n_y = model.num.n_y
    samples = synthetic.posterior_samples(6, 4, 4, seed=2)
    em = _oracle(model, samples)
    O = np.arange(n_y)
    sd_o = np.random.default_rng(1).uniform(0.0, 0.2, n_y)
    y = _synthetic_obs(model, em, O, [0.5, 0.4, 0.6], sd_o, seed=3)
    G, b, c0 = _obs(model, O, y, sd_o, samples)
    monkeypatch.setattr(cal, 'OBS_CHUNK_BYTES', 6 * 7 * 8 * 1000)            # 1000 outputs per chunk: several chunks
    Gd, bd, cd = (t.cpu().numpy() for t in cal._obs_terms(model, samples, y, None, sd_o))
    np.testing.assert_allclose(Gd, G, rtol=1e-11, atol=1e-11 * np.abs(G).max())
    np.testing.assert_allclose(bd, b, rtol=1e-11, atol=1e-11 * np.abs(b).max())
    np.testing.assert_allclose(cd, c0, rtol=1e-11)
    assert np.array_equal(Gd, Gd.transpose(0, 2, 1))
    tt = np.random.default_rng(4).uniform(0, 1, (8, 3))
    ll = cal.log_likelihood(model, samples, y, obs_sd=sd_o, t=_native(model, tt))
    ref = co.loglik(em, G, b, c0, tt)
    assert np.all(np.abs(ll - ref) <= LL_RTOL * (1 + np.abs(ref)))
    out = cal.calibrate(model, samples, y, obs_sd=sd_o, n_chains=64, n_burn=20, n_steps=20, step=0.02, seed=3)
    assert out['theta'].shape == (20, 64, 3) and np.all(np.isfinite(out['loglik']))
