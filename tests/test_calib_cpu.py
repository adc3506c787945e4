"""CPU: the calibration oracle (oracle/calib_oracle.py) -- Woodbury against the dense covariance, log-mean-exp, the replay
chain's box rejection and fixed inputs -- and the argument checks of the C entry points and of
gladsgp_b200.calibration (no device needed)."""
import ctypes

import numpy as np
import pytest
from scipy import special, stats

from helpers import make_problem, synthetic
from oracle import calib_oracle as co

WOODBURY_RTOL = 1e-12


def _obs_case(rng, pu, n_o, per_column_sd, obs_sd_kind):
    K = rng.standard_normal((pu, n_o)) * rng.uniform(0.2, 2.0, (pu, 1)) + 0.3 * rng.standard_normal((1, n_o))
    ymean = rng.standard_normal(n_o)
    ysd = rng.uniform(0.5, 3.0, n_o) if per_column_sd else np.full(n_o, 1.7)
    y = ymean + ysd * rng.standard_normal(n_o)
    obs_sd = {'scalar': 0.3, 'per_output': rng.uniform(0.0, 0.5, n_o), 'zero': 0.0}[obs_sd_kind]
    r, tau = co.standardized_obs(y, obs_sd, ymean, ysd)
    return K, r, tau


@pytest.mark.parametrize('pu', [1, 3, 10])
@pytest.mark.parametrize('n_o', [1, 5, 300])
@pytest.mark.parametrize('per_column_sd', [False, True])
@pytest.mark.parametrize('obs_sd_kind', ['scalar', 'per_output', 'zero'])
def test_woodbury_matches_dense_logpdf(pu, n_o, per_column_sd, obs_sd_kind):
    rng = np.random.default_rng(pu * 1000 + n_o + 7 * per_column_sd + len(obs_sd_kind))
    K, r, tau = _obs_case(rng, pu, n_o, per_column_sd, obs_sd_kind)
    S, N = 3, 4
    lamWOs = rng.uniform(10.0, 300.0, S)
    mu = rng.standard_normal((S, pu, N))
    var = rng.uniform(0.0, 0.5, (S, pu, N))
    var[0, 0, 0] = 0.0
    G, b, c0 = co.obs_terms(K, r, tau, lamWOs)
    got = co.loglik_woodbury(mu, var, G, b, c0)
    for s in range(S):
        for p in range(N):
            cov = np.diag(1.0 / lamWOs[s] + tau ** 2) + K.T @ (var[s, :, p][:, None] * K)
            ref = stats.multivariate_normal.logpdf(r, mean=K.T @ mu[s, :, p], cov=cov)
            assert abs(got[s, p] - ref) <= WOODBURY_RTOL * abs(ref), (s, p, got[s, p], ref)


def test_emulator_moments_are_w_pred_moments():
    pr = make_problem(m=40, q=2, pu=3, n_x=10, n_t=6, seed=4)
    num = pr['num']
    samples = synthetic.posterior_samples(3, num.d, num.pu, seed=2, f32=False)
    rng = np.random.default_rng(1)
    t = rng.uniform(0, 1, (5, 2))
    K = np.asarray(pr['K'], dtype=np.float64)
    O = np.array([0, 7, 19, 33])
    r, tau = co.standardized_obs(rng.standard_normal(O.size), 0.1, 0.0, 1.0)
    lamWOs = np.asarray(samples['lamWOs'], dtype=np.float64).reshape(-1)
    G, b, c0 = co.obs_terms(K[:, O], r, tau, lamWOs)
    mu, var = co.Emulator(num, samples).moments(t)
    wood = co.loglik_woodbury(mu, var, G, b, c0)
    for p in range(t.shape[0]):
        dense = co.loglik_dense(num, t[p], samples, K[:, O], r, tau)
        np.testing.assert_allclose(wood[:, p], dense, rtol=1e-10)


def test_log_mean_exp_with_distant_terms():
    ls = np.array([[-1000.0, -5000.0], [0.0, -4000.0], [-2000.0, -6000.0]])
    got = co.log_mean_exp(ls)
    assert np.all(np.isfinite(got))
    np.testing.assert_allclose(got, special.logsumexp(ls, axis=0) - np.log(3), rtol=1e-15)
    np.testing.assert_allclose(got[0], -np.log(3.0), rtol=1e-15)
    np.testing.assert_allclose(got[1], -4000.0 - np.log(3.0), rtol=1e-15)


def test_oracle_chain_rejects_outside_box_and_keeps_fixed_inputs():
    rng = np.random.default_rng(3)
    T, C, q = 300, 5, 3
    lo, hi = np.array([0.0, 0.0, 0.2]), np.array([1.0, 1.0, 0.8])
    step = np.array([0.6, 0.0, 0.3])                       # large steps: many proposals leave the box

    def loglik(th):
        return -0.5 * np.sum(((th - 0.5) / 0.2) ** 2, axis=1)
    theta0 = rng.uniform(lo, hi, (C, q))
    z = rng.standard_normal((T, C, q))
    logu = np.log(rng.uniform(size=(T, C)))
    out = co.chain(loglik, theta0, z, logu, lo, hi, step, n_burn=100)
    th = out['theta']
    assert np.all((th >= lo) & (th <= hi))
    np.testing.assert_array_equal(th[:, :, 1], np.broadcast_to(theta0[:, 1], (T, C)))
    assert np.all(out['L'][1] == 0.0) and np.all(out['L'][:, 1] == 0.0)
    # replay the candidates: outside the box -> never accepted, margin inf; inside -> the Metropolis rule
    prev, L = theta0, np.diag(step)
    n_out = 0
    for t in range(T):
        cand = co.propose(prev, L, z[t])
        outside = ~np.all((cand >= lo) & (cand <= hi), axis=1)
        n_out += outside.sum()
        assert not np.any(out['accepted'][t] & outside)
        assert np.all(np.isinf(out['margin'][t, outside]))
        inside = ~outside
        acc = logu[t, inside] < loglik(cand[inside]) - loglik(prev[inside])
        np.testing.assert_array_equal(out['accepted'][t, inside], acc)
        prev = th[t]
        if t == 99:
            L = co.burnin_chol(th[50:100], step)
    assert n_out > 50
    np.testing.assert_array_equal(L, out['L'])


def test_burnin_chol_falls_back_to_diagonal():
    step = np.array([0.1, 0.2])
    same = np.ones((10, 4, 2))                              # zero covariance: Cholesky fails
    np.testing.assert_array_equal(co.burnin_chol(same, step), np.diag(step))
    x = np.random.default_rng(0).standard_normal((50, 8, 2))
    L = co.burnin_chol(x, step)
    np.testing.assert_allclose(L @ L.T, np.cov(x.reshape(-1, 2), rowvar=False) * 2.38 ** 2 / 2, rtol=1e-13)


def test_calib_abi_validates_arguments_without_a_device():
    from gladsgp_b200 import _lib
    h = _lib.load()
    one = ctypes.c_void_p(8)
    # mean, var, S, pu, n, G, b, c0, ll, ll_s, stream
    args = [one, one, 4, 3, 10, one, one, one, one, None, None]
    for k in (0, 1, 5, 6, 7, 8):
        a = list(args)
        a[k] = None
        assert h.ggp_calib_loglik_f64(*a) == -1
        assert b'null pointer' in h.ggp_last_error_string()
    for k, v, msg in ((3, 0, b'pu must be'), (3, 33, b'pu must be'), (2, 0, b'must be positive'), (2, -1, b'must be positive'),
                      (4, 0, b'must be positive'), (2, 1 << 30, b'2^31')):
        a = list(args)
        a[k] = v
        assert h.ggp_calib_loglik_f64(*a) == -1
        assert msg in h.ggp_last_error_string()
    # mean, var, S, pu, C, G, b, c0, Xp, d, q, lo, hi, L, z_next, logu, theta, ll, rec_theta, rec_ll, rec_acc, stream
    sargs = [one, one, 4, 3, 10, one, one, one, one, 3, 2, one, one, one, None, one, one, one, one, one, one, None]
    for k in (0, 1, 5, 6, 7, 8, 11, 12, 13, 15, 16, 17, 18, 19, 20):
        a = list(sargs)
        a[k] = None
        assert h.ggp_calib_step_f64(*a) == -1
        assert b'null pointer' in h.ggp_last_error_string()
    for k, v, msg in ((3, 33, b'pu must be'), (3, 0, b'pu must be'), (10, 33, b'q must be'), (10, 0, b'q must be'),
                      (9, 1, b'd must be'), (2, 0, b'must be positive'), (4, 0, b'must be positive'),
                      (4, -5, b'must be positive')):
        a = list(sargs)
        a[k] = v
        assert h.ggp_calib_step_f64(*a) == -1
        assert msg in h.ggp_last_error_string()


def _model(q=2, pu=3, x_sim=False, m=40, K=None):
    from sepia.SepiaData import SepiaData
    from sepia.SepiaModel import SepiaModel
    pr = make_problem(m=m, q=q, pu=pu, n_x=10, n_t=6, seed=5)
    kw = dict(y_sim=pr['y'], y_ind_sim=np.arange(pr['y'].shape[1], dtype=float))
    if x_sim:
        kw['x_sim'] = pr['t']
    else:
        kw['t_sim'] = pr['t']
    data = SepiaData(**kw)
    data.transform_xt()
    data.standardize_y(y_mean=pr['mu'], y_sd=pr['sd'])
    data.create_K_basis(K=pr['K'] if K is None else K)
    return SepiaModel(data)


def test_calibration_value_errors():
    from gladsgp_b200 import calibration as cal
    model = _model()
    d, pu, n_y = model.num.p + model.num.q, model.num.pu, model.num.n_y
    samples = synthetic.posterior_samples(2, d, pu, seed=1)
    y = np.zeros(3)
    ok = dict(y_obs=y, obs_index=[0, 5, 9])
    bad = [
        dict(obs_index=[0, 5, n_y]),                        # out of range
        dict(obs_index=[0, -1, 9]),
        dict(obs_index=[0, 5, 5]),                          # repeated
        dict(y_obs=np.zeros(4)),                            # y_obs length mismatch
        dict(obs_sd=np.ones(2)),                            # obs_sd length mismatch
        dict(obs_sd=-0.1),                                  # negative
        dict(obs_sd=[0.1, -0.1, 0.1]),
        dict(bounds=[[0.5, 0.0], [0.5, 1.0]]),              # lo >= hi
        dict(bounds=[[0.6, 0.0], [0.5, 1.0]]),
    ]
    for kw in bad:
        args = dict(ok, **kw)
        with pytest.raises(ValueError):
            cal.calibrate(model, samples, **args)
        if 'bounds' not in kw:
            with pytest.raises(ValueError):
                cal.log_likelihood(model, samples, t=np.full((1, 2), 0.5), **args)
    with pytest.raises(ValueError):
        cal.calibrate(_model(x_sim=True), samples, **ok)    # x_sim
    with pytest.raises(ValueError):
        cal.calibrate(_model(K=np.random.default_rng(0).standard_normal((33, n_y))), synthetic.posterior_samples(2, d, 33),
                      **ok)
    with pytest.raises(ValueError):
        cal.calibrate(_model(q=33), synthetic.posterior_samples(2, 34, pu), **ok)
    with pytest.raises(ValueError):
        cal.log_likelihood(model, samples, t=np.full((1, 3), 0.5), **ok)
