"""GPU: closed-form GP sensitivity (csrc/ggp_gp_sens.cu, ops.gp_sens / ops.main_effects,
sensitivity.gp_sensitivity_indices) against the FP64 oracle, the emulator's own predictions and the Saltelli estimate."""
import numpy as np
import pytest

from helpers import synthetic, make_problem, make_scalar_problem, random_hypers
from oracle import gp_sens_oracle as gso
from oracle import sobol_oracle as sob

pytestmark = pytest.mark.gpu

M_RTOL = 1e-11        # moments: FP64 sums in another order than NumPy's
IDX_ATOL = 1e-9
# M(u) and E0^2 are sums of terms as large as (sum |a|)^2 and the indices are their differences over V: both sides carry
# a rounding error of order eps (sum |a|)^2 / V in every index, whatever the summation order
IDX_COND = 1e-10


def _weights(num, S, seed):
    """Blocks b = s*pu + j of random hyper-parameters and their mean-function weights a = S22^-1 w / lamUz from the
    cached-factor predictor.  Returns (Zin (m, q), beta (S, pu, q), a (S, pu, m)) as host arrays."""
    from gladsgp_b200 import ops
    pu, m = num.pu, num.m
    beta, lamz, lamws, lamwos = random_hypers(num, S * pu, seed=seed)
    c = 1.0 / (np.tile(num.LamSim, S) * np.repeat(lamwos[:S], pu))
    dadd = c + 1.0 / lamws
    s11 = 1.0 / lamz + 1.0 / lamws
    W = np.tile(num.wv.reshape(pu, m), (S, 1))
    P = ops.Predictor(num.zt, W, beta, lamz, dadd, s11)
    assert not P.info.any().item()
    alpha, _ = P.xval_solve(np.arange(m))
    a = (alpha / P.lamz[:, None]).cpu().numpy()
    return np.ascontiguousarray(num.zt[:, 1:]), beta[:, 1:].reshape(S, pu, -1), a.reshape(S, pu, m)


def _device(Zin, beta, a, option, grid=None):
    from gladsgp_b200 import ops
    S, pu, m = a.shape
    mode = 0 if option == 'samples' else 1
    aa = a / S if mode == 1 else a
    M, E0 = ops.gp_sens(Zin, beta.reshape(S * pu, -1), aa.reshape(S * pu, m), S, pu, mode)
    me = None if grid is None else ops.main_effects(Zin, beta.reshape(S * pu, -1), aa.reshape(S * pu, m), S, pu, grid, mode)
    return M, E0, me


def _check(Zin, beta, a, option, which=None, grid=np.linspace(0.0, 1.0, 5)):
    q = Zin.shape[1]
    M, E0, me = _device(Zin, beta, a, option, grid)
    M, E0, me = M.cpu().numpy(), E0.cpu().numpy(), me.cpu().numpy()
    funcs = gso.block_terms(Zin, beta, a, option)
    for f in (range(len(funcs)) if which is None else which):
        fa, fb, fz = funcs[f]
        ref = gso.moments(fa, fb, fz)
        scale = np.sum(np.abs(fa)) ** 2                     # bound on the absolute terms of every M
        got = gso.finish(E0[f], M[f, 2 * q], M[f, :q], M[f, q:2 * q], beta_zero=np.all(fb == 0, axis=0))
        for k, tol in (('E0', M_RTOL * np.sum(np.abs(fa))), ('Mall', M_RTOL * scale), ('M1', M_RTOL * scale),
                       ('Mt', M_RTOL * scale), ('V', M_RTOL * scale)):
            np.testing.assert_allclose(got[k], ref[k], rtol=M_RTOL, atol=tol, err_msg='%s f=%d' % (k, f))
        itol = IDX_ATOL + IDX_COND * scale / abs(ref['V'])
        np.testing.assert_allclose(got['first'], ref['first'], rtol=0, atol=itol, err_msg='first f=%d' % f)
        np.testing.assert_allclose(got['total'], ref['total'], rtol=0, atol=itol, err_msg='total f=%d' % f)
        np.testing.assert_allclose(me[f], gso.main_effects(fa, fb, fz, grid), rtol=M_RTOL,
                                   atol=M_RTOL * np.sum(np.abs(fa)), err_msg='main effect f=%d' % f)


@pytest.mark.parametrize('m,q,pu,S', [(64, 1, 1, 4), (100, 3, 3, 3), (64, 8, 10, 2), (100, 16, 3, 2), (512, 8, 2, 2),
                                      (64, 32, 1, 2)])
def test_per_sample_mode_matches_oracle(cuda, m, q, pu, S):
    num = make_problem(m=m, q=q, pu=pu)['num']
    _check(*_weights(num, S, seed=m + q), 'samples')


@pytest.mark.parametrize('m,q,pu,S', [(64, 3, 3, 4), (100, 8, 2, 3), (64, 16, 1, 4), (100, 1, 1, 5), (40, 20, 1, 3)])
def test_mean_mode_matches_oracle(cuda, m, q, pu, S):
    num = make_problem(m=m, q=q, pu=pu)['num']
    _check(*_weights(num, S, seed=m + 7 * q), 'mean')


@pytest.mark.parametrize('option', ['samples', 'mean'])
def test_cfg2_scalar_problem_matches_oracle(cuda, option):
    num = make_scalar_problem(m=1000)['num']
    _check(*_weights(num, 3, seed=2), option)


def test_cfg3_size_matches_oracle_on_a_subset(cuda):
    num = make_problem(m=512, q=8, pu=10)['num']
    _check(*_weights(num, 64, seed=11), 'samples', which=[0, 9, 137, 318, 500, 639])


def test_identical_calls_give_identical_bits(cuda):
    import torch
    num = make_problem(m=100, q=8, pu=3)['num']
    Zin, beta, a = _weights(num, 4, seed=3)
    for option in ('samples', 'mean'):
        r1 = _device(Zin, beta, a, option, np.linspace(0, 1, 9))
        r2 = _device(Zin, beta, a, option, np.linspace(0, 1, 9))
        assert all(torch.equal(x, y) for x, y in zip(r1, r2))


def _model(m=64, q=3, pu=2, seed=5):
    from sepia.SepiaData import SepiaData
    from sepia.SepiaModel import SepiaModel
    pr = make_problem(m=m, q=q, pu=pu, n_x=40, n_t=30, seed=seed)
    data = SepiaData(t_sim=pr['t'], y_sim=pr['y'], y_ind_sim=np.arange(pr['y'].shape[1], dtype=float))
    data.transform_xt(t_notrans=np.arange(q)); data.standardize_y(y_mean=pr['mu'], y_sd=pr['sd']); data.create_K_basis(K=pr['K'])
    return SepiaModel(data)


def test_weights_reproduce_predictive_means(cuda):
    import torch
    from gladsgp_b200 import sensitivity
    from sepia.SepiaPredict import SepiaEmulatorPrediction
    model = _model(m=100, q=4, pu=3)
    samples = synthetic.posterior_samples(5, model.num.p + model.num.q, 3, seed=1)
    Z, beta, a, ns = sensitivity.emulator_expansion(model, samples)
    assert ns == 5 and Z.shape == (100, 4) and beta.shape == (15, 4) and a.shape == (15, 100)
    x = synthetic.test_design(50, 4, seed=9)
    pe = SepiaEmulatorPrediction(t_pred=x, samples=samples, model=model, storeRlz=False, storeMuSigma=True)
    mu = torch.as_tensor(pe.get_mu_sigma()[0].reshape(5, 3, 50).reshape(15, 50), device='cuda')
    assert model._pred_cache is not None and pe._pred is model._pred_cache[1]
    xt = torch.as_tensor(pe.xpredt[:, 1:], device='cuda')
    d2 = (xt[None, :, None, :] - Z[None, None, :, :]) ** 2                      # (1, n, m, q)
    phi = torch.exp(-(d2 * beta[:, None, None, :]).sum(-1))                      # (B, n, m)
    mine = torch.einsum('bnm,bm->bn', phi, a)
    # two solve routes through the same factor: S21 . (L^-T L^-1 w) here, (L^-1 S21) . (L^-1 w) in predict_kernel
    assert float((mine - mu).abs().max()) <= 2e-11 * float(mu.abs().max())


def test_mean_mode_agrees_with_saltelli_estimate(cuda):
    from gladsgp_b200 import sensitivity
    model = _model(m=64, q=3, pu=2)
    samples = synthetic.posterior_samples(4, model.num.p + model.num.q, 2, seed=3)
    pcvar = np.array([0.7, 0.3])
    ex = sensitivity.gp_sensitivity_indices(model, samples, option='mean', pcvar=pcvar)
    assert ex['first'].shape == (2, 3) and ex['variance'].shape == (2,) and ex['general_first'].shape == (3,)
    func = sensitivity.emulator_mean_function(model, samples)
    first, total, gf, gt, res = sensitivity.PCA_saltelli_sensitivity_indices(
        func, 3, 12, pcvar, AB=sob.sobol_matrix(3, 12, seed=4), n_resamples=999, rng=np.random.default_rng(1))
    for est, key, rk in ((first, 'first', 'first_order'), (total, 'total', 'total_index'),
                         (gf, 'general_first', 'general_first_order'), (gt, 'general_total', 'general_total_index')):
        se = res[rk].standard_error
        assert np.all(np.abs(est - ex[key]) <= 4.0 * se), (key, est, ex[key], se)
    # the exact mean and variance of the function the Saltelli path samples
    xs = np.random.default_rng(2).uniform(size=(20000, 3))
    fx = func(xs)
    np.testing.assert_allclose(fx.mean(0), ex['mean'], atol=5 * fx.std(0).max() / np.sqrt(20000))


def test_main_effects_match_monte_carlo(cuda):
    from gladsgp_b200 import sensitivity
    model = _model(m=64, q=3, pu=2)
    samples = synthetic.posterior_samples(3, model.num.p + model.num.q, 2, seed=6)
    ex = sensitivity.gp_sensitivity_indices(model, samples, option='mean', ngrid=5)
    assert ex['main_effect'].shape == (2, 3, 5) and 'main_effect_native' not in ex
    np.testing.assert_array_equal(ex['grid'], np.linspace(0, 1, 5))
    func = sensitivity.emulator_mean_function(model, samples)
    n = 20000
    xs = np.random.default_rng(8).uniform(size=(n, 3))
    for k in range(3):
        for g in (0, 2, 4):
            x = xs.copy()
            x[:, k] = ex['grid'][g]
            fx = func(x)
            tol = 5.0 * fx.std(0) / np.sqrt(n) + 1e-12
            assert np.all(np.abs(fx.mean(0) - ex['main_effect'][:, k, g]) <= tol), (k, g)
    per = sensitivity.gp_sensitivity_indices(model, samples, option='samples', ngrid=5)
    assert per['first'].shape == (3, 2, 3) and per['main_effect'].shape == (3, 2, 3, 5)
    # the mean function's curves are the sample average of the per-sample curves
    np.testing.assert_allclose(per['main_effect'].mean(0), ex['main_effect'], rtol=1e-12,
                               atol=1e-12 * np.abs(ex['main_effect']).max())


def test_scalar_model_native_curves(cuda):
    from gladsgp_b200 import sensitivity
    from sepia.SepiaData import SepiaData
    from sepia.SepiaModel import SepiaModel
    pr = make_scalar_problem(m=200)
    data = SepiaData(t_sim=pr['t'], y_sim=pr['y'])
    data.transform_xt()
    data.standardize_y()
    model = SepiaModel(data)
    samples = synthetic.posterior_samples(4, 2, 1, seed=6)
    for option in ('samples', 'mean'):
        ex = sensitivity.gp_sensitivity_indices(model, samples, option=option)
        sd = float(np.asarray(data.sim_data.orig_y_sd).reshape(-1)[0])
        mu = float(np.asarray(data.sim_data.orig_y_mean).reshape(-1)[0])
        np.testing.assert_allclose(ex['main_effect_native'], ex['main_effect'] * sd + mu, rtol=1e-15, atol=0)
        np.testing.assert_allclose(ex['first'], 1.0, atol=1e-9)              # one input: S = T = 1
        np.testing.assert_allclose(ex['total'], 1.0, atol=1e-9)


def test_beta_zero_input_has_exactly_zero_indices(cuda):
    from gladsgp_b200 import sensitivity
    model = _model(m=64, q=3, pu=2)
    d = model.num.p + model.num.q
    samples = synthetic.posterior_samples(4, d, 2, seed=9)
    bU = np.array(samples['betaU'])
    bU[:, 2 + 1 * d] = 0.0                                  # zt column 2 (input 1) of PC 1, every sample
    samples['betaU'] = bU
    for option in ('samples', 'mean'):
        ex = sensitivity.gp_sensitivity_indices(model, samples, option=option)
        assert np.all(ex['first'][..., 1, 1] == 0.0) and np.all(ex['total'][..., 1, 1] == 0.0)
        assert np.all(ex['total'][..., 0, :] > 0.0) and np.all(ex['total'][..., 1, [0, 2]] > 0.0)


def test_argument_errors(cuda):
    from gladsgp_b200 import ops, sensitivity
    from gladsgp_b200._lib import GgpError
    Z = np.random.default_rng(0).uniform(size=(10, 3))
    beta = np.ones((2, 3))
    a = np.ones((2, 10))
    with pytest.raises(ValueError):
        ops.gp_sens(np.zeros((10, 0)), np.zeros((2, 0)), a, 2, 1)             # q = 0
    with pytest.raises(ValueError):
        ops.gp_sens(np.zeros((10, 33)), np.zeros((2, 33)), a, 2, 1)           # q > 32
    with pytest.raises(ValueError):
        ops.gp_sens(Z, beta, a, 2, 1, mode=2)
    with pytest.raises(ValueError):
        ops.gp_sens(Z, beta[:1], a, 2, 1)                                     # sizes do not match
    with pytest.raises(GgpError):
        ops.main_effects(Z, beta, a, 2, 1, grid=np.zeros(0))                  # empty grid
    model = _model(m=64, q=3, pu=2)
    samples = synthetic.posterior_samples(2, 4, 2, seed=1)
    with pytest.raises(ValueError):
        sensitivity.gp_sensitivity_indices(model, samples, option='median')
    with pytest.raises(ValueError):
        sensitivity.gp_sensitivity_indices(model, samples, ngrid=0)
    with pytest.raises(ValueError):
        sensitivity.gp_sensitivity_indices(model, samples, pcvar=[1.0, 0.0, 0.0])
    # still usable after the refusals
    ex = sensitivity.gp_sensitivity_indices(model, samples)
    assert np.all(np.isfinite(ex['first']))
