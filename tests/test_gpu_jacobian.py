"""GPU: emulator Jacobians (csrc/ggp_jacobian.cu, ops.Predictor.jacobian, gradient.emulator_jacobian) against the dense
FP64 oracle (oracle/jacobian_oracle.py), ggp_predict_f64's moments bit for bit, central differences of the prediction,
and the posterior fixtures."""
import numpy as np
import pytest

from helpers import synthetic, make_problem, make_scalar_problem
from oracle import jacobian_oracle as jo
from posterior_helpers import sepia_model_of, scalar_model_of

pytestmark = pytest.mark.gpu

PRED_RTOL = 1e-6      # the predictor's tolerance: rtol, and atol = PRED_RTOL max|.| of the compared array


def _close(got, ref, what):
    """assert_allclose at the predictor's tolerances; returns the largest error / tolerance."""
    tol = PRED_RTOL * np.abs(ref) + PRED_RTOL * np.abs(ref).max()
    ratio = float(np.max(np.abs(got - ref) / np.maximum(tol, 1e-300))) if ref.size else 0.0
    np.testing.assert_allclose(got, ref, rtol=PRED_RTOL, atol=PRED_RTOL * np.abs(ref).max(), err_msg=what)
    return ratio


def _random_blocks(m, q, B, seed):
    """A design Z (m, 1+q) with the dummy x column and B random (sample, PC) blocks."""
    rng = np.random.default_rng(seed)
    Z = np.concatenate([np.full((m, 1), 0.5), rng.uniform(0.0, 1.0, (m, q))], axis=1)
    beta = np.exp(rng.uniform(np.log(0.05), np.log(4.0), (B, q + 1)))
    lamz = rng.gamma(5.0, 0.2, B) + 0.3
    lamws = rng.uniform(200.0, 5000.0, B)
    dadd = 1.0 / lamws + rng.uniform(2e-3, 2e-2, B)
    s11 = 1.0 / lamz + 1.0 / lamws
    W = rng.standard_normal((B, m))
    return Z, W, beta, lamz, dadd, s11


def _designs(Z, n, seed):
    """n designs: training points first, then corners and edges of the box, then uniform points."""
    rng = np.random.default_rng(seed + 1)
    m, d = Z.shape
    X = np.concatenate([np.full((n, 1), 0.5), rng.uniform(0.0, 1.0, (n, d - 1))], axis=1)
    k = min(n // 3 + 1, m, n)
    X[:k] = Z[rng.permutation(m)[:k]]
    e = min(n - k, n // 3 + 1)
    if e > 0:
        X[k:k + e, 1:] = rng.integers(0, 2, (e, d - 1)).astype(np.float64)
        X[k:k + e:2, 1] = rng.uniform(0, 1, X[k:k + e:2, 1].shape)              # edges: one free coordinate
    return X


CASES = [  # m, q, pu * S blocks, n
    (1, 1, 2, 1), (31, 7, 2, 255), (33, 8, 3, 256), (512, 8, 10, 257), (1000, 15, 2, 64), (64, 16, 5, 257),
    (100, 31, 2, 33), (80, 20, 2, 40), (200, 1, 1, 2000), (4100, 3, 1, 5)]


@pytest.mark.parametrize('m,q,B,n', CASES)
def test_device_matches_oracle(cuda, m, q, B, n):
    from gladsgp_b200 import ops
    Z, W, beta, lamz, dadd, s11 = _random_blocks(m, q, B, seed=m + q)
    X = _designs(Z, n, seed=m)
    P = ops.Predictor(Z, W, beta, lamz, dadd, s11)
    assert int((P.info != 0).sum()) == 0
    mean, cov = (t.cpu().numpy() for t in P.jacobian(X, 1, full=True))
    mc, cc = (t.cpu().numpy() for t in P.jacobian(X, 1, full=False))
    assert mean.shape == (B, n, q + 1) and cov.shape == (B, n, q + 1, q + 1) and cc.shape == (B, n, 2 * q + 1)
    assert np.array_equal(cov, np.swapaxes(cov, -1, -2))
    assert np.array_equal(mean, mc) and np.array_equal(jo.compact(cov), cc)
    rm, rc = jo.blocks(Z, W, beta, lamz, dadd, s11, X, 1)
    worst = max(_close(mean[..., 0], rm[..., 0], 'mu'), _close(mean[..., 1:], rm[..., 1:], 'grad mu'),
                _close(cov, rc, 'joint covariance'), _close(cc, jo.compact(rc), 'compact'))
    # the value row is ggp_predict_f64's, bit for bit
    pm, pv = (t.cpu().numpy() for t in P.predict(X))
    assert np.array_equal(mean[..., 0], pm) and np.array_equal(cov[..., 0, 0], pv) and np.array_equal(cc[..., 0], pv)
    print('jacobian m=%d q=%d B=%d n=%d: largest error / tolerance %.3g' % (m, q, B, n, worst))


def test_identical_bits_for_any_split(cuda):
    import torch
    from gladsgp_b200 import ops
    Z, W, beta, lamz, dadd, s11 = _random_blocks(100, 8, 6, seed=1)
    X = _designs(Z, 600, seed=2)
    P = ops.Predictor(Z, W, beta, lamz, dadd, s11)
    for full in (True, False):
        m1, c1 = P.jacobian(X, 1, full=full)
        m2, c2 = P.jacobian(X, 1, full=full)
        assert torch.equal(m1, m2) and torch.equal(c1, c2)
        for a, b in ((0, 1), (17, 300), (299, 600)):
            ms, cs = P.jacobian(X[a:b], 1, full=full)
            assert torch.equal(ms, m1[:, a:b]) and torch.equal(cs, c1[:, a:b])
        ms, cs = P.jacobian(X[5:40], 1, full=full, b0=2, nb=3)
        assert torch.equal(ms, m1[2:5, 5:40]) and torch.equal(cs, c1[2:5, 5:40])


def test_beta_zero_gives_exact_zeros(cuda):
    from gladsgp_b200 import ops
    Z, W, beta, lamz, dadd, s11 = _random_blocks(70, 5, 4, seed=3)
    beta[1:3, 3] = 0.0                                     # input col 3 (row 3 of the Jacobian) in blocks 1 and 2
    X = _designs(Z, 40, seed=4)
    P = ops.Predictor(Z, W, beta, lamz, dadd, s11)
    mean, cov = (t.cpu().numpy() for t in P.jacobian(X, 1))
    _, cc = (t.cpu().numpy() for t in P.jacobian(X, 1, full=False))
    for b in (1, 2):
        assert np.all(mean[b, :, 3] == 0.0) and np.all(cov[b, :, 3, :] == 0.0) and np.all(cov[b, :, :, 3] == 0.0)
        assert np.all(cc[b, :, [3, 5 + 3]] == 0.0)
    assert np.all(np.abs(mean[0, :, 3]) > 0.0) and np.all(cov[0, :, 3, 3] > 0.0)


# --------------------------------------------------------------------------------------------------------------------
# the public call
# --------------------------------------------------------------------------------------------------------------------
def _model(m=64, q=3, pu=3, seed=5, n_x=8, n_t=4):
    return sepia_model_of(make_problem(m=m, q=q, pu=pu, n_x=n_x, n_t=n_t, seed=seed))


def _native_points(model, N, seed):
    sd = model.data.sim_data
    tt = np.random.default_rng(seed).uniform(0.05, 0.95, (N, model.num.q))
    return tt * (sd.orig_t_max - sd.orig_t_min) + sd.orig_t_min


def _oracle(model, samples, t):
    """Oracle per_sample quantities (S, N, pu, ...) in native input units."""
    from gladsgp_b200.calibration import _to_trans
    from gladsgp_b200.sensitivity import _input_span
    from gladsgp_b200.sepia.SepiaPredict import SepiaEmulatorPrediction
    q, pu = model.num.q, model.num.pu
    ns, beta, lamz, dadd, s11, W = SepiaEmulatorPrediction(t_pred=np.full((1, q), 0.5), samples=samples, model=model,
                                                           do_call=False)._blocks()
    X = np.concatenate([np.full((t.shape[0], 1), 0.5), _to_trans(model, t)], axis=1)
    mean, cov = jo.blocks(model.num.zt, W, beta, lamz, dadd, s11, X, 1)
    N = t.shape[0]
    mean = mean.reshape(ns, pu, N, q + 1).transpose(0, 2, 1, 3)
    cov = cov.reshape(ns, pu, N, q + 1, q + 1).transpose(0, 2, 1, 3, 4)
    r = jo.per_sample(mean, cov)
    span = _input_span(model)
    r['grad'] = r['grad'] / span
    r['grad_var'] = r['grad_var'] / span
    r['grad_cov'] = r['grad_cov'] / np.multiply.outer(span, span)
    return r


def test_matches_central_differences_of_the_prediction(cuda):
    """grad and grad_var against central differences of SepiaEmulatorPrediction's mean and variance in native units."""
    from gladsgp_b200 import gradient
    from gladsgp_b200.sepia.SepiaPredict import SepiaEmulatorPrediction
    model = _model(q=3, pu=2)
    sd = model.data.sim_data
    span = (sd.orig_t_max - sd.orig_t_min).reshape(-1)
    assert np.all(span != 1.0)
    samples = synthetic.posterior_samples(3, model.num.p + 3, 2, seed=2)
    t = _native_points(model, 7, seed=3)
    r = gradient.emulator_jacobian(model, samples, t)

    def moments(tp):
        p = SepiaEmulatorPrediction(t_pred=tp, samples=samples, model=model, storeRlz=False, storeMuSigma=True, joint=False)
        mu = p.mu.reshape(3, 2, -1).transpose(0, 2, 1)
        v = np.diagonal(p.sigma, axis1=1, axis2=2).reshape(3, 2, -1).transpose(0, 2, 1)
        return mu, v
    mu0, v0 = moments(t)
    np.testing.assert_array_equal(r['mean'], mu0)
    np.testing.assert_array_equal(r['var'], np.maximum(v0, 0.0))
    for k in range(3):
        h = 1e-5 * span[k]
        e = np.zeros(3)
        e[k] = h
        (mp, vp), (mm, vm) = moments(t + e), moments(t - e)
        g = (mp - mm) / (2 * h)
        gv = (vp - vm) / (2 * h)
        np.testing.assert_allclose(r['grad'][..., k], g, rtol=1e-5, atol=1e-6 * np.abs(g).max())
        np.testing.assert_allclose(r['grad_var'][..., k], gv, rtol=1e-4, atol=1e-5 * np.abs(gv).max())


def test_every_target_and_option_matches_oracle(cuda):
    from gladsgp_b200 import gradient
    model = _model(q=3, pu=3)
    samples = synthetic.posterior_samples(4, model.num.p + 3, 3, seed=4)
    t = _native_points(model, 9, seed=5)
    ref = _oracle(model, samples, t)
    worst = 0.0
    c = np.array([0.7, -1.3, 0.4])
    sd = model.data.sim_data
    K = np.asarray(sd.K, dtype=np.float64)
    ysd = np.broadcast_to(np.asarray(sd.orig_y_sd, dtype=np.float64).reshape(-1), (K.shape[1],))
    O = np.array([0, 5, 17, K.shape[1] - 1])
    coef = K[:, O] * ysd[O]
    for option in ('samples', 'mean'):
        for full in (True, False):
            for target, rr in (('pc', ref), (c, jo.linear(ref, c))):
                exp = jo.mixture(rr) if option == 'mean' else rr
                got = gradient.emulator_jacobian(model, samples, t, target=target, option=option, full=full)
                for k in ('mean', 'grad', 'grad_var'):
                    worst = max(worst, _close(got[k], exp[k], '%s %s %s' % (option, target, k)))
                worst = max(worst, _close(got['var'], np.maximum(exp['var'], 0.0), 'var'))
                if full:
                    worst = max(worst, _close(got['grad_cov'], exp['grad_cov'], 'grad_cov'))
                    assert 'grad_sd' not in got
                else:
                    sdv = np.sqrt(np.maximum(np.diagonal(exp['grad_cov'], axis1=-2, axis2=-1), 0.0))
                    worst = max(worst, _close(got['grad_sd'], sdv, 'grad_sd'))
        J, gsd = jo.field(ref, coef, option)
        got = gradient.emulator_jacobian(model, samples, t, target='field', outputs=O, option=option)
        worst = max(worst, _close(got['jacobian'], J, 'field jacobian'), _close(got['grad_sd'], gsd, 'field grad_sd'))
        ymu = np.broadcast_to(np.asarray(sd.orig_y_mean, dtype=np.float64).reshape(-1), (K.shape[1],))[O]
        ymean = ref['mean'] @ coef + ymu
        _close(got['mean'], ymean.mean(0) if option == 'mean' else ymean, 'field mean')
        allf = gradient.emulator_jacobian(model, samples, t, target='field', option=option)
        assert np.array_equal(allf['jacobian'][..., O, :], got['jacobian'])
    print('emulator_jacobian: largest error / tolerance %.3g' % worst)


def test_scalar_output_model(cuda):
    from gladsgp_b200 import gradient
    model = scalar_model_of(make_scalar_problem(m=200))
    samples = synthetic.posterior_samples(3, 2, 1, seed=6)
    sd = float(np.asarray(model.data.sim_data.orig_y_sd).reshape(-1)[0])
    t = _native_points(model, 11, seed=7)
    ref = _oracle(model, samples, t)
    for option in ('samples', 'mean'):
        pc = gradient.emulator_jacobian(model, samples, t, option=option, full=False)
        fld = gradient.emulator_jacobian(model, samples, t, target='field', option=option)
        np.testing.assert_allclose(fld['jacobian'][..., 0, :], pc['grad'][..., 0, :] * sd, rtol=1e-14, atol=0)
        np.testing.assert_allclose(fld['grad_sd'][..., 0, :], pc['grad_sd'][..., 0, :] * sd, rtol=1e-14, atol=0)
        exp = jo.mixture(ref) if option == 'mean' else ref
        _close(pc['grad'], exp['grad'], 'scalar grad')


def test_refusals(cuda, monkeypatch):
    from gladsgp_b200 import gradient
    from sepia.SepiaData import SepiaData
    from sepia.SepiaModel import SepiaModel
    pr = make_problem(m=40, q=2, pu=2, n_x=6, n_t=3)
    xs = np.random.default_rng(0).uniform(size=(40, 1))
    data = SepiaData(x_sim=xs, t_sim=pr['t'], y_sim=pr['y'], y_ind_sim=np.arange(pr['y'].shape[1], dtype=float))
    data.transform_xt()
    data.standardize_y(y_mean=pr['mu'], y_sd=pr['sd']); data.create_K_basis(K=pr['K'])
    xmodel = SepiaModel(data)
    samples = synthetic.posterior_samples(2, 3, 2, seed=1)
    with pytest.raises(ValueError, match='x_sim'):
        gradient.emulator_jacobian(xmodel, samples, np.full((2, 2), 0.5))
    big = sepia_model_of(make_problem(m=40, q=32, pu=1, n_x=6, n_t=3))
    with pytest.raises(ValueError, match='q <= 31'):
        gradient.emulator_jacobian(big, synthetic.posterior_samples(2, 33, 1, seed=1), np.full((2, 32), 0.5))
    model = _model(q=2, pu=2)
    samples = synthetic.posterior_samples(2, 3, 2, seed=1)
    t = _native_points(model, 3, seed=1)
    for kw in (dict(target='field', outputs=[10 ** 6]), dict(target='field', outputs=[]), dict(target='pc', outputs=[0]),
               dict(target='pcs'), dict(target=[1.0, 2.0, 3.0]), dict(option='median')):
        with pytest.raises(ValueError):
            gradient.emulator_jacobian(model, samples, t, **kw)
    with pytest.raises(ValueError):
        gradient.emulator_jacobian(model, samples, np.full((3, 3), 0.5))
    monkeypatch.setattr(gradient, 'FIELD_SAMPLES_BYTES', 1000)
    with pytest.raises(ValueError, match="option='mean'"):
        gradient.emulator_jacobian(model, samples, t, target='field')
    assert gradient.emulator_jacobian(model, samples, t, target='field', option='mean')['jacobian'].shape[0] == 3


# --------------------------------------------------------------------------------------------------------------------
# posterior fixtures (tests/golden/posterior_cfg*.npz): real posterior draws
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('cfg', ['cfg1', 'cfg2', 'cfg3'])
def test_posterior_draws(cuda, cfg):
    """Device against the oracle at the widest draws, at training points and inside the box; every target is finite."""
    from gladsgp_b200 import gradient
    from test_gpu_posterior_draws import _model as fixture_model, _samples, _widest
    model = fixture_model(cfg)
    samples = _samples(cfg, _widest(cfg, 3))
    q = model.num.q
    tt = np.concatenate([model.num.zt[:4, 1:], np.random.default_rng(1).uniform(0, 1, (6, q))])
    t = tt * (model.data.sim_data.orig_t_max - model.data.sim_data.orig_t_min) + model.data.sim_data.orig_t_min
    ref = _oracle(model, samples, t)
    got = gradient.emulator_jacobian(model, samples, t)
    worst = max(_close(got['grad'], ref['grad'], 'grad'), _close(got['grad_cov'], ref['grad_cov'], 'grad_cov'),
                _close(got['grad_var'], ref['grad_var'], 'grad_var'), _close(got['mean'], ref['mean'], 'mean'))
    for option in ('samples', 'mean'):
        r = gradient.emulator_jacobian(model, _samples(cfg), t, target='field', option=option)
        assert all(np.all(np.isfinite(v)) for v in r.values())
    print('jacobian %s: largest error / tolerance %.3g' % (cfg, worst))
