"""GPU: closed-form gradient outer products (csrc/ggp_grad_sens.cu, ops.grad_sens, sensitivity.gp_active_subspace) against
the FP64 oracle, quadrature of the emulator's own gradients, the field / linear targets and the posterior fixtures."""
import numpy as np
import pytest

from helpers import synthetic, make_problem, make_scalar_problem
from oracle import grad_sens_oracle as gro
from posterior_helpers import sepia_model_of, scalar_model_of
from test_gpu_gp_sens import _weights

pytestmark = pytest.mark.gpu

C_TOL = 1e-11         # |dC_kl| <= C_TOL A_kl: A is the pair sum over absolute values, the scale of the rounding error


def _omega(pu, seed):
    L = np.random.default_rng(seed).standard_normal((pu, pu + 2))
    return L @ L.T


def _device(Zin, beta, a, mode, omega=None):
    from gladsgp_b200 import ops
    S, pu, m = a.shape
    aa = a / S if mode in (1, 3) else a
    return ops.grad_sens(Zin, beta.reshape(S * pu, -1), aa.reshape(S * pu, m), S, pu, mode, omega)


def _check(Zin, beta, a, mode, omega=None, which=None):
    """Device C of every function (or of `which`) against the oracle; returns the largest |dC| / A."""
    S = a.shape[0]
    C = _device(Zin, beta, a, mode, omega).cpu().numpy()
    assert np.array_equal(C, np.swapaxes(C, 1, 2))
    funcs = gro.block_terms(Zin, beta, a / S if mode in (1, 3) else a, mode, omega)
    assert C.shape[0] == len(funcs)
    worst = 0.0
    for f in (range(len(funcs)) if which is None else which):
        ref = gro.grad_outer(*funcs[f])
        err = np.abs(C[f] - ref['C'])
        assert np.all(err <= C_TOL * ref['A']), (f, np.max(err / np.maximum(ref['A'], 1e-300)))
        worst = max(worst, float(np.max(np.where(ref['A'] > 0, err / np.maximum(ref['A'], 1e-300), 0.0))))
    return worst


@pytest.mark.parametrize('mode,m,q,pu,S', [
    (0, 64, 1, 1, 4), (0, 100, 3, 3, 3), (0, 64, 8, 10, 2), (0, 100, 16, 3, 2), (0, 512, 8, 3, 2), (0, 64, 32, 1, 2),
    (0, 1000, 3, 1, 2), (0, 64, 20, 3, 5),
    (1, 64, 3, 3, 4), (1, 100, 8, 1, 3), (1, 64, 16, 1, 2), (1, 100, 1, 1, 5), (1, 64, 20, 1, 3), (1, 64, 32, 1, 2),
    (2, 64, 3, 3, 2), (2, 100, 8, 3, 3), (2, 64, 1, 10, 2), (2, 64, 16, 3, 2), (2, 64, 32, 1, 2),
    (3, 64, 3, 3, 2), (3, 100, 8, 1, 4), (3, 64, 20, 3, 2), (3, 64, 1, 10, 2)])
def test_modes_match_oracle(cuda, mode, m, q, pu, S):
    num = make_problem(m=m, q=q, pu=pu)['num']
    omega = _omega(pu, m + q) if mode >= 2 else None
    worst = _check(*_weights(num, S, seed=m + 3 * q), mode, omega)
    print('mode %d m=%d q=%d pu=%d S=%d: largest |dC| / A %.3g' % (mode, m, q, pu, S, worst))


def test_identical_calls_give_identical_bits(cuda):
    import torch
    num = make_problem(m=100, q=8, pu=3)['num']
    Zin, beta, a = _weights(num, 4, seed=3)
    om = _omega(3, 1)
    for mode in range(4):
        r1 = _device(Zin, beta, a, mode, om)
        r2 = _device(Zin, beta, a, mode, om)
        assert torch.equal(r1, r2) and torch.equal(r1, r1.transpose(1, 2))


def test_beta_zero_input_gives_exact_zeros(cuda):
    num = make_problem(m=64, q=5, pu=3)['num']
    Zin, beta, a = _weights(num, 3, seed=4)
    beta[:, :, 2] = 0.0
    for mode in range(4):
        C = _device(Zin, beta, a, mode, _omega(3, 2)).cpu().numpy()
        assert np.all(C[:, 2, :] == 0.0) and np.all(C[:, :, 2] == 0.0), mode
        assert np.all(np.diagonal(C, axis1=1, axis2=2)[:, [0, 1, 3, 4]] > 0.0), mode


def _model(m=64, q=2, pu=2, seed=5, n_x=10, n_t=4):
    return sepia_model_of(make_problem(m=m, q=q, pu=pu, n_x=n_x, n_t=n_t, seed=seed), t_notrans=True)


def _fd_quadrature(func, q, pu, nodes=24, h=1e-3):
    """E[grad f_j grad f_j^T] (pu, q, q) by tensor Gauss-Legendre quadrature of fourth-order central differences of
    func (n, q) -> (n, pu) (a small step would amplify the predictions' rounding)."""
    x, w = np.polynomial.legendre.leggauss(nodes)
    x, w = 0.5 * (x + 1.0), 0.5 * w
    X = np.stack(np.meshgrid(*([x] * q), indexing='ij'), -1).reshape(-1, q)
    W = np.prod(np.stack(np.meshgrid(*([w] * q), indexing='ij'), -1).reshape(-1, q), axis=1)
    G = np.empty((X.shape[0], pu, q))
    for k in range(q):
        e = np.zeros(q)
        e[k] = h
        G[:, :, k] = (8.0 * (func(X + e) - func(X - e)) - (func(X + 2 * e) - func(X - 2 * e))) / (12 * h)
    return np.einsum('p,pjk,pjl->jkl', W, G, G)


@pytest.mark.parametrize('q', [1, 2])
def test_matches_quadrature_of_the_emulator_gradients(cuda, q):
    """C of 'mean' and of every sample in 'samples' against quadrature of central-difference gradients of the means the
    emulator predicts (emulator_mean_function)."""
    from gladsgp_b200 import sensitivity
    model = _model(q=q)
    S, pu = 3, model.num.pu
    samples = synthetic.posterior_samples(S, model.num.p + q, pu, seed=2)
    mean = sensitivity.gp_active_subspace(model, samples, option='mean')
    ref = _fd_quadrature(sensitivity.emulator_mean_function(model, samples), q, pu)
    np.testing.assert_allclose(mean['C'], ref, rtol=1e-6, atol=1e-6 * np.abs(ref).max())
    per = sensitivity.gp_active_subspace(model, samples, option='samples')
    assert per['C'].shape == (S, pu, q, q) and per['C_avg'].shape == (pu, q, q)
    for s in range(S):
        one = {k: v[s:s + 1] for k, v in samples.items()}
        ref = _fd_quadrature(sensitivity.emulator_mean_function(model, one), q, pu)
        np.testing.assert_allclose(per['C'][s], ref, rtol=1e-6, atol=1e-6 * np.abs(ref).max())
    np.testing.assert_allclose(per['C_avg'], per['C'].mean(0), rtol=1e-14, atol=0)


def test_result_fields(cuda):
    from gladsgp_b200 import sensitivity
    model = _model(q=3, pu=3)
    samples = synthetic.posterior_samples(4, model.num.p + 3, 3, seed=3)
    r = sensitivity.gp_active_subspace(model, samples, option='samples')
    C, lam, V = r['C'], r['eigenvalues'], r['eigenvectors']
    assert C.shape == (4, 3, 3, 3) and lam.shape == (4, 3, 3) and V.shape == (4, 3, 3, 3)
    assert np.all(np.diff(lam, axis=-1) <= 0)
    np.testing.assert_allclose(V @ (lam[..., None] * np.swapaxes(V, -1, -2)), C, rtol=0, atol=1e-12 * np.abs(C).max())
    big = np.take_along_axis(V, np.abs(V).argmax(axis=-2)[..., None, :], axis=-2)
    assert np.all(big > 0)
    np.testing.assert_array_equal(r['dgsm'], np.diagonal(C, axis1=-2, axis2=-1))
    assert r['total_bound'].shape == (4, 3, 3) and np.all((r['total_bound'] >= 0) & (r['total_bound'] <= 1))
    assert np.all(np.diff(r['eigenvalues_avg'], axis=-1) <= 0)


def test_field_target(cuda):
    """'field' equals the sum over outputs of the per-output linear targets K[:, o] sd_o, and outputs=[o] the single one,
    to 1e-11 of the pair sums over absolute values (the GP weights alternate in sign, so C is far below them)."""
    from gladsgp_b200 import design, sensitivity
    from gladsgp_b200.sensitivity import _field_omega
    model = _model(m=64, q=3, pu=3, n_x=8, n_t=4)
    samples = synthetic.posterior_samples(3, model.num.p + 3, 3, seed=4)
    sd = model.data.sim_data
    K = np.asarray(sd.K, dtype=np.float64)
    ysd = np.broadcast_to(np.asarray(sd.orig_y_sd, dtype=np.float64).reshape(-1), (K.shape[1],))
    omega = _field_omega(model, None).cpu().numpy()
    np.testing.assert_allclose(np.diag(omega), design.field_weights(model), rtol=1e-12)
    Z, beta, a, ns = sensitivity.emulator_expansion(model, samples)
    Zin, bb, aa = Z.cpu().numpy(), beta.cpu().numpy().reshape(ns, 3, -1), a.cpu().numpy().reshape(ns, 3, -1)
    for option, mode in (('samples', 2), ('mean', 3)):
        full = sensitivity.gp_active_subspace(model, samples, option=option, target='field')
        assert full['C'].shape == ((3, 3, 3) if option == 'samples' else (3, 3))
        per = [sensitivity.gp_active_subspace(model, samples, option=option, target=K[:, o] * ysd[o])['C']
               for o in range(K.shape[1])]
        scale = aa / ns if mode == 3 else aa
        A = np.array([gro.grad_outer(*f)['A'] for f in gro.block_terms(Zin, bb, scale, mode, omega)]).reshape(full['C'].shape)
        assert np.all(np.abs(full['C'] - np.sum(per, axis=0)) <= 1e-11 * A), option
        c5 = K[:, 5] * ysd[5]
        A5 = np.array([gro.grad_outer(*f)['A'] for f in gro.block_terms(Zin, bb, scale, mode, np.outer(c5, c5))])
        one = sensitivity.gp_active_subspace(model, samples, option=option, target='field', outputs=[5])
        assert np.all(np.abs(one['C'] - per[5]) <= 1e-11 * A5.reshape(one['C'].shape)), option


def test_scalar_model_field_is_sd_squared_times_pc(cuda):
    from gladsgp_b200 import sensitivity
    model = scalar_model_of(make_scalar_problem(m=200), t_notrans=True)
    samples = synthetic.posterior_samples(4, 2, 1, seed=6)
    sd = float(np.asarray(model.data.sim_data.orig_y_sd).reshape(-1)[0])
    for option in ('samples', 'mean'):
        pc = sensitivity.gp_active_subspace(model, samples, option=option, target='pc')
        fld = sensitivity.gp_active_subspace(model, samples, option=option, target='field')
        ref = pc['C'].reshape(fld['C'].shape) * sd * sd
        # mode 2 / 3 (general pair path, Omega = sd^2) against mode 0 / 1: the same sums up to rounding
        np.testing.assert_allclose(fld['C'], ref, rtol=1e-10, atol=1e-10 * np.abs(ref).max())


def test_dgsm_native_units(cuda):
    from gladsgp_b200 import sensitivity
    from sepia.SepiaData import SepiaData
    from sepia.SepiaModel import SepiaModel
    pr = make_problem(m=64, q=3, pu=2, n_x=8, n_t=4)
    t = pr['t'] * np.array([10.0, 1.0, 0.25]) + np.array([-3.0, 0.0, 7.0])
    data = SepiaData(t_sim=t, y_sim=pr['y'], y_ind_sim=np.arange(pr['y'].shape[1], dtype=float))
    data.transform_xt(t_notrans=[1])
    data.standardize_y(y_mean=pr['mu'], y_sd=pr['sd']); data.create_K_basis(K=pr['K'])
    model = SepiaModel(data)
    samples = synthetic.posterior_samples(3, model.num.p + 3, 2, seed=7)
    sd = model.data.sim_data
    span = (sd.orig_t_max - sd.orig_t_min).reshape(-1)
    assert span[1] == 1.0 and span[0] != 1.0
    r = sensitivity.gp_active_subspace(model, samples, option='mean')
    np.testing.assert_array_equal(r['dgsm_native'], r['dgsm'] / span ** 2)
    np.testing.assert_array_equal(r['dgsm_native'][..., 1], r['dgsm'][..., 1])


def test_argument_errors(cuda):
    from gladsgp_b200 import ops, sensitivity
    Z = np.random.default_rng(0).uniform(size=(10, 3))
    beta = np.ones((2, 3))
    a = np.ones((2, 10))
    for bad in (dict(mode=4), dict(mode=2), dict(mode=3, omega=np.eye(3))):
        with pytest.raises(ValueError):
            ops.grad_sens(Z, beta, a, 2, 1, **bad)
    with pytest.raises(ValueError):
        ops.grad_sens(np.zeros((10, 33)), np.zeros((2, 33)), a, 2, 1, 0)
    model = _model(q=3, pu=2)
    samples = synthetic.posterior_samples(2, 4, 2, seed=1)
    for kw in (dict(option='median'), dict(target='pcs'), dict(target=[1.0, 2.0, 3.0]), dict(target='pc', outputs=[0]),
               dict(target='field', outputs=[10 ** 6]), dict(target='field', outputs=[])):
        with pytest.raises(ValueError):
            sensitivity.gp_active_subspace(model, samples, **kw)
    assert np.all(np.isfinite(sensitivity.gp_active_subspace(model, samples)['C']))


# --------------------------------------------------------------------------------------------------------------------
# posterior fixtures (tests/golden/posterior_cfg*.npz): real posterior draws
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('cfg', ['cfg1', 'cfg2', 'cfg3'])
def test_posterior_draws(cuda, cfg):
    """Every mode at the draws is finite and PSD to rounding; the blocks of the largest betaU match the oracle (mode 0, and
    mode 1 on the 2 widest draws); total_bound bounds the device total indices."""
    from gladsgp_b200 import sensitivity
    from test_gpu_posterior_draws import _model as fixture_model, _samples, _widest
    model = fixture_model(cfg)
    samples = _samples(cfg)
    Z, beta, a, ns = sensitivity.emulator_expansion(model, samples)
    pu, m = model.num.pu, model.num.m
    Zin = Z.cpu().numpy()
    bb = beta.cpu().numpy().reshape(ns, pu, -1)
    aa = a.cpu().numpy().reshape(ns, pu, m)
    om = _omega(pu, 9)
    for mode in range(4):
        sel = np.arange(ns) if mode != 3 or cfg != 'cfg3' else _widest(cfg, 8)
        C = _device(Zin, bb[sel], aa[sel], mode, om).cpu().numpy()
        assert np.all(np.isfinite(C)) and np.array_equal(C, np.swapaxes(C, 1, 2)), mode
        lam = np.linalg.eigvalsh(C)
        assert np.all(lam[:, 0] >= -1e-9 * np.maximum(lam[:, -1], 1e-300)), (mode, lam[:, 0].min())
    wide = bb.reshape(ns * pu, -1).max(1)
    which = sorted(int(f) for f in np.argsort(wide)[-6:])
    worst = _check(Zin, bb, aa, 0, which=which)
    w2 = _widest(cfg, 2)
    worst = max(worst, _check(Zin, bb[w2], aa[w2], 1, which=list(range(min(pu, 3)))))
    print('grad_sens %s: largest |dC| / A %.3g (largest betaU %.3g)' % (cfg, worst, bb.max()))
    for option in ('samples', 'mean'):
        r = sensitivity.gp_active_subspace(model, samples, option=option)
        tot = sensitivity.gp_sensitivity_indices(model, samples, option=option)['total']
        # the device indices carry a rounding error up to about 1e-7 on ill-conditioned blocks (test_gpu_gp_sens.py)
        assert np.all(r['total_bound'] >= tot - 1e-6), (option, np.min(r['total_bound'] - tot))
