"""CPU: the emulator-Jacobian oracle (oracle/jacobian_oracle.py) against complex-step and mixed finite differences of its
own moments, exact properties, the mixture / linear / field reductions against their definitions, and the argument
checks of the C entry points and of gradient.emulator_jacobian that need no device."""
import ctypes

import numpy as np
import pytest

from helpers import ROOT  # noqa: F401  (puts the repository root on sys.path)
from oracle import jacobian_oracle as jo


def _block(m=25, q=3, seed=0):
    rng = np.random.default_rng(seed)
    Z = np.concatenate([np.full((m, 1), 0.5), rng.uniform(0, 1, (m, q))], axis=1)
    beta = np.exp(rng.uniform(np.log(0.1), np.log(3.0), q + 1))
    lamz = 0.8 + rng.uniform()
    dadd = 1e-3 + 1e-2 * rng.uniform()
    s11 = 1.0 / lamz + 1e-3
    w = rng.standard_normal(m)
    X = np.concatenate([np.full((4, 1), 0.5), rng.uniform(0, 1, (4, q))], axis=1)
    X[0] = Z[3]                                                  # a training point
    return Z, w, beta, lamz, dadd, s11, X


@pytest.mark.parametrize('seed', [0, 1, 2])
def test_gradients_match_complex_step(seed):
    """grad mu and grad v = 2 Cov(f, grad f) against complex-step derivatives of mu and v (no subtraction error)."""
    Z, w, beta, lamz, dadd, s11, X = _block(seed=seed)
    mean, cov = jo.block(Z, w, beta, lamz, dadd, s11, X, 1)
    h = 1e-30
    for t, x in enumerate(X):
        for k in range(1, Z.shape[1]):
            xc = x.astype(complex)
            xc[k] += 1j * h
            mu, v = jo.mean_var(Z, w, beta, lamz, dadd, s11, xc)
            np.testing.assert_allclose(mean[t, k], mu.imag / h, rtol=1e-12, atol=1e-12 * np.abs(mean[t]).max())
            np.testing.assert_allclose(2.0 * cov[t, k, 0], v.imag / h, rtol=1e-12,
                                       atol=1e-12 * np.abs(cov[t, 1:, 0]).max())
        mu, v = jo.mean_var(Z, w, beta, lamz, dadd, s11, x)
        # one solve with every right-hand side against separate solves: the conditioning of S22 times an ulp apart
        assert abs(mean[t, 0] - mu) <= 1e-10 * np.abs(mean[t]).max() and abs(cov[t, 0, 0] - v) <= 1e-10 * abs(v)


def test_gradient_covariance_matches_mixed_differences():
    """Sigma_grad = d^2 Sigma(x, y) / dx_k dy_l at y = x, Sigma the nugget-free predictive cross-covariance."""
    Z, w, beta, lamz, dadd, s11, X = _block(m=20, q=3, seed=4)
    _, cov = jo.block(Z, w, beta, lamz, dadd, s11, X, 1)
    h = 1e-4
    for t, x in enumerate(X):
        ref = np.empty((3, 3))
        for k in range(3):
            for l in range(3):
                ek = np.zeros(4)
                el = np.zeros(4)
                ek[k + 1] = h
                el[l + 1] = h
                S = lambda a, b: jo.cross_cov(Z, beta, lamz, dadd, a, b)   # noqa: E731
                ref[k, l] = (S(x + ek, x + el) - S(x + ek, x - el) - S(x - ek, x + el) + S(x - ek, x - el)) / (4 * h * h)
        np.testing.assert_allclose(cov[t, 1:, 1:], ref, rtol=1e-6, atol=1e-6 * np.abs(ref).max())


def test_beta_zero_psd_and_symmetry():
    Z, w, beta, lamz, dadd, s11, X = _block(m=30, q=4, seed=5)
    beta[2] = 0.0
    mean, cov = jo.block(Z, w, beta, lamz, dadd, s11, X, 1)
    assert np.all(mean[:, 2] == 0.0) and np.all(cov[:, 2, :] == 0.0) and np.all(cov[:, :, 2] == 0.0)
    beta[2] = 0.7
    mean, cov = jo.block(Z, w, beta, lamz, dadd, s11, X, 1)
    for c in cov:
        np.testing.assert_allclose(c, c.T, rtol=0, atol=1e-10 * np.abs(c).max())
        lam = np.linalg.eigvalsh(0.5 * (c + c.T))
        assert lam.min() >= -1e-12 * np.trace(c)
    cc = jo.compact(cov)
    assert np.array_equal(cc[:, 0], cov[:, 0, 0]) and np.array_equal(cc[:, 1:5], cov[:, 1:, 0])
    assert np.array_equal(cc[:, 5:], np.diagonal(cov, axis1=1, axis2=2)[:, 1:])


def _per_sample(S=4, N=3, pu=3, q=2, seed=6):
    """Oracle per-sample results of S samples x pu PCs on one design."""
    rng = np.random.default_rng(seed)
    Z = np.concatenate([np.full((15, 1), 0.5), rng.uniform(0, 1, (15, q))], axis=1)
    X = np.concatenate([np.full((N, 1), 0.5), rng.uniform(0, 1, (N, q))], axis=1)
    B = S * pu
    beta = np.exp(rng.uniform(np.log(0.2), np.log(3.0), (B, q + 1)))
    lamz = 0.8 + rng.uniform(size=B)
    dadd = 1e-3 + 1e-2 * rng.uniform(size=B)
    s11 = 1.0 / lamz + 1e-3
    W = rng.standard_normal((B, 15))
    mean, cov = jo.blocks(Z, W, beta, lamz, dadd, s11, X, 1)
    mean = mean.reshape(S, pu, N, q + 1).transpose(0, 2, 1, 3)
    cov = cov.reshape(S, pu, N, q + 1, q + 1).transpose(0, 2, 1, 3, 4)
    return jo.per_sample(mean, cov), (Z, W, beta, lamz, dadd, s11, X)


def test_mixture_matches_its_definition():
    """The mixture's var is E v + Var mu, its grad_var the complex-step derivative of that, grad_cov E Sigma + Cov(grad)."""
    r, (Z, W, beta, lamz, dadd, s11, X) = _per_sample(S=4, N=2, pu=1, q=2)
    mx = jo.mixture(r)
    S = 4
    h = 1e-30
    for t, x in enumerate(X):
        for k in (1, 2):
            xc = x.astype(complex)
            xc[k] += 1j * h
            mv = [jo.mean_var(Z, W[s], beta[s], lamz[s], dadd[s], s11[s], xc) for s in range(S)]
            mu = np.array([a for a, _ in mv])
            v = np.array([b for _, b in mv])
            var = v.mean() + (mu * mu).mean() - mu.mean() ** 2
            np.testing.assert_allclose(mx['grad_var'][t, 0, k - 1], var.imag / h, rtol=1e-10,
                                       atol=1e-12 * np.abs(mx['grad_var']).max())
            np.testing.assert_allclose(mx['grad'][t, 0, k - 1], mu.mean().imag / h, rtol=1e-10)
        g = r['grad'][:, t, 0]
        ref = r['grad_cov'][:, t, 0].mean(0) + np.cov(g.T, bias=True)
        np.testing.assert_allclose(mx['grad_cov'][t, 0], ref, rtol=1e-13, atol=1e-15)


def test_linear_and_field_reductions():
    r, _ = _per_sample(S=3, N=2, pu=3, q=2)
    c = np.array([0.5, -2.0, 1.5])
    lin = jo.linear(r, c)
    np.testing.assert_allclose(lin['grad'], sum(c[j] * r['grad'][:, :, j] for j in range(3)), rtol=1e-14)
    np.testing.assert_allclose(lin['grad_cov'], sum(c[j] ** 2 * r['grad_cov'][:, :, j] for j in range(3)), rtol=1e-14)
    np.testing.assert_allclose(lin['var'], sum(c[j] ** 2 * r['var'][:, :, j] for j in range(3)), rtol=1e-14)
    coef = np.random.default_rng(1).standard_normal((3, 4))
    for option in ('samples', 'mean'):
        J, sd = jo.field(r, coef, option)
        for o in range(4):
            lo = jo.linear(r, coef[:, o])
            if option == 'mean':
                lo = jo.mixture(lo)
            np.testing.assert_allclose(J[..., o, :], lo['grad'], rtol=1e-13, atol=1e-15)
            np.testing.assert_allclose(sd[..., o, :], np.sqrt(np.diagonal(lo['grad_cov'], axis1=-2, axis2=-1)),
                                       rtol=1e-12)


def test_jacobian_abi_validates_arguments_without_a_device():
    from gladsgp_b200 import _lib
    h = _lib.load()
    one = ctypes.c_void_p(8)
    need = h.ggp_jacobian_workspace_bytes(64, 4, 1, 10, 2)
    assert need > 0 and h.ggp_jacobian_workspace_bytes(8192, 32, 1, 10, 2) > 0
    for bad in ((0, 4, 1, 10, 2), (8193, 4, 1, 10, 2), (64, 4, 4, 10, 2), (64, 33, 1, 10, 2), (64, 4, -1, 10, 2),
                (64, 4, 1, 0, 2), (64, 4, 1, 10, 0)):
        assert h.ggp_jacobian_workspace_bytes(*bad) == -1, bad
    # X, m, d, factor, u, beta, lamz, s11, Xp, n, B, col0, full, mean, cov, workspace, bytes, stream
    args = [one, 64, 4, one, one, one, one, one, one, 10, 2, 1, 1, one, one, one, need, None]
    for k in (0, 3, 4, 5, 6, 7, 8, 13, 14, 15):
        a = list(args)
        a[k] = None
        assert h.ggp_jacobian_f64(*a) == -1
        assert b'null pointer' in h.ggp_last_error_string()
    for k, v, msg in ((1, 0, b'must be positive'), (2, 0, b'must be positive'), (9, 0, b'must be positive'),
                      (10, 0, b'must be positive'), (1, 8193, b'm must be'), (11, 4, b'[1, 31]'), (2, 33, b'[1, 31]'),
                      (11, -1, b'[1, 31]'), (12, 2, b'full')):
        a = list(args)
        a[k] = v
        assert h.ggp_jacobian_f64(*a) == -1, (k, v)
        assert msg in h.ggp_last_error_string()
    a = list(args)
    a[16] = need - 1
    assert h.ggp_jacobian_f64(*a) == -4
    assert b'workspace too small' in h.ggp_last_error_string()


def test_emulator_jacobian_refuses_before_the_device():
    from gladsgp_b200 import gradient
    from posterior_helpers import sepia_model
    from gladsgp_b200 import synthetic
    model = sepia_model(m=30, q=2, pu=2, n_x=6, n_t=3)
    samples = synthetic.posterior_samples(2, 3, 2, seed=1)
    t = np.full((3, 2), 0.5)
    for kw in (dict(target='field', outputs=[10 ** 6]), dict(target='field', outputs=[]), dict(target='pc', outputs=[0]),
               dict(target='field', outputs=[0.5]), dict(target='pcs'), dict(target=[1.0, 2.0, 3.0]),
               dict(target=[1.0, np.nan]), dict(option='median')):
        with pytest.raises(ValueError):
            gradient.emulator_jacobian(model, samples, t, **kw)
    for bad in (np.full((3, 3), 0.5), np.full((0, 2), 0.5), np.array([[0.5, np.inf]])):
        with pytest.raises(ValueError):
            gradient.emulator_jacobian(model, samples, bad)
    old = gradient.FIELD_SAMPLES_BYTES
    try:
        gradient.FIELD_SAMPLES_BYTES = 8 * 2 * 3 * 2
        with pytest.raises(ValueError, match="option='mean'"):
            gradient.emulator_jacobian(model, samples, t, target='field', outputs=[0, 1])
    finally:
        gradient.FIELD_SAMPLES_BYTES = old
