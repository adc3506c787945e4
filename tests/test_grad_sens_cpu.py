"""CPU: the closed-form gradient outer-product oracle (oracle/grad_sens_oracle.py) against adaptive and tensor Gauss-Legendre
quadrature, central differences and exact properties, and the argument checks of the C entry points (no device needed)."""
import ctypes

import numpy as np
import pytest
from scipy import integrate

from helpers import ROOT  # noqa: F401  (puts the repository root on sys.path)
from oracle import gp_sens_oracle as gso
from oracle import grad_sens_oracle as gro


def _random_function(rng, N, q, shared_beta=False):
    a = rng.standard_normal(N)
    if shared_beta:
        beta = np.broadcast_to(np.exp(rng.uniform(np.log(0.02), np.log(6.0), q)), (N, q)).copy()
    else:
        beta = np.exp(rng.uniform(np.log(0.02), np.log(6.0), (N, q)))
    Z = rng.uniform(0.0, 1.0, (N, q))
    return a, beta, Z


CASES = [(0.7, 0.3, 0.7, 0.3), (5.0, 0.9, 5.0, 0.9), (0.02, 0.0, 3.0, 1.0), (2.0, 0.4, 0.0, 0.1), (0.0, 0.6, 1.5, 0.2),
         (0.0, 0.3, 0.0, 0.8), (1e4, 0.0, 1e4, 1.0), (1e4, 0.5, 3.0, 0.49), (1e4, 1.0, 1e4, 1.0), (0.3, 1.0, 8.0, 0.0),
         (40.0, 0.1, 0.5, 0.95)]


@pytest.mark.filterwarnings('ignore::scipy.integrate.IntegrationWarning')
@pytest.mark.parametrize('b,z,b2,z2', CASES)
def test_integrals_match_adaptive_quadrature(b, z, b2, z2):
    def phi(x, bb, zz):
        return np.exp(-bb * (x - zz) ** 2)

    def dphi(x, bb, zz):
        return -2.0 * bb * (x - zz) * phi(x, bb, zz)

    pts = [z, z2]

    def quad(f):
        return integrate.quad(f, 0.0, 1.0, epsabs=0, epsrel=2e-14, limit=400, points=pts)[0]

    I2, G12, G21, H = gro.integrals(b, z, b2, z2)
    refs = (quad(lambda x: phi(x, b, z) * phi(x, b2, z2)), quad(lambda x: dphi(x, b, z) * phi(x, b2, z2)),
            quad(lambda x: phi(x, b, z) * dphi(x, b2, z2)), quad(lambda x: dphi(x, b, z) * dphi(x, b2, z2)))
    for got, ref, name in zip((I2, G12, G21, H), refs, ('I2', 'G12', 'G21', 'H')):
        # relative to the value; values far below the integrand's size (cancelling +/- lobes) to that size
        size = quad(lambda x, n=name: abs({'I2': phi(x, b, z) * phi(x, b2, z2), 'G12': dphi(x, b, z) * phi(x, b2, z2),
                                            'G21': phi(x, b, z) * dphi(x, b2, z2),
                                            'H': dphi(x, b, z) * dphi(x, b2, z2)}[n]))
        np.testing.assert_allclose(got, ref, rtol=1e-13, atol=1e-13 * size + 1e-300, err_msg=name)
    if b == 0.0:
        assert G12 == 0.0 and H == 0.0
    if b2 == 0.0:
        assert G21 == 0.0 and H == 0.0
    if b == b2 == 0.0:
        assert I2 == 1.0
    np.testing.assert_allclose(I2, gso.I2(b, z, b2, z2), rtol=1e-15)


@pytest.mark.parametrize('q', [1, 2, 3])
@pytest.mark.parametrize('shared_beta', [False, True])
def test_closed_form_matches_tensor_quadrature(q, shared_beta):
    rng = np.random.default_rng(20 * q + shared_beta)
    a, beta, Z = _random_function(rng, 9, q, shared_beta)
    r = gro.grad_outer(a, beta, Z)
    ref = gro.quad_grad_outer(a, beta, Z, nodes=60)
    np.testing.assert_allclose(r['C'], ref, rtol=1e-12, atol=1e-12 * np.abs(ref).max())


def test_weighted_pcs_match_tensor_quadrature():
    """Mode-2/3 pair weights: sum_{j,j'} Omega_jj' E[grad g_j grad g_j'^T] with a non-diagonal Omega."""
    rng = np.random.default_rng(7)
    S, pu, m, q = 2, 3, 6, 2
    Zin = rng.uniform(0, 1, (m, q))
    beta = np.exp(rng.uniform(-2, 1.5, (S, pu, q)))
    a = rng.standard_normal((S, pu, m))
    L = rng.standard_normal((pu, 5))
    omega = L @ L.T
    for mode in (2, 3):
        aa = a / S if mode == 3 else a
        funcs = gro.block_terms(Zin, beta, aa, mode, omega)
        for f, (fa, fb, fz, pw) in enumerate(funcs):
            pc = np.tile(np.repeat(np.arange(pu), m), S if mode == 3 else 1)
            ref = gro.quad_grad_outer(fa, fb, fz, pc=pc, omega=omega, nodes=60)
            got = gro.grad_outer(fa, fb, fz, pw)['C']
            np.testing.assert_allclose(got, ref, rtol=1e-12, atol=1e-12 * np.abs(ref).max(), err_msg='mode %d' % mode)


def test_analytic_gradient_matches_central_differences():
    rng = np.random.default_rng(3)
    a, beta, Z = _random_function(rng, 12, 4)
    x = rng.uniform(0, 1, (5, 4))
    g = gro.gradient(a, beta, Z, x)

    def f(p):
        return np.sum(a[None] * np.exp(-np.sum(beta[None] * (p[:, None, :] - Z[None]) ** 2, axis=2)), axis=1)

    h = 1e-5
    for k in range(4):
        e = np.zeros(4)
        e[k] = h
        fd = (f(x + e) - f(x - e)) / (2 * h)
        np.testing.assert_allclose(g[:, k], fd, rtol=1e-7, atol=1e-8 * np.abs(g).max())


def test_symmetric_positive_semidefinite():
    rng = np.random.default_rng(4)
    a, beta, Z = _random_function(rng, 30, 6)
    r = gro.grad_outer(a, beta, Z)
    C = r['C']
    assert np.array_equal(C, C.T)
    lam = np.linalg.eigvalsh(C)
    assert lam.min() >= -1e-12 * r['A'].max()
    assert np.all(np.abs(C) <= r['A'] * (1 + 1e-15))


def test_beta_zero_input_has_exactly_zero_row_and_column():
    rng = np.random.default_rng(5)
    a, beta, Z = _random_function(rng, 14, 4)
    beta[:, 2] = 0.0
    C = gro.grad_outer(a, beta, Z)['C']
    assert np.all(C[2, :] == 0.0) and np.all(C[:, 2] == 0.0)
    assert np.all(np.diag(C)[[0, 1, 3]] > 0)


@pytest.mark.parametrize('q', [1, 2, 3])
def test_dgsm_bounds_the_total_index(q):
    """T_k V <= nu_k / pi^2 (Sobol' and Kucherenko 2009, uniform inputs on [0, 1])."""
    rng = np.random.default_rng(30 + q)
    for _ in range(4):
        a, beta, Z = _random_function(rng, 10, q)
        nu = np.diag(gro.grad_outer(a, beta, Z)['C'])
        mo = gso.moments(a, beta, Z)
        assert np.all(mo['total'] * mo['V'] <= nu / np.pi ** 2 * (1 + 1e-12)), (mo['total'] * mo['V'], nu / np.pi ** 2)


def test_unit_omega_pick_equals_the_per_block_function():
    """Mode 2 with Omega = e_j e_j^T is mode 0's block (s, j); Omega = c c^T is mode 0 of the weights c_j a_j summed."""
    rng = np.random.default_rng(6)
    S, pu, m, q = 2, 3, 7, 3
    Zin = rng.uniform(0, 1, (m, q))
    beta = np.exp(rng.uniform(-2, 1.5, (S, pu, q)))
    a = rng.standard_normal((S, pu, m))
    per = gro.block_terms(Zin, beta, a, 0)
    for j in range(pu):
        e = np.zeros((pu, pu))
        e[j, j] = 1.0
        for s, (fa, fb, fz, pw) in enumerate(gro.block_terms(Zin, beta, a, 2, e)):
            ref = gro.grad_outer(*per[s * pu + j][:3])['C']
            got = gro.grad_outer(fa, fb, fz, pw)['C']
            np.testing.assert_allclose(got, ref, rtol=1e-13, atol=1e-14 * np.abs(ref).max())
    c = rng.standard_normal(pu)
    for s, (fa, fb, fz, pw) in enumerate(gro.block_terms(Zin, beta, a, 2, np.outer(c, c))):
        # the same function written as terms with weights c_j a_sji and no pair weight
        ca = (c[:, None] * a[s]).reshape(-1)
        ref = gro.grad_outer(ca, fb, fz)['C']
        got = gro.grad_outer(fa, fb, fz, pw)['C']
        np.testing.assert_allclose(got, ref, rtol=1e-13, atol=1e-14 * np.abs(ref).max())


def test_grad_sens_abi_validates_arguments_without_a_device():
    from gladsgp_b200 import _lib
    h = _lib.load()
    one = ctypes.c_void_p(8)
    need = h.ggp_grad_sens_workspace_bytes(64, 3, 4, 2, 0)
    assert need > 0 and all(h.ggp_grad_sens_workspace_bytes(64, 3, 4, 2, md) > 0 for md in (1, 2, 3))
    for bad in ((64, 0, 4, 2, 0), (64, 33, 4, 2, 0), (0, 3, 4, 2, 0), (64, 3, 0, 2, 0), (64, 3, 4, 0, 0), (64, 3, 4, 2, 4),
                (64, 3, 4, 2, -1), (1 << 20, 3, 1 << 12, 1, 1), (1 << 12, 3, 1 << 10, 1 << 10, 3), (1 << 16, 3, 2, 1 << 15, 2),
                (8, 3, 1 << 16, 1 << 15, 0)):
        assert h.ggp_grad_sens_workspace_bytes(*bad) == -1, bad
    assert h.ggp_grad_sens_workspace_bytes(1 << 12, 3, 1 << 10, 1 << 10, 0) > 0    # per block: m terms
    # Z, m, q, beta, a, S, pu, mode, omega, C, workspace, bytes, stream
    args = [one, 64, 3, one, one, 4, 2, 0, None, one, one, need, None]
    for k in (0, 3, 4, 9, 10):
        a = list(args)
        a[k] = None
        assert h.ggp_grad_sens_f64(*a) == -1
        assert b'null pointer' in h.ggp_last_error_string()
    for md in (2, 3):
        a = list(args)
        a[7] = md
        a[11] = h.ggp_grad_sens_workspace_bytes(64, 3, 4, 2, md)
        assert h.ggp_grad_sens_f64(*a) == -1
        assert b'omega' in h.ggp_last_error_string()
    for k, v, msg in ((2, 0, b'q must be'), (2, 33, b'q must be'), (1, 0, b'must be positive'), (5, -1, b'must be positive'),
                      (6, 0, b'must be positive'), (7, 4, b'mode'), (7, -1, b'mode')):
        a = list(args)
        a[k] = v
        assert h.ggp_grad_sens_f64(*a) == -1
        assert msg in h.ggp_last_error_string()
    a = list(args)
    a[1], a[5], a[6], a[7], a[8] = 1 << 12, 1 << 10, 1 << 10, 3, one
    assert h.ggp_grad_sens_f64(*a) == -1
    assert b'2^31' in h.ggp_last_error_string()
    a = list(args)
    a[11] = need - 1
    assert h.ggp_grad_sens_f64(*a) == -4
    assert b'workspace too small' in h.ggp_last_error_string()
    a = list(args)
    a[7], a[8] = 3, one
    a[11] = h.ggp_grad_sens_workspace_bytes(64, 3, 4, 2, 3) - 8
    assert h.ggp_grad_sens_f64(*a) == -4
