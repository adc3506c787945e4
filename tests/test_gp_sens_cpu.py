"""CPU: the closed-form GP sensitivity oracle (oracle/gp_sens_oracle.py) against tensor Gauss-Legendre quadrature and
exact properties, and the argument checks of the C entry points (no device needed)."""
import ctypes

import numpy as np
import pytest
from scipy import integrate

from helpers import ROOT  # noqa: F401  (puts the repository root on sys.path)
from oracle import gp_sens_oracle as gso

QUAD_RTOL = 1e-10


def _random_function(rng, N, q, shared_beta=False):
    a = rng.standard_normal(N)
    if shared_beta:
        beta = np.broadcast_to(np.exp(rng.uniform(np.log(0.02), np.log(6.0), q)), (N, q)).copy()
    else:
        beta = np.exp(rng.uniform(np.log(0.02), np.log(6.0), (N, q)))
    Z = rng.uniform(0.0, 1.0, (N, q))
    return a, beta, Z


@pytest.mark.parametrize('q', [1, 2, 3])
@pytest.mark.parametrize('shared_beta', [False, True])
def test_closed_forms_match_tensor_quadrature(q, shared_beta):
    rng = np.random.default_rng(10 * q + shared_beta)
    a, beta, Z = _random_function(rng, 9, q, shared_beta)
    grid = np.linspace(0.0, 1.0, 7)
    c = gso.moments(a, beta, Z)
    r = gso.quad_moments(a, beta, Z, nodes=60, grid=grid)
    for k in ('E0', 'Mall', 'M1', 'Mt', 'V'):
        np.testing.assert_allclose(c[k], r[k], rtol=QUAD_RTOL, atol=QUAD_RTOL * abs(r['Mall']), err_msg=k)
    np.testing.assert_allclose(c['first'], r['first'], rtol=0, atol=1e-9)
    np.testing.assert_allclose(c['total'], r['total'], rtol=0, atol=1e-9)
    me = gso.main_effects(a, beta, Z, grid)
    np.testing.assert_allclose(me, r['main_effect'], rtol=QUAD_RTOL, atol=QUAD_RTOL * np.abs(r['main_effect']).max())
    # the main-effect curve integrates to E0 and its square to M({k})
    x, w = np.polynomial.legendre.leggauss(60)
    x, w = 0.5 * (x + 1.0), 0.5 * w
    curves = gso.main_effects(a, beta, Z, x)
    np.testing.assert_allclose(curves @ w, c['E0'], rtol=QUAD_RTOL, atol=1e-14)
    np.testing.assert_allclose((curves * curves) @ w, c['M1'], rtol=QUAD_RTOL)


def test_one_input_gives_first_and_total_one():
    rng = np.random.default_rng(1)
    a, beta, Z = _random_function(rng, 12, 1)
    c = gso.moments(a, beta, Z)
    np.testing.assert_allclose(c['first'], [1.0], rtol=0, atol=1e-12)
    np.testing.assert_allclose(c['total'], [1.0], rtol=0, atol=1e-12)


def test_beta_zero_input_has_zero_indices_and_unit_integrals():
    rng = np.random.default_rng(2)
    a, beta, Z = _random_function(rng, 10, 3)
    beta[:, 1] = 0.0
    assert np.all(gso.I1(0.0, Z[:, 1]) == 1.0)
    assert np.all(gso.I2(0.0, Z[:, 1], 0.0, Z[::-1, 1]) == 1.0)
    c = gso.moments(a, beta, Z)
    assert c['first'][1] == 0.0 and c['total'][1] == 0.0
    assert np.all(c['first'][[0, 2]] > 0) and np.all(c['total'][[0, 2]] > 0)


def test_additive_function_has_equal_first_and_total():
    """Every term depends on one input only (beta = 0 on the others): f is additive, so S_k = T_k and sum S_k = 1."""
    rng = np.random.default_rng(3)
    q, N = 3, 12
    a, beta, Z = _random_function(rng, N, q)
    keep = np.arange(N) % q
    beta = np.where(np.arange(q)[None, :] == keep[:, None], beta, 0.0)
    c = gso.moments(a, beta, Z)
    np.testing.assert_allclose(c['first'], c['total'], rtol=0, atol=1e-12)
    np.testing.assert_allclose(c['first'].sum(), 1.0, rtol=0, atol=1e-12)


@pytest.mark.parametrize('b,z,b2,z2', [(0.7, 0.3, 0.7, 0.3), (5.0, 0.9, 5.0, 0.9), (0.02, 0.0, 3.0, 1.0), (2.0, 0.4, 0.0, 0.1)])
def test_integrals_match_adaptive_quadrature(b, z, b2, z2):
    ref2, _ = integrate.quad(lambda x: np.exp(-b * (x - z) ** 2 - b2 * (x - z2) ** 2), 0.0, 1.0, epsabs=0, epsrel=1e-13)
    np.testing.assert_allclose(gso.I2(b, z, b2, z2), ref2, rtol=1e-13)
    ref1, _ = integrate.quad(lambda x: np.exp(-b * (x - z) ** 2), 0.0, 1.0, epsabs=0, epsrel=1e-13)
    np.testing.assert_allclose(gso.I1(b, z), ref1, rtol=1e-13)


def test_mean_mode_terms_are_the_sample_average():
    """block_terms('mean') is the average over samples of the per-sample functions: E0 is the mean of their E0."""
    rng = np.random.default_rng(4)
    S, pu, m, q = 3, 2, 5, 2
    Zin = rng.uniform(0, 1, (m, q))
    beta = np.exp(rng.uniform(-2, 1, (S, pu, q)))
    a = rng.standard_normal((S, pu, m))
    per = gso.block_terms(Zin, beta, a, 'samples')
    mean = gso.block_terms(Zin, beta, a, 'mean')
    for j in range(pu):
        e = np.mean([gso.moments(*per[s * pu + j])['E0'] for s in range(S)])
        np.testing.assert_allclose(gso.moments(*mean[j])['E0'], e, rtol=1e-13)


def test_gp_sens_abi_validates_arguments_without_a_device():
    from gladsgp_b200 import _lib
    h = _lib.load()
    one = ctypes.c_void_p(8)
    need = h.ggp_gp_sens_workspace_bytes(64, 3, 4, 2, 0)
    assert need > 0 and h.ggp_gp_sens_workspace_bytes(64, 3, 4, 2, 1) > 0
    for bad in ((64, 0, 4, 2, 0), (64, 33, 4, 2, 0), (0, 3, 4, 2, 0), (64, 3, 0, 2, 0), (64, 3, 4, 0, 0), (64, 3, 4, 2, 2),
                (1 << 20, 3, 1 << 12, 1, 1)):
        assert h.ggp_gp_sens_workspace_bytes(*bad) == -1, bad
    # Z, m, q, beta, a, S, pu, mode, M, E0, workspace, bytes, stream
    args = [one, 64, 3, one, one, 4, 2, 0, one, one, one, need, None]
    for k in (0, 3, 4, 8, 9, 10):
        a = list(args)
        a[k] = None
        assert h.ggp_gp_sens_f64(*a) == -1
        assert b'null pointer' in h.ggp_last_error_string()
    for k, v, msg in ((2, 0, b'q must be'), (2, 33, b'q must be'), (1, 0, b'must be positive'), (5, -1, b'must be positive'),
                      (6, 0, b'must be positive'), (7, 2, b'mode')):
        a = list(args)
        a[k] = v
        assert h.ggp_gp_sens_f64(*a) == -1
        assert msg in h.ggp_last_error_string()
    a = list(args)
    a[11] = need - 1
    assert h.ggp_gp_sens_f64(*a) == -4
    assert b'workspace too small' in h.ggp_last_error_string()
    # Z, m, q, beta, a, S, pu, mode, grid, ngrid, out, workspace, bytes, stream
    margs = [one, 64, 3, one, one, 4, 2, 0, one, 21, one, one, need, None]
    for k in (0, 3, 4, 8, 10, 11):
        a = list(margs)
        a[k] = None
        assert h.ggp_main_effects_f64(*a) == -1
        assert b'null pointer' in h.ggp_last_error_string()
    for k, v, msg in ((9, 0, b'ngrid'), (2, 40, b'q must be'), (7, -1, b'mode')):
        a = list(margs)
        a[k] = v
        assert h.ggp_main_effects_f64(*a) == -1
        assert msg in h.ggp_last_error_string()
    a = list(margs)
    a[12] = 0
    assert h.ggp_main_effects_f64(*a) == -4
