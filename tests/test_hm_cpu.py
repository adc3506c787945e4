"""CPU: the history-matching oracle (oracle/hm_oracle.py) -- the feature route against the direct route -- and the
argument checks of the C entry points and of gladsgp_b200.history (no device needed)."""
import ctypes

import numpy as np
import pytest

from helpers import make_problem, synthetic
from oracle import hm_oracle as ho

ROUTE_RTOL = 1e-12


def _moments(S, pu, N, n_o, seed):
    rng = np.random.default_rng(seed)
    mu = rng.standard_normal((S, pu, N)) * rng.uniform(0.1, 2.0, (1, pu, 1))
    var = rng.uniform(0.0, 0.5, (S, pu, N))
    var[0, 0, :3] = -1e-17                                    # clamped at 0, as the device does
    K_O = rng.standard_normal((pu, n_o)) * 0.5
    r = rng.standard_normal(n_o) * 2.0
    c = rng.uniform(0.01, 0.2, n_o)
    return mu, var, K_O, r, c


@pytest.mark.parametrize('S,pu,N,n_o', [(1, 1, 50, 1), (1, 3, 40, 17), (4, 1, 30, 9), (8, 10, 60, 100), (3, 32, 20, 45),
                                        (16, 2, 33, 7)])
def test_feature_route_matches_direct_route(S, pu, N, n_o):
    mu, var, K_O, r, c = _moments(S, pu, N, n_o, seed=S * 100 + pu + n_o)
    ea, Va = ho.route_features(mu, var, K_O, r, c)
    eb, Vb = ho.route_direct(mu, var, K_O, r, c)
    m, _ = ho.mixture(mu, var)
    te = np.abs(r)[None, :] + np.abs(m) @ np.abs(K_O)        # the size of e's terms
    assert np.all(np.abs(ea - eb) <= ROUTE_RTOL * te)
    np.testing.assert_allclose(Va, Vb, rtol=ROUTE_RTOL, atol=0)
    Ia, Ib = ho.implausibility(ea, Va), ho.implausibility(eb, Vb)
    sc = ho.scale(mu, var, K_O, r, c)
    assert np.all(np.abs(Ia - Ib) <= ROUTE_RTOL * (Ia + sc[:, None]))
    for order in range(1, min(8, n_o) + 1):
        a, b = ho.reduce(Ia, order, 1.5), ho.reduce(Ib, order, 1.5)
        assert np.all(np.diff(a['impl'], axis=1) <= 0)
        np.testing.assert_allclose(a['impl'], b['impl'], rtol=1e-11, atol=0)
        far = a['edge'] > 1e-9
        np.testing.assert_array_equal(a['n_over'][far], b['n_over'][far])
        np.testing.assert_array_equal(a['nroy'], a['impl'][:, order - 1] <= 1.5)


def test_mixture_is_the_law_of_total_variance():
    mu, var, _, _, _ = _moments(6, 3, 5, 1, seed=2)
    m, M = ho.mixture(mu, var)
    for n in range(5):
        cov = np.cov(mu[:, :, n].T, ddof=0) + np.diag(np.maximum(var[:, :, n], 0).mean(0))
        np.testing.assert_allclose(M[n], cov, rtol=1e-13, atol=1e-15)
        np.testing.assert_allclose(m[n], mu[:, :, n].mean(0), rtol=1e-14)


def test_implausibility_edge_rules():
    e = np.array([[0.0, 1.0, np.nan, 2.0]])
    V = np.array([[0.0, 0.0, 1.0, 4.0]])
    I = ho.implausibility(e, V)                               # a NaN (here 0 / 0) counts as +inf
    np.testing.assert_array_equal(I, [[np.inf, np.inf, np.inf, 1.0]])
    out = ho.reduce(I, 2, 3.0)
    assert out['n_over'][0] == 3 and not out['nroy'][0]


def test_hm_abi_validates_arguments_without_a_device():
    from gladsgp_b200 import _lib
    h = _lib.load()
    assert h.ggp_hm_workspace_bytes(0, 5, 3, 2) == -1 and h.ggp_hm_workspace_bytes(5, 0, 3, 2) == -1
    assert h.ggp_hm_workspace_bytes(5, 5, 0, 2) == -1 and h.ggp_hm_workspace_bytes(5, 5, 33, 2) == -1
    assert h.ggp_hm_workspace_bytes(5, 5, 3, 0) == -1 and h.ggp_hm_workspace_bytes(5, 5, 32, 1 << 26) == -1
    need = h.ggp_hm_workspace_bytes(100, 1000, 10, 8)
    assert need >= 100 * (16 + 56) * 8
    one = ctypes.c_void_p(8)
    # mean, var, S, pu, n, K_O, r, c, n_o, order, cutoff, impl, nover, workspace, workspace_bytes, stream
    args = [one, one, 8, 10, 100, one, one, one, 1000, 3, 3.0, one, one, one, need, None]
    for k in (0, 1, 5, 6, 7, 11, 12, 13):
        a = list(args)
        a[k] = None
        assert h.ggp_hm_impl_f64(*a) == -1
        assert b'null pointer' in h.ggp_last_error_string()
    for k, v, msg in ((2, 0, b'must be positive'), (4, 0, b'must be positive'), (8, -1, b'must be positive'),
                      (3, 0, b'pu must be'), (3, 33, b'pu must be'), (9, 0, b'order must be'), (9, 9, b'order must be'),
                      (10, 0.0, b'cutoff'), (10, -1.0, b'cutoff'), (10, float('nan'), b'cutoff'),
                      (10, float('inf'), b'cutoff'), (2, 1 << 28, b'S * pu'), (14, need - 1, b'workspace too small')):
        a = list(args)
        a[k] = v
        assert h.ggp_hm_impl_f64(*a) == -1, (k, v)
        assert msg in h.ggp_last_error_string()
    a = list(args)
    a[8], a[9] = 2, 3                                        # order above n_o
    assert h.ggp_hm_impl_f64(*a) == -1 and b'order must be' in h.ggp_last_error_string()


def _model(q=2, pu=3, x_sim=False, m=40):
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
    data.create_K_basis(K=pr['K'])
    return SepiaModel(data)


def test_history_match_value_errors():
    from gladsgp_b200 import history
    model = _model()
    samples = synthetic.posterior_samples(2, 3, 3, seed=1)
    n_y = model.num.n_y
    O = np.arange(0, n_y, 7)
    y = np.zeros(O.size)
    t = np.random.default_rng(0).uniform(0, 1, (20, 2))
    bad = [
        dict(obs_index=np.r_[O, O[:1]]), dict(obs_index=np.r_[O[:-1], n_y]), dict(obs_index=np.r_[-1, O[1:]]),
        dict(y_obs=np.zeros(O.size + 1)),
        dict(obs_sd=-0.1), dict(obs_sd=np.inf), dict(obs_sd=np.nan), dict(obs_sd=np.ones(O.size - 1)),
        dict(disc_sd=-0.1), dict(disc_sd=np.inf), dict(disc_sd=np.nan), dict(disc_sd=np.ones(2)),
        dict(disc_sd=np.r_[np.ones(O.size - 1), -1.0]),
        dict(order=0), dict(order=9), dict(order=2.5), dict(order=True),
        dict(cutoff=0.0), dict(cutoff=-1.0), dict(cutoff=np.inf), dict(cutoff=np.nan),
        dict(t=t[:, :1]), dict(t=np.zeros((0, 2))), dict(t=np.where(t == t[3, 1], np.nan, t)),
    ]
    for kw in bad:
        args = dict(dict(y_obs=y, t=t, obs_index=O), **kw)
        with pytest.raises(ValueError):
            history.history_match(model, samples, **args)
    with pytest.raises(ValueError):                             # order above n_o
        history.history_match(model, samples, np.zeros(2), t, obs_index=O[:2], order=3)
    with pytest.raises(ValueError):
        history.history_match(_model(x_sim=True), samples, y, t, obs_index=O)
