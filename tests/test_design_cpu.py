"""CPU: the sequential-design oracle (oracle/design_oracle.py) -- the rank-one route against re-factoring the enlarged
S22, the integrated-variance identity -- and the argument checks of the C entry points and of gladsgp_b200.design (no
device needed)."""
import ctypes

import numpy as np
import pytest

from helpers import make_problem, make_scalar_problem, synthetic
from oracle import design_oracle as do

ROUTE_RTOL = 1e-10


def _case(m, q, pu, S, n_ref, n_cand, seed):
    rng = np.random.default_rng(seed)
    zt = do.designs(rng.uniform(0, 1, (m, q)))
    samples = synthetic.posterior_samples(S, 1 + q, pu, seed=seed, f32=False)
    LamSim = rng.uniform(0.5, 3.0, pu)
    XC = do.designs(rng.uniform(-0.2, 1.2, (n_cand, q)))
    XR = XC if n_ref is None else do.designs(rng.uniform(0, 1, (n_ref, q)))
    return zt, LamSim, samples, XR, XC, rng.uniform(0.1, 2.0, pu)


@pytest.mark.parametrize('m,q,pu,S,n_ref,n_cand,k', [(20, 1, 1, 1, 17, 25, 5), (48, 2, 2, 2, 31, 60, 5),
                                                     (33, 3, 3, 2, None, 40, 4), (48, 8, 2, 1, 50, 60, 3)])
def test_rank_one_matches_direct_route(m, q, pu, S, n_ref, n_cand, k):
    zt, LamSim, samples, XR, XC, w = _case(m, q, pu, S, n_ref, n_cand, seed=m + n_cand)
    a = do.greedy_rank_one(zt, LamSim, samples, XR, XC, k, w)
    b = do.greedy_direct(zt, LamSim, samples, XR, XC, k, w)
    np.testing.assert_array_equal(a['index'], b['index'])
    np.testing.assert_allclose(a['imse'], b['imse'], rtol=ROUTE_RTOL, atol=0)
    np.testing.assert_allclose(a['score'], b['score'], rtol=ROUTE_RTOL, atol=0)
    for t in range(k):                                        # every unselected candidate's score, not only the winner's
        live = np.isfinite(b['scores'][t]) & (b['scores'][t] != 0)
        np.testing.assert_allclose(a['scores'][t][live], b['scores'][t][live], rtol=ROUTE_RTOL, atol=0)
    assert np.all(a['margin'] > 0)


def test_imse_identity_and_monotone():
    zt, LamSim, samples, XR, XC, w = _case(40, 2, 3, 3, 70, 90, seed=1)
    a = do.greedy_rank_one(zt, LamSim, samples, XR, XC, 10, w)
    np.testing.assert_allclose(a['imse'][:-1] - a['imse'][1:], a['score'], rtol=1e-9, atol=1e-14 * a['imse'][0])
    assert np.all(a['score'] > 0) and np.all(np.diff(a['imse']) < 0)
    assert np.unique(a['index']).size == 10


def test_design_abi_validates_arguments_without_a_device():
    from gladsgp_b200 import _lib
    h = _lib.load()
    one = ctypes.c_void_p(8)
    assert h.ggp_design_workspace_bytes(0, 4) == -1 and h.ggp_design_workspace_bytes(10, 0) == -1
    assert h.ggp_design_workspace_bytes(10, 4) == (40 + 4) * 8
    # XR, n_ref, XC, n_cand, d, beta, lamz, dadd, s11, wgt, V_R, V_C, m, A_R, A_C, Kp, t, B, accumulate, score, imse,
    # workspace, workspace_bytes, stream
    args = [one, 7, one, 10, 3, one, one, one, one, one, one, one, 40, one, one, 8, 2, 4, 0, one, one, one, 1 << 20, None]
    for k in (0, 2, 5, 6, 7, 8, 9, 10, 11, 13, 14, 20, 21):
        a = list(args)
        a[k] = None
        assert h.ggp_design_score_f64(*a) == -1
        assert b'null pointer' in h.ggp_last_error_string()
    for k, v, msg in ((1, 0, b'must be positive'), (3, 0, b'must be positive'), (4, 0, b'must be positive'),
                      (12, -1, b'must be positive'), (15, 0, b'must be positive'), (17, 0, b'must be positive'),
                      (15, 12, b'multiple of 8'), (12, 8193, b'm must be'), (16, 9, b't must be'), (16, -1, b't must be'),
                      (22, 8 * 43, b'workspace too small')):
        a = list(args)
        a[k] = v
        assert h.ggp_design_score_f64(*a) == -1, (k, v)
        assert msg in h.ggp_last_error_string()
    # XR, n_ref, XC, n_cand, d, beta, lamz, dadd, V_R, V_C, m, A_R, A_C, Kp, t, B, index, stream
    two = ctypes.c_void_p(16)
    cargs = [one, 7, two, 10, 3, one, one, one, one, two, 40, one, two, 8, 2, 4, 3, None]
    for k in (0, 2, 5, 6, 7, 8, 9, 11, 12):
        a = list(cargs)
        a[k] = None
        assert h.ggp_design_condition_f64(*a) == -1
        assert b'null pointer' in h.ggp_last_error_string()
    for k, v, msg in ((1, -3, b'must be positive'), (15, 0, b'must be positive'), (13, 4, b'multiple of 8'),
                      (14, 8, b't must be'), (14, -1, b't must be'), (16, 10, b'index out of range'),
                      (16, -1, b'index out of range')):
        a = list(cargs)
        a[k] = v
        assert h.ggp_design_condition_f64(*a) == -1, (k, v)
        assert msg in h.ggp_last_error_string()
    same = list(cargs)                                        # a shared reference / candidate set of another size
    same[2], same[9], same[12] = one, one, one
    assert h.ggp_design_condition_f64(*same) == -1
    assert b'n_ref == n_cand' in h.ggp_last_error_string()


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


def test_next_runs_value_errors():
    from gladsgp_b200 import design
    model = _model()
    samples = synthetic.posterior_samples(2, 3, 3, seed=1)
    cand = np.random.default_rng(0).uniform(0, 1, (20, 2))
    bad = [
        dict(n_new=0), dict(n_new=21), dict(n_new=2.5), dict(n_new=True),
        dict(candidates=cand[:, :1]), dict(candidates=cand[0]), dict(candidates=np.zeros((0, 2))),
        dict(reference=np.zeros((5, 3))),
        dict(candidates=np.where(np.arange(40).reshape(20, 2) == 7, np.nan, cand)),
        dict(reference=np.full((3, 2), np.inf)),
        dict(pc_weights=np.ones(2)), dict(pc_weights=np.ones((3, 1))), dict(pc_weights=[1.0, np.nan, 1.0]),
        dict(pc_weights=[1.0, -1.0, 1.0]),
    ]
    for kw in bad:
        args = dict(dict(candidates=cand, n_new=3), **kw)
        with pytest.raises(ValueError):
            design.next_runs(model, samples, **args)
    big = np.random.default_rng(1).uniform(0, 1, (200, 2))
    with pytest.raises(ValueError):
        design.next_runs(model, samples, big, n_new=design.MAX_NEW + 1)
    with pytest.raises(ValueError):
        design.next_runs(_model(x_sim=True), samples, cand, 3)


def test_next_runs_rejects_a_model_without_inputs():
    from gladsgp_b200 import design

    class Data:
        dummy_x = True

    class Num:
        q, pu = 0, 1

    class M:
        data, num = Data(), Num()
    with pytest.raises(ValueError):
        design.next_runs(M(), None, np.zeros((3, 0)), 1)


def test_field_weights():
    from gladsgp_b200 import design
    model = _model(pu=3)
    sd = model.data.sim_data
    K = np.asarray(sd.K, dtype=np.float64)
    ysd = np.broadcast_to(np.asarray(sd.orig_y_sd, dtype=np.float64).reshape(-1), (K.shape[1],))
    np.testing.assert_allclose(design.field_weights(model), [np.sum((K[j] * ysd) ** 2) for j in range(3)], rtol=1e-13)
    from sepia.SepiaData import SepiaData
    from sepia.SepiaModel import SepiaModel
    pr = make_scalar_problem(m=30)
    data = SepiaData(t_sim=pr['t'], y_sim=pr['y'])
    data.transform_xt(); data.standardize_y()
    scalar = SepiaModel(data)
    np.testing.assert_allclose(design.field_weights(scalar), [float(np.asarray(scalar.data.sim_data.orig_y_sd).reshape(-1)[0]) ** 2])
