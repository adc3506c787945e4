"""GPU: greedy ALC sequential design (csrc/ggp_design.cu, ops.design_score / ops.design_condition, gladsgp_b200.design)
against the FP64 oracle (oracle/design_oracle.py): indices, scores and integrated variances, determinism, chunking over
blocks, prefixes of a longer design and a one-input model with an empty half."""
import numpy as np
import pytest

from helpers import make_scalar_problem, synthetic
from oracle import design_oracle as do
from posterior_helpers import sepia_model as _model

pytestmark = pytest.mark.gpu

SCORE_RTOL = 1e-9
CANCEL_TOL = 1e-11


def _scalar_model(t=None, m=200):
    from sepia.SepiaData import SepiaData
    from sepia.SepiaModel import SepiaModel
    if t is None:
        pr = make_scalar_problem(m=m)
        t, y = pr['t'], pr['y']
    else:
        y = (t[:, 0] * np.sin(2 * np.pi * t[:, 0]))[:, None]
    data = SepiaData(t_sim=t, y_sim=y)
    data.transform_xt(); data.standardize_y()
    return SepiaModel(data)


def _points(model, n, seed):
    sd = model.data.sim_data
    lo, hi = np.asarray(sd.orig_t_min, dtype=np.float64).reshape(-1), np.asarray(sd.orig_t_max, dtype=np.float64).reshape(-1)
    return np.random.default_rng(seed).uniform(lo, hi, (n, lo.size))


def _oracle(model, samples, C, R, k, w):
    from gladsgp_b200 import calibration as cal
    XC = do.designs(cal._to_trans(model, C))
    XR = XC if R is None else do.designs(cal._to_trans(model, R))
    return do.greedy_rank_one(model.num.zt, model.num.LamSim, samples, XR, XC, k, w)


def _cancel_tol(samples, w):
    """CANCEL_TOL * sum_b w_j / lamUz_b^2: the rounding of k - V.V, whose terms are as large as 1/lamUz."""
    lamUz = np.asarray(samples['lamUz'], dtype=np.float64).reshape(-1, w.size)
    return CANCEL_TOL * float(np.sum(w[None, :] / lamUz ** 2))


def _check(out, ref, samples):
    """Indices equal while the oracle's top-two margins exceed the tolerance; scores and imse within it up to there.
    Returns the number of steps compared and the largest error relative to the tolerance's second term."""
    tol_c = _cancel_tol(samples, out['pc_weights'])
    k = out['index'].size
    n = 0
    worst = 0.0
    for t in range(k):
        tol = SCORE_RTOL * abs(ref['score'][t]) + tol_c
        err_i = abs(out['imse'][t] - ref['imse'][t])
        assert err_i <= SCORE_RTOL * abs(ref['imse'][t]) + tol_c, (t, out['imse'][t], ref['imse'][t])
        worst = max(worst, err_i / tol_c)
        if ref['margin'][t] <= tol:
            return n, worst
        assert out['index'][t] == ref['index'][t], (t, out['index'], ref['index'], ref['margin'])
        err = abs(out['score'][t] - ref['score'][t])
        assert err <= tol, (t, out['score'][t], ref['score'][t])
        worst = max(worst, err / tol_c)
        n += 1
    assert abs(out['imse'][k] - ref['imse'][k]) <= SCORE_RTOL * abs(ref['imse'][k]) + tol_c
    return n, worst


@pytest.mark.parametrize('m,q,pu,S,n_ref,n_cand,k,given', [
    (32, 2, 1, 1, 45, 70, 8, False),
    (200, 3, 3, 4, 101, 150, 8, True),
    (512, 8, 10, 16, 130, 257, 6, False),
    (200, 4, 10, 4, None, 99, 8, True),
    (512, 2, 3, 1, 77, 200, 5, True),
    (32, 1, 3, 16, 33, 65, 8, False),
])
def test_next_runs_match_oracle(cuda, m, q, pu, S, n_ref, n_cand, k, given):
    from gladsgp_b200 import design
    model = _model(m=m, q=q, pu=pu, seed=m + pu)
    samples = synthetic.posterior_samples(S, 1 + q, pu, seed=m + S)
    C = _points(model, n_cand, seed=1)
    R = None if n_ref is None else _points(model, n_ref, seed=2)
    w = np.random.default_rng(3).uniform(0.2, 3.0, pu) if given else None
    out = design.next_runs(model, samples, C, k, reference=R, pc_weights=w)
    if not given:
        np.testing.assert_allclose(out['pc_weights'], design.field_weights(model), rtol=0)
    ref = _oracle(model, samples, C, R, k, out['pc_weights'])
    n, worst = _check(out, ref, samples)
    assert n >= min(k, 3), (n, ref['margin'])
    print('m=%d pu=%d S=%d: %d steps compared, max error %.3g x the cancellation term' % (m, pu, S, n, worst))
    np.testing.assert_array_equal(out['t'], C[out['index']])
    # imse_t - imse_{t+1} = score_t
    tol = SCORE_RTOL * np.abs(out['score']) + 2 * _cancel_tol(samples, out['pc_weights'])
    assert np.all(np.abs(out['imse'][:-1] - out['imse'][1:] - out['score']) <= tol)
    assert np.unique(out['index']).size == k


@pytest.mark.parametrize('reference', [False, True])
def test_cfg2_scalar_model(cuda, reference):
    from gladsgp_b200 import design
    model = _scalar_model()
    samples = synthetic.posterior_samples(4, 2, 1, seed=9)
    C = np.linspace(-0.1, 1.1, 83)[:, None]
    R = np.linspace(0.0, 1.0, 57)[:, None] if reference else None
    out = design.next_runs(model, samples, C, 8, reference=R)
    ref = _oracle(model, samples, C, R, 8, out['pc_weights'])
    n, worst = _check(out, ref, samples)
    assert n >= 3
    print('cfg2 reference=%s: %d steps compared, max error %.3g x the cancellation term' % (reference, n, worst))


def _mid_problem():
    model = _model(m=200, q=3, pu=3, seed=8)
    samples = synthetic.posterior_samples(4, 4, 3, seed=4)
    return model, samples, _points(model, 131, seed=5), _points(model, 70, seed=6)


def _same(a, b, j=None):
    j = a['index'].size if j is None else j
    np.testing.assert_array_equal(a['index'][:j], b['index'][:j])
    np.testing.assert_array_equal(a['score'][:j], b['score'][:j])
    np.testing.assert_array_equal(a['imse'][:j + 1], b['imse'][:j + 1])


def test_identical_calls_give_identical_bits(cuda):
    from gladsgp_b200 import design
    model, samples, C, R = _mid_problem()
    a = design.next_runs(model, samples, C, 6, reference=R)
    model._pred_cache = None                                 # a fresh factorisation too
    b = design.next_runs(model, samples, C, 6, reference=R)
    _same(a, b)


@pytest.mark.parametrize('reference', [False, True])
def test_several_chunks_give_identical_bits(cuda, monkeypatch, reference):
    from gladsgp_b200 import design
    model, samples, C, R = _mid_problem()
    R = R if reference else None
    a = design.next_runs(model, samples, C, 6, reference=R)
    Mp = (model.num.m + 31) // 32 * 32
    per = ((R.shape[0] if reference else 0) + C.shape[0]) * Mp * 8
    for blocks in (1, 5):                                    # 12 blocks in chunks of 1 and of 5 (5, 5, 2)
        monkeypatch.setattr(design, 'DESIGN_V_BYTES', blocks * per)
        _same(a, design.next_runs(model, samples, C, 6, reference=R))


def test_prefix_of_a_longer_design(cuda):
    from gladsgp_b200 import design
    model, samples, C, R = _mid_problem()
    long = design.next_runs(model, samples, C, 12, reference=R)
    for j in (1, 5, 8):
        _same(long, design.next_runs(model, samples, C, j, reference=R), j)


def test_first_run_fills_the_empty_half(cuda):
    from gladsgp_b200 import design
    t = np.sort(np.random.default_rng(0).uniform(0.0, 0.5, 40))[:, None]
    t[0, 0], t[-1, 0] = 0.0, 0.5
    model = _scalar_model(t=t)
    rng = np.random.default_rng(1)
    S = 4
    samples = dict(betaU=np.column_stack([np.full(S, 1.0), rng.uniform(1.0, 3.0, S)]),
                   lamUz=rng.uniform(0.8, 1.2, (S, 1)), lamWs=np.full((S, 1), 1000.0), lamWOs=np.full((S, 1), 100.0))
    C = np.linspace(0.0, 1.0, 101)[:, None]
    out = design.next_runs(model, samples, C, 3)
    assert 0.5 < out['t'][0, 0] <= 1.0, out['t']
    assert np.all(out['score'] > 0) and np.all(np.diff(out['imse']) < 0)
