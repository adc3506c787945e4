"""GPU: history matching (csrc/ggp_hm.cu, ops.hm_impl, gladsgp_b200.history) against the FP64 oracle
(oracle/hm_oracle.py): implausibilities, counts and the region not ruled out, the kernel's edge rules and output slabs,
determinism under identical calls, point chunks and point permutations, a known input that must not be ruled out, and a
second wave chosen by design.next_runs on that region.

Tolerance: impl within IMPL_RTOL impl + SCALE_TOL scale per point, with
  scale = max_i [(|r_i| + sum_j |K_ji m_j|) / sqrt(V_i) + I_i (sum_j sqrt(M_jj) |K_ji|)^2 / V_i]
(hm_oracle.scale): the terms of e_i over sqrt(V_i), and the terms of V_i (|M_jk| <= sqrt(M_jj M_kk), so their sum is at
most (sum_j sqrt(M_jj) |K_ji|)^2) times dI/dV = I / (2 V).  Counts and nroy are compared exactly where the oracle's
distance to the cutoff exceeds that tolerance."""
import numpy as np
import pytest

from helpers import synthetic
from oracle import hm_oracle as ho
from posterior_helpers import at as _at, emulator as _emulator, hm_obs as _obs_terms, mean_field as _mean_field, \
    native as _native, scalar_model as _scalar_model, sepia_model as _model

pytestmark = pytest.mark.gpu

IMPL_RTOL = 1e-10
SCALE_TOL = 1e-12


def _check(out, ref, cutoff):
    """impl within the tolerance; n_over and nroy exact away from the cutoff.  Returns the largest impl error over the
    scale term."""
    tol = IMPL_RTOL * ref['impl'] + SCALE_TOL * ref['scale'][:, None]
    err = np.abs(out['impl'] - ref['impl'])
    assert np.all(err <= tol), (np.max(err - tol), np.argmax(np.max(err - tol, axis=1)))
    tp = IMPL_RTOL * cutoff + SCALE_TOL * ref['scale']
    far = ref['edge'] > tp
    np.testing.assert_array_equal(out['n_over'][far], ref['n_over'][far])
    clear = ref['margin'] > tp
    np.testing.assert_array_equal(out['nroy'][clear], ref['nroy'][clear])
    assert np.all(np.diff(out['impl'], axis=1) <= 0)
    np.testing.assert_array_equal(out['nroy'], out['impl'][:, -1] <= cutoff)
    assert out['nroy_fraction'] == out['nroy'].mean()
    return float(np.max(err / np.maximum(ref['scale'][:, None], 1e-300)))


# (m, q, pu, S, N, n_o or None for every output, order, obs_sd per output, disc_sd per output)
CASES = [
    (64, 1, 2, 3, 200, 37, 1, False, False),
    (200, 3, 10, 8, 777, 1000, 3, True, True),
    (100, 3, 32, 4, 150, None, 2, False, True),
    (64, 2, 3, 1, 300, 50, 8, True, False),
    (64, 8, 10, 7, 129, None, 1, False, False),
]


@pytest.mark.parametrize('m,q,pu,S,N,n_o,order,sd_vec,disc_vec', CASES)
def test_history_match_matches_oracle(cuda, m, q, pu, S, N, n_o, order, sd_vec, disc_vec):
    from gladsgp_b200 import history
    rng = np.random.default_rng(m + q + pu + S)
    K = None
    n_x, n_t = (50, 20) if n_o and n_o > 200 else (20, 10)
    if pu > 25:                                              # beyond make_problem's 25 singular vectors
        K = (rng.standard_normal((pu, n_x * n_t)) * 0.3).astype(np.float32)
    model = _model(m=m, q=q, pu=pu, n_x=n_x, n_t=n_t, K=K)
    samples = synthetic.posterior_samples(S, 1 + q, pu, seed=m + S)
    em = _emulator(model, samples)
    n_y = model.num.n_y
    O = np.arange(n_y) if n_o is None else np.sort(rng.choice(n_y, size=n_o, replace=False))
    ysd = _at(model, model.data.sim_data.orig_y_sd, O)
    obs_sd = rng.uniform(0.01, 0.1, O.size) * ysd if sd_vec else 0.05 * float(np.mean(ysd))
    disc_sd = rng.uniform(0.0, 0.2, O.size) * ysd if disc_vec else 0.1 * float(np.mean(ysd))
    y = _mean_field(model, em, O, rng.uniform(0.2, 0.8, q)) + rng.standard_normal(O.size) * 0.05 * ysd
    tt = rng.uniform(0, 1, (N, q))
    cutoff = 3.0
    out = history.history_match(model, samples, y, _native(model, tt), obs_index=None if n_o is None else O,
                                obs_sd=obs_sd, disc_sd=disc_sd, order=order, cutoff=cutoff)
    assert out['impl'].shape == (N, order) and out['n_over'].dtype == np.int64 and out['nroy'].dtype == bool
    K_O, r, c = _obs_terms(model, samples, O, y, obs_sd, disc_sd)
    ref = ho.history_match(em, tt, K_O, r, c, order, cutoff)
    worst = _check(out, ref, cutoff)
    print('pu=%d S=%d n_o=%d order=%d: max impl error %.3g x scale, nroy %.3f'
          % (pu, S, O.size, order, worst, out['nroy_fraction']))


def test_scalar_model_matches_oracle(cuda):
    from gladsgp_b200 import history
    model = _scalar_model()
    samples = synthetic.posterior_samples(5, 2, 1, seed=4)
    em = _emulator(model, samples)
    O = np.array([0])
    y = _mean_field(model, em, O, [0.3])
    tt = np.linspace(0.0, 1.0, 301)[:, None]
    out = history.history_match(model, samples, y, _native(model, tt), obs_sd=0.01, disc_sd=0.02)
    K_O, r, c = _obs_terms(model, samples, O, y, 0.01, 0.02)
    ref = ho.history_match(em, tt, K_O, r, c, 1, 3.0)
    _check(out, ref, 3.0)
    assert out['nroy'][90] and 0.0 < out['nroy_fraction'] < 1.0


def test_kernel_edge_rules_and_slabs(cuda):
    """ops.hm_impl on given moments: V = 0 (0 for e = 0, +inf otherwise), NaN moments counted as +inf, exact ties, and
    output counts that split into many slabs, against the feature route on the same moments."""
    import torch
    from gladsgp_b200 import ops
    rng = np.random.default_rng(7)
    for S, pu, N, n_o, order in ((3, 4, 5, 5000, 8), (2, 1, 70, 1, 1), (1, 7, 40000, 130, 4), (4, 32, 65, 700, 3)):
        mu = rng.standard_normal((S, pu, N))
        var = rng.uniform(-1e-3, 0.3, (S, pu, N))
        K_O = rng.standard_normal((pu, n_o)) * 0.4
        r = rng.standard_normal(n_o) * 3.0
        c = rng.uniform(0.05, 0.3, n_o)
        if n_o >= 130:
            c[:2] = 0.0
            K_O[:, :2] = 0.0                                 # V = 0 at outputs 0 and 1
            r[0] = 0.0                                       # ... with e = 0 at output 0
            K_O[:, 5], r[5], c[5] = K_O[:, 4], r[4], c[4]    # a tie
        mu[:, 0, 3 % N] = np.nan                             # every output of point 3 is NaN
        def dev(a):
            return torch.as_tensor(np.ascontiguousarray(a), device='cuda')
        impl, nover = ops.hm_impl(dev(mu.reshape(S * pu, N)), dev(var.reshape(S * pu, N)), dev(K_O), dev(r), dev(c),
                                  order, 2.0)
        impl, nover = impl.cpu().numpy(), nover.cpu().numpy()
        e, V = ho.route_features(mu, var, K_O, r, c)
        I = ho.implausibility(e, V)
        if n_o >= 130:
            I[:, 0] = np.where(np.isnan(mu[:, 0, :]).any(0), np.inf, 0.0)   # the device's rule for V = 0, e = 0
        ref = ho.reduce(I, order, 2.0)
        sc = ho.scale(mu, var, K_O, r, c)
        assert np.all(np.isinf(impl[3 % N])) and nover[3 % N] == n_o
        ok = np.isfinite(ref['impl'])
        np.testing.assert_array_equal(np.isfinite(impl), ok)
        assert np.all(np.abs(impl - ref['impl'])[ok] <= (1e-12 * ref['impl'] + 1e-13 * sc[:, None])[ok])
        far = ref['edge'] > 1e-12 * (2.0 + sc)
        np.testing.assert_array_equal(nover[far], ref['n_over'][far])


def _mid_problem():
    model = _model(m=100, q=3, pu=5, seed=8, n_x=20, n_t=15)
    samples = synthetic.posterior_samples(6, 4, 5, seed=4)
    em = _emulator(model, samples)
    rng = np.random.default_rng(11)
    O = np.sort(rng.choice(model.num.n_y, size=120, replace=False))
    y = _mean_field(model, em, O, [0.3, 0.6, 0.5])
    t = _native(model, rng.uniform(0, 1, (1500, 3)))
    return model, samples, O, y, t


def _same(a, b):
    np.testing.assert_array_equal(a['impl'], b['impl'])
    np.testing.assert_array_equal(a['n_over'], b['n_over'])
    np.testing.assert_array_equal(a['nroy'], b['nroy'])


def test_identical_calls_chunks_and_permutations_give_identical_bits(cuda, monkeypatch):
    from gladsgp_b200 import history
    model, samples, O, y, t = _mid_problem()
    kw = dict(obs_index=O, obs_sd=0.01, disc_sd=0.02, order=3)
    a = history.history_match(model, samples, y, t, **kw)
    model._pred_cache = None                                 # a fresh factorisation too
    _same(a, history.history_match(model, samples, y, t, **kw))
    perm = np.random.default_rng(2).permutation(t.shape[0])
    p = history.history_match(model, samples, y, t[perm], **kw)
    _same(dict(impl=a['impl'][perm], n_over=a['n_over'][perm], nroy=a['nroy'][perm]), p)
    for pts in (1, 97):                                      # chunks of 1 and of 97 points
        monkeypatch.setattr(history, 'POINT_CHUNK_BYTES', 16 * 6 * 5 * pts)
        _same(a, history.history_match(model, samples, y, t, **kw))


def test_known_input_is_not_ruled_out_and_waves(cuda):
    from gladsgp_b200 import design, history
    model, samples, O, y, t = _mid_problem()
    star = _native(model, np.array([[0.3, 0.6, 0.5]]))
    t = np.concatenate([star, t])
    out = history.history_match(model, samples, y, t, obs_index=O, obs_sd=0.01)
    assert out['nroy'][0] and out['impl'][0, 0] < 1e-6, out['impl'][0]
    fr = [history.history_match(model, samples, y, t, obs_index=O, obs_sd=0.01, cutoff=cut)['nroy_fraction']
          for cut in (1.0, 2.0, 3.0, 5.0, 10.0)]
    assert np.all(np.diff(fr) >= 0) and fr[0] < fr[-1], fr
    keep = t[out['nroy']]
    assert 4 <= keep.shape[0] < t.shape[0]
    wave = design.next_runs(model, samples, keep, 4)
    assert np.unique(wave['index']).size == 4
    np.testing.assert_array_equal(wave['t'], keep[wave['index']])
