"""CPU: betaU elements of constant input columns are marked likelihood-neutral in the sampler's fixed table, and the
oracle's log-likelihood under such a proposal is bit for bit the current one (the rule the device applies there)."""
import numpy as np

from helpers import so, make_problem
from gladsgp_b200.ops import mark_neutral_sites, FIXED_NEUTRAL


def _model(pr, x_sim=None, q=3):
    from sepia.SepiaData import SepiaData
    from sepia.SepiaModel import SepiaModel
    d = SepiaData(x_sim=x_sim, t_sim=pr['t'], y_sim=pr['y'], y_ind_sim=np.linspace(0, 1, pr['y'].shape[1]))
    d.transform_xt(t_notrans=np.arange(q))
    d.standardize_y(y_mean=pr['mu'], y_sd=pr['sd'])
    d.create_K_basis(K=pr['K'])
    return SepiaModel(d)


def _marked(model):
    tb = model._tables()
    fx = mark_neutral_sites(model.num.zt, tb['fixed'], model.num.pu)
    return tb, fx


def test_dummy_x_marks_first_input_of_every_pc():
    pr = make_problem(m=40, q=3, pu=2)
    model = _model(pr)
    tb, fx = _marked(model)
    d, pu = model.num.zt.shape[1], model.num.pu
    want = np.zeros_like(tb['fixed'])
    want[[j * d for j in range(pu)]] = FIXED_NEUTRAL
    np.testing.assert_array_equal(fx, want)
    assert np.all(tb['fixed'] == 0)                     # the model's own table is not changed


def test_constant_real_column_is_marked_and_varying_x_is_not():
    pr = make_problem(m=40, q=3, pu=2)
    m = pr['t'].shape[0]
    x = np.stack([np.linspace(0.0, 1.0, m), np.full(m, 7.25)], axis=1)     # column 1 constant
    model = _model(pr, x_sim=x)
    _, fx = _marked(model)
    d, pu = model.num.zt.shape[1], model.num.pu
    assert d == 5
    want = np.zeros(fx.size, dtype=np.uint8)
    want[[j * d + 1 for j in range(pu)]] = FIXED_NEUTRAL
    np.testing.assert_array_equal(fx, want)
    model2 = _model(pr, x_sim=x[:, :1])
    _, fx2 = _marked(model2)
    assert not np.any(fx2 == FIXED_NEUTRAL)


def test_only_sampled_betau_elements_are_marked():
    X = np.concatenate([np.full((6, 1), 0.5), np.linspace(0, 1, 6)[:, None], np.full((6, 1), np.inf)], axis=1)
    pu = 2
    P = 3 * pu + 2 * pu + 1
    fixed = np.zeros(P, dtype=np.uint8)
    fixed[3] = 1                                        # betaU[0, 1] fixed: stays fixed
    fx = mark_neutral_sites(X, fixed, pu)
    want = np.zeros(P, dtype=np.uint8)
    want[0] = FIXED_NEUTRAL
    want[3] = 1                                         # a constant but infinite column is not neutral
    np.testing.assert_array_equal(fx, want)
    fixed[:3 * pu] = 2                                  # betaU outside mcmcList
    np.testing.assert_array_equal(mark_neutral_sites(X, fixed, pu), fixed)


def test_oracle_loglik_unchanged_at_neutral_sites():
    pr = make_problem(m=48, q=3, pu=3)
    num = pr['num']
    assert np.all(num.zt[:, 0] == num.zt[0, 0])
    mod = so.OracleModel(num)
    rng = np.random.default_rng(2)
    mod.betaU.val[:] = rng.uniform(0.05, 2.0, size=mod.betaU.val.shape)
    mod.log_lik()
    for j in range(num.pu):
        ll_old = mod.SigWl[j]
        for cand in (1e-3, 0.37, 5.0, 80.0):
            mod.betaU.val[0, j] = cand
            mod.log_lik('betaU', j * num.d)
            assert mod.SigWl[j].tobytes() == ll_old.tobytes()
        mod.betaU.val[1, j] *= 1.5                      # a varying column does change the term
        mod.log_lik('betaU', j * num.d + 1)
        assert mod.SigWl[j] != ll_old
