"""GPU: the chain diagnostics (csrc/ggp_chain_diag.cu) against oracle/chain_diag_oracle.py -- R-hat to 1e-12 and ESS to
1e-10 relative, on inputs whose Geyer sign tests sit at least 1e-9 from a flip (the monotone comparisons are continuous in
rho and tie exactly on indicator series; see oracle.chain_diag_oracle.diagnose_all) -- and the
public routes: SepiaModel.mcmc_diagnostics, do_mcmc_chains(device=True) and ModelBatch.mcmc_diagnostics."""
import io
from contextlib import redirect_stdout

import numpy as np
import pytest

from helpers import make_problem, synthetic
from oracle import chain_diag_oracle as cdo

pytestmark = pytest.mark.gpu

MARGIN = 1e-9


def _dev(torch, x):
    return torch.as_tensor(np.ascontiguousarray(x), dtype=torch.float64, device='cuda')


def _sticky_ar1(rng, n, C, E, phi=0.8, stick=0.7):
    """AR(1) draws that repeat the previous value with probability `stick`, as Metropolis rejections do."""
    x = np.empty((n, C, E))
    x[0] = rng.standard_normal((C, E))
    for i in range(1, n):
        move = rng.random((C, E)) >= stick
        x[i] = np.where(move, phi * x[i - 1] + rng.standard_normal((C, E)), x[i - 1])
    return x


def _check(torch, x_dev, x_host):
    from gladsgp_b200 import ops
    r, eb, et, margin, _ = cdo.diagnose_all(x_host)
    assert margin >= MARGIN, margin
    dr, deb, det = (t.cpu().numpy() for t in ops.chain_diagnostics(x_dev))
    np.testing.assert_allclose(dr, r, rtol=1e-12, atol=0, equal_nan=True)
    np.testing.assert_allclose(deb, eb, rtol=1e-10, atol=0, equal_nan=True)
    np.testing.assert_allclose(det, et, rtol=1e-10, atol=0, equal_nan=True)
    return dr, deb, det


@pytest.mark.parametrize('C', [1, 2, 3, 8, 64])
@pytest.mark.parametrize('n', [4, 5, 7, 64, 1001])
def test_matches_oracle_over_chains_and_draws(cuda, C, n):
    rng = np.random.default_rng(1000 * C + n)
    x = np.concatenate([rng.standard_normal((n, C, 1)),
                        _sticky_ar1(rng, n, C, 1),
                        np.round(_sticky_ar1(rng, n, C, 1) * 2) / 2,                 # quantised: heavy ties
                        rng.standard_normal((n, C, 1)) + np.arange(C)[None, :, None] * 0.5],
                       axis=2)
    _check(cuda, _dev(cuda, x), x)


def test_ties_signed_zeros_constant_and_non_finite_elements(cuda):
    rng = np.random.default_rng(3)
    n, C = 200, 4
    x = _sticky_ar1(rng, n, C, 8, stick=0.9)
    x[:, :, 1] = np.round(x[:, :, 1])                                               # a handful of distinct values
    x[:, :, 2] = np.where(rng.random((n, C)) < 0.5, -0.0, 0.0) + (rng.random((n, C)) < 0.3)   # +-0.0 mixture
    x[:, :, 3] = 1.25                                                                # constant
    x[:, :, 4] = 0.0
    x[::2, :, 4] = -0.0                                                              # constant up to the sign of zero
    x[17, 2, 5] = np.nan
    x[0, 0, 6] = -np.inf
    dr, deb, det = _check(cuda, _dev(cuda, x), x)
    assert np.isnan(dr[3]) and deb[3] == det[3] == 2 * C * (n // 2)
    assert np.isnan(dr[4]) and deb[4] == 2 * C * (n // 2)
    assert all(np.isnan(v[k]) for v in (dr, deb, det) for k in (5, 6))


def test_layouts(cuda):
    torch = cuda
    rng = np.random.default_rng(5)
    n, C, P = 301, 6, 9
    x = _sticky_ar1(rng, n, C, P)
    _check(torch, _dev(torch, x), x)                                                # (n, C, P)
    xt = _dev(torch, np.ascontiguousarray(x.transpose(2, 1, 0))).permute(2, 1, 0)   # element-major storage
    assert xt.stride() == (1, n, n * C)
    _check(torch, xt, x)
    big = _dev(torch, _sticky_ar1(rng, n, 2 * C, 3 * P))
    view = big[:, ::2, 1::3]                                                        # strided view
    _check(torch, view, view.cpu().numpy())
    models = _dev(torch, x.reshape(n, 1, C * P))                                   # one chain per element
    _check(torch, models, x.reshape(n, 1, C * P))


def test_long_geyer_sequences(cuda):
    torch = cuda
    rng = np.random.default_rng(7)
    C, n, phi = 2, 20000, 0.999
    e = rng.standard_normal((C, n))
    a = np.empty((C, n))
    a[:, 0] = e[:, 0] * 20
    for i in range(1, n):
        a[:, i] = phi * a[:, i - 1] + e[:, i]
    info = {}
    cdo.ess_raw(cdo.z_scale(cdo.split_chains(a)), info=info)
    assert info['max_t'] > 2 * 256                                                  # past two lag blocks
    x = a.T[:, :, None]
    _check(torch, _dev(torch, x), x)
    w = np.cumsum(np.random.default_rng(1).standard_normal((1, 64)), axis=1)       # random walk: runs to h - 3
    cdo.ess_raw(cdo.z_scale(cdo.split_chains(w)), info=info)
    assert info['max_t'] >= 32 - 5
    _check(torch, _dev(torch, w.T[:, :, None]), w.T[:, :, None])


def _build(pr, q):
    from sepia.SepiaData import SepiaData
    from sepia.SepiaModel import SepiaModel
    d = SepiaData(t_sim=pr['t'], y_sim=pr['y'], y_ind_sim=np.linspace(0, 1, pr['y'].shape[1]))
    d.transform_xt(t_notrans=np.arange(q))
    d.standardize_y(y_mean=pr['mu'], y_sd=pr['sd'])
    d.create_K_basis(K=pr['K'])
    return SepiaModel(d)


def _flat(model, res):
    """{name: dict} of mcmc_diagnostics -> three flat arrays in the sampler's element order (logPost last)."""
    blocks = model._blocks()[0]
    return [np.concatenate([np.asarray(res[b.name][k]).reshape(-1, order='F') for b in blocks] +
                           [np.atleast_1d(res['logPost'][k])]) for k in ('rhat', 'ess_bulk', 'ess_tail')]


def test_real_sampler_draws_and_device_draws(cuda):
    torch = cuda
    model = _build(make_problem(m=64, q=3, pu=2), 3)
    d_host, l_host = model.do_mcmc_chains(300, 16, seed=3)
    d_dev, l_dev = model.do_mcmc_chains(300, 16, seed=3, device=True)
    assert torch.is_tensor(d_dev) and d_dev.is_cuda and torch.is_tensor(l_dev) and l_dev.is_cuda
    assert np.array_equal(d_dev.cpu().numpy(), d_host) and np.array_equal(l_dev.cpu().numpy(), l_host)
    res = model.mcmc_diagnostics(d_dev, l_dev, nburn=50)
    assert res['betaU']['rhat'].shape == model.params.betaU.val_shape
    x = np.concatenate([d_host, l_host[:, :, None]], axis=2)[50:]
    r, eb, et, margin, _ = cdo.diagnose_all(x)
    assert margin >= MARGIN, margin
    got = _flat(model, res)
    np.testing.assert_allclose(got[0], r, rtol=1e-12, atol=0, equal_nan=True)
    np.testing.assert_allclose(got[1], eb, rtol=1e-10, atol=0)
    np.testing.assert_allclose(got[2], et, rtol=1e-10, atol=0)
    for k, v in zip(('rhat', 'ess_bulk', 'ess_tail'), _flat(model, model.mcmc_diagnostics(d_host, l_host, nburn=50))):
        assert np.array_equal(v, got[('rhat', 'ess_bulk', 'ess_tail').index(k)], equal_nan=True)
    # the recorded chain: one chain split in two
    model.do_mcmc(120, prog=False, seed=4)
    own = model.mcmc_diagnostics()
    s = model.get_samples()
    xs = np.concatenate([s['betaU'], s['lamUz'], s['lamWs'], s['lamWOs'], s['logPost']], axis=1)[:, None, :]
    r, eb, et, margin, _ = cdo.diagnose_all(xs)
    assert margin >= MARGIN, margin
    got = _flat(model, own)
    np.testing.assert_allclose(got[0], r, rtol=1e-12, atol=0, equal_nan=True)
    np.testing.assert_allclose(got[1], eb, rtol=1e-10, atol=0)
    np.testing.assert_allclose(got[2], et, rtol=1e-10, atol=0)


def test_full_scale_subset_against_oracle(cuda):
    torch = cuda
    from gladsgp_b200 import ops
    rng = np.random.default_rng(11)
    n, C, E = 1000, 944, 112
    x = _sticky_ar1(rng, n, C, E)
    xd = _dev(torch, x)
    dr, deb, det = (t.cpu().numpy() for t in ops.chain_diagnostics(xd))
    assert np.all(np.isfinite(dr)) and np.all(np.isfinite(deb)) and np.all(np.isfinite(det))
    pick = np.sort(np.random.default_rng(12).choice(E, 8, replace=False))
    r, eb, et, margin, _ = cdo.diagnose_all(x[:, :, pick])
    assert margin >= MARGIN, margin
    np.testing.assert_allclose(dr[pick], r, rtol=1e-12, atol=0)
    np.testing.assert_allclose(deb[pick], eb, rtol=1e-10, atol=0)
    np.testing.assert_allclose(det[pick], et, rtol=1e-10, atol=0)


def test_deterministic_and_independent_of_chunking(cuda, monkeypatch):
    torch = cuda
    from gladsgp_b200 import ops
    rng = np.random.default_rng(13)
    x = _dev(torch, _sticky_ar1(rng, 3000, 5, 17))
    a = [t.cpu().numpy() for t in ops.chain_diagnostics(x)]
    b = [t.cpu().numpy() for t in ops.chain_diagnostics(x)]
    per = ops._lib.load().ggp_chain_diag_workspace_bytes(3000, 5, 1)
    monkeypatch.setattr(ops, 'CHAIN_DIAG_WS_BYTES', 3 * per + 1)                    # 6 launches of at most 3 elements
    c = [t.cpu().numpy() for t in ops.chain_diagnostics(x)]
    for u, v, w in zip(a, b, c):
        assert np.array_equal(u, v, equal_nan=True) and np.array_equal(u, w, equal_nan=True)


def test_model_batch_equals_each_model(cuda):
    from sepia.SepiaData import SepiaData
    from sepia.SepiaModel import SepiaModel
    from gladsgp_b200.batch import ModelBatch
    rng = np.random.default_rng(4)
    m, q = 48, 3
    t = synthetic.design(m, q, seed=9)
    ys = [np.sin(3 * t[:, 0]) + 0.1 * rng.standard_normal(m), t[:, 1] ** 2 - t[:, 2] + 0.05 * rng.standard_normal(m),
          np.cos(2 * t[:, 2]) * t[:, 0] + 0.2 * rng.standard_normal(m)]

    def make(y):
        d = SepiaData(t_sim=t, y_sim=y.astype(np.float32))
        d.transform_xt()
        d.standardize_y()
        return SepiaModel(d)
    models = [make(y) for y in ys]
    batch = ModelBatch(models, seeds=[1, 2, 3])
    with redirect_stdout(io.StringIO()):
        batch.tune_step_sizes(4, 3)
    batch.do_mcmc(512)
    together = batch.mcmc_diagnostics(nburn=12)
    for mm, res in zip(models, together):
        own = mm.mcmc_diagnostics(nburn=12)
        assert set(own) == set(res) == {'betaU', 'lamUz', 'lamWs', 'lamWOs', 'logPost'}
        for name in own:
            for k in ('rhat', 'ess_bulk', 'ess_tail'):
                assert np.array_equal(np.asarray(own[name][k]), np.asarray(res[name][k]), equal_nan=True), (name, k)
