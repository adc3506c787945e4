"""GPU: every code path of the covariance distance product against FP64 references built from coordinate differences.

The kernels form squared distances as a rank-(d+2) product on the FP64 tensor cores in cov_ksteps(d) = (d + 5) >> 2
DMMA steps: register-resident forms for 1-5 steps (d <= 18) and a runtime loop for d >= 19.  The dimensions below reach
every step count, with d + 2 both a multiple of 4 and not, the last specialised d (18), the first generic one (19) and
the sampler's limit (64).  DESIGN.md section 4 bounds the product form: a covariance entry is within
8 eps (1 + |x~_i|^2 + |x~_j|^2) of its value relative, x~ = sqrt(beta) o x."""
import numpy as np
import pytest
import scipy.linalg

from helpers import so, make_problem, tables_from_oracle, replay_from_trace

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps
DIMS = [2, 3, 6, 10, 11, 14, 18, 19, 22, 33, 64]
LL_RTOL = 1e-8
PRED_RTOL = 1e-6


def _hypers(d, B, seed):
    """Length scales that keep the correlations of unit-cube inputs away from 0 and 1 at every d."""
    rng = np.random.default_rng(seed)
    beta = rng.uniform(0.05, 3.0, size=(B, d)) * min(1.0, 8.0 / d)
    lamz = rng.uniform(0.5, 2.0, size=B)
    dadd = rng.uniform(1e-3, 1e-2, size=B)
    return beta, lamz, dadd


def _sqdist(A, Bm, beta):
    """sum_k beta_k (a_k - b_k)^2 from coordinate differences, (len(A), len(Bm))."""
    D = np.zeros((A.shape[0], Bm.shape[0]))
    for k in range(A.shape[1]):
        D += beta[k] * (A[:, None, k] - Bm[None, :, k]) ** 2
    return D


def _product_form_bound(A, Bm, beta, Cref):
    na = (A ** 2) @ beta
    nb = (Bm ** 2) @ beta
    return 8 * EPS * (1.0 + na[:, None] + nb[None, :]) * np.abs(Cref)


def _dense_cov(X, beta, lamz, dadd):
    C = np.exp(-_sqdist(X, X, beta)) / lamz
    np.fill_diagonal(C, 1.0 / lamz + dadd)
    return C


@pytest.mark.parametrize('m', [128, 100])           # whole 64-row blocks: row-block kernel; otherwise the tile kernel
@pytest.mark.parametrize('d', DIMS)
def test_cov_build_and_cross_cov_every_distance_path(cuda, d, m):
    from gladsgp_b200 import ops
    rng = np.random.default_rng(1000 * d + m)
    X = rng.uniform(0, 1, size=(m, d))
    Xp = rng.uniform(0, 1, size=(37, d))
    B = 2
    beta, lamz, dadd = _hypers(d, B, seed=d)
    Cg = ops.cov_build(X, beta, lamz, dadd).cpu().numpy()
    Sg = ops.cross_cov(X, Xp, beta, lamz).cpu().numpy()
    for b in range(B):
        C = _dense_cov(X, beta[b], lamz[b], dadd[b])
        err = np.abs(Cg[b] - C)
        bound = _product_form_bound(X, X, beta[b], C)
        assert np.all(err <= bound), (b, np.max(err / bound))
        S = np.exp(-_sqdist(X, Xp, beta[b])) / lamz[b]
        err = np.abs(Sg[b] - S)
        bound = _product_form_bound(X, Xp, beta[b], S)
        assert np.all(err <= bound), (b, np.max(err / bound))


@pytest.mark.parametrize('d', DIMS)
def test_loglik_every_distance_path_in_every_schedule(cuda, monkeypatch, d):
    """m = 257 (ragged last panel): log-likelihood against SciPy, u and the factor against the dense solve, and the
    look-ahead, plain and cluster schedules bit for bit."""
    from gladsgp_b200 import ops, _lib
    h = _lib.load()
    m, B = 257, 2
    rng = np.random.default_rng(d)
    X = rng.uniform(0, 1, size=(m, d))
    W = rng.standard_normal((B, m))
    beta, lamz, dadd = _hypers(d, B, seed=d + 1)
    res = {}
    old = h.ggp_set_lookahead(1)
    try:
        for key, g, la in (('la', '1', 1), ('plain', '1', 0), ('cluster', '4', 0)):
            monkeypatch.setenv('GGP_CLUSTER', g)
            h.ggp_set_lookahead(la)
            out = ops.loglik_batched(X, W, beta, lamz, dadd, want_factor=True, want_u=True)
            assert np.all(out['info'].cpu().numpy() == 0), key
            res[key] = (out['loglik'].cpu().numpy(), ops.factor_unpack(out['factor'], m).cpu().numpy(),
                        out['u'].cpu().numpy())
    finally:
        h.ggp_set_lookahead(old)
    for key in ('plain', 'cluster'):
        for a, b in zip(res['la'], res[key]):
            assert np.array_equal(a, b), key
    ll, Lg, ug = res['la']
    for b in range(B):
        L = scipy.linalg.cholesky(_dense_cov(X, beta[b], lamz[b], dadd[b]), lower=True)
        u = scipy.linalg.solve_triangular(L, W[b], lower=True)
        ref = -np.sum(np.log(np.diag(L))) - 0.5 * u @ u
        assert abs(ll[b] - ref) <= LL_RTOL * abs(ref), (b, ll[b], ref)
        np.testing.assert_allclose(Lg[b], L, rtol=0, atol=1e-9 * np.abs(L).max())
        np.testing.assert_allclose(ug[b, :m], u, rtol=0, atol=1e-8 * np.abs(u).max())


@pytest.mark.parametrize('d', DIMS)
def test_predict_every_distance_path(cuda, d):
    """Predictor.predict (n = 37, with V) and pred_cov against S21^T S22^-1 w and S11 - S21^T S22^-1 S21."""
    from gladsgp_b200 import ops
    m, n, B = 100, 37, 2
    rng = np.random.default_rng(500 + d)
    X = rng.uniform(0, 1, size=(m, d))
    Xp = rng.uniform(0, 1, size=(n, d))
    W = rng.standard_normal((B, m))
    beta, lamz, dadd = _hypers(d, B, seed=d + 2)
    lamws = rng.uniform(300, 3000, size=B)
    s11 = 1.0 / lamz + 1.0 / lamws
    P = ops.Predictor(X, W, beta, lamz, dadd, s11)
    assert not P.info.any().item()
    mean, var, V = P.predict(Xp, want_V=True)
    Sg = P.pred_cov(Xp, V).cpu().numpy()
    mean, var = mean.cpu().numpy(), var.cpu().numpy()
    for b in range(B):
        cf = scipy.linalg.cho_factor(_dense_cov(X, beta[b], lamz[b], dadd[b]), lower=True)
        S21 = np.exp(-_sqdist(X, Xp, beta[b])) / lamz[b]
        S11 = np.exp(-_sqdist(Xp, Xp, beta[b])) / lamz[b]
        np.fill_diagonal(S11, s11[b])
        mu = S21.T @ scipy.linalg.cho_solve(cf, W[b])
        Sig = S11 - S21.T @ scipy.linalg.cho_solve(cf, S21)
        np.testing.assert_allclose(mean[b], mu, rtol=PRED_RTOL, atol=PRED_RTOL * np.abs(mu).max())
        np.testing.assert_allclose(var[b], np.diag(Sig), rtol=PRED_RTOL)
        np.testing.assert_allclose(Sg[b], Sig, rtol=PRED_RTOL, atol=PRED_RTOL * np.abs(Sig).max())


def _oracle_chain(d, n_steps):
    pr = make_problem(m=64, q=d - 1, pu=2)
    num = pr['num']
    assert num.d == d
    mod = so.OracleModel(num)
    tb = tables_from_oracle(mod)
    P = tb['theta'].size
    mod.trace = []
    mod.do_mcmc(n_steps, rng=np.random.RandomState(d))
    replay, acc = replay_from_trace(mod.trace, n_steps, P)
    ref = mod.get_samples()
    draws = np.concatenate([ref['betaU'], ref['lamUz'], ref['lamWs'], ref['lamWOs']], axis=1)
    return num, tb, replay, acc, draws, ref['logPost'][:, 0]


@pytest.mark.parametrize('chains,spec', [(1, None), (1, '0'), (3, None), (160, None)])
@pytest.mark.parametrize('d', [13, 19, 64])
def test_sampler_replay_every_distance_path(cuda, monkeypatch, d, chains, spec):
    """5 replayed oracle steps: one chain (cluster / speculative step kernels, and GGP_SPEC=0), 3 chains (cluster step
    kernel), 160 chains (one CTA per matrix, look-ahead step kernel); d = 64 fills beta_sm[64] of the step kernels."""
    from gladsgp_b200 import ops
    if spec is not None:
        monkeypatch.setenv('GGP_SPEC', spec)
    n_steps = 5
    num, tb, replay, acc_ref, draws_ref, lp_ref = _oracle_chain(d, n_steps)
    rep = {k: np.repeat(v, chains, axis=1) for k, v in replay.items()}
    eng = ops.McmcEngine(num.zt, num.w.T.copy(), num.LamSim, tb, n_chains=chains)
    eng.set_state(tb['theta'])
    out = eng.run(n_steps, tb['step'], replay=rep, record_accept=True)
    acc = out['accepted'].cpu().numpy()
    draws = out['draws'].cpu().numpy()
    lp = out['lp'].cpu().numpy()
    for c in range(chains):
        assert np.array_equal(acc[:, c:c + 1], acc_ref), c
        assert np.array_equal(draws[:, c], draws_ref), c
        np.testing.assert_allclose(lp[:, c], lp_ref, rtol=1e-9)
    if chains == 1:
        # the same chain with its PCs swept by two shards, one after the other
        eng.set_state(tb['theta'])
        out = eng.run_by_pc(n_steps, tb['step'], replay=replay, record_accept=True, shards=[(0, 1), (1, 1)])
        assert np.array_equal(out['accepted'].cpu().numpy(), acc_ref)
        assert np.array_equal(out['draws'].cpu().numpy()[:, 0], draws_ref)


def test_sampler_rejects_d_above_64(cuda):
    """d = 65 overflows the step kernels' per-block parameter arrays: the argument check refuses it before any launch,
    for the whole-step entry point and for the PC-shard entry points."""
    import torch
    from gladsgp_b200 import ops, _lib
    pr = make_problem(m=64, q=64, pu=2)
    num = pr['num']
    assert num.d == 65
    tb = tables_from_oracle(so.OracleModel(num))
    eng = ops.McmcEngine(num.zt, num.w.T.copy(), num.LamSim, tb, n_chains=1)
    eng.set_state(tb['theta'])
    ws0 = eng.ws.clone()
    theta0 = eng.theta.clone()
    us = np.random.default_rng(0).random((1, 2 * tb['theta'].size * 2))
    with pytest.raises(_lib.GgpError, match='d must be <= 64'):
        eng.run(2, tb['step'], uniforms=us)
    with pytest.raises(_lib.GgpError, match='d must be <= 64'):
        eng.run_by_pc(2, tb['step'], uniforms=us, shards=[(0, 1), (1, 1)])
    torch.cuda.synchronize()
    assert torch.equal(eng.theta, theta0) and torch.equal(eng.ws, ws0)
