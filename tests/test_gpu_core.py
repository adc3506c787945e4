"""GPU parity: covariance build, fused log-likelihood, MCMC replay vs the CPU oracle (through the C ABI)."""
import numpy as np
import pytest

from helpers import so, make_problem, make_scalar_problem, random_hypers, tables_from_oracle, replay_from_trace

pytestmark = pytest.mark.gpu

LL_RTOL = 1e-8        # north_star: log-likelihoods within 1e-8 relative in FP64


def _oracle_ll(num, beta, lamz, lamws, lamwos, j):
    C = so.block_cov(num, beta, lamz, lamws, lamwos, j)
    return C, so.do_loglik(C, num.wv[j * num.m:(j + 1) * num.m, 0])


@pytest.mark.parametrize('m,q,pu', [(33, 2, 1), (64, 3, 2), (100, 8, 5), (257, 4, 2), (512, 8, 3)])
def test_cov_and_loglik_match_oracle(cuda, m, q, pu):
    from gladsgp_b200 import ops
    pr = make_problem(m=m, q=q, pu=pu)
    num = pr['num']
    B = 2 * pu
    beta, lamz, lamws, lamwos = random_hypers(num, B, seed=m)
    js = np.arange(B) % pu
    dadd = 1.0 / (num.LamSim[js] * lamwos) + 1.0 / lamws
    W = np.stack([num.wv[j * m:(j + 1) * m, 0] for j in js])
    Cg = ops.cov_build(num.zt, beta, lamz, dadd).cpu().numpy()
    out = ops.loglik_batched(num.zt, W, beta, lamz, dadd, want_factor=True, want_u=True)
    ll = out['loglik'].cpu().numpy()
    Lg = ops.factor_unpack(out['factor'], m).cpu().numpy()
    ug = out['u'].cpu().numpy()[:, :m]
    assert np.all(out['info'].cpu().numpy() == 0)
    for b in range(B):
        C, ref = _oracle_ll(num, beta[b], lamz[b], lamws[b], lamwos[b], js[b])
        np.testing.assert_allclose(Cg[b], C, rtol=1e-13, atol=1e-300)
        assert abs(ll[b] - ref) <= LL_RTOL * abs(ref), (b, ll[b], ref)
        L = np.linalg.cholesky(C)
        np.testing.assert_allclose(Lg[b], L, rtol=0, atol=1e-9 * np.abs(L).max())
        u = np.linalg.solve(L, W[b])
        np.testing.assert_allclose(ug[b], u, rtol=0, atol=1e-8 * np.abs(u).max())


def test_loglik_scalar_1d_m1000(cuda):
    """cfg 2 shape: m=1000, d=2, pu=1 (multi-pass panels)."""
    from gladsgp_b200 import ops
    pr = make_scalar_problem(m=1000)
    num = pr['num']
    beta = np.array([[0.1, 30.0], [0.5, 80.0]]); lamz = np.array([0.8, 1.3])
    dadd = 1.0 / (1.0 * np.array([150.0, 90.0])) + 1.0 / np.array([800.0, 2000.0])
    W = np.stack([num.wv[:, 0]] * 2)
    ll = ops.loglik_batched(num.zt, W, beta, lamz, dadd)['loglik'].cpu().numpy()
    for b in range(2):
        C = so.cov_self(num, beta[b], lamz[b]); np.fill_diagonal(C, C.diagonal() + dadd[b])
        ref = so.do_loglik(C, num.wv[:, 0])
        assert abs(ll[b] - ref) <= LL_RTOL * abs(ref), (ll[b], ref)


def test_loglik_not_positive_definite_is_minus_inf(cuda):
    from gladsgp_b200 import ops
    pr = make_problem(m=64, q=3, pu=2)
    num = pr['num']
    beta = np.full((1, num.d), 1e-6); lamz = np.array([1.0]); dadd = np.array([-0.999999])
    out = ops.loglik_batched(num.zt, num.wv[:64, 0][None, :], beta, lamz, dadd)
    assert out['loglik'].cpu().numpy()[0] == -np.inf
    assert out['info'].cpu().numpy()[0] > 0


def test_cross_cov_matches_oracle(cuda):
    from gladsgp_b200 import ops
    pr = make_problem(m=100, q=8, pu=2)
    num = pr['num']
    rng = np.random.default_rng(1)
    xp = np.concatenate([0.5 * np.ones((37, 1)), rng.uniform(size=(37, 8))], axis=1)
    beta, lamz, _, _ = random_hypers(num, 3, seed=9)
    S = ops.cross_cov(num.zt, xp, beta, lamz).cpu().numpy()
    for b in range(3):
        np.testing.assert_allclose(S[b], so.cov_cross(num.zt, xp, beta[b], lamz[b]), rtol=1e-13)


@pytest.mark.parametrize('override', [False, True])
def test_mcmc_replay_matches_oracle_chain(cuda, override):
    """Chains identical given the same proposals and uniforms (north_star)."""
    from gladsgp_b200 import ops
    pr = make_problem(m=64, q=3, pu=2)
    num = pr['num']
    mod = so.OracleModel(num)
    if override:
        mod.override_lamWOs(50.0)
    tb = tables_from_oracle(mod)
    P = tb['theta'].size
    n_steps = 12
    rng = np.random.RandomState(11)
    mod.trace = []
    mod.do_mcmc(n_steps, rng=rng)
    replay, acc_ref = replay_from_trace(mod.trace, n_steps, P)
    ref = mod.get_samples()
    ref_draws = np.concatenate([ref['betaU'], ref['lamUz'], ref['lamWs'], ref['lamWOs']], axis=1)
    eng = ops.McmcEngine(num.zt, num.w.T.copy(), num.LamSim, tb, n_chains=1)
    eng.set_state(tb['theta'])
    out = eng.run(n_steps, tb['step'], replay=replay, record_accept=True)
    acc = out['accepted'].cpu().numpy()
    draws = out['draws'].cpu().numpy()[:, 0, :]
    lp = out['lp'].cpu().numpy()[:, 0]
    assert np.array_equal(acc, acc_ref)
    assert np.array_equal(draws, ref_draws)            # bit-identical chain under replay
    np.testing.assert_allclose(lp, ref['logPost'][:, 0], rtol=1e-9)


def test_mcmc_uniform_stream_matches_oracle(cuda):
    """Device-side proposal generation from the same U[0,1) stream as np.random."""
    from gladsgp_b200 import ops
    pr = make_problem(m=64, q=3, pu=2)
    num = pr['num']
    mod = so.OracleModel(num)
    tb = tables_from_oracle(mod)
    P = tb['theta'].size
    n_steps = 10
    rs = np.random.RandomState(123)
    stream = rs.random_sample(2 * P * n_steps)
    rs = np.random.RandomState(123)
    mod.trace = []
    mod.do_mcmc(n_steps, rng=rs)
    used = sum(1 + int(tr['valid']) for tr in mod.trace)
    ref = mod.get_samples()
    ref_draws = np.concatenate([ref['betaU'], ref['lamUz'], ref['lamWs'], ref['lamWOs']], axis=1)
    eng = ops.McmcEngine(num.zt, num.w.T.copy(), num.LamSim, tb, n_chains=1)
    eng.set_state(tb['theta'])
    out = eng.run(n_steps, tb['step'], uniforms=stream[None, :], record_accept=True)
    assert int(out['consumed'].cpu().numpy()[0]) == used
    acc_ref = np.array([tr['accept'] for tr in mod.trace], dtype=np.uint8).reshape(n_steps, 1, P)
    assert np.array_equal(out['accepted'].cpu().numpy(), acc_ref)
    np.testing.assert_allclose(out['draws'].cpu().numpy()[:, 0, :], ref_draws, rtol=1e-12)


def test_in_kernel_exponential_accuracy(cuda):
    """The fused kernels use their own exp for y <= 0 (64-entry table + degree-5 polynomial): ~1 ulp."""
    import torch
    from gladsgp_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(0)
    y = -np.concatenate([rng.uniform(0, 1e-3, 20000), rng.uniform(0, 5, 50000), rng.uniform(5, 680, 30000), [0.0]])
    yd = torch.as_tensor(y, device='cuda'); out = torch.empty_like(yd)
    _lib.check(lib.ggp_debug_exp_neg_f64(_lib.ptr(yd), _lib.ptr(out), y.size, _lib.stream_ptr()))
    got = out.cpu().numpy()
    ref = np.exp(y)
    rel = np.abs(got - ref) / ref
    assert rel.max() < 4.5e-16, rel.max()
    assert got[-1] == 1.0


def test_loglik_large_m_many_inputs(cuda):
    """cfg 5 shape class (m in the thousands, d = 17): single-CTA path, multi-pass panels."""
    import scipy.linalg
    from gladsgp_b200 import ops, synthetic
    m, q = 1500, 16
    t = synthetic.design(m, q)
    X = np.concatenate([0.5 * np.ones((m, 1)), t.astype(np.float64)], axis=1)
    rng = np.random.default_rng(0)
    beta = np.exp(rng.uniform(np.log(0.05), np.log(1.0), size=(2, q + 1)))
    lamz = np.array([0.9, 1.4]); dadd = np.array([2e-3, 5e-3])
    W = rng.standard_normal((2, m))
    out = ops.loglik_batched(X, W, beta, lamz, dadd)
    ll = out['loglik'].cpu().numpy()
    for b in range(2):
        D = ((X[:, None, :] - X[None, :, :]) ** 2) @ beta[b]
        C = np.exp(-D) / lamz[b]
        np.fill_diagonal(C, 1 / lamz[b] + dadd[b])
        L = scipy.linalg.cholesky(C, lower=True)
        u = scipy.linalg.solve_triangular(L, W[b], lower=True)
        ref = -np.sum(np.log(np.diag(L))) - 0.5 * u @ u
        assert abs(ll[b] - ref) <= LL_RTOL * abs(ref)


def test_loglik_cfg5_size_against_scipy_and_across_schedules(cuda, monkeypatch):
    """BASELINE.json configs[4] at full size (m = 4096, d = 17): log-likelihood against SciPy's Cholesky at 1e-8, and the
    16-CTA cluster schedule (what one chain of 20 PCs runs) bit-identical to the one-CTA look-ahead schedule."""
    import scipy.linalg
    from gladsgp_b200 import ops, synthetic
    m, q = 4096, 16
    t = synthetic.design(m, q)
    X = np.concatenate([0.5 * np.ones((m, 1)), t.astype(np.float64)], axis=1)
    rng = np.random.default_rng(4)
    beta = np.exp(rng.uniform(np.log(0.05), np.log(1.0), size=(1, q + 1)))
    lamz = np.array([1.1]); dadd = np.array([3e-3])
    W = rng.standard_normal((1, m))
    D = np.zeros((m, m))
    for k in range(q + 1):
        D += beta[0, k] * (X[:, None, k] - X[None, :, k]) ** 2
    C = np.exp(-D) / lamz[0]
    np.fill_diagonal(C, 1 / lamz[0] + dadd[0])
    L = scipy.linalg.cholesky(C, lower=True)
    u = scipy.linalg.solve_triangular(L, W[0], lower=True)
    ref = -np.sum(np.log(np.diag(L))) - 0.5 * u @ u
    res = {}
    for key, g in (('cluster16', '16'), ('la', '1')):
        monkeypatch.setenv('GGP_CLUSTER', g)
        out = ops.loglik_batched(X, W, beta, lamz, dadd, want_u=True)
        res[key] = (out['loglik'].cpu().numpy(), out['u'].cpu().numpy())
        assert int(out['info'].cpu().numpy()[0]) == 0
    assert abs(res['cluster16'][0][0] - ref) <= LL_RTOL * abs(ref)
    np.testing.assert_allclose(res['cluster16'][1][0, :m], u, rtol=1e-7, atol=1e-9)
    for a, b in zip(res['cluster16'], res['la']):
        assert np.array_equal(a, b)


def test_cluster_and_single_cta_variants_agree_bitwise(cuda, monkeypatch):
    """Small batches run one matrix per thread-block cluster (up to 8 CTAs); the per-unit arithmetic is the same
    as in the one-CTA-per-matrix variant, so results must be bit-identical."""
    from gladsgp_b200 import ops
    pr = make_problem(m=257, q=4, pu=2)
    num = pr['num']
    beta, lamz, lamws, lamwos = random_hypers(num, 2, seed=5)
    dadd = 1.0 / (num.LamSim * lamwos) + 1.0 / lamws
    W = num.w.T.copy()
    res = {}
    for g in ('1', '2', '8'):
        monkeypatch.setenv('GGP_CLUSTER', g)
        out = ops.loglik_batched(num.zt, W, beta, lamz, dadd, want_factor=True, want_u=True)
        res[g] = (out['loglik'].cpu().numpy(), ops.factor_unpack(out['factor'], 257).cpu().numpy(), out['u'].cpu().numpy())
    for g in ('2', '8'):
        for a, b in zip(res['1'], res[g]):
            assert np.array_equal(a, b)
    # failure is reported consistently by every CTA of the cluster
    monkeypatch.setenv('GGP_CLUSTER', '8')
    bad = ops.loglik_batched(num.zt, W, np.full((2, num.d), 1e-6), np.ones(2), np.full(2, -0.999999))
    assert np.all(bad['loglik'].cpu().numpy() == -np.inf) and np.all(bad['info'].cpu().numpy() > 0)


@pytest.mark.parametrize('m,q,pu', [(32, 2, 1), (100, 8, 3), (257, 4, 2), (512, 8, 2), (1100, 16, 1), (2049, 12, 1)])
def test_lookahead_and_cluster_schedules_agree_bitwise(cuda, monkeypatch, m, q, pu):
    """The look-ahead schedule (diagonal block of panel j+1 factored while panel j is finished; dynamic pool of pairs)
    reorders work, not arithmetic: factor, u and log-likelihood equal the cluster variant's bit for bit."""
    from gladsgp_b200 import ops
    pr = make_problem(m=m, q=q, pu=pu)
    num = pr['num']
    beta, lamz, lamws, lamwos = random_hypers(num, pu, seed=11)
    dadd = 1.0 / (num.LamSim * lamwos) + 1.0 / lamws
    W = num.w.T.copy()
    res = {}
    infos = []
    for g in ('1', '4'):
        monkeypatch.setenv('GGP_CLUSTER', g)
        out = ops.loglik_batched(num.zt, W, beta, lamz, dadd, want_factor=True, want_u=True)
        res[g] = (out['loglik'].cpu().numpy(), ops.factor_unpack(out['factor'], m).cpu().numpy(), out['u'].cpu().numpy())
        # not positive definite: same failing pivot reported
        bad = ops.loglik_batched(num.zt, W, np.full((pu, num.d), 1e-6), np.ones(pu), np.full(pu, -0.999999))
        assert np.all(bad['loglik'].cpu().numpy() == -np.inf)
        infos.append(bad['info'].cpu().numpy())
    for a, b in zip(res['1'], res['4']):
        assert np.array_equal(a, b)
    assert np.array_equal(infos[0], infos[1]) and np.all(infos[0] > 0)


def test_lookahead_repeated_runs_are_bit_identical(cuda):
    """The look-ahead schedule hands pairs to warps through a shared-memory counter and orders its phases with named barriers;
    which warp takes which pair varies from run to run, the result must not (compute-sanitizer is not available on this
    pool: a data race would show up here as run-to-run differences).  More matrices than one wave of CTAs, ragged size."""
    from gladsgp_b200 import ops
    import torch
    pr = make_problem(m=257, q=4, pu=2)
    num = pr['num']
    B = 700
    rng = np.random.default_rng(3)
    beta = np.exp(rng.uniform(np.log(0.05), np.log(3.0), size=(B, num.d)))
    lamz = rng.uniform(0.5, 2.0, B); dadd = rng.uniform(1e-3, 1e-2, B)
    W = np.tile(num.w.T, (B // 2, 1))
    Xd, Wd, bd, ld, dd = [torch.as_tensor(np.ascontiguousarray(a), device='cuda') for a in (num.zt, W, beta, lamz, dadd)]
    ref = None
    for rep in range(6):
        out = ops.loglik_batched(Xd, Wd, bd, ld, dd, want_factor=True, want_u=True)
        got = (out['loglik'].clone(), out['u'].clone(), out['factor'][:, :4096].clone())
        if ref is None:
            ref = got
            assert torch.isfinite(ref[0]).all()
        else:
            for a, b in zip(ref, got):
                assert torch.equal(a, b), rep
