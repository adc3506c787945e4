"""GPU parity: prediction moments, reconstruction and rSVD passes vs the CPU oracle."""
import numpy as np
import pytest

from helpers import so, svd_oracle, synthetic, make_problem, make_scalar_problem

pytestmark = pytest.mark.gpu

PRED_RTOL = 1e-6      # north_star: predictive means and variances within 1e-6 relative


def _blocks(num, samples):
    """(sample, PC) hyper-parameter blocks in (s, j) order, as float64."""
    d, pu, m = num.d, num.pu, num.m
    ns = samples['lamWs'].shape[0]
    beta = np.zeros((ns * pu, d)); lamz = np.zeros(ns * pu); dadd = np.zeros(ns * pu); s11 = np.zeros(ns * pu)
    W = np.zeros((ns * pu, m))
    for s in range(ns):
        bU = np.asarray(samples['betaU'][s], dtype=np.float64).reshape((d, pu), order='F')
        for j in range(pu):
            b = s * pu + j
            lz = float(samples['lamUz'][s, j]); lw = float(samples['lamWs'][s, j]); lo = float(samples['lamWOs'][s, 0])
            beta[b] = bU[:, j]; lamz[b] = lz
            dadd[b] = 1.0 / (num.LamSim[j] * lo) + 1.0 / lw
            s11[b] = 1.0 / lz + 1.0 / lw
            W[b] = num.wv[j * m:(j + 1) * m, 0]
    return beta, lamz, dadd, s11, W


@pytest.mark.parametrize('m,q,pu,npred,ns', [(64, 3, 2, 5, 6), (100, 8, 5, 4, 6), (257, 4, 2, 37, 6),
                                             (512, 8, 10, 256, 2)])      # last: cfg3 model at the reference's largest call size
def test_predict_moments_match_oracle(cuda, m, q, pu, npred, ns):
    from gladsgp_b200 import ops
    pr = make_problem(m=m, q=q, pu=pu)
    num = pr['num']
    samples = synthetic.posterior_samples(ns, num.d, pu, seed=m)
    tp = synthetic.test_design(npred, q)
    _, mu, Sig = so.w_pred(num, tp, samples, draw=False)
    beta, lamz, dadd, s11, W = _blocks(num, samples)
    P = ops.Predictor(num.zt, W, beta, lamz, dadd, s11)
    xp = np.concatenate([0.5 * np.ones((npred, 1)), tp.astype(np.float64)], axis=1)
    mean, var, V = P.predict(xp, want_V=True)
    Sg = P.pred_cov(xp, V).cpu().numpy()
    mean = mean.cpu().numpy(); var = var.cpu().numpy()
    scale = np.abs(mu).max()
    for s in range(ns):
        for j in range(pu):
            b = s * pu + j
            sl = slice(j * npred, (j + 1) * npred)
            np.testing.assert_allclose(mean[b], mu[s, sl], rtol=PRED_RTOL, atol=PRED_RTOL * scale)
            np.testing.assert_allclose(var[b], np.diag(Sig[s, sl, sl]), rtol=PRED_RTOL)
            np.testing.assert_allclose(Sg[b], Sig[s, sl, sl], rtol=PRED_RTOL, atol=PRED_RTOL * np.abs(Sig[s, sl, sl]).max())


def test_predict_many_designs_blocks(cuda):
    """More designs than one 512-row task; moments must not depend on the blocking."""
    from gladsgp_b200 import ops
    pr = make_problem(m=64, q=3, pu=2)
    num = pr['num']
    samples = synthetic.posterior_samples(3, num.d, 2, seed=1)
    tp = synthetic.test_design(1100, 3)
    xp = np.concatenate([0.5 * np.ones((1100, 1)), tp.astype(np.float64)], axis=1)
    beta, lamz, dadd, s11, W = _blocks(num, samples)
    P = ops.Predictor(num.zt, W, beta, lamz, dadd, s11)
    mean, var = P.predict(xp)
    m2, v2 = P.predict(xp[500:600])
    assert np.array_equal(mean.cpu().numpy()[:, 500:600], m2.cpu().numpy())
    assert np.array_equal(var.cpu().numpy()[:, 500:600], v2.cpu().numpy())
    _, mu, Sig = so.w_pred(num, tp[:8], samples, draw=False)
    np.testing.assert_allclose(mean.cpu().numpy()[0, :8], mu[0, :8], rtol=PRED_RTOL, atol=1e-6 * np.abs(mu).max())


@pytest.mark.parametrize('n_y', [1000, 4099])
def test_reconstruct_matches_get_y(cuda, n_y):
    from gladsgp_b200 import ops
    rng = np.random.default_rng(0)
    R, pu = 37, 10
    w = rng.standard_normal((R, pu)).astype(np.float32)
    K = rng.standard_normal((pu, n_y)).astype(np.float32)
    sd = rng.uniform(0.1, 2.0, n_y).astype(np.float32); mu = rng.standard_normal(n_y).astype(np.float32)
    ref = so.get_y(w[None], K, sd, mu)[0]
    y = ops.reconstruct(w, K, sd, mu).cpu().numpy()
    np.testing.assert_allclose(y, ref, rtol=2e-5, atol=2e-5)
    y1 = ops.reconstruct(w, K, np.float32(1.7), np.float32(0.3)).cpu().numpy()
    np.testing.assert_allclose(y1, so.get_y(w[None], K, np.float32(1.7), np.float32(0.3))[0], rtol=2e-5, atol=2e-5)


@pytest.mark.parametrize('m,n,r', [(64, 1000, 25), (100, 5003, 25), (128, 3000, 40)])
def test_rsvd_passes_match_numpy(cuda, m, n, r):
    from gladsgp_b200 import ops
    torch = cuda
    rng = np.random.default_rng(m)
    X = rng.standard_normal((m, n)).astype(np.float32)
    om = rng.standard_normal((n, r)).astype(np.float32)
    Xd = torch.as_tensor(X, device='cuda')
    Y = ops.rsvd_sketch(Xd, torch.as_tensor(om.T.copy(), device='cuda')).cpu().numpy()
    ref = X.astype(np.float64) @ om.astype(np.float64)
    np.testing.assert_allclose(Y, ref, rtol=0, atol=3e-5 * np.abs(ref).max())
    Yq = rng.standard_normal((m, r)).astype(np.float32)
    Bt = ops.rsvd_xty(Xd, torch.as_tensor(Yq, device='cuda')).cpu().numpy()
    refB = Yq.astype(np.float64).T @ X.astype(np.float64)
    np.testing.assert_allclose(Bt, refB, rtol=0, atol=3e-5 * np.abs(refB).max())


@pytest.mark.parametrize('nsamp,npred,n_y,q', [(64, 4, 3001, 0.025), (128, 1, 1000, 0.025), (16, 3, 2048, 0.05)])
def test_fused_stats_match_numpy_postprocessing(cuda, nsamp, npred, n_y, q):
    """assess_all_models.py:493-500: mean of get_y over samples, quantiles of get_y + sd_y * N(0, 1/lamWOs[s])."""
    from gladsgp_b200 import ops
    rng = np.random.default_rng(3)
    pu = 10
    w = rng.standard_normal((nsamp, npred, pu)).astype(np.float32)
    K = rng.standard_normal((pu, n_y)).astype(np.float32)
    sd = rng.uniform(0.1, 2.0, n_y).astype(np.float32); mu = rng.standard_normal(n_y).astype(np.float32)
    noise = (rng.standard_normal((nsamp, npred)) / np.sqrt(rng.uniform(20, 200, (nsamp, 1)))).astype(np.float32)
    y = so.get_y(w, K, sd, mu)                                   # (nsamp, npred, n_y)
    z = y + sd[None, None, :] * noise[:, :, None]
    ref_mean = np.mean(y, axis=0)
    ref_lo = np.quantile(z, q, axis=0); ref_hi = np.quantile(z, 1 - q, axis=0)
    m_, lo, hi = [t.cpu().numpy() for t in ops.reconstruct_stats(w, K, sd, mu, q=q, noise=noise)]
    np.testing.assert_allclose(m_, ref_mean, rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(lo, ref_lo, rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(hi, ref_hi, rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize('nsamp,npred,n_y,q', [(64, 4, 3001, 0.025), (128, 2, 1500, 0.025), (16, 5, 2048, 0.05)])
def test_fused_error_statistics_match_assess_all_models(cuda, nsamp, npred, n_y, q):
    """assess_all_models.py:489-538 in one pass (ggp_reconstruct_errstats_f32): RMSE, MAPE above the 10 % quantile of the test
    matrix, coverage, mean limits, integrated interval width.  The reference works in float32 (ypreds, np.mean, np.quantile on
    float32 arrays); the kernel forms float32 fields and sums in FP64: tolerance 2e-5 relative, coverage within the few outputs
    whose limit lies within float32 round-off of the test value."""
    from gladsgp_b200 import ops
    from oracle import assess_oracle as ao
    rng = np.random.default_rng(11)
    pu = 10
    w = rng.standard_normal((nsamp, npred, pu)).astype(np.float32)
    K = rng.standard_normal((pu, n_y)).astype(np.float32)
    sd = rng.uniform(0.1, 0.3, n_y).astype(np.float32); mu = (2.0 + rng.standard_normal(n_y) * 0.2).astype(np.float32)
    noise = (rng.standard_normal((nsamp, npred)) / np.sqrt(rng.uniform(20, 200, (nsamp, 1)))).astype(np.float32)
    ym, ylq, yuq = ao.fields(w, K, sd, mu, noise, q)
    y_test = (ym + 0.4 * rng.standard_normal(ym.shape) * sd).astype(np.float32)
    ref = ao.error_statistics(ym, ylq, yuq, y_test)
    err, fl = ops.reconstruct_errstats(w, K, sd, mu, y_test, float(ref['mape_floor']), q=q, noise=noise, want_fields=True)
    np.testing.assert_allclose(np.sqrt(err[:, 0] / n_y), ref['rmse'], rtol=2e-5)
    np.testing.assert_allclose(err[:, 1] / err[:, 2], ref['mape'], rtol=2e-5)
    np.testing.assert_allclose(err[:, 4] / n_y, ref['lq'], rtol=2e-5)
    np.testing.assert_allclose(err[:, 5] / n_y, ref['uq'], rtol=2e-5)
    assert np.all(np.abs(err[:, 3] - ref['frac_covered'] * n_y) <= 3)
    assert np.array_equal(err[:, 2], np.sum(y_test >= ref['mape_floor'], axis=1))
    np.testing.assert_allclose(np.mean((err[:, 5] - err[:, 4]) / n_y), ref['integrated_ci'], rtol=2e-5)
    # fields, when asked for, are those of reconstruct_stats; without them the sums are identical (and deterministic)
    m_, lo, hi = [t.cpu().numpy() for t in ops.reconstruct_stats(w, K, sd, mu, q=q, noise=noise)]
    assert np.array_equal(fl[0].cpu().numpy(), m_) and np.array_equal(fl[1].cpu().numpy(), lo) and np.array_equal(fl[2].cpu().numpy(), hi)
    err2, none = ops.reconstruct_errstats(w, K, sd, mu, y_test, float(ref['mape_floor']), q=q, noise=noise)
    assert none is None and np.array_equal(err, err2)


def test_get_y_error_stats_api(cuda):
    """SepiaEmulatorPrediction.get_y_error_stats: default MAPE floor = np.quantile(y_test, 0.1)."""
    from oracle import assess_oracle as ao
    from sepia.SepiaData import SepiaData
    from sepia.SepiaModel import SepiaModel
    from sepia.SepiaPredict import SepiaEmulatorPrediction
    pr = make_problem(m=64, q=3, pu=2, n_x=40, n_t=30)
    data = SepiaData(t_sim=pr['t'], y_sim=pr['y'], y_ind_sim=np.arange(pr['y'].shape[1], dtype=float))
    data.transform_xt(t_notrans=np.arange(3)); data.standardize_y(y_mean=pr['mu'], y_sd=pr['sd']); data.create_K_basis(K=pr['K'])
    model = SepiaModel(data)
    samples = synthetic.posterior_samples(64, model.num.p + model.num.q, 2, seed=4)
    tp = synthetic.test_design(4, 3)
    np.random.seed(0)
    pe = SepiaEmulatorPrediction(t_pred=tp, samples=samples, model=model)
    pe.w = pe.w.astype(np.float32)
    rng = np.random.default_rng(1)
    noise = (rng.standard_normal((64, 4)) / np.sqrt(np.asarray(samples['lamWOs'], dtype=np.float64).reshape(-1, 1))).astype(np.float32)
    y_test = (pe.get_y().mean(axis=0) + 0.05 * rng.standard_normal((4, pr['y'].shape[1]))).astype(np.float32)
    got = pe.get_y_error_stats(y_test, quantile=0.025, noise=noise)
    ym, ylq, yuq = ao.fields(pe.w, pr['K'], np.asarray(pr['sd'], dtype=np.float32), np.asarray(pr['mu'], dtype=np.float32), noise, 0.025)
    ref = ao.error_statistics(ym, ylq, yuq, y_test)
    assert abs(got['mape_floor'] - ref['mape_floor']) <= 1e-6 * abs(ref['mape_floor'])
    for k in ('rmse', 'mape', 'lq', 'uq'):
        np.testing.assert_allclose(got[k], ref[k], rtol=5e-5, err_msg=k)
    assert np.all(np.abs(got['frac_covered'] - ref['frac_covered']) <= 4.0 / y_test.shape[1])
    assert abs(got['integrated_ci'] - ref['integrated_ci']) <= 5e-5 * abs(ref['integrated_ci'])


@pytest.mark.parametrize('n,B', [(1, 3), (4, 7), (31, 5), (32, 5), (33, 5), (100, 6), (256, 9), (300, 3), (1000, 2)])
def test_chol_draw_matches_numpy_cholesky(cuda, n, B):
    """dev = L z with Sigma = L L^T (the draw step of wPred) against numpy.linalg.cholesky, over block sizes around the
    32-wide panels; entries of a Cholesky factor are unique, so the product must agree to rounding."""
    import torch
    from gladsgp_b200 import ops
    rng = np.random.default_rng(n * 100 + B)
    A = rng.standard_normal((B, n, n + 3))
    Sig = A @ A.transpose(0, 2, 1) / n + 0.05 * np.eye(n)[None]
    z = rng.standard_normal((B, n))
    ref = np.einsum('bij,bj->bi', np.linalg.cholesky(Sig), z)
    dev, info = ops.chol_draw(torch.as_tensor(Sig, device='cuda'), torch.as_tensor(z, device='cuda'))
    assert not info.any().item()
    np.testing.assert_allclose(dev.cpu().numpy(), ref, rtol=1e-10, atol=1e-12)


def test_chol_draw_chunked_workspace_and_rejection(cuda, monkeypatch):
    """A workspace smaller than B scratch factors gives the same result in several launches; a block that is not positive
    definite is reported in info and leaves the other blocks untouched."""
    import torch
    from gladsgp_b200 import ops
    rng = np.random.default_rng(5)
    n, B = 96, 11
    A = rng.standard_normal((B, n, n))
    Sig = A @ A.transpose(0, 2, 1) / n + 0.1 * np.eye(n)[None]
    Sig[4] -= 3.0 * np.eye(n)                      # indefinite
    z = rng.standard_normal((B, n))
    Sd, zd = torch.as_tensor(Sig, device='cuda'), torch.as_tensor(z, device='cuda')
    dev1, info1 = ops.chol_draw(Sd, zd)
    one = int(ops._lib.load().ggp_chol_draw_workspace_bytes(n, 1))
    monkeypatch.setattr(ops, 'CHOL_DRAW_WS_BYTES', 3 * one + 8)          # 3 blocks per launch
    dev2, info2 = ops.chol_draw(Sd, zd)
    i1 = info1.cpu().numpy()
    assert i1[4] > 0 and not np.delete(i1, 4).any()
    assert np.array_equal(i1, info2.cpu().numpy())
    good = np.delete(np.arange(B), 4)
    assert np.array_equal(dev1.cpu().numpy()[good], dev2.cpu().numpy()[good])
    ref = np.einsum('bij,bj->bi', np.linalg.cholesky(Sig[good]), z[good])
    np.testing.assert_allclose(dev1.cpu().numpy()[good], ref, rtol=1e-10, atol=1e-12)


def test_full_size_prediction_is_invariant_to_the_call_split(cuda):
    """cfg4 shape (m = 512, pu = 10) at 20 000 designs per call: moments are bit-identical whether the designs go through in
    one call, in the reference's 4-design calls or in ragged pieces (size-independent property at a size the oracle
    cannot reach), and the variances stay within (0, s11]."""
    from gladsgp_b200 import ops
    pr = make_problem(m=512, q=8, pu=10)
    num = pr['num']
    samples = synthetic.posterior_samples(4, num.d, 10, seed=21)
    n = 20000
    tp = synthetic.test_design(n, 8)
    xp = np.concatenate([0.5 * np.ones((n, 1)), tp.astype(np.float64)], axis=1)
    beta, lamz, dadd, s11, W = _blocks(num, samples)
    P = ops.Predictor(num.zt, W, beta, lamz, dadd, s11)
    mean, var = (a.cpu().numpy() for a in P.predict(xp))
    assert np.isfinite(mean).all() and (var > 0).all() and (var <= s11[:, None] * (1 + 1e-12)).all()
    for lo, hi in ((0, 4), (4, 8), (9996, 10000), (255, 769), (19999, 20000), (12345, 13370)):
        m2, v2 = (a.cpu().numpy() for a in P.predict(xp[lo:hi]))
        assert np.array_equal(mean[:, lo:hi], m2) and np.array_equal(var[:, lo:hi], v2), (lo, hi)


def test_full_size_reconstruction(cuda):
    """get_y at the full field size of cfg3 / cfg4 (n_y = 1 460 000), 256 rows: against the float32 expression on the device."""
    import torch
    from gladsgp_b200 import ops
    g = torch.Generator(device='cuda'); g.manual_seed(9)
    R, pu, n_y = 256, 10, 1460000
    w = torch.randn((R, pu), dtype=torch.float32, device='cuda', generator=g)
    K = torch.randn((pu, n_y), dtype=torch.float32, device='cuda', generator=g)
    sd = torch.rand((n_y,), dtype=torch.float32, device='cuda', generator=g) * 1.9 + 0.1
    mu = torch.randn((n_y,), dtype=torch.float32, device='cuda', generator=g)
    y = ops.reconstruct(w, K, sd, mu)
    ref = (w.double() @ K.double()) * sd.double() + mu.double()
    assert float((y.double() - ref).abs().max()) <= 2e-5 * float(ref.abs().max())


def test_scalar_gp_cfg2_size_10000_designs_against_oracle(cuda):
    """BASELINE.json configs[1]: 1-D GP with 1000 training points, 10 000 test designs in one call; moments of 60 designs
    spread over the call against the oracle's SEPIA-style solve (one fresh S22 factorisation per sample)."""
    from gladsgp_b200 import ops
    pr = make_scalar_problem(m=1000)
    num = pr['num']
    samples = synthetic.posterior_samples(3, num.d, 1, seed=12)
    samples['betaU'] = np.clip(samples['betaU'], 0.5, None) * 10.0           # length scales that resolve x sin(2 pi x)
    npred = 10000
    tp = np.linspace(0.0, 1.0, npred)[:, None]
    beta, lamz, dadd, s11, W = _blocks(num, samples)
    P = ops.Predictor(num.zt, W, beta, lamz, dadd, s11)
    xp = np.concatenate([0.5 * np.ones((npred, 1)), tp], axis=1)
    mean, var = (a.cpu().numpy() for a in P.predict(xp))
    idx = np.unique(np.concatenate([np.arange(0, npred, 173), [npred - 1]]))[:60]
    _, mu, Sig = so.w_pred(num, tp[idx], samples, draw=False)
    for s in range(3):
        np.testing.assert_allclose(mean[s, idx], mu[s], rtol=PRED_RTOL, atol=PRED_RTOL * np.abs(mu).max())
        np.testing.assert_allclose(var[s, idx], np.diag(Sig[s]), rtol=PRED_RTOL, atol=1e-9)


def _dense_posterior_device(X, Xp, W, beta, lamz, dadd):
    """Dense FP64 references on the device from coordinate differences and torch's Cholesky: L of S22, Vr = L^-1 S21
    (m, n) and u = L^-1 w."""
    import torch
    Xd, Xpd = torch.as_tensor(X, device='cuda'), torch.as_tensor(Xp, device='cuda')
    bd = torch.as_tensor(beta, device='cuda')

    def sq(A, Bm):
        D = torch.zeros((A.shape[0], Bm.shape[0]), dtype=torch.float64, device='cuda')
        for k in range(A.shape[1]):
            D += bd[k] * (A[:, None, k] - Bm[None, :, k]) ** 2
        return D
    C = torch.exp(-sq(Xd, Xd)) / lamz
    C.diagonal().fill_(1.0 / lamz + dadd)
    L = torch.linalg.cholesky(C)
    del C
    Vr = torch.linalg.solve_triangular(L, torch.exp(-sq(Xd, Xpd)) / lamz, upper=False)
    u = torch.linalg.solve_triangular(L, torch.as_tensor(W, device='cuda')[:, None], upper=False)[:, 0]
    return L, Vr, u, torch.exp(-sq(Xpd, Xpd)) / lamz


def _check_xval_rows(P, b, L, u, rows):
    import torch
    m = L.shape[0]
    E = torch.zeros((m, len(rows)), dtype=torch.float64, device='cuda')
    E[torch.as_tensor(rows, device='cuda'), torch.arange(len(rows), device='cuda')] = 1.0
    Zr = torch.linalg.solve_triangular(L, E, upper=False).T                     # row i = L^-1 e_i
    alpha, p, Z = P.xval_solve(rows, want_Z=True, b0=b, nb=1)
    assert float((Z[0, :, :m] - Zr).abs().max()) <= PRED_RTOL * float(Zr.abs().max())
    assert not Z[0, :, m:].any().item()
    ra = Zr @ u
    assert float((alpha[0] - ra).abs().max()) <= PRED_RTOL * float(ra.abs().max())
    assert float(((p[0] - (Zr * Zr).sum(1)) / (Zr * Zr).sum(1)).abs().max()) <= PRED_RTOL


def test_prediction_at_cfg5_size_against_dense_fp64(cuda):
    """BASELINE.json configs[4] shape (m = 4096, d = 17), 2 blocks, 257 designs (a second 256-design task holding one
    design): mean, var and V against the dense solve, pred_cov on the first 65 designs, xval_solve rows against L^-1 e_i."""
    import torch
    from gladsgp_b200 import ops
    m, q, B, n = 4096, 16, 2, 257
    X = np.concatenate([0.5 * np.ones((m, 1)), synthetic.design(m, q).astype(np.float64)], axis=1)
    Xp = np.concatenate([0.5 * np.ones((n, 1)), synthetic.test_design(n, q).astype(np.float64)], axis=1)
    rng = np.random.default_rng(17)
    beta = np.exp(rng.uniform(np.log(0.05), np.log(1.0), size=(B, q + 1)))
    lamz = np.array([1.1, 0.8]); lamws = np.array([900.0, 2500.0])
    dadd = 3e-3 + 1.0 / lamws; s11 = 1.0 / lamz + 1.0 / lamws
    W = rng.standard_normal((B, m))
    P = ops.Predictor(X, W, beta, lamz, dadd, s11)
    assert not P.info.any().item()
    mean, var, V = P.predict(Xp, want_V=True)
    Sg = P.pred_cov(Xp[:65], V[:, :65].contiguous())
    for b in range(B):
        L, Vr, u, S11 = _dense_posterior_device(X, Xp, W[b], beta[b], lamz[b], dadd[b])
        mu = Vr.T @ u
        vr = s11[b] - (Vr * Vr).sum(0)
        assert float((mean[b] - mu).abs().max()) <= PRED_RTOL * float(mu.abs().max())
        assert float(((var[b] - vr) / vr).abs().max()) <= PRED_RTOL
        assert float((V[b, :, :m] - Vr.T).abs().max()) <= PRED_RTOL * float(Vr.abs().max())
        assert not V[b, :, m:].any().item()
        S11 = S11[:65, :65].clone()
        S11.diagonal().fill_(s11[b])
        Sig = S11 - Vr[:, :65].T @ Vr[:, :65]
        assert float((Sg[b] - Sig).abs().max()) <= PRED_RTOL * float(Sig.abs().max())
        _check_xval_rows(P, b, L, u, [0, 1, 31, 32, 2047, 4064, 4095])
        del L, Vr
        torch.cuda.empty_cache()


def test_prediction_at_the_largest_supported_m(cuda):
    """m = 8192 fills the kernels' 1024-entry slab-offset table (256 panels x 4 sub-slabs): moments and xval_solve rows
    against torch FP64 on the device; m = 8193 is refused by both entry points."""
    import torch
    from gladsgp_b200 import ops, _lib
    m, q, n = 8192, 8, 5
    X = np.concatenate([0.5 * np.ones((m, 1)), synthetic.design(m, q).astype(np.float64)], axis=1)
    Xp = np.concatenate([0.5 * np.ones((n, 1)), synthetic.test_design(n, q).astype(np.float64)], axis=1)
    rng = np.random.default_rng(8192)
    beta = np.exp(rng.uniform(np.log(0.1), np.log(2.0), size=(1, q + 1)))
    lamz = np.array([1.3]); lamws = np.array([1500.0])
    dadd = 2e-3 + 1.0 / lamws; s11 = 1.0 / lamz + 1.0 / lamws
    W = rng.standard_normal((1, m))
    P = ops.Predictor(X, W, beta, lamz, dadd, s11)
    assert not P.info.any().item()
    mean, var = P.predict(Xp)
    L, Vr, u, _ = _dense_posterior_device(X, Xp, W[0], beta[0], lamz[0], dadd[0])
    mu = Vr.T @ u
    vr = s11[0] - (Vr * Vr).sum(0)
    assert float((mean[0] - mu).abs().max()) <= PRED_RTOL * float(mu.abs().max())
    assert float(((var[0] - vr) / vr).abs().max()) <= PRED_RTOL
    _check_xval_rows(P, 0, L, u, [0, 4095, 8160, 8191])
    del L, Vr, P
    torch.cuda.empty_cache()
    lib = _lib.load()
    x = torch.zeros(64, dtype=torch.float64, device='cuda')
    idx = torch.zeros(1, dtype=torch.int32, device='cuda')
    p = _lib.ptr
    rc = lib.ggp_predict_f64(p(x), 8193, 1, p(x), p(x), p(x), p(x), p(x), p(x), 1, 1, p(x), p(x), None, p(x), x.numel() * 8,
                             _lib.stream_ptr())
    assert rc == -1 and b'8192' in lib.ggp_last_error_string()
    rc = lib.ggp_xval_solve_f64(p(x), p(x), 8193, 1, p(idx), 1, p(x), p(x), None, p(x), x.numel() * 8, _lib.stream_ptr())
    assert rc == -1 and b'8192' in lib.ggp_last_error_string()


@pytest.mark.parametrize('d', [17, 22])
@pytest.mark.parametrize('n', [1, 31, 32, 33, 63, 64, 65, 129, 1024])
def test_pred_cov_ragged_tile_edges(cuda, n, d):
    """pred_cov walks the lower triangle in 64 x 32 tiles (row tile rt holds min(n_ct, 2 rt + 2) column tiles): every
    entry, both triangles, against S11 - S21^T S22^-1 S21 at sizes around the tile edges and at 1024 designs."""
    import scipy.linalg
    from gladsgp_b200 import ops
    m, B = 100, 2
    rng = np.random.default_rng(n * 7 + d)
    X = rng.uniform(0, 1, size=(m, d))
    Xp = rng.uniform(0, 1, size=(n, d))
    beta = rng.uniform(0.05, 1.0, size=(B, d)); lamz = rng.uniform(0.5, 2.0, size=B)
    lamws = rng.uniform(300, 3000, size=B); dadd = 1.0 / lamws + 1e-3
    P = ops.Predictor(X, rng.standard_normal((B, m)), beta, lamz, dadd, 1.0 / lamz + 1.0 / lamws)
    _, _, V = P.predict(Xp, want_V=True)
    Sg = P.pred_cov(Xp, V).cpu().numpy()
    for b in range(B):
        def cov(A, Bm):
            D = np.zeros((A.shape[0], Bm.shape[0]))
            for k in range(d):
                D += beta[b, k] * (A[:, None, k] - Bm[None, :, k]) ** 2
            return np.exp(-D) / lamz[b]
        S22 = cov(X, X)
        np.fill_diagonal(S22, 1.0 / lamz[b] + dadd[b])
        S21 = cov(X, Xp)
        S11 = cov(Xp, Xp)
        np.fill_diagonal(S11, 1.0 / lamz[b] + 1.0 / lamws[b])
        Sig = S11 - S21.T @ scipy.linalg.cho_solve(scipy.linalg.cho_factor(S22, lower=True), S21)
        np.testing.assert_allclose(Sg[b], Sig, rtol=PRED_RTOL, atol=PRED_RTOL * np.abs(Sig).max())
