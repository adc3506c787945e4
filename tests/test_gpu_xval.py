"""GPU: cross-validated predictions from the cached factor (ggp_xval_solve_f64, Predictor.xval,
SepiaXvalEmulatorPrediction) against the literal per-fold refit of the oracle and dense FP64 algebra."""
import numpy as np
import pytest

from helpers import synthetic, make_problem, make_scalar_problem
from oracle import xval_oracle as xo

pytestmark = pytest.mark.gpu

PRED_RTOL = 1e-6      # the tolerances of test_predict_moments_match_oracle


def _blocks(num, samples):
    """(sample, PC) blocks in (s, j) order: beta, lamz, dadd, s11, W and c = 1 / (LamSim_j lamWOs_s)."""
    d, pu, m = num.d, num.pu, num.m
    ns = samples['lamWs'].shape[0]
    beta = np.zeros((ns * pu, d)); lamz = np.zeros(ns * pu); dadd = np.zeros(ns * pu); s11 = np.zeros(ns * pu)
    W = np.zeros((ns * pu, m)); c = np.zeros(ns * pu)
    for s in range(ns):
        bU = np.asarray(samples['betaU'][s], dtype=np.float64).reshape((d, pu), order='F')
        for j in range(pu):
            b = s * pu + j
            lz = float(samples['lamUz'][s, j]); lw = float(samples['lamWs'][s, j]); lo = float(samples['lamWOs'][s, 0])
            beta[b] = bU[:, j]; lamz[b] = lz
            c[b] = 1.0 / (num.LamSim[j] * lo)
            dadd[b] = c[b] + 1.0 / lw
            s11[b] = 1.0 / lz + 1.0 / lw
            W[b] = num.wv[j * m:(j + 1) * m, 0]
    return beta, lamz, dadd, s11, W, c


def _predictor(num, samples):
    from gladsgp_b200 import ops
    beta, lamz, dadd, s11, W, c = _blocks(num, samples)
    P = ops.Predictor(num.zt, W, beta, lamz, dadd, s11)
    assert not P.info.any().item()
    return P, c


def _check_folds(P, c, num, samples, folds, ref_mu, ref_Sig):
    """Predictor.xval against the oracle's per-fold mu / Sigma (PC-major per sample)."""
    ns, pu = samples['lamWs'].shape[0], num.pu
    mu, var, Sig = P.xval(folds, c)
    mu = mu.cpu().numpy().reshape(ns, pu, -1); var = var.cpu().numpy().reshape(ns, pu, -1)
    scale = max(np.abs(r).max() for r in ref_mu)
    off = 0
    for k, f in enumerate(folds):
        n = len(f)
        rm = ref_mu[k].reshape(ns, pu, n)
        rS = np.stack([ref_Sig[k][:, j * n:(j + 1) * n, j * n:(j + 1) * n] for j in range(pu)], axis=1)   # (ns, pu, n, n)
        np.testing.assert_allclose(mu[:, :, off:off + n], rm, rtol=PRED_RTOL, atol=PRED_RTOL * scale)
        np.testing.assert_allclose(var[:, :, off:off + n], np.diagonal(rS, axis1=-2, axis2=-1), rtol=PRED_RTOL)
        if n > 1:
            g = Sig[k].cpu().numpy().reshape(ns, pu, n, n)
            np.testing.assert_allclose(g, rS, rtol=PRED_RTOL, atol=PRED_RTOL * np.abs(rS).max())
        else:
            assert Sig[k] is None
        off += n


@pytest.mark.parametrize('m,q,pu,ns,lamws', [(64, 3, 2, 6, None), (100, 8, 5, 6, None), (257, 4, 2, 4, None),
                                             (512, 8, 10, 4, None), (96, 3, 2, 4, 1e5)])
def test_leave_one_out_moments_match_oracle(cuda, m, q, pu, ns, lamws):
    pr = make_problem(m=m, q=q, pu=pu)
    num = pr['num']
    samples = synthetic.posterior_samples(ns, num.d, pu, seed=m)
    if lamws is not None:                                    # small nugget: S22 close to the noise-free covariance
        samples['lamWs'] = np.full_like(samples['lamWs'], lamws)
    P, c = _predictor(num, samples)
    folds = [[i] for i in range(m)]
    # the literal refit costs one m x m solve per (fold, sample, PC): at m = 512 the oracle checks a spread of rows
    check = list(range(m)) if m <= 257 else sorted({0, 1, 31, 32, 100, 255, 256, 300, 480, 510, m - 1})
    _, ref_mu, ref_Sig = xo.xval_pred(num, samples, [[i] for i in check], draw=False)
    mu, var, Sig = P.xval(folds, c)
    assert all(s is None for s in Sig)
    mu = mu.cpu().numpy().reshape(ns, pu, m)[:, :, check]
    var = var.cpu().numpy().reshape(ns, pu, m)[:, :, check]
    rm = np.stack([r.reshape(ns, pu) for r in ref_mu], axis=-1)
    rv = np.stack([r.reshape(ns, pu) for r in [np.diagonal(S, axis1=1, axis2=2) for S in ref_Sig]], axis=-1)
    np.testing.assert_allclose(mu, rm, rtol=PRED_RTOL, atol=PRED_RTOL * np.abs(rm).max())
    np.testing.assert_allclose(var, rv, rtol=PRED_RTOL)


def test_kernel_against_dense_fp64(cuda):
    """alpha = z.u and p = z.z against the dense inverse of the unpacked factor, Z rows against a triangular solve, and
    identical bits for ascending and permuted indices (the skipped panels would only add exact zeros)."""
    import torch
    from gladsgp_b200 import ops
    m = 300
    pr = make_problem(m=m, q=4, pu=3)
    num = pr['num']
    samples = synthetic.posterior_samples(2, num.d, 3, seed=7)
    P, _ = _predictor(num, samples)
    L = ops.factor_unpack(P.factor, m)
    Linv = torch.linalg.inv(L)
    u = P.u[:, :m]
    idx = np.arange(m)
    alpha, p, Z = P.xval_solve(idx, want_Z=True)
    ref_a = torch.einsum('bki,bk->bi', Linv, u)
    ref_p = (Linv * Linv).sum(1)
    assert float((alpha - ref_a).abs().max()) <= 1e-9 * float(ref_a.abs().max())
    assert float(((p - ref_p) / ref_p).abs().max()) <= 1e-9
    eye = torch.eye(m, dtype=torch.float64, device='cuda').expand(P.B, m, m)
    ref_Z = torch.linalg.solve_triangular(L, eye, upper=False).transpose(1, 2)       # row i = L^-1 e_i
    assert float((Z[:, :, :m] - ref_Z).abs().max()) <= 1e-9 * float(ref_Z.abs().max())
    assert not Z[:, :, m:].any().item()
    rng = np.random.default_rng(3)
    perm = rng.permutation(m)
    a2, p2, Z2 = P.xval_solve(perm, want_Z=True)
    assert torch.equal(a2, alpha[:, perm]) and torch.equal(p2, p[:, perm]) and torch.equal(Z2, Z[:, perm])
    sub = np.sort(rng.choice(m, 37, replace=False))[::-1].copy()                 # a descending subset, no Z
    a3, p3 = P.xval_solve(sub)
    assert torch.equal(a3, alpha[:, sub]) and torch.equal(p3, p[:, sub])


@pytest.mark.parametrize('case', ['kfold5', 'unsorted_overlap', 'fold_over_256'])
def test_folds_match_oracle(cuda, case):
    m = {'kfold5': 100, 'unsorted_overlap': 90, 'fold_over_256': 600}[case]
    pr = make_problem(m=m, q=3, pu=2)
    num = pr['num']
    samples = synthetic.posterior_samples(3, num.d, 2, seed=m)
    rng = np.random.default_rng(m)
    if case == 'kfold5':
        folds = [list(f) for f in np.array_split(rng.permutation(m), 5)]
    elif case == 'unsorted_overlap':
        folds = [[40, 3, 77, 12], [3, 89, 0], [55], [12, 40, 61, 8, 30, 31, 33]]
    else:                                                    # one fold spans several 256-row kernel tasks
        folds = [list(rng.permutation(m)[:300]), list(range(599, 259, -1))]
    P, c = _predictor(num, samples)
    _, ref_mu, ref_Sig = xo.xval_pred(num, samples, folds, draw=False)
    _check_folds(P, c, num, samples, folds, ref_mu, ref_Sig)


def test_folds_chunked_over_blocks(cuda, monkeypatch):
    """Z chunked over blocks gives the same moments as one launch."""
    from gladsgp_b200 import ops
    pr = make_problem(m=80, q=3, pu=3)
    num = pr['num']
    samples = synthetic.posterior_samples(5, num.d, 3, seed=2)
    P, c = _predictor(num, samples)
    folds = [[1, 5, 9], [70, 2], [33]]
    mu1, var1, S1 = P.xval(folds, c)
    monkeypatch.setattr(ops, 'XVAL_Z_BYTES', 4 * 6 * 96 * 8)               # 4 blocks per launch
    mu2, var2, S2 = P.xval(folds, c)
    # the kernel is deterministic; the batched Gram / Cholesky products may pick other algorithms for other batch sizes
    np.testing.assert_allclose(mu2.cpu().numpy(), mu1.cpu().numpy(), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(var2.cpu().numpy(), var1.cpu().numpy(), rtol=1e-12)
    for a, b in zip(S1, S2):
        assert (a is None) == (b is None)
        if a is not None:
            np.testing.assert_allclose(b.cpu().numpy(), a.cpu().numpy(), rtol=1e-12, atol=1e-12)


def _model(m=64, q=3, pu=2):
    from sepia.SepiaData import SepiaData
    from sepia.SepiaModel import SepiaModel
    pr = make_problem(m=m, q=q, pu=pu, n_x=40, n_t=30)
    data = SepiaData(t_sim=pr['t'], y_sim=pr['y'], y_ind_sim=np.arange(pr['y'].shape[1], dtype=float))
    data.transform_xt(t_notrans=np.arange(q)); data.standardize_y(y_mean=pr['mu'], y_sd=pr['sd']); data.create_K_basis(K=pr['K'])
    return pr, data, SepiaModel(data)


def test_public_class(cuda):
    from sepia.SepiaPredict import SepiaEmulatorPrediction, SepiaXvalEmulatorPrediction
    from oracle import sepia_oracle as so
    pr, data, model = _model()
    m, pu, ns = 64, 2, 8
    samples = synthetic.posterior_samples(ns, model.num.p + model.num.q, pu, seed=4)
    # an ordinary prediction first: cross-validation re-uses its factors
    np.random.seed(0)
    pe = SepiaEmulatorPrediction(t_pred=synthetic.test_design(4, 3), samples=samples, model=model)
    pred_obj = model._pred_cache[1]
    folds = [[5, 2, 9], [0], [63, 10]]
    np.random.seed(1)
    xv = SepiaXvalEmulatorPrediction(samples=samples, model=model, leave_out_inds=folds, storeMuSigma=True)
    assert xv._pred is pred_obj and model._pred_cache[1] is pred_obj
    st = np.random.RandomState(); st.seed(1); st.normal(size=ns * 6 * pu)
    assert np.random.normal() == st.normal()
    assert xv.w.shape == (ns, 6, pu) and xv.w.dtype == np.float64
    rows = [5, 2, 9, 0, 63, 10]
    np.testing.assert_array_equal(xv.xpred, data.sim_data.x_trans[rows])
    np.testing.assert_array_equal(xv.t_pred, data.sim_data.t_trans[rows])
    assert [list(f) for f in xv.leave_out_inds] == folds
    assert [a.shape for a in xv.mu] == [(ns, 6), (ns, 2), (ns, 4)]
    assert [a.shape for a in xv.sigma] == [(ns, 6, 6), (ns, 2, 2), (ns, 4, 4)]
    num = so.OracleNum(data.sim_data.t_trans, data.sim_data.y_std, pr['K'])
    _, ref_mu, ref_Sig = xo.xval_pred(num, samples, folds, draw=False)
    for k in range(3):
        np.testing.assert_allclose(xv.mu[k], ref_mu[k], rtol=1e-6, atol=1e-6 * np.abs(ref_mu[k]).max())
        np.testing.assert_allclose(xv.sigma[k], ref_Sig[k], rtol=1e-6, atol=1e-6 * np.abs(ref_Sig[k]).max())
    assert xv.get_y().shape == (ns, 6, pr['y'].shape[1])
    xv.w = xv.w.astype(np.float32)
    err = xv.get_y_error_stats(y_test=pr['y'][rows].astype(np.float32))
    assert err['rmse'].shape == (6,) and np.isfinite(err['rmse']).all()
    # default folds: leave-one-out, one row per training simulation
    loo = SepiaXvalEmulatorPrediction(samples=samples, model=model, storeRlz=False, storeMuSigma=True)
    assert loo.w is None and len(loo.mu) == m and loo.mu[7].shape == (ns, pu) and loo.sigma[7].shape == (ns, pu, pu)
    np.testing.assert_array_equal(loo.t_pred, data.sim_data.t_trans)
    # addResidVar: the variance gains 1 / (LamSim lamWOs)
    ar = SepiaXvalEmulatorPrediction(samples=samples, model=model, leave_out_inds=[[7]], addResidVar=True, storeRlz=False,
                                     storeMuSigma=True)
    lo = np.asarray(samples['lamWOs'], dtype=np.float64).reshape(-1, 1)
    np.testing.assert_allclose(np.diagonal(ar.sigma[0], axis1=1, axis2=2) - np.diagonal(loo.sigma[7], axis1=1, axis2=2),
                               1.0 / (model.num.LamSim[None, :] * lo), rtol=1e-6)


@pytest.mark.parametrize('bad', [[[]], [[1, 1]], [list(range(64))], [[64]], [[-1]], [], [[0.5]]])
def test_public_class_rejects_bad_folds(cuda, bad):
    from sepia.SepiaPredict import SepiaXvalEmulatorPrediction
    _, _, model = _model()
    samples = synthetic.posterior_samples(2, model.num.p + model.num.q, 2, seed=4)
    model._pred_cache = None
    with pytest.raises(ValueError):
        SepiaXvalEmulatorPrediction(samples=samples, model=model, leave_out_inds=bad)
    assert model._pred_cache is None                        # rejected before anything ran on the device


def test_public_class_scalar_model(cuda):
    from sepia.SepiaData import SepiaData
    from sepia.SepiaModel import SepiaModel
    from sepia.SepiaPredict import SepiaXvalEmulatorPrediction
    from oracle import sepia_oracle as so
    pr = make_scalar_problem(m=100)
    data = SepiaData(t_sim=pr['t'], y_sim=pr['y'])
    data.transform_xt()
    data.standardize_y()
    model = SepiaModel(data)
    samples = synthetic.posterior_samples(5, 2, 1, seed=6)
    samples['betaU'] = np.clip(samples['betaU'], 0.5, None) * 10.0
    folds = [[3], [50, 20, 70]]
    xv = SepiaXvalEmulatorPrediction(samples=samples, model=model, leave_out_inds=folds, storeMuSigma=True)
    assert xv.w.shape == (5, 4, 1) and xv.get_y().shape == (5, 4, 1)
    num = so.OracleNum(data.sim_data.t_trans, data.sim_data.y_std, None)
    _, ref_mu, ref_Sig = xo.xval_pred(num, samples, folds, draw=False)
    for k in range(2):
        np.testing.assert_allclose(xv.mu[k], ref_mu[k], rtol=1e-6, atol=1e-6 * np.abs(ref_mu[k]).max())
        np.testing.assert_allclose(xv.sigma[k], ref_Sig[k], rtol=1e-6, atol=1e-6 * np.abs(ref_Sig[k]).max())


def test_realisation_distribution(cuda):
    """4000 copies of one posterior sample: whitened draws (by sqrt(var) for one-row folds, by the Cholesky factor of
    Sig_F for a larger fold) have mean 0 and variance 1 within 5 sigma."""
    from sepia.SepiaPredict import SepiaXvalEmulatorPrediction
    _, _, model = _model(m=40)
    pu, R = 2, 4000
    one = synthetic.posterior_samples(1, model.num.p + model.num.q, pu, seed=8)
    samples = {k: np.repeat(np.asarray(v), R, axis=0) for k, v in one.items()}
    folds = [[i] for i in range(0, 40, 4)] + [[9, 3, 21]]
    np.random.seed(5)
    xv = SepiaXvalEmulatorPrediction(samples=samples, model=model, leave_out_inds=folds, storeMuSigma=True)
    for k, f in enumerate(folds):
        n = len(f)
        mu = xv.mu[k][0].reshape(pu, n)
        for j in range(pu):
            S = xv.sigma[k][0, j * n:(j + 1) * n, j * n:(j + 1) * n]
            d = xv.w[:, sum(len(g) for g in folds[:k]):][:, :n, j] - mu[j]          # (R, n)
            wz = np.linalg.solve(np.linalg.cholesky(S), d.T).T
            assert np.all(np.abs(wz.mean(0)) < 5.0 / np.sqrt(R)), (k, j)
            assert np.all(np.abs(wz.var(0) - 1.0) < 5.0 * np.sqrt(2.0 / R)), (k, j)
