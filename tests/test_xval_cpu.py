"""CPU: the literal cross-validation route (one sub-model per fold) against the closed form the GPU path computes, and the
argument checks of the cross-validation C ABI."""
import ctypes

import numpy as np
import pytest
import scipy.linalg

from helpers import so, synthetic, make_problem
from oracle import xval_oracle as xo


def _closed_form(num, samples, folds, add_resid=False):
    """Per fold: mu_F = w_F - G^-1 alpha_F, Sig_F = G^-1 - c I with G = Z_F Z_F^T, rows z_i = L^-1 e_i, alpha = L^-T L^-1 w,
    c = 1 / (LamSim_j lamWOs_s) (0 with addResidVar).  Same layouts as the oracle (PC-major per sample)."""
    d, pu, m = num.d, num.pu, num.m
    ns = samples['lamWs'].shape[0]
    mus = [np.zeros((ns, pu * len(f))) for f in folds]
    Sigs = [np.zeros((ns, pu * len(f), pu * len(f))) for f in folds]
    for s in range(ns):
        bU = np.asarray(samples['betaU'][s], dtype=np.float64).reshape((d, pu), order='F')
        lo = float(samples['lamWOs'][s, 0])
        for j in range(pu):
            S22 = so.block_cov(num, bU[:, j], float(samples['lamUz'][s, j]), float(samples['lamWs'][s, j]), lo, j)
            L = scipy.linalg.cholesky(S22, lower=True)
            Zc = scipy.linalg.solve_triangular(L, np.eye(m), lower=True)          # column i = z_i
            w = num.wv[j * m:(j + 1) * m, 0]
            alpha = Zc.T @ scipy.linalg.solve_triangular(L, w, lower=True)
            c = 0.0 if add_resid else 1.0 / (num.LamSim[j] * lo)
            for k, f in enumerate(folds):
                f = np.asarray(f)
                n = f.size
                Gi = np.linalg.inv(Zc[:, f].T @ Zc[:, f])
                sl = slice(j * n, (j + 1) * n)
                mus[k][s, sl] = w[f] - Gi @ alpha[f]
                Sigs[k][s, sl, sl] = Gi - c * np.eye(n)
    return mus, Sigs


def _assert_close(got, ref, tol=1e-10):
    for g, r in zip(got, ref):
        np.testing.assert_allclose(g, r, rtol=tol, atol=tol * np.abs(r).max())


@pytest.mark.parametrize('case', ['loo', 'folds3', 'fold32', 'small_nugget'])
def test_literal_xval_matches_closed_form(case):
    m = {'loo': 24, 'folds3': 30, 'fold32': 70, 'small_nugget': 40}[case]
    pr = make_problem(m=m, q=3, pu=2, n_x=8, n_t=6)
    num = pr['num']
    samples = synthetic.posterior_samples(2, num.d, 2, seed=m)
    if case == 'small_nugget':
        samples['lamWs'] = np.full_like(samples['lamWs'], 1e5)
    rng = np.random.default_rng(m)
    if case == 'loo':
        folds = [[i] for i in range(m)]
    elif case == 'folds3':
        folds = [list(p) for p in rng.permutation(m).reshape(10, 3)]
    elif case == 'fold32':
        folds = [rng.permutation(m)[:32], [5, 1]]
    else:
        folds = [[i] for i in range(0, m, 3)] + [[2, 7, 11]]
    w, mu, Sig = xo.xval_pred(num, samples, folds, draw=False)
    assert w is None and len(mu) == len(folds) == len(Sig)
    ref_mu, ref_Sig = _closed_form(num, samples, folds)
    _assert_close(mu, ref_mu)
    _assert_close(Sig, ref_Sig)


def test_literal_xval_defaults_and_draw_order():
    """Default folds are leave-one-out; the draws consume rng.normal fold by fold, sample by sample, pu |F| values each."""
    pr = make_problem(m=20, q=2, pu=2, n_x=6, n_t=5)
    num = pr['num']
    samples = synthetic.posterior_samples(3, num.d, 2, seed=1)
    rs = np.random.RandomState(4)
    w, mu, _ = xo.xval_pred(num, samples, rng=rs)
    assert w.shape == (3, 20, 2) and len(mu) == 20
    assert rs.normal() == np.random.RandomState(4).normal(size=3 * 20 * 2 + 1)[-1]
    folds = [[3, 1], [0]]
    w2, mu2, Sig2 = xo.xval_pred(num, samples, folds, rng=np.random.RandomState(4))
    assert w2.shape == (3, 3, 2)
    z = np.random.RandomState(4).normal(size=3 * 3 * 2)
    U, sv, _ = np.linalg.svd(Sig2[0][0])
    np.testing.assert_allclose(w2[0, :2], (mu2[0][0] + U @ (np.sqrt(sv) * z[:4])).reshape(2, 2).T, rtol=1e-12)


def test_xval_abi_validates_arguments_without_a_device():
    from gladsgp_b200 import _lib
    h = _lib.load()
    one = ctypes.c_void_p(8)
    assert h.ggp_xval_workspace_bytes(0, 4, 2) == -1 and h.ggp_xval_workspace_bytes(8, 0, 2) == -1
    args = [one, one, 8, 2, one, 4, one, one, None, one, 1 << 20, None]     # fake pointers: only rejected calls are made
    for k, bad in ((0, None), (1, None), (4, None), (6, None), (7, None), (9, None)):
        a = list(args)
        a[k] = bad
        assert h.ggp_xval_solve_f64(*a) == -1
        assert b'null pointer' in h.ggp_last_error_string()
    for k, bad in ((2, 0), (5, 0), (5, -3), (3, 0)):
        a = list(args)
        a[k] = bad
        assert h.ggp_xval_solve_f64(*a) == -1
        assert b'must be positive' in h.ggp_last_error_string()
