"""The backward-error bars of tests/backward_helpers.py on the host: the device's factorisation algorithm, emulated in
FP64 NumPy, meets them with margin over the conditioning posteriors reach; LAPACK's outputs meet them; and outputs that
are wrong by 1e-12 relative in one place fail them.

The emulation follows csrc/ggp_chol.cuh: left-looking, 32-column panels, the matrix padded to a multiple of 32 with the
identity.  Per panel: P = C[rows, panel] - L[rows, :32j] L[panel, :32j]^T; the 32x32 diagonal block of P is factored
column by column (pivot d, r = 1/sqrt(d), L_kk = d r, L_ik = P_ik r, right-looking update); its inverse M_j is formed by
forward substitution of every unit vector (rows scaled by r); the rows below are X = P M_j^T (an inverse-based
triangular solve, whose error grows with cond(L_jj), unlike LAPACK's substitution).  u = L^-1 w substitutes in the
diagonal block and updates the rest with X u_j; the prediction rows V and the cross-validation rows z_i run the same
panel loop with M_j."""
import numpy as np
import pytest
import scipy.linalg
import torch

import backward_helpers as bh
from helpers import synthetic

SCALES = [3.0, 0.3, 0.03, 0.003]
NUGGETS = [1e-2, 1e-4, 1e-6, 1e-8, 1e-10]
EMU_MAX = 0.25              # the emulated algorithm must stay this far below every bar


# --------------------------------------------------------------------------------------------------------------------
# host emulation of the device algorithm
# --------------------------------------------------------------------------------------------------------------------
def _pad(C):
    m = C.shape[0]
    Mp = bh.round_up32(m)
    Cp = np.eye(Mp)
    Cp[:m, :m] = C
    return Cp


def _chol32(P):
    """The kernel's 32x32 block factorisation (warp 0, lane = row): L and r = 1/sqrt(pivot) per column."""
    A = P.copy()
    L = np.zeros((32, 32))
    r = np.zeros(32)
    for k in range(32):
        d = A[k, k]
        if not d > 0.0:
            raise np.linalg.LinAlgError('pivot %d' % k)
        r[k] = 1.0 / np.sqrt(d)
        col = A[k:, k] * r[k]
        col[0] = d * r[k]
        L[k:, k] = col
        A[k + 1:, k + 1:] -= np.outer(col[1:], col[1:])
    return L, r


def _inv32(L, r):
    """The kernel's inverse of the block (warp 1, lane k solves L y = e_k row by row, y_i scaled by r_i)."""
    Y = np.zeros((32, 32))
    eye = np.eye(32)
    for i in range(32):
        Y[i] = (eye[i] - L[i, :i] @ Y[:i]) * r[i]
    return Y


def emulate_factor(C):
    """Packed-factor equivalents of the device: L (Mp, Mp), the inverted diagonal blocks M (nP, 32, 32) and r (Mp,)."""
    Cp = _pad(C)
    Mp = Cp.shape[0]
    nP = Mp // 32
    L = np.zeros((Mp, Mp))
    M = np.zeros((nP, 32, 32))
    r = np.zeros(Mp)
    for j in range(nP):
        r0 = 32 * j
        P = Cp[r0:, r0:r0 + 32] - L[r0:, :r0] @ L[r0:r0 + 32, :r0].T
        Ljj, rj = _chol32(P[:32])
        M[j] = _inv32(Ljj, rj)
        L[r0:r0 + 32, r0:r0 + 32] = Ljj
        L[r0 + 32:, r0:r0 + 32] = P[32:] @ M[j].T
        r[r0:r0 + 32] = rj
    return L, M, r


def emulate_u(L, r, w):
    Mp = L.shape[0]
    b = np.zeros(Mp)
    b[:w.size] = w
    u = np.zeros(Mp)
    for j in range(Mp // 32):
        r0 = 32 * j
        bj = b[r0:r0 + 32].copy()
        for c in range(32):
            u[r0 + c] = bj[c] * r[r0 + c]
            bj[c + 1:] -= L[r0 + c + 1:r0 + 32, r0 + c] * u[r0 + c]
        b[r0 + 32:] -= L[r0 + 32:, r0:r0 + 32] @ u[r0:r0 + 32]
    return u


def emulate_rows(L, M, R, skip=None):
    """Rows V (n, Mp) with L V^T = R^T, R (n, m): the prediction / cross-validation panel loop.  skip = (row, j, k):
    that row's panel j leaves out the update from panel k."""
    Mp = L.shape[0]
    Rp = np.zeros((R.shape[0], Mp))
    Rp[:, :R.shape[1]] = R
    V = np.zeros_like(Rp)
    for j in range(Mp // 32):
        r0 = 32 * j
        S = V[:, :r0] @ L[r0:r0 + 32, :r0].T
        if skip is not None and skip[1] == j:
            i, k = skip[0], skip[2]
            S[i] -= V[i, 32 * k:32 * k + 32] @ L[r0:r0 + 32, 32 * k:32 * k + 32].T
        V[:, r0:r0 + 32] = (Rp[:, r0:r0 + 32] - S) @ M[j].T
    return V


# --------------------------------------------------------------------------------------------------------------------
# inputs
# --------------------------------------------------------------------------------------------------------------------
def design(m, q=8, dup_pairs=0, gap=1e-7, exact=False, seed=3):
    """[dummy 0.5, synthetic.design(m, q)]; dup_pairs > 0: that many rows, spread over the design, are replaced by a
    neighbour's coordinates moved by `gap` along a random direction (exact: not moved)."""
    X = np.concatenate([0.5 * np.ones((m, 1)), synthetic.design(m, q).astype(np.float64)], axis=1)
    if dup_pairs:
        rng = np.random.default_rng(seed)
        rows = np.linspace(0, m - 1, 2 * dup_pairs).astype(int)
        src, dst = rows[0::2], rows[1::2]
        X[dst] = X[src]
        if not exact:
            v = rng.standard_normal((dup_pairs, q))
            X[dst, 1:] += gap * v / np.linalg.norm(v, axis=1, keepdims=True)
    return X


def prediction_designs(X, n_train, n_lhs=64):
    """The first n_train training rows, the same rows moved by 1e-7 in every input, and n_lhs LHS points: near the data
    is where s11 - |V|^2 cancels."""
    T = X[:n_train].copy()
    off = T.copy()
    off[:, 1:] += 1e-7
    lhs = np.concatenate([0.5 * np.ones((n_lhs, 1)), synthetic.test_design(n_lhs, X.shape[1] - 1).astype(np.float64)],
                         axis=1)
    return np.concatenate([T, off, lhs])


def hypers(d, scales, nuggets, seed=11):
    """Blocks of every (scale, nugget): beta_k = scale r_k with fixed r_k in [0.3, 1] (r = 1 for the dummy column),
    lamz = 1, S22 nugget delta, s11 = 1 + delta / 2 (the part of the nugget a prediction keeps)."""
    r = np.exp(np.random.default_rng(seed).uniform(np.log(0.3), 0.0, size=d))
    r[0] = 1.0
    beta = np.array([s * r for s in scales for _ in nuggets])
    dadd = np.array([n for _ in scales for n in nuggets])
    lamz = np.ones(beta.shape[0])
    return beta, lamz, dadd, 1.0 / lamz + 0.5 * dadd


def _t(a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64)


def _ratios(X, Xp, beta, lamz, dadd, s11, w, L, M, u, V, Z, rows, ll, mean, var):
    """Every helper ratio of one block (host tensors); L (m, m) or padded, M (nP, 32, 32), u, V (n, .), Z (k, .)."""
    m = X.shape[0]
    Xt, Xpt, bt = _t(X), _t(Xp), _t(beta[None])
    lz, dd = _t([lamz]), _t([dadd])
    C = bh.dense_cov(Xt, bt, lz, dd)
    Lt = _t(L[:m, :m])[None]
    S21 = bh.cross_cov(Xt, Xpt, bt, lz)
    E = torch.eye(m, dtype=torch.float64)[:, rows][None]
    Ld = _t(np.stack([L[32 * j:32 * j + 32, 32 * j:32 * j + 32] for j in range(M.shape[0])]))[None]
    Mt = _t(M)[None]
    Vt = _t(V[:, :m])[None]
    Zt = _t(Z[:, :m])[None]
    ut = _t(u[:m])[None]
    return dict(
        factor=float(bh.factor_ratio(C, Lt, bh.pf_bound(Xt, Xt, bt, C, self_cov=True), bh.factor_trsm_term(Lt, Ld, Mt))),
        u=float(bh.solve_ratio(Lt, ut[:, :, None], _t(w)[None, :, None])),
        V=float(bh.solve_ratio(Lt, Vt.transpose(1, 2), S21, bh.pf_bound(Xt, Xpt, bt, S21),
                               bh.trsm_term(Vt, Ld, Mt).transpose(1, 2))),
        Z=float(bh.solve_ratio(Lt, Zt.transpose(1, 2), E, None, bh.trsm_term(Zt, Ld, Mt).transpose(1, 2))),
        inverse=float(bh.inverse_ratio(Ld, _t(M)[None])),
        ll=float(bh.ll_ratio(_t([ll]), Lt, ut)),
        mean=float(bh.mean_ratio(_t(mean)[None], Vt, ut)),
        var=float(bh.var_ratio(_t(var)[None], Vt, _t([s11]))))


def _lapack(X, Xp, beta, lamz, dadd, w, rows):
    C = np.exp(-((X[:, None, :] - X[None, :, :]) ** 2) @ beta) / lamz
    np.fill_diagonal(C, 1.0 / lamz + dadd)
    S21 = np.exp(-((X[:, None, :] - Xp[None, :, :]) ** 2) @ beta) / lamz
    L = np.linalg.cholesky(C)
    u = scipy.linalg.solve_triangular(L, w, lower=True)
    V = scipy.linalg.solve_triangular(L, S21, lower=True).T
    Z = scipy.linalg.solve_triangular(L, np.eye(X.shape[0])[:, rows], lower=True).T
    Lp = _pad(L)
    M = np.stack([scipy.linalg.solve_triangular(Lp[32 * j:32 * j + 32, 32 * j:32 * j + 32], np.eye(32), lower=True)
                  for j in range(Lp.shape[0] // 32)])
    return C, S21, L, u, V, Z, M


def _case(m, scale, nugget, dup=0, exact=False):
    X = design(m, dup_pairs=dup, exact=exact)
    beta, lamz, dadd, s11 = hypers(X.shape[1], [scale], [nugget])
    Xp = prediction_designs(X, 48)
    return X, Xp, beta[0], lamz[0], dadd[0], s11[0], np.random.default_rng(m).standard_normal(m)


def _rows(m):
    return sorted({0, 31, 32, m // 2, m - 1} & set(range(m)))


def _emulated(X, Xp, beta, lamz, dadd, s11, w):
    m = X.shape[0]
    C = np.exp(-((X[:, None, :] - X[None, :, :]) ** 2) @ beta) / lamz
    np.fill_diagonal(C, 1.0 / lamz + dadd)
    S21 = np.exp(-((X[:, None, :] - Xp[None, :, :]) ** 2) @ beta) / lamz
    L, M, r = emulate_factor(C)
    u = emulate_u(L, r, w)
    V = emulate_rows(L, M, S21.T)
    rows = _rows(m)
    Z = emulate_rows(L, M, np.eye(m)[rows])
    ll = -np.sum(np.log(np.diag(L)[:m])) - 0.5 * u @ u
    mean = V @ u
    var = s11 - np.sum(V * V, axis=1)
    return dict(C=C, S21=S21, L=L, M=M, r=r, u=u, V=V, Z=Z, rows=rows, ll=ll, mean=mean, var=var)


# --------------------------------------------------------------------------------------------------------------------
# 1. the device's algorithm meets the bars with margin
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('m,dup', [(33, 0), (257, 0), (512, 0), (1000, 0), (512, 16)])
def test_emulated_device_algorithm_meets_the_bars(m, dup):
    """Every (beta scale, nugget) of the sweep, cond(S22) from ~1 to ~1e12: every ratio <= 0.25.  dup = 16: sixteen
    pairs of rows 1e-7 apart."""
    worst = {}
    for scale in SCALES:
        for nugget in NUGGETS:
            X, Xp, beta, lamz, dadd, s11, w = _case(m, scale, nugget, dup)
            e = _emulated(X, Xp, beta, lamz, dadd, s11, w)
            r = _ratios(X, Xp, beta, lamz, dadd, s11, w, e['L'], e['M'], e['u'], e['V'], e['Z'], e['rows'], e['ll'],
                        e['mean'], e['var'])
            for k, v in r.items():
                assert v <= EMU_MAX, (k, v, scale, nugget)
                worst[k] = max(worst.get(k, 0.0), v)
            # the padded rows and columns of the last block are the identity, in L and in M
            mask = bh.padded_identity_mask(m, 'cpu').numpy()
            Mp = e['L'].shape[0]
            Lb = np.stack([e['L'][32 * j:32 * j + 32, 32 * j:32 * j + 32] for j in range(Mp // 32)])
            eye = np.broadcast_to(np.eye(32), Lb.shape)
            assert np.array_equal(Lb[mask], eye[mask]) and np.array_equal(e['M'][mask], eye[mask])
    print('emulation m=%d dup=%d: %s' % (m, dup, ' '.join('%s %.3g' % kv for kv in sorted(worst.items()))))


def test_lapack_outputs_meet_the_bars():
    """LAPACK's factor, substitution solves and triangular inverses, at a well- and an ill-conditioned block."""
    for scale, nugget in ((3.0, 1e-2), (0.003, 1e-10)):
        X, Xp, beta, lamz, dadd, s11, w = _case(257, scale, nugget)
        rows = _rows(257)
        C, S21, L, u, V, Z, M = _lapack(X, Xp, beta, lamz, dadd, w, rows)
        ll = -np.sum(np.log(np.diag(L))) - 0.5 * u @ u
        r = _ratios(X, Xp, beta, lamz, dadd, s11, w, _pad(L), M, u, V, Z, rows, ll, V @ u, s11 - np.sum(V * V, axis=1))
        assert max(r.values()) <= 1.0, r


# --------------------------------------------------------------------------------------------------------------------
# 2. the bars bite: outputs wrong by 1e-12 relative in one place fail
# --------------------------------------------------------------------------------------------------------------------
def _ill():
    X, Xp, beta, lamz, dadd, s11, w = _case(512, 0.03, 1e-6)
    return X, Xp, beta, lamz, dadd, s11, w, _emulated(X, Xp, beta, lamz, dadd, s11, w)


def test_perturbed_factor_entry_fails():
    X, _, beta, lamz, dadd, _, _, e = _ill()
    L = np.linalg.cholesky(e['C'])
    Xt, bt = _t(X), _t(beta[None])
    C = _t(e['C'])[None]
    E = bh.pf_bound(Xt, Xt, bt, C, self_cov=True)
    assert float(bh.factor_ratio(C, _t(L)[None], E)) <= 0.05
    i, j = np.unravel_index(np.argmax(np.abs(L)), L.shape)
    L[i, j] *= 1.0 + 1e-12
    assert float(bh.factor_ratio(C, _t(L)[None], E)) > 1.0


def test_perturbed_inverse_block_entry_fails():
    e = _ill()[-1]
    Mp = e['L'].shape[0]
    Ld = np.stack([e['L'][32 * j:32 * j + 32, 32 * j:32 * j + 32] for j in range(Mp // 32)])
    M = e['M'].copy()
    assert float(bh.inverse_ratio(_t(Ld)[None], _t(M)[None])) <= EMU_MAX
    # the entry whose change moves L_jj M_j most: |L_jj[a, a] M_j[a, b]| largest
    j, a, b = np.unravel_index(np.argmax(np.abs(np.diagonal(Ld, axis1=1, axis2=2)[:, :, None] * M)), M.shape)
    M[j, a, b] *= 1.0 + 1e-12
    assert float(bh.inverse_ratio(_t(Ld)[None], _t(M)[None])) > 1.0


def test_stale_panel_in_one_prediction_row_fails():
    X, Xp, beta, lamz, dadd, s11, w, e = _ill()
    m = X.shape[0]
    Xt, Xpt, bt = _t(X), _t(Xp), _t(beta[None])
    Lt = _t(e['L'][:m, :m])[None]
    S21 = _t(e['S21'])[None]
    E = bh.pf_bound(Xt, Xpt, bt, S21)
    assert float(bh.solve_ratio(Lt, _t(e['V'][:, :m]).T[None], S21, E)) <= EMU_MAX
    V = emulate_rows(e['L'], e['M'], e['S21'].T, skip=(100, 9, 4))
    assert np.array_equal(np.delete(V, 100, 0), np.delete(e['V'], 100, 0))
    assert float(bh.solve_ratio(Lt, _t(V[:, :m]).T[None], S21, E)) > 1.0


def test_loglik_off_by_1e_11_of_its_terms_fails():
    X, _, _, _, _, _, _, e = _ill()
    m = X.shape[0]
    Lt = _t(e['L'][:m, :m])[None]
    ut = _t(e['u'][:m])[None]
    terms = np.sum(np.abs(np.log(np.diag(e['L'])[:m]))) + 0.5 * e['u'] @ e['u']
    assert float(bh.ll_ratio(_t([e['ll']]), Lt, ut)) <= EMU_MAX
    assert float(bh.ll_ratio(_t([e['ll'] + 1e-11 * terms]), Lt, ut)) > 1.0
