"""CPU oracle of the emulator Jacobians (csrc/ggp_jacobian.cu, gladsgp_b200.gradient).  TEST INFRASTRUCTURE ONLY.

Dense FP64 restatement per (sample, PC) block, from explicit solves with S22 (not from its Cholesky factor): with
k(x, z) = exp(-sum_k beta_k (x_k - z_k)^2) / lamz and G = [k(x, Z); g_1; ...; g_q], g_k = d k(x, Z) / d x_k,
    mean vector [mu, grad mu] = G S22^-1 w,     joint covariance of [f, grad f] = P - G S22^-1 G^T,
P = diag(s11, 2 beta_1 / lamz, ..., 2 beta_q / lamz).  The functions accept complex designs (complex-step checks:
k^T S22^-1 k without conjugation is holomorphic), and the posterior mixture and linear / field reductions of
gladsgp_b200.gradient are restated from their definitions.
"""
import numpy as np

from oracle import sepia_oracle as so


def s22(Z, beta, lamz, dadd):
    """S22 of a block: sepia_oracle's covariance of the training design plus the nugget dadd on the diagonal."""
    C = so.cov_cross(Z, Z, beta, lamz)
    return C + dadd * np.eye(Z.shape[0])


def rows(Z, beta, lamz, x, cols):
    """G (q+1, m) at one design x (d,): k(x, Z) and its derivatives along the inputs `cols` (real or complex x)."""
    k = np.exp(-(((x[None, :] - Z) ** 2) @ beta)) / lamz
    g = [-2.0 * beta[c] * (x[c] - Z[:, c]) * k for c in cols]
    return np.stack([k] + g)


def block(Z, w, beta, lamz, dadd, s11, X, col0):
    """Mean vectors (n, q+1) and joint covariances (n, q+1, q+1) of one block at designs X (n, d)."""
    d = Z.shape[1]
    cols = list(range(col0, d))
    n, r, m = X.shape[0], len(cols) + 1, Z.shape[0]
    S = s22(Z, beta, lamz, dadd)
    G = np.stack([rows(Z, beta, lamz, x, cols) for x in X])                   # (n, q+1, m)
    sol = np.linalg.solve(S, np.concatenate([w[:, None], G.reshape(n * r, m).T], axis=1))
    P = np.diag(np.concatenate([[s11], 2.0 * beta[cols] / lamz]))
    mean = G @ sol[:, 0]
    cov = P - np.einsum('tkm,mtl->tkl', G, sol[:, 1:].reshape(m, n, r))
    return mean, cov


def mean_var(Z, w, beta, lamz, dadd, s11, x):
    """Predictive mean and variance at one design x (complex allowed: no conjugation anywhere)."""
    S = s22(Z, beta, lamz, dadd)
    k = np.exp(-(((x[None, :] - Z) ** 2) @ beta)) / lamz
    return k @ np.linalg.solve(S, w), s11 - k @ np.linalg.solve(S, k)


def cross_cov(Z, beta, lamz, dadd, x, y):
    """Nugget-free predictive cross-covariance Sigma(x, y) = c(x, y) - k(x)^T S22^-1 k(y)."""
    S = s22(Z, beta, lamz, dadd)
    kx = np.exp(-(((x[None, :] - Z) ** 2) @ beta)) / lamz
    ky = np.exp(-(((y[None, :] - Z) ** 2) @ beta)) / lamz
    return np.exp(-np.sum(beta * (x - y) ** 2)) / lamz - kx @ np.linalg.solve(S, ky)


def blocks(Z, W, beta, lamz, dadd, s11, X, col0):
    """Every block b of (B, .) hyper-parameters -> mean (B, n, q+1), cov (B, n, q+1, q+1)."""
    out = [block(Z, W[b], beta[b], lamz[b], dadd[b], s11[b], X, col0) for b in range(beta.shape[0])]
    return np.stack([o[0] for o in out]), np.stack([o[1] for o in out])


def compact(cov):
    """(..., q+1, q+1) -> (..., 2q+1) = [v, Cov(f, d_k f), Var(d_k f)]."""
    dg = np.diagonal(cov, axis1=-2, axis2=-1)
    return np.concatenate([dg[..., :1], cov[..., 1:, 0], dg[..., 1:]], axis=-1)


def per_sample(mean, cov):
    """Per-(sample, point, PC) quantities from mean (S, N, pu, q+1), cov (S, N, pu, q+1, q+1), transformed scale."""
    return dict(mean=mean[..., 0], var=cov[..., 0, 0], grad=mean[..., 1:], grad_var=2.0 * cov[..., 1:, 0],
                grad_cov=cov[..., 1:, 1:])


def mixture(r):
    """Posterior mixture over the sample axis 0 of per_sample / linear results (law of total (co)variance)."""
    S = r['mean'].shape[0]
    m = r['mean'].mean(0)
    g = r['grad'].mean(0)
    dm = r['mean'] - m
    dg = r['grad'] - g
    return dict(mean=m, grad=g, var=r['var'].mean(0) + (dm * dm).mean(0),
                grad_var=r['grad_var'].mean(0) + (2.0 / S) * np.sum(dm[..., None] * dg, axis=0),
                grad_cov=r['grad_cov'].mean(0) + np.einsum('s...k,s...l->...kl', dg, dg) / S)


def linear(r, c):
    """The linear target sum_j c_j f_j of per_sample results (PC axis -1 of mean / var, -2 of grad, -3 of grad_cov):
    given a sample the PCs are independent."""
    c = np.asarray(c, dtype=np.float64)
    c2 = c * c
    return dict(mean=r['mean'] @ c, var=r['var'] @ c2, grad=np.einsum('...jk,j->...k', r['grad'], c),
                grad_var=np.einsum('...jk,j->...k', r['grad_var'], c2),
                grad_cov=np.einsum('...jkl,j->...kl', r['grad_cov'], c2))


def field(r, coef, option):
    """Native-output Jacobians dy_c/dt (transformed scale) for coef (pu, n_O) = K_O diag(sd_O), and the marginal sd of
    every entry: option 'samples' -> (S, N, n_O, q); 'mean' -> (N, n_O, q), the mixture sd."""
    gv = np.diagonal(r['grad_cov'], axis1=-2, axis2=-1)                      # (S, N, pu, q)
    J = np.einsum('snjk,jc->snck', r['grad'], coef)
    V = np.einsum('snjk,jc->snck', gv, coef * coef)
    if option == 'samples':
        return J, np.sqrt(np.maximum(V, 0.0))
    Jm = J.mean(0)
    dJ = J - Jm
    return Jm, np.sqrt(np.maximum(V.mean(0) + (dJ * dJ).mean(0), 0.0))
