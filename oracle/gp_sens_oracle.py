"""CPU oracle for the closed-form GP sensitivity indices (csrc/ggp_gp_sens.cu).  TEST INFRASTRUCTURE ONLY.

The function analysed is a weighted sum of product squared-exponential kernels on [0,1]^q with independent uniform inputs,
  f(x) = sum_n a_n prod_k exp(-beta_nk (x_k - z_nk)^2),
for which every Sobol' integral has a closed form in erf and exp:
  I1(b, z)         = int_0^1 e^{-b(x-z)^2} dx
  I2(b, z; b', z') = int_0^1 e^{-b(x-z)^2 - b'(x-z')^2} dx
  M(u) = E_{x_u}[(E_{x_~u} f)^2] = sum_{n,n'} a_n a_n' prod_{k in u} I2_k(n,n') prod_{k not in u} I1_k(n) I1_k(n')
  E0 = sum_n a_n prod_k I1_k(n),  V = M(all) - E0^2,  S_k = (M({k}) - E0^2) / V,  T_k = 1 - (M(all\\k) - E0^2) / V.
Both integrals are exactly 1 at beta = 0.  Products over all inputs but one are formed from prefix and suffix products,
never by dividing.  quad_moments() recomputes M(u) and the main-effect curves by tensor Gauss-Legendre quadrature, as an
independent check of the closed forms for q <= 3.
"""
import numpy as np
from scipy import special


def I1(b, z):
    """int_0^1 exp(-b (x - z)^2) dx, elementwise; exactly 1 where b == 0."""
    b, z = np.broadcast_arrays(np.asarray(b, dtype=np.float64), np.asarray(z, dtype=np.float64))
    out = np.ones(b.shape)
    nz = b != 0
    sb = np.sqrt(b[nz])
    out[nz] = 0.5 * np.sqrt(np.pi / b[nz]) * (special.erf(sb * (1.0 - z[nz])) + special.erf(sb * z[nz]))
    return out


def I2(b, z, b2, z2):
    """int_0^1 exp(-b (x - z)^2 - b2 (x - z2)^2) dx, elementwise; exactly 1 where b == b2 == 0."""
    b, z, b2, z2 = np.broadcast_arrays(*(np.asarray(v, dtype=np.float64) for v in (b, z, b2, z2)))
    out = np.ones(b.shape)
    B = b + b2
    nz = B != 0
    Bn = B[nz]
    c = (b[nz] * z[nz] + b2[nz] * z2[nz]) / Bn
    sB = np.sqrt(Bn)
    out[nz] = (np.exp(-b[nz] * b2[nz] * np.square(z[nz] - z2[nz]) / Bn) * 0.5 * np.sqrt(np.pi / Bn) *
               (special.erf(sB * (1.0 - c)) + special.erf(sB * c)))
    return out


def _excl_prod(x):
    """prod over the last axis of x with entry k left out, for every k (prefix x suffix products, no division)."""
    q = x.shape[-1]
    pre = np.ones(x.shape)
    suf = np.ones(x.shape)
    for k in range(1, q):
        pre[..., k] = pre[..., k - 1] * x[..., k - 1]
        suf[..., q - 1 - k] = suf[..., q - k] * x[..., q - k]
    return pre * suf


def moments(a, beta, Z):
    """Closed-form moments of f = sum_n a_n phi_n.  a (N,), beta (N, q) per term, Z (N, q) centres.
    Returns dict(E0, Mall, M1 (q,) = M({k}), Mt (q,) = M(all\\k), V, first (q,), total (q,))."""
    a = np.asarray(a, dtype=np.float64)
    beta = np.asarray(beta, dtype=np.float64)
    Z = np.asarray(Z, dtype=np.float64)
    i1 = I1(beta, Z)                                                        # (N, q)
    A = i1[:, None, :] * i1[None, :, :]                                     # (N, N, q)
    B = I2(beta[:, None, :], Z[:, None, :], beta[None, :, :], Z[None, :, :])
    w = a[:, None] * a[None, :]
    E0 = float(np.sum(a * np.prod(i1, axis=1)))
    Mall = float(np.sum(w * np.prod(B, axis=2)))
    M1 = np.einsum('nl,nlk->k', w, _excl_prod(A) * B)
    Mt = np.einsum('nl,nlk->k', w, _excl_prod(B) * A)
    return finish(E0, Mall, M1, Mt, beta_zero=np.all(beta == 0, axis=0))


def finish(E0, Mall, M1, Mt, beta_zero=None):
    """Indices from the moments.  An input with beta = 0 in every term does not enter f: its indices are exactly 0."""
    V = Mall - E0 * E0
    first = (M1 - E0 * E0) / V
    total = 1.0 - (Mt - E0 * E0) / V
    if beta_zero is not None:
        first = np.where(beta_zero, 0.0, first)
        total = np.where(beta_zero, 0.0, total)
    return dict(E0=E0, Mall=Mall, M1=np.asarray(M1), Mt=np.asarray(Mt), V=V, first=first, total=total)


def main_effects(a, beta, Z, grid):
    """E[f | x_k = g] for every input k and grid value g -> (q, ngrid)."""
    a = np.asarray(a, dtype=np.float64)
    beta = np.asarray(beta, dtype=np.float64)
    Z = np.asarray(Z, dtype=np.float64)
    ex = _excl_prod(I1(beta, Z))                                            # (N, q)
    g = np.asarray(grid, dtype=np.float64)
    ker = np.exp(-beta[:, :, None] * np.square(g[None, None, :] - Z[:, :, None]))     # (N, q, ngrid)
    return np.einsum('n,nk,nkg->kg', a, ex, ker)


def block_terms(Zin, beta_blocks, a_blocks, option):
    """The functions of one call: option 'samples' -> one (a, beta, Z) per (sample, PC) block b = s * pu + j; 'mean' ->
    one per PC j over the terms n = (s, i) with weights a / S.  beta_blocks (S, pu, q), a_blocks (S, pu, m)."""
    S, pu, m = a_blocks.shape
    if option == 'samples':
        return [(a_blocks[s, j], np.broadcast_to(beta_blocks[s, j], Zin.shape), Zin) for s in range(S) for j in range(pu)]
    out = []
    for j in range(pu):
        a = (a_blocks[:, j, :] / S).reshape(-1)
        beta = np.repeat(beta_blocks[:, j, :], m, axis=0)
        out.append((a, beta, np.tile(Zin, (S, 1))))
    return out


def quad_moments(a, beta, Z, nodes=60, grid=None):
    """Tensor Gauss-Legendre quadrature (q <= 3) of E0, M(u) for u = {k} and all\\k and all, and of the main-effect
    curves on `grid` (for those the pinned input is set to the grid value and the others integrated)."""
    a = np.asarray(a, dtype=np.float64)
    beta = np.asarray(beta, dtype=np.float64)
    Z = np.asarray(Z, dtype=np.float64)
    q = Z.shape[1]
    assert q <= 3
    x, wq = np.polynomial.legendre.leggauss(nodes)
    x = 0.5 * (x + 1.0)
    wq = 0.5 * wq
    # factor of every term along every axis: phi[n, k, node]
    phi = np.exp(-beta[:, :, None] * np.square(x[None, None, :] - Z[:, :, None]))

    def cond_mean(u):
        """E_{x_~u} f as an array over the nodes of the inputs in u (sorted)."""
        f = a.copy().reshape(-1, *([1] * len(u)))
        for k in range(q):
            if k in u:
                pos = u.index(k)
                shape = [1] * len(u)
                shape[pos] = nodes
                f = f * phi[:, k, :].reshape(-1, *shape)
            else:
                f = f * (phi[:, k, :] @ wq).reshape(-1, *([1] * len(u)))
        return f.sum(axis=0)

    def second(u):
        g = cond_mean(u)
        W = np.ones([nodes] * len(u))
        for pos in range(len(u)):
            shape = [1] * len(u)
            shape[pos] = nodes
            W = W * wq.reshape(shape)
        return float(np.sum(W * g * g))

    E0 = float(cond_mean([]))
    M1 = np.array([second([k]) for k in range(q)])
    Mt = np.array([second([r for r in range(q) if r != k]) for k in range(q)])
    Mall = second(list(range(q)))
    out = finish(E0, Mall, M1, Mt)
    if grid is not None:
        g = np.asarray(grid, dtype=np.float64)
        me = np.zeros((q, g.size))
        for k in range(q):
            f = a[:, None] * np.exp(-beta[:, k, None] * np.square(g[None, :] - Z[:, k, None]))
            for r in range(q):
                if r != k:
                    f = f * (phi[:, r, :] @ wq)[:, None]
            me[k] = f.sum(axis=0)
        out['main_effect'] = me
    return out

