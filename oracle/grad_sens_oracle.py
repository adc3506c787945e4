"""CPU oracle for the closed-form gradient outer-product matrices (csrc/ggp_grad_sens.cu).  TEST INFRASTRUCTURE ONLY.

The function analysed is g(x) = sum_n a_n phi_n(x), phi_n(x) = prod_k exp(-beta_nk (x_k - z_nk)^2), on [0,1]^q with
independent uniform inputs, where pairs of terms may carry an extra weight Omega_{pc(n) pc(n')}:
  C = E[grad g grad g^T] = sum_{n,n'} a_n a_n' Omega_{pc(n) pc(n')} int grad phi_n grad phi_n'^T dx.
Per input, with phi = exp(-b (x-z)^2), phi' = exp(-b' (x-z')^2), B = b + b', c = (b z + b' z') / B, e = exp(-b b' (z-z')^2/B):
  I2 = int phi phi' = e It,  It = 1/2 sqrt(pi/B) [erf(sqrt(B)(1-c)) + erf(sqrt(B) c)]
  G(n,n') = int d phi phi' = -2 b e (m1 + (c-z) It),    H = int d phi d phi' = 4 b b' e (m2 + m1 (2c-z-z') + (c-z)(c-z') It)
  m1 = (E0 - E1) / 2B,  m2 = It / 2B - ((1-c) E1 + c E0) / 2B,  E0 = e^{-B c^2},  E1 = e^{-B (1-c)^2}.
Then, over every ordered pair (n, n'):
  C_kl = sum a a' Omega G_k(n,n') G_l(n',n) prod_{r != k,l} I2_r,   C_kk = sum a a' Omega H_k prod_{r != k} I2_r.
This restates C the direct way: each input's integrals with their own factor e_r, the explicit products over the inputs
other than k and l, no ratio of integrals.  `A` is the same sums over absolute values: the scale of the rounding error.
quad_grad_outer() recomputes C by tensor Gauss-Legendre quadrature of the analytic gradient, for q <= 3.
"""
import numpy as np
from scipy import special


def integrals(b, z, b2, z2):
    """(I2, G(n,n'), G(n',n), H) elementwise for phi = exp(-b (x-z)^2), phi' = exp(-b2 (x-z2)^2) on [0, 1].
    I2 is exactly 1 and G, H exactly 0 where b == b2 == 0.  E0 - E1 is the larger exponential times expm1 of the
    exponent difference (no cancellation at small B)."""
    b, z, b2, z2 = np.broadcast_arrays(*(np.asarray(v, dtype=np.float64) for v in (b, z, b2, z2)))
    I2 = np.ones(b.shape)
    G12 = np.zeros(b.shape)
    G21 = np.zeros(b.shape)
    H = np.zeros(b.shape)
    nz = (b + b2) != 0
    b, z, b2, z2 = b[nz], z[nz], b2[nz], z2[nz]
    B = b + b2
    c = (b * z + b2 * z2) / B
    e = np.exp(-b * b2 * np.square(z - z2) / B)
    sB = np.sqrt(B)
    It = 0.5 * np.sqrt(np.pi / B) * (special.erf(sB * (1.0 - c)) + special.erf(sB * c))
    t = B * (1.0 - 2.0 * c)
    lo = t >= 0
    Ebig = np.exp(-B * np.where(lo, c * c, (1.0 - c) ** 2))
    em = np.expm1(-np.abs(t))
    Esmall = Ebig + Ebig * em
    E0 = np.where(lo, Ebig, Esmall)
    E1 = np.where(lo, Esmall, Ebig)
    m1 = np.where(lo, -Ebig, Ebig) * em / (2.0 * B)
    m2 = It / (2.0 * B) - ((1.0 - c) * E1 + c * E0) / (2.0 * B)
    I2[nz] = e * It
    G12[nz] = -2.0 * b * e * (m1 + (c - z) * It)
    G21[nz] = -2.0 * b2 * e * (m1 + (c - z2) * It)
    H[nz] = 4.0 * b * b2 * e * (m2 + m1 * (2.0 * c - z - z2) + (c - z) * (c - z2) * It)
    return I2, G12, G21, H


def grad_outer(a, beta, Z, pair_weight=None):
    """C and A (q, q) of g = sum_n a_n phi_n.  a (N,), beta (N, q), Z (N, q); pair_weight (N, N) multiplies the pair
    (n, n') (Omega_{pc(n) pc(n')}; default 1)."""
    a = np.asarray(a, dtype=np.float64)
    beta = np.asarray(beta, dtype=np.float64)
    Z = np.asarray(Z, dtype=np.float64)
    q = Z.shape[1]
    I2, G12, G21, H = integrals(beta[:, None, :], Z[:, None, :], beta[None, :, :], Z[None, :, :])     # (N, N, q)
    w = a[:, None] * a[None, :]
    if pair_weight is not None:
        w = w * np.asarray(pair_weight, dtype=np.float64)
    C = np.zeros((q, q))
    A = np.zeros((q, q))
    for k in range(q):
        for l in range(k, q):
            rest = np.ones(q, dtype=bool)
            rest[[k, l]] = False
            P = np.prod(I2[:, :, rest], axis=2)
            t = w * (H[:, :, k] if k == l else G12[:, :, k] * G21[:, :, l]) * P
            C[k, l] = C[l, k] = np.sum(t)
            A[k, l] = A[l, k] = np.sum(np.abs(t))
    return dict(C=C, A=A)


def block_terms(Zin, beta_blocks, a_blocks, mode, omega=None):
    """The functions of one call as (a, beta, Z, pair_weight) per function, in the device's order.  beta_blocks (S, pu, q),
    a_blocks (S, pu, m), weights as given (the caller scales them by 1/S in modes 1 and 3).
    mode 0: one per block (s, j); 1: one per PC j over (s, i); 2: one per sample s over (j, i), Omega; 3: one over (s, j, i)."""
    S, pu, m = a_blocks.shape
    q = Zin.shape[1]
    if mode == 0:
        return [(a_blocks[s, j], np.broadcast_to(beta_blocks[s, j], (m, q)), Zin, None) for s in range(S) for j in range(pu)]
    if mode == 1:
        return [(a_blocks[:, j, :].reshape(-1), np.repeat(beta_blocks[:, j, :], m, axis=0), np.tile(Zin, (S, 1)), None)
                for j in range(pu)]
    omega = np.asarray(omega, dtype=np.float64)
    if mode == 2:
        pc = np.repeat(np.arange(pu), m)
        return [(a_blocks[s].reshape(-1), np.repeat(beta_blocks[s], m, axis=0), np.tile(Zin, (pu, 1)),
                 omega[pc[:, None], pc[None, :]]) for s in range(S)]
    pc = np.tile(np.repeat(np.arange(pu), m), S)
    return [(a_blocks.reshape(-1), np.repeat(beta_blocks.reshape(S * pu, q), m, axis=0), np.tile(Zin, (S * pu, 1)),
             omega[pc[:, None], pc[None, :]])]


def gradient(a, beta, Z, x):
    """Analytic gradient of g at points x (n, q) -> (n, q)."""
    d = x[:, None, :] - Z[None, :, :]                                            # (n, N, q)
    phi = np.exp(-np.sum(beta[None] * d * d, axis=2))                            # (n, N)
    return np.einsum('n,pn,pnk->pk', a, phi, -2.0 * beta[None] * d)


def quad_grad_outer(a, beta, Z, pc=None, omega=None, nodes=40):
    """C by tensor Gauss-Legendre quadrature (q <= 3) of the analytic gradients: sum_{j,j'} Omega_jj' E[grad g_j grad g_j'^T]
    with g_j the terms of PC j (pc (N,) the PC of each term; default one PC, Omega = 1)."""
    a = np.asarray(a, dtype=np.float64)
    beta = np.asarray(beta, dtype=np.float64)
    Z = np.asarray(Z, dtype=np.float64)
    q = Z.shape[1]
    assert q <= 3
    x, wq = np.polynomial.legendre.leggauss(nodes)
    x, wq = 0.5 * (x + 1.0), 0.5 * wq
    X = np.stack(np.meshgrid(*([x] * q), indexing='ij'), axis=-1).reshape(-1, q)
    W = np.prod(np.stack(np.meshgrid(*([wq] * q), indexing='ij'), axis=-1).reshape(-1, q), axis=1)
    if pc is None:
        pc, omega = np.zeros(a.size, dtype=int), np.ones((1, 1))
    omega = np.asarray(omega, dtype=np.float64)
    grads = [gradient(a[pc == j], beta[pc == j], Z[pc == j], X) for j in range(omega.shape[0])]
    C = np.zeros((q, q))
    for j in range(omega.shape[0]):
        for j2 in range(omega.shape[0]):
            C += omega[j, j2] * np.einsum('p,pk,pl->kl', W, grads[j], grads[j2])
    return C
