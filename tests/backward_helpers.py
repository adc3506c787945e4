"""Scaled residuals (backward errors) of the FP64 evaluator, its solves and the predictive moments.

A forward-error bar against a plain FP64 solve only holds while S22 is well conditioned; at the conditioning real
posteriors reach (nuggets of 1e-6 .. 1e-10 against a nearly rank-one correlation, cond(S22) up to ~5e12) two correct
FP64 factors already differ in the 4th to 7th digit.  The measures below are the ones LAPACK's own test suite uses for
Cholesky: residuals scaled by what a backward-stable algorithm leaves, O(m eps) whatever the conditioning.  Every
function returns max |residual| / bar per block (a (B,) tensor); a value <= 1 passes.  eps = 2^-52.

  factor      |C - L L^T| / (eps (m max|C| + E_pf + T))
  solve       |L y - b| / (eps (m max|L| max|y| + E_pf(b) + T))    u (b = w), V rows (b = S21), xval rows (b = e_i)
  inverse     |L_jj M_j - I| / (32 eps max(|L_jj| |M_j|))            every 32x32 diagonal block and its stored inverse
  consistency device value against the same expression formed from the device's own L, u, V: bar 4 m eps times the sum
              of the absolute values of the terms

E_pf = max_ij 8 (1 + |x~_i|^2 + |x~_j|^2) |C_ij|, x~ = sqrt(beta) o x, is the bound of DESIGN.md section 4 on the error of
the covariance entries the kernels form as a rank-(d+2) product on the tensor cores (the diagonal of S22 is set exactly
and is left out).  C itself is built from coordinate differences.

T is the term of the inverse-based panel solve (DESIGN.md section 2): the kernels solve the 32 columns of panel j for
the rows below its diagonal block (and for every prediction / cross-validation row) as X = P M_j^T with the stored
inverse M_j instead of substituting.  With |L_jj M_j - I| <= 32 eps |L_jj| |M_j| and the rounding of the product, the
residual of such a row is at most 64 eps |x| (|L_jj| |M_j| |L_jj|)^T: entrywise, zero in the diagonal blocks and for the
substitution solve of u.  It grows with cond(L_jj) and is what keeps the bars from holding only at large m.

The residuals are formed in FP64 with batched torch matmuls, on whatever device the tensors live on (LAPACK's practice:
the bar absorbs the residual's own rounding)."""
import torch

EPS = 2.0 ** -52
NB = 32                      # panel width of the factorisation (csrc/ggp_common.cuh)


# --------------------------------------------------------------------------------------------------------------------
# packed factor layout (csrc/ggp_common.cuh)
# --------------------------------------------------------------------------------------------------------------------
def round_up32(m):
    return (m + 31) & ~31


def panel_off(kb, Mp):
    return 32 * (kb * Mp - 16 * kb * (kb - 1))


def minv_off(Mp):
    return panel_off(Mp // 32, Mp)


def packed_blocks(factor, m):
    """Diagonal blocks L_jj and their stored inverses M_j, read from the packed workspace (B, >= minv_off + 1024 nP):
    two (B, nP, 32, 32) tensors.  L[r][32kb + 8ks + c] lives at panel_off(kb) + ks (Mp - 32kb) 8 + (r - 32kb) 8 + c,
    M_j at minv_off(Mp) + 1024 j, row-major."""
    Mp = round_up32(m)
    nP = Mp // NB
    dev = factor.device
    j = torch.arange(nP, device=dev)[:, None, None]
    r = torch.arange(NB, device=dev)[None, :, None]
    c = torch.arange(NB, device=dev)[None, None, :]
    poff = 32 * (j * Mp - 16 * j * (j - 1))
    idx_l = poff + (c // 8) * (Mp - 32 * j) * 8 + r * 8 + c % 8
    idx_m = minv_off(Mp) + 1024 * j + 32 * r + c
    B = factor.shape[0]
    Ld = factor[:, idx_l.reshape(-1)].reshape(B, nP, NB, NB)
    M = factor[:, idx_m.reshape(-1)].reshape(B, nP, NB, NB)
    return Ld, M


def diag_blocks(L):
    """Diagonal blocks of dense factors L (B, m, m), padded with the identity to (B, nP, 32, 32)."""
    B, m, _ = L.shape
    Mp = round_up32(m)
    Lp = torch.eye(Mp, dtype=torch.float64, device=L.device).repeat(B, 1, 1)
    Lp[:, :m, :m] = L
    nP = Mp // NB
    return torch.stack([Lp[:, NB * j:NB * j + NB, NB * j:NB * j + NB] for j in range(nP)], dim=1)


def padded_identity_mask(m, device):
    """(nP, 32, 32) bool: entries of the diagonal blocks that lie in a padded row or column (index >= m)."""
    Mp = round_up32(m)
    g = torch.arange(Mp, device=device).reshape(Mp // NB, NB)
    return (g[:, :, None] >= m) | (g[:, None, :] >= m)


# --------------------------------------------------------------------------------------------------------------------
# references from coordinate differences
# --------------------------------------------------------------------------------------------------------------------
def sqdist(A, Bm, beta):
    """sum_k beta_k (a_k - b_k)^2: A (m, d), Bm (n, d), beta (B, d) -> (B, m, n)."""
    D = torch.zeros((beta.shape[0], A.shape[0], Bm.shape[0]), dtype=torch.float64, device=A.device)
    for k in range(A.shape[1]):
        D += beta[:, k, None, None] * ((A[:, None, k] - Bm[None, :, k]) ** 2)[None]
    return D


def cross_cov(A, Bm, beta, lamz):
    return torch.exp(-sqdist(A, Bm, beta)) / lamz[:, None, None]


def dense_cov(X, beta, lamz, dadd):
    C = cross_cov(X, X, beta, lamz)
    C.diagonal(dim1=-2, dim2=-1).copy_((1.0 / lamz + dadd)[:, None].expand(-1, X.shape[0]))
    return C


def pf_bound(A, Bm, beta, C, self_cov=False):
    """E_pf / eps per block: max_ij 8 (1 + |x~_i|^2 + |x~_j|^2) |C_ij| (off the diagonal when self_cov)."""
    na = (A ** 2) @ beta.T                        # (m, B)
    nb = (Bm ** 2) @ beta.T
    E = 8.0 * (1.0 + na.T[:, :, None] + nb.T[:, None, :]) * C.abs()
    if self_cov:
        E.diagonal(dim1=-2, dim2=-1).zero_()
    return E.amax(dim=(-2, -1))


# --------------------------------------------------------------------------------------------------------------------
# ratios
# --------------------------------------------------------------------------------------------------------------------
def _amax(t):
    return t.abs().flatten(1).amax(1)


def trsm_term(Y, Ld, M):
    """T / eps of rows solved panel by panel with the inverted diagonal blocks: Y (B, n, m) rows, Ld and M (B, nP, 32, 32)
    -> (B, n, m), 64 (|y_j| (|L_jj| |M_j| |L_jj|)^T) in the 32 columns of panel j."""
    B, n, m = Y.shape
    nP = Ld.shape[1]
    Yp = torch.zeros((B, n, 32 * nP), dtype=torch.float64, device=Y.device)
    Yp[:, :, :m] = Y.abs()
    G = Ld.abs() @ M.abs() @ Ld.abs()
    T = torch.einsum('bnpk,bpck->bnpc', Yp.reshape(B, n, nP, NB), G)
    return 64.0 * T.reshape(B, n, 32 * nP)[:, :, :m]


def factor_trsm_term(L, Ld, M):
    """T / eps of the factor, (B, m, m) symmetric: trsm_term of the rows of L below each diagonal block."""
    m = L.shape[-1]
    T = trsm_term(L, Ld, M)
    i = torch.arange(m, device=L.device)
    T = T * (i[:, None] >= NB * (i[None, :] // NB + 1))
    return T + T.transpose(-1, -2)


def factor_ratio(C, L, E_pf=None, T=None):
    """|C - L L^T| / (eps (m max|C| + E_pf + T)); E_pf in units of eps (pf_bound), None for a given matrix; T
    (factor_trsm_term) entrywise."""
    m = C.shape[-1]
    bar = m * _amax(C)
    if E_pf is not None:
        bar = bar + E_pf
    bar = bar[:, None, None] if T is None else bar[:, None, None] + T
    return _amax(torch.baddbmm(C, L, L.transpose(-1, -2), alpha=-1.0) / (EPS * bar))


def solve_ratio(L, Y, Bm, E_pf=None, T=None):
    """|L Y - B| / (eps (m max|L| max|Y| + E_pf + T)): L (B, m, m), Y and Bm (B, m, k) (columns = right-hand sides), T
    (trsm_term of the rows Y^T, transposed) entrywise."""
    m = L.shape[-1]
    bar = m * _amax(L) * _amax(Y)
    if E_pf is not None:
        bar = bar + E_pf
    bar = bar[:, None, None] if T is None else bar[:, None, None] + T
    return _amax(torch.baddbmm(Bm, L, Y, alpha=-1.0) / (EPS * bar))


def inverse_ratio(Ld, M):
    """max over the panels of |L_jj M_j - I| / (32 eps max(|L_jj| |M_j|)); Ld, M (B, nP, 32, 32)."""
    eye = torch.eye(NB, dtype=torch.float64, device=Ld.device)
    R = (Ld @ M - eye).abs().amax(dim=(-2, -1))
    bar = NB * EPS * (Ld.abs() @ M.abs()).amax(dim=(-2, -1))
    return (R / bar).amax(1)


def ll_ratio(ll, L, u):
    """ll against -sum log L_ii - u.u / 2; L (B, m, m), u (B, m)."""
    m = L.shape[-1]
    lg = torch.log(L.diagonal(dim1=-2, dim2=-1))
    q = 0.5 * (u * u).sum(1)
    ref = -lg.sum(1) - q
    return (ll - ref).abs() / (4 * m * EPS * (lg.abs().sum(1) + q))


def mean_ratio(mean, V, u):
    """mean (B, n) against V u; V (B, n, m), u (B, m)."""
    m = V.shape[-1]
    ref = (V @ u[:, :, None])[..., 0]
    bar = 4 * m * EPS * (V.abs() @ u.abs()[:, :, None])[..., 0]
    return ((mean - ref).abs() / bar).amax(1)


def var_ratio(var, V, s11):
    """var (B, n) against s11 - sum V^2."""
    m = V.shape[-1]
    sq = (V * V).sum(-1)
    return ((var - (s11[:, None] - sq)).abs() / (4 * m * EPS * (s11[:, None].abs() + sq))).amax(1)


def cov_ratio(Sig, S11, V):
    """Sig (B, n, n) against S11 - V V^T."""
    m = V.shape[-1]
    ref = torch.baddbmm(S11, V, V.transpose(-1, -2), alpha=-1.0)
    bar = 4 * m * EPS * (S11.abs() + V.abs() @ V.abs().transpose(-1, -2))
    return ((Sig - ref).abs() / bar).flatten(1).amax(1)
