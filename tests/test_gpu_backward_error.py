"""GPU: the FP64 evaluator, its solves and the predictive moments by backward error (tests/backward_helpers.py) across the
conditioning posteriors reach.

Every consumer reads the packed factor of csrc/ggp_chol.cuh: L, and the inverted 32x32 diagonal blocks M_j.  The
forward-error tests of the suite (L to 1e-9, u to 1e-8 of a plain FP64 solve) only hold while S22 is well conditioned;
the scaled residuals here hold one fixed bar from cond(S22) ~ 1 to ~1e12 and fail on an output wrong by 1e-12 relative
in one place (tests/test_backward_error_cpu.py).

Inputs.  Constructed: m in {33, 257, 512, 1000}, d = 9 ([dummy 0.5, synthetic.design(m, 8)]), beta scale in
{3, 0.3, 0.03, 0.003}, nugget 1e-2 .. 1e-10 with lamz = 1; the m = 512 design with 16 pairs of rows 1e-7 apart; the cfg5
shape (m = 4096, d = 17) at the two most ill-conditioned blocks of the sweep.  Posterior: every (draw, PC) block of
tests/golden/posterior_cfg1/2/3.npz.

Checks.  (1) loglik_batched: info, the factor, u and diagonal-block inverse ratios, ll against -sum log L_ii - u.u/2, and
bit-identical results under GGP_CLUSTER = 1, 4 (and 16 at m = 4096); the padded rows and columns of the last diagonal
block, in L and in M_j, are exactly the identity: the kernel factors the padding as an identity block (pivot 1,
r = 1, nothing coupled to the real rows), so the inverse of that block is the identity too.  (2) Predictor.predict: V
ratio, zeros beyond m, mean against V u, var against s11 - |V|^2 and var >= -4 m eps s11, at the training rows, the rows
moved by 1e-7 and 64 LHS points.  (3) pred_cov against S11 - V V^T, exactly symmetric.  (4) xval_solve: z_i ratios at
rows {0, 31, 32, m/2, m-1}, alpha = z.u and p = |z|^2.  (5) chol_draw of item 3's matrix at the moved rows, L read
column by column (B = n copies, z_b = e_b).  (6) positive-definiteness decisions at 16 exactly duplicated rows."""
import numpy as np
import pytest

import backward_helpers as bh
from test_backward_error_cpu import NUGGETS, SCALES, design, hypers, prediction_designs
from test_gpu_posterior_draws import _fixture, _samples
from test_gpu_predict import _blocks

pytestmark = pytest.mark.gpu

EPS = bh.EPS


def _report(item, r):
    print('%s: largest ratio %.3g' % (item, r))


def _dev(a):
    import torch
    return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device='cuda')


def _evaluate(monkeypatch, X, W, beta, lamz, dadd, schedules):
    """loglik_batched under every schedule: the same info and loglik everywhere, and the same factor and u bit for bit in
    every block that factors.  Returns the first schedule's output."""
    import torch
    from gladsgp_b200 import _lib, ops
    lib = _lib.load()
    m = X.shape[0]
    n_factor = lib.ggp_factor_doubles(m) - lib.ggp_padded_m(m) - 64       # panels + inverted blocks (no cluster scratch)
    res = []
    for g in schedules:
        monkeypatch.setenv('GGP_CLUSTER', g)
        res.append(ops.loglik_batched(X, W, beta, lamz, dadd, want_factor=True, want_u=True))
    monkeypatch.delenv('GGP_CLUSTER')
    a = res[0]
    ok = a['info'] == 0
    for b in res[1:]:
        assert torch.equal(a['info'], b['info'])
        assert torch.equal(a['loglik'], b['loglik'])
        assert torch.equal(a['factor'][ok, :n_factor], b['factor'][ok, :n_factor])
        assert torch.equal(a['u'][ok], b['u'][ok])
    return a


def _check_evaluator(X, W, beta, lamz, dadd, out, idx, chunk):
    """Ratios of item 1 over the blocks idx (all of which factored).  -> dict of maxima."""
    import torch
    from gladsgp_b200 import ops
    m = X.shape[0]
    Xd = _dev(X)
    mask = bh.padded_identity_mask(m, 'cuda')
    eye = torch.eye(32, dtype=torch.float64, device='cuda').expand_as(mask)
    r = dict(factor=0.0, u=0.0, inverse=0.0, ll=0.0)
    idx = torch.as_tensor(np.asarray(idx), device='cuda')
    for c0 in range(0, idx.numel(), chunk):
        ib = idx[c0:c0 + chunk]
        F = out['factor'][ib]
        L = ops.factor_unpack(F, m)
        Ld, M = bh.packed_blocks(F, m)
        assert torch.equal(Ld[:, mask], eye[mask].expand(ib.numel(), -1))
        assert torch.equal(M[:, mask], eye[mask].expand(ib.numel(), -1))
        bt = _dev(beta)[ib]
        C = bh.dense_cov(Xd, bt, _dev(lamz)[ib], _dev(dadd)[ib])
        u = out['u'][ib]
        assert not u[:, m:].any().item()
        u = u[:, :m]
        r['factor'] = max(r['factor'], float(bh.factor_ratio(C, L, bh.pf_bound(Xd, Xd, bt, C, self_cov=True),
                                                             bh.factor_trsm_term(L, Ld, M)).max()))
        del C
        r['u'] = max(r['u'], float(bh.solve_ratio(L, u[:, :, None], _dev(W)[ib][:, :, None]).max()))
        r['inverse'] = max(r['inverse'], float(bh.inverse_ratio(Ld, M).max()))
        r['ll'] = max(r['ll'], float(bh.ll_ratio(out['loglik'][ib], L, u).max()))
    for k, v in r.items():
        assert v <= 1.0, (k, v)
    return r


def _check_prediction(X, Xp, W, beta, lamz, dadd, s11, rows):
    """Items 2-4 on one Predictor.  -> (dict of maxima, pred_cov output)."""
    import torch
    from gladsgp_b200 import ops
    m, n = X.shape[0], Xp.shape[0]
    P = ops.Predictor(X, W, beta, lamz, dadd, s11)
    assert not P.info.any().item()
    L = ops.factor_unpack(P.factor, m)
    Ld, M = bh.packed_blocks(P.factor, m)
    u = P.u[:, :m]
    Xd, Xpd, bt, lz, s1 = _dev(X), _dev(Xp), _dev(beta), _dev(lamz), _dev(s11)
    r = {}
    mean, var, V = P.predict(Xp, want_V=True)
    assert not V[:, :, m:].any().item()
    Vm = V[:, :, :m]
    S21 = bh.cross_cov(Xd, Xpd, bt, lz)
    r['V'] = float(bh.solve_ratio(L, Vm.transpose(1, 2), S21, bh.pf_bound(Xd, Xpd, bt, S21),
                                  bh.trsm_term(Vm, Ld, M).transpose(1, 2)).max())
    del S21
    r['mean'] = float(bh.mean_ratio(mean, Vm, u).max())
    r['var'] = float(bh.var_ratio(var, Vm, s1).max())
    r['var floor'] = float((-var / (4 * m * EPS * s1[:, None])).max())
    Sig = P.pred_cov(Xp, V)
    assert torch.equal(Sig, Sig.transpose(1, 2))
    S11 = bh.cross_cov(Xpd, Xpd, bt, lz)
    S11.diagonal(dim1=-2, dim2=-1).copy_(s1[:, None].expand(-1, n))
    r['pred_cov'] = float(bh.cov_ratio(Sig, S11, Vm).max())
    del S11, V, Vm
    alpha, p, Z = P.xval_solve(rows, want_Z=True)
    assert not Z[:, :, m:].any().item()
    Zm = Z[:, :, :m]
    E = torch.zeros((1, m, len(rows)), dtype=torch.float64, device='cuda')
    E[0, torch.as_tensor(rows, device='cuda'), torch.arange(len(rows), device='cuda')] = 1.0
    r['Z'] = float(bh.solve_ratio(L, Zm.transpose(1, 2), E.expand(Zm.shape[0], -1, -1), None,
                                  bh.trsm_term(Zm, Ld, M).transpose(1, 2)).max())
    r['alpha'] = float(bh.mean_ratio(alpha, Zm, u).max())
    zz = (Zm * Zm).sum(-1)
    r['p'] = float(((p - zz).abs() / (4 * m * EPS * zz)).max())
    for k, v in r.items():
        assert v <= 1.0, (k, v)
    return r, Sig


def _check_chol_draw(Sig):
    """chol_draw of each matrix of Sig (k, n, n): B = n copies with z_b = e_b give the columns of L."""
    import torch
    from gladsgp_b200 import ops
    worst = 0.0
    n = Sig.shape[-1]
    eye = torch.eye(n, dtype=torch.float64, device='cuda')
    for S in Sig:
        S = S.contiguous()
        out, info = ops.chol_draw(S.expand(n, n, n).contiguous(), eye)
        assert not info.any().item()
        L = out.T.contiguous()[None]
        assert torch.equal(L, L.tril())
        Ld = bh.diag_blocks(L)
        M = torch.linalg.solve_triangular(Ld, torch.eye(32, dtype=torch.float64, device='cuda').expand_as(Ld),
                                          upper=False)
        worst = max(worst, float(bh.factor_ratio(S[None], L, None, bh.factor_trsm_term(L, Ld, M))))
    assert worst <= 1.0, worst
    return worst


def _rows(m):
    return sorted({0, 31, 32, m // 2, m - 1} & set(range(m)))


# --------------------------------------------------------------------------------------------------------------------
# constructed sweep
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('m,dup', [(33, 0), (257, 0), (512, 0), (1000, 0), (512, 16)])
def test_constructed_sweep(cuda, monkeypatch, m, dup):
    """Every (beta scale, nugget) block of the sweep at one design: items 1-5."""
    X = design(m, dup_pairs=dup)
    beta, lamz, dadd, s11 = hypers(X.shape[1], SCALES, NUGGETS)
    W = np.random.default_rng(m + dup).standard_normal((beta.shape[0], m))
    out = _evaluate(monkeypatch, X, W, beta, lamz, dadd, ['1', '4'])
    assert not out['info'].any().item()
    tag = 'sweep m=%d%s' % (m, ' 16 pairs 1e-7 apart' if dup else '')
    r = _check_evaluator(X, W, beta, lamz, dadd, out, np.arange(beta.shape[0]), 20)
    Xp = prediction_designs(X, m)
    rp, Sig = _check_prediction(X, Xp, W, beta, lamz, dadd, s11, _rows(m))
    # item 5: the joint covariance at the moved training rows, nugget 1e-8, beta scales 3, 0.03, 0.003
    n = min(m, 256)
    sel = [SCALES.index(s) * len(NUGGETS) + NUGGETS.index(1e-8) for s in (3.0, 0.03, 0.003)]
    r['chol_draw'] = _check_chol_draw(Sig[sel][:, m:m + n, m:m + n])
    r.update(rp)
    for k, v in sorted(r.items()):
        _report('%s: %s' % (tag, k), v)


def test_cfg5_shape_at_the_worst_blocks(cuda, monkeypatch):
    """m = 4096, d = 17, beta scale 0.003 and 0.03 at nugget 1e-10 (cond(S22) ~ 1e12), schedules 1, 4 and 16."""
    m = 4096
    X = design(m, q=16)
    beta, lamz, dadd, s11 = hypers(X.shape[1], [0.003, 0.03], [1e-10])
    W = np.random.default_rng(4096).standard_normal((2, m))
    out = _evaluate(monkeypatch, X, W, beta, lamz, dadd, ['1', '4', '16'])
    assert not out['info'].any().item()
    r = _check_evaluator(X, W, beta, lamz, dadd, out, [0, 1], 1)
    rp, _ = _check_prediction(X, prediction_designs(X, 64), W, beta, lamz, dadd, s11, _rows(m))
    r.update(rp)
    for k, v in sorted(r.items()):
        _report('cfg5 shape: %s' % k, v)


def test_positive_definiteness_decisions(cuda, monkeypatch):
    """m = 257 with 16 exactly duplicated rows: lambda_min(C) = delta, swept from 1e-4 to 1e-14 (lamz = 1).  Above
    delta = 4 eps (m + 16 max|x~|^2) / lamz every block must factor with a finite ll and the bars of item 1 (a false -inf
    would make the sampler reject a valid proposal); below it either outcome is allowed, an accepted factor must still
    meet the bars, and every schedule reports the same info."""
    m = 257
    X = design(m, dup_pairs=16, exact=True)
    deltas = [10.0 ** -k for k in range(4, 15)]
    beta, lamz, dadd, _ = hypers(X.shape[1], SCALES, deltas)
    W = np.random.default_rng(257).standard_normal((beta.shape[0], m))
    out = _evaluate(monkeypatch, X, W, beta, lamz, dadd, ['1', '2', '4', '8'])
    info = out['info'].cpu().numpy()
    ll = out['loglik'].cpu().numpy()
    xn = ((X ** 2) @ beta.T).max(0)
    need = dadd > 4 * EPS * (m + 16 * xn) / lamz
    assert need.sum() >= 30
    bad = np.nonzero(need & ((info != 0) | ~np.isfinite(ll)))[0]
    assert bad.size == 0, [(beta[b, 0], dadd[b], info[b]) for b in bad]
    acc = np.nonzero(info == 0)[0]
    assert np.all(np.isfinite(ll[acc]))
    assert np.all(np.isneginf(ll[info != 0]))
    r = _check_evaluator(X, W, beta, lamz, dadd, out, acc, 44)
    print('  %d of %d blocks factored (%d required); smallest delta factored %.0e' %
          (acc.size, info.size, need.sum(), dadd[acc].min()))
    for k, v in sorted(r.items()):
        _report('positive definiteness m=257: %s' % k, v)


# --------------------------------------------------------------------------------------------------------------------
# posterior fixtures
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('cfg', ['cfg1', 'cfg2', 'cfg3'])
def test_posterior_blocks(cuda, monkeypatch, cfg):
    """Every (draw, PC) block: item 1 under both schedules, items 2-4 at the training rows, the rows moved by 1e-7 and
    64 LHS points, in groups of 64 blocks."""
    _, pr, d, pu = _fixture(cfg)
    num = pr['num']
    m = num.m
    beta, lamz, dadd, s11, W = _blocks(num, _samples(cfg))
    X = np.asarray(num.zt, dtype=np.float64)
    out = _evaluate(monkeypatch, X, W, beta, lamz, dadd, ['1', '4'])
    assert not out['info'].any().item()
    B = beta.shape[0]
    r = _check_evaluator(X, W, beta, lamz, dadd, out, np.arange(B), 64)
    Xp = prediction_designs(X, m)
    for b0 in range(0, B, 64):
        sl = slice(b0, min(B, b0 + 64))
        rp, _ = _check_prediction(X, Xp, W[sl], beta[sl], lamz[sl], dadd[sl], s11[sl], _rows(m))
        for k, v in rp.items():
            r[k] = max(r.get(k, 0.0), v)
    for k, v in sorted(r.items()):
        _report('posterior %s (%d blocks, smallest nugget %.2g): %s' % (cfg, B, dadd.min(), k), v)
