"""GPU: PC-basis reconstruction and the fused predictive statistics across their template instantiations
(reconstruct_kernel: PUMAX 4/8/12/16/24/32 x vector / scalar stores; reconstruct_stats_kernel: PUMAX 4/8/12/16 x KQ 4/8)
against FP64 fields formed from the same float32 inputs.

Bounds.  A float32 field entry y = (sum_p w_p K_p) sd + mu is within F = (pu+2) eps32 (|sd| sum_p |w_p K_p| + |mu|) of
its exact value; z = y + sd noise adds eps32 |sd noise|.  Order statistics are 1-Lipschitz in the max norm, so a
quantile is within that bound plus two float32 ulp of the interpolation; the mean adds nsamp eps32 max|y| for the
sequential float32 sum over samples."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

EPS32 = float(np.finfo(np.float32).eps)
STATS_PU = [3, 8, 12, 16]
# (nsamp, q): the order-statistic position i0 = floor(q (nsamp - 1)) runs through 0..6 (KQ = 4 for i0 <= 2, KQ = 8 above);
# (41, 0.025) sits exactly on an order statistic; 722 and 723 samples at pu 16 and every case from 1000 samples at pu >= 9
# need more than the default 48 KB of shared memory (staged samples plus the kernel's static reduction buffer)
STATS_CASES = [((2, 0.3), 0), ((64, 0.01), 0), ((41, 0.025), 1), ((101, 0.025), 2), ((128, 0.025), 3), ((1000, 0.005), 4),
               ((3000, 0.002), 5), ((256, 0.025), 6), ((722, 0.009), 6), ((723, 0.009), 6)]


def _fields64(w, K, sd, mu, noise):
    """FP64 y (nsamp, npred, n_y), z = y + sd noise, and the per-entry formation bounds of y and z."""
    w64, K64 = w.astype(np.float64), K.astype(np.float64)
    sd64 = np.broadcast_to(np.asarray(sd, dtype=np.float64), (K.shape[1],))
    mu64 = np.broadcast_to(np.asarray(mu, dtype=np.float64), (K.shape[1],))
    pu = w.shape[-1]
    y = np.einsum('stp,pc->stc', w64, K64) * sd64 + mu64
    absum = np.einsum('stp,pc->stc', np.abs(w64), np.abs(K64))
    fy = (pu + 2) * EPS32 * (np.abs(sd64) * absum + np.abs(mu64))
    if noise is None:
        return y, y, fy, fy
    sn = np.abs(sd64)[None, None, :] * np.abs(noise.astype(np.float64))[:, :, None]
    return y, y + sd64 * noise.astype(np.float64)[:, :, None], fy, fy + EPS32 * sn


def _stats_problem(nsamp, npred, n_y, pu, seed, noise=True, scalar=False, ties=True):
    rng = np.random.default_rng(seed)
    w = rng.standard_normal((nsamp, npred, pu)).astype(np.float32)
    K = rng.standard_normal((pu, n_y)).astype(np.float32)
    if scalar:
        sd, mu = np.float32(1.7), np.float32(0.3)
    else:
        sd = rng.uniform(0.1, 2.0, n_y).astype(np.float32)
        mu = (2.0 + rng.standard_normal(n_y)).astype(np.float32)
    nz = (rng.standard_normal((nsamp, npred)) / np.sqrt(rng.uniform(20, 200, (nsamp, 1)))).astype(np.float32) if noise else None
    if ties and nsamp >= 4:
        w[nsamp // 2] = w[0]                     # exact ties among the sample values
        w[nsamp - 1] = w[1]
        if nz is not None:
            nz[nsamp // 2] = nz[0]
            nz[nsamp - 1] = nz[1]
    return w, K, sd, mu, nz


def _check_stats(w, K, sd, mu, nz, q, got):
    nsamp = w.shape[0]
    y, z, fy, fz = _fields64(w, K, sd, mu, nz)
    ym, lo, hi = [t.cpu().numpy().astype(np.float64) for t in got]
    mabs = np.abs(y).max(axis=0)
    assert np.all(np.abs(ym - y.mean(axis=0)) <= fy.max(axis=0) + nsamp * EPS32 * mabs)
    zmax = np.abs(z).max(axis=0)
    tol = fz.max(axis=0) + 2 * EPS32 * zmax
    ref_lo = np.quantile(z, q, axis=0, method='linear')
    ref_hi = np.quantile(z, 1 - q, axis=0, method='linear')
    assert np.all(np.abs(lo - ref_lo) <= tol), np.max(np.abs(lo - ref_lo) / tol)
    assert np.all(np.abs(hi - ref_hi) <= tol), np.max(np.abs(hi - ref_hi) / tol)


def _check_errstats(w, K, sd, mu, nz, q, fields, seed):
    """reconstruct_errstats: the fields must be those of reconstruct_stats bit for bit, and the six sums those of the
    fields, with test values placed exactly on ylo, on yhi (covered) and on the MAPE floor (counted)."""
    from gladsgp_b200 import ops
    ym, lo, hi = [t.cpu().numpy() for t in fields]
    npred, n_y = ym.shape
    rng = np.random.default_rng(seed)
    yt = (ym + 0.5 * (hi - lo) * rng.standard_normal(ym.shape)).astype(np.float32)
    floor = np.float32(np.quantile(yt, 0.1))
    cols = rng.permutation(n_y)
    k = max(1, n_y // 10)
    on_lo, on_hi, on_floor = cols[:k], cols[k:2 * k], cols[2 * k:3 * k]
    yt[:, on_lo] = lo[:, on_lo]
    yt[:, on_hi] = hi[:, on_hi]
    yt[:, on_floor] = floor
    err, fl = ops.reconstruct_errstats(w, K, sd, mu, yt, float(floor), q=q, noise=nz, want_fields=True)
    for a, b in zip(fl, (ym, lo, hi)):
        assert np.array_equal(a.cpu().numpy(), b)
    res = ym - yt                                           # float32, as in the kernel
    ape = np.abs(res / yt)
    take = ~(yt < floor)
    cov = (yt >= lo) & (yt <= hi)
    assert cov[:, on_lo].all() and cov[:, on_hi].all() and take[:, on_floor].all()
    ref = np.stack([(res * res).astype(np.float64).sum(1),
                    np.where(take, ape, 0).astype(np.float64).sum(1), take.sum(1), cov.sum(1),
                    lo.astype(np.float64).sum(1), hi.astype(np.float64).sum(1)], axis=1)
    np.testing.assert_array_equal(err[:, 2:4], ref[:, 2:4])
    np.testing.assert_allclose(err[:, [0, 1, 4, 5]], ref[:, [0, 1, 4, 5]], rtol=1e-12)


@pytest.mark.parametrize('case,i0', STATS_CASES, ids=['n%d-q%g' % c for c, _ in STATS_CASES])
@pytest.mark.parametrize('pu', STATS_PU)
def test_stats_every_template_and_order_statistic(cuda, pu, case, i0):
    """n_y = 1024 k + 1 (a one-column last tile), two designs, noise, per-output sd / mean, tied samples."""
    from gladsgp_b200 import ops
    nsamp, q = case
    assert int(np.floor(q * (nsamp - 1))) == i0                # the kernel's own position arithmetic
    npred, n_y = 2, 1025
    w, K, sd, mu, nz = _stats_problem(nsamp, npred, n_y, pu, seed=nsamp * 31 + pu)
    got = ops.reconstruct_stats(w, K, sd, mu, q=q, noise=nz)
    _check_stats(w, K, sd, mu, nz, q, got)
    _check_errstats(w, K, sd, mu, nz, q, got, seed=pu)


@pytest.mark.parametrize('case', [(64, 0.025), (128, 0.025)], ids=['kq4', 'kq8'])
@pytest.mark.parametrize('noise,scalar,npred,n_y', [(False, False, 3, 700), (True, True, 3, 700), (True, False, 300, 129)],
                         ids=['no_noise', 'scalar_sd_mean', 'npred300'])
def test_stats_without_noise_scalar_scaling_and_many_designs(cuda, case, noise, scalar, npred, n_y):
    """noise=None (the default of get_y_stats), scalar sd / mean, fewer outputs than one tile, 300 designs."""
    from gladsgp_b200 import ops
    nsamp, q = case
    w, K, sd, mu, nz = _stats_problem(nsamp, npred, n_y, 8, seed=npred + n_y, noise=noise, scalar=scalar)
    got = ops.reconstruct_stats(w, K, sd, mu, q=q, noise=nz)
    _check_stats(w, K, sd, mu, nz, q, got)
    _check_errstats(w, K, sd, mu, nz, q, got, seed=n_y)


def test_stats_guards_launch_nothing(cuda):
    """pu > 16, an order statistic beyond the eighth, and more than 200 KB of staged samples come back as
    GGP_ERR_UNSUPPORTED (-3) from both entry points, with the outputs untouched."""
    import torch
    from gladsgp_b200 import _lib, ops
    lib = _lib.load()
    p = _lib.ptr
    for pu, nsamp, q in ((17, 64, 0.025), (8, 300, 0.025), (16, 3100, 0.001)):
        n_y, npred = 1025, 2
        assert int(np.floor(q * (nsamp - 1))) + 2 <= nsamp
        w = torch.zeros((nsamp, npred, pu), dtype=torch.float32, device='cuda')
        K = torch.zeros((pu, n_y), dtype=torch.float32, device='cuda')
        one = torch.ones(1, dtype=torch.float32, device='cuda')
        outs = [torch.full((npred, n_y), 7.0, dtype=torch.float32, device='cuda') for _ in range(3)]
        rc = lib.ggp_reconstruct_stats_f32(p(w), p(K), p(one), 1, p(one), 1, None, nsamp, npred, pu, n_y, q,
                                           p(outs[0]), p(outs[1]), p(outs[2]), _lib.stream_ptr())
        assert rc == -3, (pu, nsamp, q)
        yt = torch.zeros((npred, n_y), dtype=torch.float32, device='cuda')
        need = lib.ggp_errstats_workspace_bytes(npred, n_y)
        ws = torch.zeros(need, dtype=torch.uint8, device='cuda')
        err = torch.full((npred, 6), 7.0, dtype=torch.float64, device='cuda')
        rc = lib.ggp_reconstruct_errstats_f32(p(w), p(K), p(one), 1, p(one), 1, None, nsamp, npred, pu, n_y, q, p(yt), 0.0,
                                              p(outs[0]), p(outs[1]), p(outs[2]), p(err), p(ws), need, _lib.stream_ptr())
        assert rc == -3, (pu, nsamp, q)
        torch.cuda.synchronize()
        assert all(bool((o == 7.0).all()) for o in outs) and bool((err == 7.0).all()) and not ws.any().item()
        with pytest.raises(_lib.GgpError, match=r'\(-3\)'):
            ops.reconstruct_stats(w, K, one, one, q=q)


def test_get_y_stats_with_1000_samples(cuda):
    """SepiaEmulatorPrediction.get_y_stats at the 0.5 % quantile of 1000 posterior samples (52 KB of staged samples at
    pu = 10)."""
    from helpers import make_problem, synthetic
    from sepia.SepiaData import SepiaData
    from sepia.SepiaModel import SepiaModel
    from sepia.SepiaPredict import SepiaEmulatorPrediction
    pr = make_problem(m=64, q=3, pu=10, n_x=40, n_t=30)
    data = SepiaData(t_sim=pr['t'], y_sim=pr['y'], y_ind_sim=np.arange(pr['y'].shape[1], dtype=float))
    data.transform_xt(t_notrans=np.arange(3)); data.standardize_y(y_mean=pr['mu'], y_sd=pr['sd']); data.create_K_basis(K=pr['K'])
    model = SepiaModel(data)
    ns = 1000
    samples = synthetic.posterior_samples(ns, model.num.p + model.num.q, 10, seed=8)
    np.random.seed(0)
    pe = SepiaEmulatorPrediction(t_pred=synthetic.test_design(3, 3), samples=samples, model=model)
    pe.w = pe.w.astype(np.float32)
    rng = np.random.default_rng(2)
    noise = (rng.standard_normal((ns, 3)) / np.sqrt(np.asarray(samples['lamWOs'], dtype=np.float64).reshape(-1, 1))).astype(np.float32)
    got = pe.get_y_stats(quantile=0.005, noise=noise, device=True)
    sd = np.asarray(pr['sd'], dtype=np.float32); mu = np.asarray(pr['mu'], dtype=np.float32)
    _check_stats(pe.w, np.asarray(pr['K'], dtype=np.float32), sd, mu, noise, 0.005, (got['mean'], got['lq'], got['uq']))


RECON_PU = [1, 3, 4, 5, 8, 9, 12, 13, 16, 17, 24, 25, 32]


@pytest.mark.parametrize('scalar', [False, True])
@pytest.mark.parametrize('pu', RECON_PU)
def test_reconstruct_every_template_and_store_path(cuda, pu, scalar):
    """n_y % 4 == 0: an aligned output takes the 16-byte store path, the same output one float off alignment the scalar
    path; both against the FP64 field and bit-identical to each other."""
    import torch
    from gladsgp_b200 import ops
    rng = np.random.default_rng(pu * 2 + scalar)
    R, n_y = 37, 4100
    w = rng.standard_normal((R, pu)).astype(np.float32)
    K = rng.standard_normal((pu, n_y)).astype(np.float32)
    if scalar:
        sd, mu = np.float32(1.7), np.float32(-0.3)
    else:
        sd = rng.uniform(0.1, 2.0, n_y).astype(np.float32); mu = rng.standard_normal(n_y).astype(np.float32)
    y, _, fy, _ = _fields64(w[None], K, sd, mu, None)
    out = torch.empty((R, n_y), dtype=torch.float32, device='cuda')
    assert out.data_ptr() % 16 == 0
    ya = ops.reconstruct(w, K, sd, mu, out=out)
    buf = torch.empty(R * n_y + 1, dtype=torch.float32, device='cuda')
    mis = buf[1:].view(R, n_y)
    assert mis.data_ptr() % 16 != 0
    ys = ops.reconstruct(w, K, sd, mu, out=mis)
    assert torch.equal(ya, ys)
    assert np.all(np.abs(ya.cpu().numpy() - y[0]) <= fy[0])


def test_reconstruct_many_rows_per_cta(cuda):
    """n_y = 1 220 001 (odd: scalar stores) and 300 rows: the grid covers the columns alone, so one CTA stages all 300 rows
    in three tiles of at most 128; against the FP64 field on the device."""
    import torch
    from gladsgp_b200 import ops
    g = torch.Generator(device='cuda'); g.manual_seed(5)
    R, pu, n_y = 300, 13, 1220001
    w = torch.randn((R, pu), dtype=torch.float32, device='cuda', generator=g)
    K = torch.randn((pu, n_y), dtype=torch.float32, device='cuda', generator=g)
    sd = torch.rand((n_y,), dtype=torch.float32, device='cuda', generator=g) * 1.9 + 0.1
    mu = torch.randn((n_y,), dtype=torch.float32, device='cuda', generator=g)
    y = ops.reconstruct(w, K, sd, mu)
    ref = (w.double() @ K.double()) * sd.double() + mu.double()
    bound = (pu + 2) * EPS32 * ((w.double().abs() @ K.double().abs()) * sd.double() + mu.double().abs())
    assert bool(((y.double() - ref).abs() <= bound).all())
