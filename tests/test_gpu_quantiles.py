"""GPU: exact quantile fields (ggp_reconstruct_quantiles_f32), error sums from fields (ggp_fields_errstats_f32) and the
public get_y_quantiles / get_y_stats / get_y_error_stats routes that use them.

The reference for every quantile is np.quantile (or its float32 restatement in quantile_helpers) of z formed on the device
from ops.reconstruct and `y + sd * noise` in torch float32 -- the same float32 operations the kernel performs -- so the
quantiles are compared bit for bit.  The mean is an FP64 sum rounded once: within one float32 ulp of the exact mean."""
import numpy as np
import pytest

from helpers import make_problem, make_scalar_problem, synthetic
from quantile_helpers import quantile_sorted

pytestmark = pytest.mark.gpu

BASE_Q = [0.0, 1.0, 0.5, 0.025, 0.975, 0.25, 0.3]


def _quantile_list(n):
    """BASE_Q plus a position with t exactly 0.5 (when n-1 is odd, q = 0.5 gives it) and one with t just below 0.5."""
    qs = list(BASE_Q)
    if n > 1:
        half = np.float32((max(0, (n - 1) // 3) + 0.5) / (n - 1))
        qs += [float(half), float(np.nextafter(half, np.float32(0)))]
    return qs


def _problem(nsamp, npred, n_y, pu, seed, noise=True, scalar=False, ties=True):
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
        w[nsamp // 2] = w[0]
        w[nsamp - 1] = w[1]
        if nz is not None:
            nz[nsamp // 2] = nz[0]
            nz[nsamp - 1] = nz[1]
    return w, K, sd, mu, nz


def _fields(w, K, sd, mu, nz):
    """y (nsamp, npred, n_y) from ops.reconstruct and z = y + sd * noise in torch float32, on the device."""
    import torch
    from gladsgp_b200 import ops
    nsamp, npred, pu = w.shape
    n_y = K.shape[1]
    y = ops.reconstruct(w.reshape(nsamp * npred, pu), K, sd, mu).reshape(nsamp, npred, n_y)
    if nz is None:
        return y, y
    sdt = torch.as_tensor(np.asarray(sd, dtype=np.float32).reshape(-1), device='cuda')
    nzt = torch.as_tensor(nz, device='cuda')
    return y, y + sdt * nzt[:, :, None]


def _check_mean(got, y):
    ref = np.mean(y.astype(np.float64), axis=0)
    got = got.astype(np.float64)
    ulp = np.spacing(np.abs(ref).astype(np.float32)).astype(np.float64)
    ok = (np.abs(got - ref) <= ulp) | (np.isnan(got) & np.isnan(ref))
    assert ok.all(), np.max(np.abs(got - ref) / ulp)


def _check_exact(w, K, sd, mu, nz, qs):
    from gladsgp_b200 import ops
    y, z = _fields(w, K, sd, mu, nz)
    yh, zh = y.cpu().numpy(), z.cpu().numpy()
    ym, yq = ops.reconstruct_quantiles(w, K, sd, mu, qs, noise=nz)
    yq = yq.cpu().numpy()
    for k, q in enumerate(qs):
        np.testing.assert_array_equal(yq[k], np.quantile(zh, q, axis=0), err_msg='q=%r' % q)
    _check_mean(ym.cpu().numpy(), yh)
    return ym, yq


@pytest.mark.parametrize('pu', [1, 3, 16, 17, 20, 32])
@pytest.mark.parametrize('nsamp', [1, 2, 3, 64, 281, 1000, 4096, 16384])
def test_quantiles_bit_exact(cuda, nsamp, pu):
    """Two designs, noise, per-output sd / mean, tied samples, n_y with a ragged last tile for every tile width."""
    n_y = 37 if nsamp >= 4096 else 301
    w, K, sd, mu, nz = _problem(nsamp, 2, n_y, pu, seed=nsamp * 7 + pu)
    _check_exact(w, K, sd, mu, nz, _quantile_list(nsamp))


@pytest.mark.parametrize('nsamp', [3, 281, 1000])
@pytest.mark.parametrize('noise,scalar', [(False, False), (False, True), (True, True)], ids=['no_noise', 'scalar', 'noise_scalar'])
def test_quantiles_without_noise_and_scalar_scaling(cuda, nsamp, noise, scalar):
    w, K, sd, mu, nz = _problem(nsamp, 3, 517, 10, seed=nsamp, noise=noise, scalar=scalar)
    _check_exact(w, K, sd, mu, nz, _quantile_list(nsamp))


def test_quantiles_nan_sample_and_determinism(cuda):
    """A NaN weight makes every quantile and the mean of its design NaN (as np.quantile / np.mean); other designs are
    unaffected.  Two runs give identical bits."""
    from gladsgp_b200 import ops
    w, K, sd, mu, nz = _problem(300, 3, 1030, 8, seed=1)
    w[17, 1, 2] = np.nan
    ym, yq = _check_exact(w, K, sd, mu, nz, _quantile_list(300))
    assert np.isnan(yq[:, 1]).all() and np.isnan(ym.cpu().numpy()[1]).all()
    assert not np.isnan(yq[:, [0, 2]]).any()
    ym2, yq2 = ops.reconstruct_quantiles(w, K, sd, mu, _quantile_list(300), noise=nz)
    np.testing.assert_array_equal(ym.cpu().numpy(), ym2.cpu().numpy())
    np.testing.assert_array_equal(yq, yq2.cpu().numpy())


def test_quantiles_70000_designs_in_one_call(cuda):
    w, K, sd, mu, nz = _problem(16, 70000, 5, 3, seed=2)
    _check_exact(w, K, sd, mu, nz, [0.025, 0.5, 0.975])


def test_quantiles_at_cfg4_size(cuda):
    """nsamp = 1000, npred = 4, n_y = 1 460 000, pu = 10, noise: against torch.sort + the float32 lerp on the device in
    column chunks; the mean within one ulp of an FP64 mean, and identical across two runs."""
    import torch
    from gladsgp_b200 import ops
    g = torch.Generator(device='cuda'); g.manual_seed(3)
    ns, npred, pu, n_y = 1000, 4, 10, 1460000
    w = torch.randn((ns, npred, pu), dtype=torch.float32, device='cuda', generator=g)
    K = torch.randn((pu, n_y), dtype=torch.float32, device='cuda', generator=g)
    sd = torch.rand((n_y,), dtype=torch.float32, device='cuda', generator=g) * 1.9 + 0.1
    mu = torch.randn((n_y,), dtype=torch.float32, device='cuda', generator=g)
    nz = torch.randn((ns, npred), dtype=torch.float32, device='cuda', generator=g) * 0.1
    qs = [0.025, 0.25, 0.5, 0.75, 0.975]
    ym, yq = ops.reconstruct_quantiles(w, K, sd, mu, qs, noise=nz)
    ym2, _ = ops.reconstruct_quantiles(w, K, sd, mu, qs, noise=nz)
    assert torch.equal(ym, ym2)
    bad = 0
    for c0 in range(0, n_y, 200000):
        c1 = min(n_y, c0 + 200000)
        y = ops.reconstruct(w.reshape(ns * npred, pu), K[:, c0:c1], sd[c0:c1], mu[c0:c1]).reshape(ns, npred, -1)
        zs = torch.sort(y + sd[c0:c1] * nz[:, :, None], dim=0).values
        for k, q in enumerate(qs):
            bad += int((quantile_sorted(zs, q) != yq[k, :, c0:c1]).sum().item())
        ref = y.double().mean(dim=0)
        ulp = torch.as_tensor(np.spacing(ref.abs().float().cpu().numpy()), device='cuda').double()
        assert bool(((ym[:, c0:c1].double() - ref).abs() <= ulp).all())
        del y, zs
    assert bad == 0


def _sepia_model(pu, ns, seed=4):
    from sepia.SepiaData import SepiaData
    from sepia.SepiaModel import SepiaModel
    pr = make_problem(m=64, q=3, pu=pu, n_x=40, n_t=30)
    data = SepiaData(t_sim=pr['t'], y_sim=pr['y'], y_ind_sim=np.arange(pr['y'].shape[1], dtype=float))
    data.transform_xt(t_notrans=np.arange(3)); data.standardize_y(y_mean=pr['mu'], y_sd=pr['sd']); data.create_K_basis(K=pr['K'])
    model = SepiaModel(data)
    samples = synthetic.posterior_samples(ns, model.num.p + model.num.q, pu, seed=seed)
    return pr, model, samples


def _noise(samples, npred, seed):
    rng = np.random.default_rng(seed)
    ns = np.asarray(samples['lamWOs']).shape[0]
    return (rng.standard_normal((ns, npred)) / np.sqrt(np.asarray(samples['lamWOs'], dtype=np.float64).reshape(-1, 1))).astype(np.float32)


def _api_reference(pe, noise, qs):
    """z from the object's own get_y (float32 w) and its sd_y, on the device; np.quantile on the host."""
    import torch
    y = pe.get_y(device=True)
    sd = np.asarray(pe.model.data.sim_data.orig_y_sd, dtype=np.float32).reshape(-1)
    z = y if noise is None else y + torch.as_tensor(sd, device='cuda') * torch.as_tensor(noise, device='cuda')[:, :, None]
    zh = z.cpu().numpy()
    return y.cpu().numpy(), [np.quantile(zh, q, axis=0) for q in qs]


def test_get_y_quantiles_pu20(cuda):
    from sepia.SepiaPredict import SepiaEmulatorPrediction
    _, model, samples = _sepia_model(20, 100)
    np.random.seed(0)
    pe = SepiaEmulatorPrediction(t_pred=synthetic.test_design(5, 3), samples=samples, model=model)
    pe.w = pe.w.astype(np.float32)
    noise = _noise(samples, 5, 1)
    got = pe.get_y_quantiles(noise=noise)
    assert got['quantiles'].shape == (3, 5, pe.get_y().shape[2]) and list(got['q']) == [0.025, 0.5, 0.975]
    y, ref = _api_reference(pe, noise, got['q'])
    for k in range(3):
        np.testing.assert_array_equal(got['quantiles'][k], ref[k])
    _check_mean(got['mean'], y)
    # get_y_stats at pu = 20 (beyond the fused kernel) routes here: the same bits as (q, 1-q)
    st = pe.get_y_stats(quantile=0.025, noise=noise)
    np.testing.assert_array_equal(st['lq'], ref[0])
    np.testing.assert_array_equal(st['uq'], ref[2])
    np.testing.assert_array_equal(st['mean'], got['mean'])


def test_get_y_quantiles_scalar_model(cuda):
    """A scalar-output model (pu = 1) goes through the 1 x 1 unit basis: the quantiles of get_y() (w sd + mean)."""
    from sepia.SepiaData import SepiaData
    from sepia.SepiaModel import SepiaModel
    from sepia.SepiaPredict import SepiaEmulatorPrediction
    pr = make_scalar_problem(m=100)
    data = SepiaData(t_sim=pr['t'], y_sim=pr['y'])
    data.transform_xt()
    data.standardize_y()
    model = SepiaModel(data)
    samples = synthetic.posterior_samples(300, model.num.p + model.num.q, 1, seed=6)
    np.random.seed(1)
    pe = SepiaEmulatorPrediction(model=model, t_pred=np.linspace(0.05, 0.95, 40)[:, None], samples=samples)
    pe.w = pe.w.astype(np.float32)
    noise = _noise(samples, 40, 2)
    qs = (0.025, 0.1, 0.5, 0.9, 0.975)
    got = pe.get_y_quantiles(quantiles=qs, noise=noise)
    assert got['mean'].shape == (40, 1) and got['quantiles'].shape == (5, 40, 1)
    y, ref = _api_reference(pe, noise, qs)
    for k in range(5):
        np.testing.assert_array_equal(got['quantiles'][k], ref[k])
    _check_mean(got['mean'], y)
    st = pe.get_y_stats(quantile=0.025, noise=noise)                 # 300 samples: the general kernel
    np.testing.assert_array_equal(st['lq'], ref[0])
    yt = (y.mean(axis=0) + 0.1).astype(np.float32)
    err = pe.get_y_error_stats(yt, quantile=0.025, noise=noise)
    assert err['rmse'].shape == (40,) and np.isfinite(err['rmse']).all()


def test_get_y_quantiles_on_xval_prediction(cuda):
    from sepia.SepiaPredict import SepiaXvalEmulatorPrediction
    _, model, samples = _sepia_model(3, 64)
    np.random.seed(2)
    xv = SepiaXvalEmulatorPrediction(samples=samples, model=model, leave_out_inds=[[5, 2], [9], [40]])
    xv.w = xv.w.astype(np.float32)
    qs = (0.05, 0.5, 0.95)
    got = xv.get_y_quantiles(quantiles=qs)
    y, ref = _api_reference(xv, None, qs)
    for k in range(3):
        np.testing.assert_array_equal(got['quantiles'][k], ref[k])
    _check_mean(got['mean'], y)


def test_get_y_stats_1000_samples_at_2_5_percent(cuda):
    """cfg4's sample count at the reference's own 2.5 %: beyond the fused kernel, served exactly by the general one."""
    from gladsgp_b200 import ops
    from sepia.SepiaPredict import SepiaEmulatorPrediction
    _, model, samples = _sepia_model(10, 1000, seed=8)
    np.random.seed(0)
    pe = SepiaEmulatorPrediction(t_pred=synthetic.test_design(3, 3), samples=samples, model=model)
    pe.w = pe.w.astype(np.float32)
    assert not ops.stats_supported(1000, 10, 0.025)
    noise = _noise(samples, 3, 3)
    st = pe.get_y_stats(quantile=0.025, noise=noise)
    y, ref = _api_reference(pe, noise, (0.025, 1 - 0.025))
    np.testing.assert_array_equal(st['lq'], ref[0])
    np.testing.assert_array_equal(st['uq'], ref[1])
    _check_mean(st['mean'], y)


def test_get_y_stats_keeps_the_fused_kernel_where_it_serves(cuda):
    from gladsgp_b200 import ops
    from sepia.SepiaPredict import SepiaEmulatorPrediction
    _, model, samples = _sepia_model(10, 64)
    np.random.seed(0)
    pe = SepiaEmulatorPrediction(t_pred=synthetic.test_design(4, 3), samples=samples, model=model)
    pe.w = pe.w.astype(np.float32)
    assert ops.stats_supported(64, 10, 0.025)
    noise = _noise(samples, 4, 4)
    st = pe.get_y_stats(quantile=0.025, noise=noise)
    sdd, mud = model.data.sim_data.stats_device()
    ref = ops.reconstruct_stats(pe.w, pe._basis_device(), sdd, mud, q=0.025, noise=noise)
    for a, b in zip((st['mean'], st['lq'], st['uq']), ref):
        np.testing.assert_array_equal(a, b.cpu().numpy())
    with pytest.raises(Exception, match=r'q must be in \(0, 0.5\)'):
        pe.get_y_stats(quantile=0.7)


def test_get_y_error_stats_pu20_matches_assess_oracle(cuda):
    """get_y_error_stats at pu = 20 (field route): the error table equals assess_oracle.error_statistics of the same float32
    fields, and the fields are those of get_y_stats."""
    from oracle import assess_oracle as ao
    from sepia.SepiaPredict import SepiaEmulatorPrediction
    pr, model, samples = _sepia_model(20, 200, seed=5)
    np.random.seed(0)
    pe = SepiaEmulatorPrediction(t_pred=synthetic.test_design(4, 3), samples=samples, model=model)
    pe.w = pe.w.astype(np.float32)
    noise = _noise(samples, 4, 5)
    rng = np.random.default_rng(6)
    y_test = (pe.get_y().mean(axis=0) + 0.05 * rng.standard_normal((4, pr['y'].shape[1]))).astype(np.float32)
    got = pe.get_y_error_stats(y_test, quantile=0.025, noise=noise, fields=True)
    st = pe.get_y_stats(quantile=0.025, noise=noise)
    for k, f in (('mean', 'mean'), ('lq_field', 'lq'), ('uq_field', 'uq')):
        np.testing.assert_array_equal(got[k].cpu().numpy(), st[f])
    ref = ao.error_statistics(st['mean'], st['lq'], st['uq'], y_test)
    assert abs(got['mape_floor'] - ref['mape_floor']) <= 1e-6 * abs(ref['mape_floor'])
    for k in ('rmse', 'mape', 'lq', 'uq'):
        np.testing.assert_allclose(got[k], ref[k], rtol=1e-5, err_msg=k)
    assert np.all(np.abs(got['frac_covered'] - ref['frac_covered']) <= 1.0 / y_test.shape[1])
    np.testing.assert_allclose(got['integrated_ci'], ref['integrated_ci'], rtol=1e-5)
    nof = pe.get_y_error_stats(y_test, quantile=0.025, noise=noise)             # chunked, no fields kept
    for k in ('rmse', 'mape', 'lq', 'uq', 'frac_covered'):
        np.testing.assert_array_equal(nof[k], got[k])


def test_fields_errstats_sums_and_fused_parity(cuda):
    from gladsgp_b200 import ops
    rng = np.random.default_rng(9)
    npred, n_y = 3, 5000
    ym = rng.standard_normal((npred, n_y)).astype(np.float32) + 3.0
    lo = (ym - rng.uniform(0.1, 1.0, ym.shape)).astype(np.float32)
    hi = (ym + rng.uniform(0.1, 1.0, ym.shape)).astype(np.float32)
    yt = (ym + 0.7 * rng.standard_normal(ym.shape)).astype(np.float32)
    floor = np.float32(np.quantile(yt, 0.1))
    cols = rng.permutation(n_y)
    yt[:, cols[:300]] = lo[:, cols[:300]]
    yt[:, cols[300:600]] = hi[:, cols[300:600]]
    yt[:, cols[600:900]] = floor
    err = ops.fields_errstats(ym, lo, hi, yt, float(floor))
    res = ym - yt
    take = ~(yt < floor)
    cov = (yt >= lo) & (yt <= hi)
    ref = np.stack([(res * res).astype(np.float64).sum(1), np.where(take, np.abs(res / yt), 0).astype(np.float64).sum(1),
                    take.sum(1), cov.sum(1), lo.astype(np.float64).sum(1), hi.astype(np.float64).sum(1)], axis=1)
    np.testing.assert_array_equal(err[:, 2:4], ref[:, 2:4])
    np.testing.assert_allclose(err[:, [0, 1, 4, 5]], ref[:, [0, 1, 4, 5]], rtol=1e-12)
    # fed the fused kernel's own fields, the same sums bit for bit
    w, K, sd, mu, nz = _problem(64, 3, 3001, 10, seed=10)
    yt2 = (rng.standard_normal((3, 3001)) + 2.0).astype(np.float32)
    e_fused, fl = ops.reconstruct_errstats(w, K, sd, mu, yt2, 1.5, q=0.025, noise=nz, want_fields=True)
    np.testing.assert_array_equal(ops.fields_errstats(fl[0], fl[1], fl[2], yt2, 1.5), e_fused)


def test_quantiles_refusals_leave_outputs_untouched(cuda):
    import ctypes
    import torch
    from gladsgp_b200 import _lib
    lib = _lib.load()
    p = _lib.ptr
    npred, n_y = 2, 100

    def call(nsamp, pu, qs, nq=None, null=None):
        w = torch.zeros((nsamp, npred, pu), dtype=torch.float32, device='cuda')
        K = torch.zeros((pu, n_y), dtype=torch.float32, device='cuda')
        one = torch.ones(1, dtype=torch.float32, device='cuda')
        ym = torch.full((npred, n_y), 7.0, dtype=torch.float32, device='cuda')
        yq = torch.full((max(len(qs), 1), npred, n_y), 7.0, dtype=torch.float32, device='cuda')
        qa = (ctypes.c_double * max(len(qs), 1))(*qs)
        args = [p(w), p(K), p(one), 1, p(one), 1, None, nsamp, npred, pu, n_y, qa, len(qs) if nq is None else nq,
                p(ym), p(yq), _lib.stream_ptr()]
        if null is not None:
            args[null] = None
        rc = lib.ggp_reconstruct_quantiles_f32(*args)
        torch.cuda.synchronize()
        assert bool((ym == 7.0).all()) and bool((yq == 7.0).all())
        return rc
    assert call(16385, 3, [0.5]) == -3
    assert call(64, 33, [0.5]) == -3
    assert call(64, 3, [0.5] * 33) == -1
    assert call(64, 3, [0.5], nq=0) == -1
    assert call(64, 3, [0.5, 1.5]) == -1
    assert call(64, 3, [-0.1]) == -1
    for k in (0, 1, 2, 4, 14):
        assert call(64, 3, [0.5], null=k) == -1
