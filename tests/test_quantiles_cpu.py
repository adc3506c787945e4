"""CPU: the argument checks of the quantile and field-error C ABI, the fused-statistics support predicate at its boundaries,
and the torch float32 quantile reference against np.quantile."""
import ctypes

import numpy as np
import pytest

from quantile_helpers import numpy_rank, quantile_sorted


def _q(*vals):
    return (ctypes.c_double * len(vals))(*vals)


def test_quantiles_abi_validates_arguments_without_a_device():
    from gladsgp_b200 import _lib
    h = _lib.load()
    one = ctypes.c_void_p(8)
    q2 = _q(0.025, 0.975)
    # w, K, sd, sd_len, mean, mean_len, noise, nsamp, npred, pu, n_y, q_host, nq, ymean, yq, stream (fake device pointers:
    # only rejected calls are made)
    args = [one, one, one, 1, one, 1, None, 64, 2, 10, 100, q2, 2, one, one, None]
    for k in (0, 1, 2, 4, 11, 14):
        a = list(args)
        a[k] = None
        assert h.ggp_reconstruct_quantiles_f32(*a) == -1
        assert b'null pointer' in h.ggp_last_error_string()
    for k, bad in ((7, 0), (8, 0), (9, 0), (10, 0), (7, -5)):
        a = list(args)
        a[k] = bad
        assert h.ggp_reconstruct_quantiles_f32(*a) == -1
        assert b'must be positive' in h.ggp_last_error_string()
    for k, bad in ((3, 7), (5, 99)):
        a = list(args)
        a[k] = bad
        assert h.ggp_reconstruct_quantiles_f32(*a) == -1
        assert b'length' in h.ggp_last_error_string()
    for nq in (0, 33, -1):
        a = list(args)
        a[11], a[12] = _q(*([0.5] * max(nq, 1))), nq
        assert h.ggp_reconstruct_quantiles_f32(*a) == -1
        assert b'nq must be' in h.ggp_last_error_string()
    for bad in (-1e-9, 1.0 + 1e-9, float('nan'), float('inf')):
        a = list(args)
        a[11] = _q(0.5, bad)
        assert h.ggp_reconstruct_quantiles_f32(*a) == -1
        assert b'in [0, 1]' in h.ggp_last_error_string()
    for k, bad in ((7, 16385), (9, 33)):
        a = list(args)
        a[k] = bad
        assert h.ggp_reconstruct_quantiles_f32(*a) == -3
        assert b'unsupported' in h.ggp_last_error_string()


def test_fields_errstats_abi_validates_arguments_without_a_device():
    from gladsgp_b200 import _lib
    h = _lib.load()
    one = ctypes.c_void_p(8)
    need = h.ggp_errstats_workspace_bytes(3, 2049)
    assert need == 3 * 3 * 6 * 8
    args = [one, one, one, one, 3, 2049, 0.1, one, one, need, None]
    for k in (0, 1, 2, 3, 7, 8):
        a = list(args)
        a[k] = None
        assert h.ggp_fields_errstats_f32(*a) == -1
        assert b'null pointer' in h.ggp_last_error_string()
    for k in (4, 5):
        a = list(args)
        a[k] = 0
        assert h.ggp_fields_errstats_f32(*a) == -1
        assert b'must be positive' in h.ggp_last_error_string()
    a = list(args)
    a[9] = need - 1
    assert h.ggp_fields_errstats_f32(*a) == -4
    assert b'workspace too small' in h.ggp_last_error_string()


@pytest.mark.parametrize('nsamp,pu,q,ok', [
    (280, 10, 0.025, 1), (281, 10, 0.025, 0),          # 2.5 %: the eighth order statistic is the last one kept
    (700, 10, 0.01, 1), (701, 10, 0.01, 0), (140, 10, 0.05, 1), (141, 10, 0.05, 0),
    (64, 16, 0.025, 1), (64, 17, 0.025, 0),
    (3011, 16, 0.001, 1), (3012, 16, 0.001, 0),        # 17 floats per staged sample within 200 KB
    (2, 3, 0.3, 1), (1, 3, 0.3, 0)])                    # two order statistics are needed
def test_stats_supported_boundaries(nsamp, pu, q, ok):
    from gladsgp_b200 import _lib
    assert _lib.load().ggp_reconstruct_stats_supported(nsamp, pu, q) == ok


@pytest.mark.parametrize('n', [1, 2, 3, 7, 64, 281, 1000, 4096])
def test_torch_lerp_matches_numpy_quantile(n):
    import torch
    rng = np.random.default_rng(n)
    z = (rng.standard_normal((n, 257)) * rng.uniform(0.1, 50.0, 257)).astype(np.float32)
    z[:, 3] = 1.5                                       # all tied
    if n > 2:
        z[n // 2, 5] = np.nan
        z[:, 7] = np.round(z[:, 7])                     # many ties
    zs = torch.sort(torch.as_tensor(z), dim=0).values
    qs = [0.0, 1.0, 0.5, 0.025, 0.975, 0.25, 0.75, 0.01, 0.3, 1 / 3]
    i = max(0, (n - 1) // 2 - 1)
    if n > 1:
        half = np.float32((i + 0.5) / (n - 1))
        qs += [float(half), float(np.nextafter(half, np.float32(0)))]
    for q in qs:
        ref = np.quantile(z, q, axis=0)
        assert ref.dtype == np.float32
        np.testing.assert_array_equal(quantile_sorted(zs, q).numpy(), ref, err_msg='n=%d q=%r' % (n, q))
    assert numpy_rank(5, 0.75) == (3, 4, np.float32(0.0))
