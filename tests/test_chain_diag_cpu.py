"""CPU: the chain-diagnostics oracle (rank-normalized split R-hat, bulk / tail ESS; DESIGN.md section 2) on cases worked out
by hand and on processes with known answers, and the argument checks of the C ABI without a device."""
import ctypes

import numpy as np
import pytest
from scipy.special import ndtri

from oracle import chain_diag_oracle as cdo


def test_hand_computed_two_chains_four_draws_with_ties():
    x = np.array([[1., 2., 2., 3.],
                  [2., 4., 1., 1.]])
    # split (h = 2): [1, 2], [2, 4], [2, 3], [1, 1]; pooled sorted 1 1 1 2 2 2 3 4 -> ranks 2 (x3), 5 (x3), 7, 8
    z = {r: ndtri((r - 0.375) / 8.25) for r in (2.0, 5.0, 7.0, 8.0)}
    bulk = np.array([[z[2], z[5]], [z[5], z[8]], [z[5], z[7]], [z[2], z[2]]])
    # median 2; folded |x - 2|: [1, 0], [0, 2], [0, 1], [1, 1]; sorted 0 0 0 1 1 1 1 2 -> ranks 2 (x3), 5.5 (x4), 8
    zf = {r: ndtri((r - 0.375) / 8.25) for r in (2.0, 5.5, 8.0)}
    fold = np.array([[zf[5.5], zf[2]], [zf[2], zf[8]], [zf[2], zf[5.5]], [zf[5.5], zf[5.5]]])

    def rhat(a):                           # h = 2: a chain's variance (ddof 1) is (a0 - a1)^2 / 2
        means = (a[:, 0] + a[:, 1]) / 2
        W = np.mean((a[:, 0] - a[:, 1]) ** 2 / 2)
        B = 2 * np.sum((means - means.mean()) ** 2) / 3
        return np.sqrt((B / W + 1) / 2)
    want_rhat = max(rhat(bulk), rhat(fold))
    # h = 2 < 4: Geyer's loop never runs, max_t = -1, rho[0] = 1, tau = 0 -> 1 / log10(8); every series is non-constant
    # (q05 = 1: 1(x <= 1) = [1, 0], [0, 0], [0, 0], [1, 1]; q95 = 3 + 0.65 = 3.65: only the 4 is above)
    want_ess = 8 * np.log10(8)
    r, eb, et = cdo.diagnose(x)
    assert r == pytest.approx(want_rhat, rel=1e-14)
    assert r == pytest.approx(1.40252025163189, rel=1e-12)
    assert eb == pytest.approx(want_ess, rel=1e-14) and et == pytest.approx(want_ess, rel=1e-14)
    assert want_ess == pytest.approx(7.224719895935548, rel=1e-14)


def test_constant_and_non_finite_elements():
    r, eb, et = cdo.diagnose(np.full((3, 7), 2.5))
    assert np.isnan(r) and eb == 18 and et == 18            # S = 2 C floor(n / 2)
    x = np.random.default_rng(0).standard_normal((2, 10))
    for bad in (np.nan, np.inf, -np.inf):
        y = x.copy()
        y[1, 4] = bad
        assert all(np.isnan(v) for v in cdo.diagnose(y))


def test_odd_n_drops_the_middle_draw_from_ranks_but_not_from_the_quantiles():
    x = np.array([[0.0, 1.0, -100.0, 2.0, 3.0],
                  [0.5, 1.5, 100.0, 2.5, 3.5]])
    r, eb, et = cdo.diagnose(x)
    r4, eb4, et4 = cdo.diagnose(np.delete(x, 2, axis=1))
    assert r == r4 and eb == eb4                            # ranks see only the split draws
    # q05 = -55 and q95 = 56.575 come from all ten draws: no split draw lies below q05 or above q95 -> both constant
    assert et == 8.0
    assert et4 == pytest.approx(8 * np.log10(8))


def test_max_rule_keeps_bulk_when_the_folded_array_is_constant():
    x = np.array([[0., 1., 0., 1.], [1., 0., 1., 0.]])      # median 0.5: |x - 0.5| is constant
    s = cdo.split_chains(x)
    bulk = cdo.rhat_raw(cdo.z_scale(s))
    assert np.isnan(cdo.rhat_raw(cdo.z_scale(np.abs(s - np.median(s)))))
    assert np.isfinite(bulk)
    assert cdo.diagnose(x)[0] == bulk


def _ar1(rng, C, n, phi):
    e = rng.standard_normal((C, n))
    x = np.empty((C, n))
    x[:, 0] = e[:, 0] / np.sqrt(1 - phi * phi)
    for i in range(1, n):
        x[:, i] = phi * x[:, i - 1] + e[:, i]
    return x


def test_known_processes():
    rng = np.random.default_rng(2024)
    phi = 0.9
    x = _ar1(rng, 8, 20000, phi)
    _, eb, _ = cdo.diagnose(x)
    want = 8 * 20000 * (1 - phi) / (1 + phi)
    assert abs(eb / want - 1) < 0.1, (eb, want)
    iid = rng.standard_normal((8, 1000))
    assert cdo.diagnose(iid)[0] < 1.005
    shifted = iid.copy()
    shifted[3] += 1.0
    assert cdo.diagnose(shifted)[0] > 1.01


def test_margins_are_reported():
    m = []
    cdo.diagnose(_ar1(np.random.default_rng(1), 4, 400, 0.5), m)
    assert len(m) == 6 and all(v > 0 for v in m)


def test_chain_diag_abi_validates_arguments_without_a_device():
    from gladsgp_b200 import _lib
    h = _lib.load()
    one = ctypes.c_void_p(8)
    need = h.ggp_chain_diag_workspace_bytes(100, 4, 3)
    assert need > 0 and need == 3 * h.ggp_chain_diag_workspace_bytes(100, 4, 1)
    assert h.ggp_chain_diag_workspace_bytes(3, 4, 3) == -1
    # x, n_draws, n_chains, n_elem, s_draw, s_chain, s_elem, rhat, ess_bulk, ess_tail, workspace, bytes, stream
    args = [one, 100, 4, 3, 12, 3, 1, one, one, one, one, need, None]
    for k in (0, 7, 8, 9, 10):
        a = list(args)
        a[k] = None
        assert h.ggp_chain_diag_f64(*a) == -1
        assert b'null pointer' in h.ggp_last_error_string()
    for bad in (3, 0, -1):
        a = list(args)
        a[1] = bad
        assert h.ggp_chain_diag_f64(*a) == -1
        assert b'at least 4' in h.ggp_last_error_string()
    for k in (2, 3):
        a = list(args)
        a[k] = 0
        assert h.ggp_chain_diag_f64(*a) == -1
        assert b'must be positive' in h.ggp_last_error_string()
    a = list(args)
    a[1], a[2] = 1 << 16, 1 << 15                           # n_chains * n_draws = 2^31
    assert h.ggp_chain_diag_f64(*a) == -1
    assert b'below 2^31' in h.ggp_last_error_string()
    a = list(args)
    a[11] = need - 1
    assert h.ggp_chain_diag_f64(*a) == -1
    assert b'workspace too small' in h.ggp_last_error_string()
