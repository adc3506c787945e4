"""The golden posterior draws (tests/golden/posterior_cfg*.npz, made by tests/golden/make_golden_posterior.py): inside the
prior support of their tables, reproducible from the script, and reaching the betaU values the posterior consumers must
handle."""
import os
import subprocess
import sys

import numpy as np
import pytest

from posterior_helpers import GOLD, load_posterior

SCRIPT = os.path.join(GOLD, 'make_golden_posterior.py')


@pytest.mark.parametrize('cfg', ['cfg1', 'cfg2', 'cfg3'])
def test_draws_inside_prior_bounds(cfg):
    g = load_posterior(cfg)
    lo, hi = g['tb_lo'], g['tb_hi']
    for key in ('draws', 'state', 'chain_draws'):
        x = np.atleast_2d(g[key])
        assert x.dtype == np.float64 and x.shape[-1] == lo.size
        assert np.all((x >= lo) & (x <= hi)), key
    assert g['draws'].shape[0] == 64
    n = int(g['n_burn'])
    assert np.all(g['draw_steps'] >= n // 2) and np.all(np.diff(g['draw_steps']) > 0)
    assert np.array_equal(g['chain_acc'].shape, g['rp_cand'].shape)


def test_cfg1_regenerates_bit_for_bit(tmp_path):
    subprocess.run([sys.executable, SCRIPT, 'cfg1', '--out', str(tmp_path)], check=True, capture_output=True)
    new = np.load(os.path.join(str(tmp_path), 'posterior_cfg1.npz'))
    old = load_posterior('cfg1')
    assert sorted(new.files) == sorted(old)
    for k in old:
        assert new[k].dtype == old[k].dtype and np.array_equal(new[k], old[k]), k


def test_cfg1_betaU_reaches_beyond_the_synthetic_range():
    """synthetic.posterior_samples draws betaU log-uniform on [0.01, 5] and lamWOs on [10, 200]: the chain goes above 5
    and sits at the lower prior bound 60 of lamWOs, where no consumer test ran before."""
    g = load_posterior('cfg1')
    nb = int(np.sum(g['tb_prior_kind'] == 2))                  # the betaU sites: Beta prior on rho = exp(-beta / 4)
    assert g['draws'][:, :nb].max() >= 5.0
    assert g['draws'][:, :nb].min() < 0.01
    assert np.all(g['draws'][:, -1] < 61.0)
