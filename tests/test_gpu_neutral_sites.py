"""Likelihood-neutral betaU sites (constant input columns, include/gladsgp_b200.h fixed code 3) are decided without an
evaluation in every step kernel.  The chain is the oracle's (tests/golden/chain_cfg3.npz: d = 9 with the dummy x first),
the uniform stream is consumed as before, and exactly the in-bounds neutral proposals leave the evaluation count."""
import copy
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def _golden(cfg, steps=None):
    g = np.load(os.path.join(GOLD, 'chain_%s.npz' % cfg))
    n = int(g['n_steps']) if steps is None else steps
    tb = {k[3:]: g[k] for k in g.files if k.startswith('tb_')}
    rp = {k[3:]: g[k][:n] for k in g.files if k.startswith('rp_')}
    return g, tb, rp, n


def _engine(g, tb, n_chains, neutral=True):
    from gladsgp_b200 import ops
    eng = ops.McmcEngine(g['zt'], np.ascontiguousarray(g['w'].T), g['LamSim'], tb, n_chains=n_chains)
    if not neutral:                                     # the table as given: every site evaluated
        eng.t_fixed.copy_(eng.torch.as_tensor(np.asarray(tb['fixed'], dtype=np.uint8), device='cuda'))
    eng.set_state(tb['theta'])
    return eng


def _neutral_mask(g, tb):
    d = g['zt'].shape[1]
    pu = g['w'].shape[1]
    mask = np.zeros(tb['theta'].size, dtype=bool)
    const = np.all(g['zt'] == g['zt'][:1], axis=0)
    for j in range(pu):
        mask[j * d:(j + 1) * d] = const
    return mask


def _np(o, k):
    return o[k].cpu().numpy()


@pytest.mark.parametrize('chains,spec', [(1, '0'), (1, '1'), (16, '0'), (80, '0')])
def test_replay_skips_exactly_the_in_bounds_neutral_proposals(cuda, monkeypatch, chains, spec):
    """cfg3 replay under the single-chain (speculative / cluster) and the many-chain (look-ahead) step kernels.  The
    speculative kernel counts the evaluations of its three lanes per round, so there the count only has to fall."""
    monkeypatch.setenv('GGP_SPEC', spec)
    g, tb, rp, n = _golden('cfg3')
    mask = _neutral_mask(g, tb)
    assert mask.sum() == 10                            # betaU[0, j] of the 10 PCs
    rep = {k: np.repeat(v, chains, axis=1) for k, v in rp.items()}
    outs = {}
    for neutral in (True, False):
        eng = _engine(g, tb, chains, neutral)
        outs[neutral] = eng.run(n, tb['step'], replay=rep, record_accept=True, time_kernels=True)
    o, ref = outs[True], outs[False]
    for c in range(chains):
        assert np.array_equal(_np(o, 'draws')[:, c, :], g['chain_draws'])
        assert np.array_equal(_np(o, 'accepted')[:, c, :], g['chain_acc'][:, 0, :])
    np.testing.assert_allclose(_np(o, 'lp')[:, 0], g['chain_lp'], rtol=1e-9)
    skipped = int((rp['valid'][:, 0, mask] != 0).sum()) * chains
    assert skipped > 0
    if spec == '0':
        assert int(ref['eval_count'][0]) - int(o['eval_count'][0]) == skipped
    else:
        assert int(ref['eval_count'][0]) > int(o['eval_count'][0])
    assert int(ref['eval_count'][1]) == int(o['eval_count'][1])


def test_stream_mode_consumes_and_draws_as_before(cuda):
    """Uniform stream at the bench's shape (cfg3 model, look-ahead kernel): the same draws are consumed and the chains
    agree with the all-evaluated run, log-posteriors to the last bits of the parent's noisy neutral terms."""
    g, tb, _, _ = _golden('cfg3')
    P = tb['theta'].size
    steps, chains = 12, 96
    us = np.random.RandomState(17).random_sample((chains, 2 * P * steps))
    outs = {}
    for neutral in (True, False):
        eng = _engine(g, tb, chains, neutral)
        o = eng.run(steps, tb['step'], uniforms=us, record_accept=True, time_kernels=True)
        outs[neutral] = {k: _np(o, k) for k in ('draws', 'lp', 'accepted', 'consumed')}
        outs[neutral]['eval_count'] = o['eval_count']
    a, b = outs[True], outs[False]
    assert np.array_equal(a['consumed'], b['consumed'])
    assert np.array_equal(a['draws'], b['draws'])
    assert np.array_equal(a['accepted'], b['accepted'])
    np.testing.assert_allclose(a['lp'], b['lp'], rtol=1e-12)
    assert a['eval_count'][0] < b['eval_count'][0]
    assert a['eval_count'][1] == b['eval_count'][1]


@pytest.mark.parametrize('spec', ['0', '1'])
def test_accepted_neutral_site_leaves_the_pc_term(cuda, monkeypatch, spec):
    """One replayed step in which only the neutral sites are proposed: no evaluation, every candidate accepted by the
    prior rule lands in theta and the per-PC terms stay bit for bit the same (also through the PC-shard path)."""
    monkeypatch.setenv('GGP_SPEC', spec)
    g, tb, rp, _ = _golden('cfg3', steps=1)
    mask = _neutral_mask(g, tb)
    rep = {k: v.copy() for k, v in rp.items()}
    rep['valid'][:] = 0
    rep['valid'][0, 0, mask] = 1
    rep['cand'][0, 0, mask] = np.linspace(0.02, 3.0, mask.sum())
    rep['logacorr'][0, 0, :] = 0.0
    rep['logu'][0, 0, mask] = np.log(np.linspace(0.05, 0.95, mask.sum()))
    for by_pc in (False, True):
        eng = _engine(g, tb, 1)
        eng.run(0, tb['step'], uniforms=np.full((1, 1), 0.5))                      # sigwl of the start state
        sig0 = eng.sigwl.clone()
        if by_pc:
            o = eng.run_by_pc(1, tb['step'], replay=rep, record_accept=True, init_sigwl=False, shards=[(0, 4), (4, 6)])
        else:
            o = eng.run(1, tb['step'], replay=rep, record_accept=True, init_sigwl=False, time_kernels=True)
            assert int(o['eval_count'][0]) == 0
        acc = _np(o, 'accepted')[0, 0].astype(bool)
        assert acc.any() and not acc.all() and not acc[~mask].any()
        th = _np(o, 'draws')[0, 0]
        np.testing.assert_array_equal(th[acc], rep['cand'][0, 0, acc])
        np.testing.assert_array_equal(th[~acc], tb['theta'][~acc])
        assert eng.torch.equal(eng.sigwl, sig0)


@pytest.mark.parametrize('spec', ['0', '1'])
def test_pc_sharded_stepping_with_neutral_sites(cuda, monkeypatch, spec):
    monkeypatch.setenv('GGP_SPEC', spec)
    g, tb, rp, n = _golden('cfg3', steps=12)
    eng = _engine(g, tb, 1)
    o = eng.run_by_pc(n, tb['step'], replay=rp, record_accept=True, shards=[(0, 3), (3, 7)])
    assert np.array_equal(_np(o, 'accepted'), g['chain_acc'][:n])
    assert np.array_equal(_np(o, 'draws')[:, 0, :], g['chain_draws'][:n])
    np.testing.assert_allclose(_np(o, 'lp')[:, 0], g['chain_lp'][:n], rtol=1e-9)


def test_model_batch_marks_and_matches_the_all_evaluated_run(cuda):
    from helpers import make_problem
    from sepia.SepiaData import SepiaData
    from sepia.SepiaModel import SepiaModel
    from gladsgp_b200.batch import ModelBatch
    from gladsgp_b200.ops import FIXED_NEUTRAL
    pr = make_problem(m=64, q=3, pu=2)
    models = []
    for i in range(3):
        d = SepiaData(t_sim=pr['t'], y_sim=pr['y'] * (1.0 + 0.1 * i), y_ind_sim=np.linspace(0, 1, pr['y'].shape[1]))
        d.transform_xt(t_notrans=np.arange(3))
        d.standardize_y()
        d.create_K_basis(K=pr['K'])
        models.append(SepiaModel(d))
    res = []
    for neutral in (True, False):
        mb = ModelBatch([copy.deepcopy(m) for m in models], seeds=[3, 4, 5])
        assert (mb.engine.t_fixed.cpu().numpy() == FIXED_NEUTRAL).sum() == 2       # betaU[0, j] of the 2 PCs
        if not neutral:
            mb.engine.t_fixed.zero_()
        mb.do_mcmc(20)
        res.append([mm.get_samples() for mm in mb.models])
    for a, b in zip(*res):
        for k in ('betaU', 'lamUz', 'lamWs', 'lamWOs'):
            assert np.array_equal(a[k], b[k])
        np.testing.assert_allclose(a['logPost'], b['logPost'], rtol=1e-12)
