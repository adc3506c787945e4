"""CPU: host-side mirror of the SEPIA surface (no compute calls) and the C-ABI library exports."""
import ctypes
import os
import re
import numpy as np
import pytest

from helpers import so, make_problem, make_scalar_problem, tables_from_oracle, ROOT


def _data(pr, q):
    from sepia.SepiaData import SepiaData
    d = SepiaData(t_sim=pr['t'], y_sim=pr['y'], y_ind_sim=np.linspace(0, 1, pr['y'].shape[1]))
    d.transform_xt(t_notrans=np.arange(q))
    d.standardize_y(y_mean=pr['mu'], y_sd=pr['sd'])
    d.create_K_basis(K=pr['K'])
    return d


def test_reference_imports_resolve():
    """The exact import lines of src/model.py:13-15, assess_all_models.py:30-32, include_trunc_error.py:16."""
    from sepia.SepiaModel import SepiaModel                                     # noqa: F401
    from sepia.SepiaData import SepiaData                                       # noqa: F401
    from sepia import SepiaParam
    from sepia import SepiaPlot                                                 # noqa: F401
    from sepia.SepiaPredict import SepiaEmulatorPrediction, SepiaXvalEmulatorPrediction   # noqa: F401
    from sepia.SepiaPrior import SepiaPrior                                     # noqa: F401
    prm = SepiaParam(val=3.0, name='lamWOs', val_shape=(1, 1), dist='Gamma', params=[50, 50 / 3.0],
                     bounds=[1., np.inf], mcmcStepParam=10, mcmcStepType='Uniform')   # src/model.py:227-229
    assert prm.val.shape == (1, 1) and prm.prior.dist == 'Gamma' and prm.mcmc.stepType == 'Uniform'
    assert prm.prior.params[1][0, 0] == 50 / 3.0 and prm.mcmc.stepParam[0, 0] == 10.0


def test_sepiadata_str_matches_notebook_output():
    pr = make_problem(m=32, q=8, pu=6, n_x=73, n_t=5)
    d = _data(pr, 8)
    exp = ('This SepiaData instance implies the following:\n'
           'This is a simulator (eta)-only model, y dimension 365\n'
           'm  =    32 (number of simulated data)\n'
           'p  =     1 (number of inputs)\n'
           'q  =     8 (number of additional simulation inputs)\n'
           'pu =     6 (transformed response dimension)\n')
    assert str(d) == exp                      # examples/04_*.ipynb:255-260 (m differs)
    from sepia.SepiaData import SepiaData
    ps = make_scalar_problem(m=20)
    ds = SepiaData(t_sim=ps['t'], y_sim=ps['y'][:, 0])       # 1-D y_sim as sensitivity_indices.py:183
    assert str(ds).splitlines()[-1] == 'pu =     1 (univariate response dimension)'   # 03_*.ipynb:166
    assert ds.sim_data.y.shape == (20, 1) and ds.scalar_out


def test_transform_and_standardize_rules():
    from sepia.SepiaData import SepiaData
    rng = np.random.default_rng(0)
    t = rng.uniform(2, 5, size=(15, 3)); y = rng.normal(size=(15, 4))
    d = SepiaData(t_sim=t, y_sim=y, y_ind_sim=np.arange(4))
    d.transform_xt(t_notrans=[1])
    tt = d.sim_data.t_trans
    assert np.allclose(tt[:, [0, 2]].min(0), 0) and np.allclose(tt[:, [0, 2]].max(0), 1)
    np.testing.assert_array_equal(tt[:, 1], t[:, 1])            # notrans column untouched
    np.testing.assert_array_equal(d.sim_data.x_trans, 0.5)      # dummy x stays 0.5 (zero range)
    _, t2 = d.transform_xt(t=t[:4])
    np.testing.assert_allclose(t2, tt[:4])
    d.standardize_y()
    assert np.ndim(d.sim_data.orig_y_sd) == 0                   # scalar sd by default
    np.testing.assert_allclose(d.sim_data.y_std.mean(0), 0, atol=1e-12)
    d.create_K_basis(n_pc=2)
    assert d.sim_data.K.shape == (2, 4)
    with pytest.raises(ValueError):
        d.create_K_basis(K=np.ones((2, 5)))
    with pytest.raises(NotImplementedError):
        SepiaData(t_sim=t, y_sim=y, y_ind_sim=np.arange(4), y_obs=y[:2])


def test_model_setup_matches_oracle_without_gpu():
    pr = make_problem(m=40, q=3, pu=2)
    from sepia.SepiaModel import SepiaModel
    model = SepiaModel(_data(pr, 3))
    num = pr['num']
    np.testing.assert_allclose(model.num.w, num.wv, rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(model.num.LamSim, num.LamSim, rtol=1e-5)
    np.testing.assert_array_equal(model.num.zt, num.zt)
    tb = model._tables()
    ref = tables_from_oracle(so.OracleModel(num))
    for k in ('prior_kind', 'prior_a', 'lo', 'prop_kind', 'fixed', 'step', 'theta'):
        np.testing.assert_array_equal(np.asarray(tb[k], dtype=float), np.asarray(ref[k], dtype=float))
    np.testing.assert_allclose(tb['prior_b'], ref['prior_b'], rtol=1e-5)
    # printing surface used by mcmc_diagnostics_advanced.py:46-47
    model.print_value_info(); model.print_mcmc_info(); model.print_prior_info()


def test_samples_bookkeeping_and_pickle_roundtrip(tmp_path):
    pr = make_problem(m=24, q=2, pu=2, n_x=6, n_t=5)
    from sepia.SepiaModel import SepiaModel
    model = SepiaModel(_data(pr, 2))
    P = model._tables()['theta'].size
    rng = np.random.default_rng(1)
    draws = rng.uniform(1, 2, size=(20, P)); lps = rng.normal(size=20)
    model._record(draws, lps)
    s = model.get_samples()
    assert s['betaU'].shape == (20, 6) and s['logPost'].shape == (20, 1)
    np.testing.assert_array_equal(s['betaU'], draws[:, :6])          # engine order == SEPIA flat (Fortran) order
    np.testing.assert_array_equal(model.params.betaU.val, draws[-1, :6].reshape((3, 2), order='F'))
    sub = model.get_samples(5, nburn=4)                               # positional numsamples (assess_all_models.py:471)
    idx = [int(i) for i in np.linspace(4, 19, 5)]
    np.testing.assert_array_equal(sub['lamUz'], s['lamUz'][idx])
    assert model.get_samples(numsamples=64, nburn=0)['lamWs'].shape[0] == 20
    path = os.path.join(tmp_path, 'm')
    model.save_model_info(path)
    import pickle
    raw = pickle.load(open(path + '.pkl', 'rb'))
    assert np.array(raw['samples']['betaU']).shape == (20, 3, 2)      # mcmc_diagnostics_simple.py:31-35
    m2 = SepiaModel(_data(pr, 2))
    m2.restore_model_info(path)
    np.testing.assert_array_equal(m2.get_samples()['betaU'], s['betaU'])
    m2.clear_samples()
    assert m2.get_num_samples() == 0


def test_compute_paths_fail_loudly_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip('CUDA present')
    from gladsgp_b200._lib import GgpError
    from gladsgp_b200 import svd
    pr = make_problem(m=24, q=2, pu=2, n_x=6, n_t=5)
    from sepia.SepiaModel import SepiaModel
    model = SepiaModel(_data(pr, 2))
    from gladsgp_b200 import sensitivity
    for fn in (lambda: model.do_mcmc(2, prog=False), lambda: model.logLik(), lambda: model.tune_step_sizes(2, 2),
               lambda: model.tune_step_sizes(2, 2, parallel=True),
               lambda: svd.randomized_svd(pr['y_std'], 3, k=0),
               lambda: sensitivity.saltelli_sensitivity_indices(lambda x: x[:, :1] + x[:, 1:2], 2, 3, n_resamples=9)):
        with pytest.raises(GgpError):
            fn()


def test_logit_glm_recovers_known_coefficients():
    from gladsgp_b200.sepia.SepiaModel import _logit_glm
    x = np.log(np.array([0.025, 0.05, 0.1, 0.2, 0.4]))
    p = 1 / (1 + np.exp(-(-1.0 - 0.8 * x)))
    b = _logit_glm(x, 1000 * p, 1000)
    np.testing.assert_allclose(b, [-1.0, -0.8], atol=1e-6)


def test_library_exports_every_declared_symbol():
    from gladsgp_b200 import _lib
    hdr = open(os.path.join(ROOT, 'include', 'gladsgp_b200.h')).read()
    declared = sorted(set(re.findall(r'\b(ggp_[a-z0-9_]+)\s*\(', hdr)))
    assert len(declared) >= 15
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert sorted(_lib.SIGNATURES) == declared               # ctypes table mirrors the header one to one
    h = _lib.load()
    assert h.ggp_version() == 202
    assert h.ggp_padded_m(100) == 128 and h.ggp_factor_doubles(512) == 139264 + 16 * 1024 + 512 + 64
    # argument validation happens before any CUDA call
    assert h.ggp_cov_build_f64(None, 4, 2, None, None, None, 1, None, None) == -1
    assert b'null pointer' in h.ggp_last_error_string()
    assert ctypes.sizeof(_lib.McmcArgs) == h.ggp_sizeof_mcmc_args()


def test_legacy_normal_stream_is_call_size_invariant():
    """SepiaPredict draws the realisations of all samples with ONE np.random.normal call where SEPIA makes one call per
    sample: the legacy global stream (polar Box-Muller with its cached second value) gives the same numbers either way."""
    for per_call in (1, 3, 7, 10):
        np.random.seed(11)
        a = np.concatenate([np.random.normal(size=per_call) for _ in range(9)])
        np.random.seed(11)
        b = np.random.normal(size=9 * per_call)
        assert np.array_equal(a, b)
        assert np.random.random_sample() == (np.random.seed(11), np.random.normal(size=9 * per_call), np.random.random_sample())[2]


def test_normal_proposals_are_rejected_loudly():
    """The device sampler implements the proposal kinds of the GladsGP path (Uniform, BetaRho, PropMH); a parameter with
    a Normal step type must not be mis-sampled silently."""
    from gladsgp_b200.ops import PROP_KIND
    assert 'Normal' not in PROP_KIND and set(PROP_KIND) == {'Uniform', 'BetaRho', 'PropMH'}
    src = open(os.path.join(ROOT, 'gladsgp_b200', 'sepia', 'SepiaModel.py')).read()
    assert "if b.mcmc.stepType not in PROP_KIND:" in src and 'raise NotImplementedError' in src


def test_sepia_mirror_takes_the_reference_call_arguments():
    """The functions GladsGP's drivers call exist with the argument names they pass (src/model.py:57-106,225-238;
    assess_all_models.py:468-492)."""
    import inspect
    from sepia.SepiaModel import SepiaModel
    from sepia.SepiaData import SepiaData
    from sepia.SepiaPredict import SepiaEmulatorPrediction
    from sepia import SepiaParam
    assert {'t_sim', 'y_sim', 'y_ind_sim'} <= set(inspect.signature(SepiaData.__init__).parameters)
    assert {'y_mean', 'y_sd'} <= set(inspect.signature(SepiaData.standardize_y).parameters)
    assert 'K' in inspect.signature(SepiaData.create_K_basis).parameters
    assert list(inspect.signature(SepiaModel.tune_step_sizes).parameters)[1:3] == ['n_burn', 'n_levels']
    assert {'numsamples', 'nburn'} <= set(inspect.signature(SepiaModel.get_samples).parameters)
    assert {'t_pred', 'samples', 'model'} <= set(inspect.signature(SepiaEmulatorPrediction.__init__).parameters)
    assert {'val', 'name', 'val_shape', 'dist', 'params', 'bounds', 'mcmcStepParam', 'mcmcStepType'} <= \
        set(inspect.signature(SepiaParam.__init__).parameters)
