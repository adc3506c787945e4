"""Shared builders of the posterior-consumer tests (calibration, history matching, sequential design, GP sensitivity and
the posterior-draw tests): SEPIA models of the tests/helpers.py problems, the oracle emulator on exactly a model's design,
PC weights and LamSim, observation terms, and the golden posterior draws of tests/golden/posterior_cfg*.npz."""
import os

import numpy as np

from helpers import make_problem, make_scalar_problem
from oracle import calib_oracle as co
from oracle import sepia_oracle as so

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


# --------------------------------------------------------------------------------------------------------------------
# models and the oracle emulator
# --------------------------------------------------------------------------------------------------------------------
def sepia_model_of(pr, K=None, t_notrans=False):
    """SepiaModel of a make_problem result.  t_notrans: keep the design as it is (zt equal to the oracle problem's)."""
    from sepia.SepiaData import SepiaData
    from sepia.SepiaModel import SepiaModel
    q = pr['t'].shape[1]
    data = SepiaData(t_sim=pr['t'], y_sim=pr['y'], y_ind_sim=np.arange(pr['y'].shape[1], dtype=float))
    if t_notrans:
        data.transform_xt(t_notrans=np.arange(q))
    else:
        data.transform_xt()
    data.standardize_y(y_mean=pr['mu'], y_sd=pr['sd']); data.create_K_basis(K=pr['K'] if K is None else K)
    return SepiaModel(data)


def sepia_model(m=64, q=3, pu=2, seed=5, n_x=20, n_t=10, K=None):
    pr = make_problem(m=m, q=q, pu=min(pu, 25), n_x=n_x, n_t=n_t, seed=seed)
    return sepia_model_of(pr, K=K)


def scalar_model_of(pr, t_notrans=False):
    from sepia.SepiaData import SepiaData
    from sepia.SepiaModel import SepiaModel
    data = SepiaData(t_sim=pr['t'], y_sim=pr['y'])
    if t_notrans:
        data.transform_xt(t_notrans=np.arange(1))
    else:
        data.transform_xt()
    data.standardize_y()
    return SepiaModel(data)


def scalar_model(m=200):
    return scalar_model_of(make_scalar_problem(m=m))


def oracle_num(model):
    """Oracle problem on exactly the model's design, PC weights and LamSim."""
    sd = model.data.sim_data
    K = None if model.data.scalar_out else np.asarray(sd.K, dtype=np.float64)
    num = so.OracleNum(model.num.zt[:, 1:], np.asarray(sd.y_std, dtype=np.float64), K)
    num.w = model._w_pcs.T.copy()
    num.wv = num.w.reshape((-1, 1), order='F')
    num.LamSim = np.asarray(model.num.LamSim, dtype=np.float64)
    return num


def emulator(model, samples):
    """Oracle emulator on exactly the model's design, PC weights and LamSim."""
    return co.Emulator(oracle_num(model), samples)


def native(model, tt):
    """Transformed inputs [0, 1] -> the model's native inputs."""
    sd = model.data.sim_data
    return tt * (sd.orig_t_max - sd.orig_t_min) + sd.orig_t_min


def basis(model):
    sd = model.data.sim_data
    return np.ones((1, 1)) if model.data.scalar_out else np.asarray(sd.K, dtype=np.float64)


def at(model, v, O):
    """A scalar or per-output standardisation vector at outputs O."""
    v = np.asarray(v, dtype=np.float64).reshape(-1)
    return np.broadcast_to(v, (basis(model).shape[1],))[O]


def mean_field(model, em, O, theta_star):
    """Native outputs O of the oracle's mixture mean at theta_star (transformed)."""
    sd = model.data.sim_data
    mu, _ = em.moments(np.asarray(theta_star, dtype=np.float64)[None])
    return (mu[:, :, 0].mean(0) @ basis(model)[:, O]) * at(model, sd.orig_y_sd, O) + at(model, sd.orig_y_mean, O)


def calib_obs(model, O, y_obs, obs_sd, samples):
    """Oracle Woodbury terms G, b, c0 of native observations at outputs O."""
    sd = model.data.sim_data
    r, tau = co.standardized_obs(y_obs, obs_sd, at(model, sd.orig_y_mean, O), at(model, sd.orig_y_sd, O))
    return co.obs_terms(basis(model)[:, O], r, tau, np.asarray(samples['lamWOs'], dtype=np.float64).reshape(-1))


def hm_obs(model, samples, O, y, obs_sd, disc_sd):
    """K_O, r, c of the history-matching oracle for native observations y at outputs O."""
    sd = model.data.sim_data
    ysd = at(model, sd.orig_y_sd, O)
    r, tau = co.standardized_obs(y, obs_sd, at(model, sd.orig_y_mean, O), ysd)
    delta = np.broadcast_to(np.asarray(disc_sd, dtype=np.float64), (O.size,)) / ysd
    rho = np.mean(1.0 / np.asarray(samples['lamWOs'], dtype=np.float64).reshape(-1))
    return basis(model)[:, O], r, rho + tau ** 2 + delta ** 2


# --------------------------------------------------------------------------------------------------------------------
# golden posterior draws (tests/golden/make_golden_posterior.py)
# --------------------------------------------------------------------------------------------------------------------
def load_posterior(cfg):
    g = np.load(os.path.join(GOLD, 'posterior_%s.npz' % cfg))
    return {k: g[k] for k in g.files}


def fixture_problem(g):
    """The tests/helpers.py problem a posterior fixture was drawn on."""
    args = {k[4:]: g[k].item() for k in g if k.startswith('arg_')}
    return make_problem(**args) if str(g['kind']) == 'pca' else make_scalar_problem(**args)


def split_draws(draws, d, pu):
    """(S, P) draws in sampling order -> the samples dict of SepiaEmulatorPrediction and the consumers."""
    draws = np.asarray(draws, dtype=np.float64)
    nb = d * pu
    return dict(betaU=draws[:, :nb].copy(), lamUz=draws[:, nb:nb + pu].copy(), lamWs=draws[:, nb + pu:nb + 2 * pu].copy(),
                lamWOs=draws[:, nb + 2 * pu:nb + 2 * pu + 1].copy())
