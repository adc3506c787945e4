#!/usr/bin/env python
"""End-to-end walk through the reference workflow on a synthetic GlaDS-shaped ensemble (cfg 1 shape:
m = 100 simulations, 8 parameters, 5 PCs), on the GPU:

    fit   : gladsgp_b200.model.fit_models  (mirror of /root/reference/src/model.py:152-245: rSVD -> K basis ->
            SepiaModel -> lamWOs override -> tune_step_sizes(100, 5) -> do_mcmc(512) -> pickle + timing.csv)
    assess: the prediction pattern of experiments/synthetic/analysis/assess_all_models.py:468-500
            (get_samples(64, nburn=256), batches of 4 test designs, get_y, truncation noise, mean / quantiles)

Usage: python examples/synthetic_fit_predict.py [workdir] [--nx 200 --nt 36 --mcmc 512]
"""
import argparse
import os
import sys
import tempfile
import time
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from gladsgp_b200 import model as gmodel, synthetic          # noqa: E402
from sepia.SepiaPredict import SepiaEmulatorPrediction, SepiaXvalEmulatorPrediction   # noqa: E402


def make_config(workdir, m, q, n_x, n_t, tag, seed):
    """Writes X_standard (csv with header) and Y_physical ((n_y, m) .npy, the layout of
    src/aggregate_outputs.py:61-68) and returns a config module like experiments/synthetic/train_config.py."""
    t = synthetic.design(m, q, seed=seed) if tag == 'train' else synthetic.test_design(m, q, seed=seed)
    y = synthetic.ensemble(t, n_x=n_x, n_t=n_t, seed=20240318)
    os.makedirs(workdir, exist_ok=True)
    xs = os.path.join(workdir, '%s_standard.csv' % tag)
    np.savetxt(xs, t, delimiter=',', header=','.join('p%d' % i for i in range(q)), comments='')
    yp = os.path.join(workdir, '%s_ff.npy' % tag)
    np.save(yp, y.T)
    cfg = types.SimpleNamespace(exp='synthetic', m=m, p=5, X_standard=xs, Y_physical=yp, data_dir=os.path.join(workdir, 'data'))
    return cfg, t, y


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('workdir', nargs='?', default=None)
    ap.add_argument('--m', type=int, default=100)
    ap.add_argument('--nx', type=int, default=200)
    ap.add_argument('--nt', type=int, default=36)
    ap.add_argument('--mcmc', type=int, default=512)
    ap.add_argument('--tune', type=int, default=100)
    ap.add_argument('--ntest', type=int, default=16)
    args = ap.parse_args()
    workdir = args.workdir or tempfile.mkdtemp(prefix='gladsgp_')
    q, pu = 8, 5
    train, t_train, y_train = make_config(workdir, args.m, q, args.nx, args.nt, 'train', 20240318)
    test, t_test, y_test = make_config(workdir, args.ntest, q, args.nx, args.nt, 'test', 42186)
    np.random.seed(0)
    t0 = time.perf_counter()
    gmodel.fit_models(train, [args.m], [pu], n_tune=(args.tune, 5), n_mcmc=args.mcmc)
    print('fit_models: %.2f s' % (time.perf_counter() - t0))

    data, model = gmodel.load_model(train, args.m, pu)
    n_samp = min(64, args.mcmc // 2)
    samples = model.get_samples(n_samp, nburn=args.mcmc // 2)
    for key in samples.keys():
        samples[key] = samples[key].astype(np.float32)                       # assess_all_models.py:473-474
    sd_y = np.std(model.data.sim_data.y, ddof=1, axis=0); sd_y[sd_y < 1e-6] = 1e-6
    ypred_mean = np.zeros_like(y_test); lq = np.zeros_like(y_test); uq = np.zeros_like(y_test)
    t0 = time.perf_counter()
    for j0 in range(0, args.ntest, 4):                                      # batches of 4 (assess_all_models.py:481)
        tj = t_test[j0:j0 + 4]
        preds = SepiaEmulatorPrediction(t_pred=tj, samples=samples, model=model)
        preds.w = preds.w.astype(np.float32)
        noise = np.random.normal(size=(n_samp, len(tj))) / np.sqrt(samples['lamWOs'][:, :1])
        st = preds.get_y_stats(quantile=0.025, noise=noise.astype(np.float32))   # fused get_y + mean + quantiles
        ypred_mean[j0:j0 + 4], lq[j0:j0 + 4], uq[j0:j0 + 4] = st['mean'], st['lq'], st['uq']
    print('prediction + statistics for %d designs: %.2f s' % (args.ntest, time.perf_counter() - t0))
    rmse = np.sqrt(np.mean((ypred_mean - y_test) ** 2))
    cover = np.mean((y_test >= lq) & (y_test <= uq))
    print('test RMSE %.4f (field sd %.3f), 95%% interval coverage %.3f' % (rmse, y_test.std(), cover))
    # leave-one-out cross-validation on the training set: no test ensemble needed, same samples (cached factors)
    t0 = time.perf_counter()
    xv = SepiaXvalEmulatorPrediction(samples=samples, model=model)
    xv.w = xv.w.astype(np.float32)
    err = xv.get_y_error_stats(y_test=y_train.astype(np.float32))
    print('leave-one-out over %d simulations: %.2f s, RMSE %.4f, 95%% interval coverage %.3f'
          % (args.m, time.perf_counter() - t0, float(np.sqrt(np.mean(err['rmse'] ** 2))), float(np.mean(err['frac_covered']))))
    print('artefacts in', os.path.join(workdir, 'data', 'models'), sorted(os.listdir(os.path.join(workdir, 'data', 'models'))))
    return rmse, cover


if __name__ == '__main__':
    main()
