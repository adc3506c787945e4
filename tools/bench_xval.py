"""Developer benchmark: leave-one-out cross-validation at cfg3 (m = 512, q = 8, pu = 10, 64 posterior samples).

Times ggp_xval_solve_f64 with ascending indices (each row skips the panels above it: 640 * m^3/3 flop) and with the
same indices permuted (the skip is lost: up to 640 * m^3 flop), the whole SepiaXvalEmulatorPrediction call cold (factors
built) and warm (factors cached with the model), and SEPIA's refit route -- a sub-model Predictor per fold -- on 16 folds,
extrapolated to 512; reports the largest difference between the two routes.  Prints one JSON line."""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
from gladsgp_b200 import ops, synthetic                     # noqa: E402
from helpers import make_problem                             # noqa: E402


def ev(fn, iters=10, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), float(np.min(ts))


def wall(fn, iters=3):
    ts = []
    for _ in range(iters):
        torch.cuda.synchronize()
        t0 = time.perf_counter(); fn(); torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def main():
    from sepia.SepiaData import SepiaData
    from sepia.SepiaModel import SepiaModel
    from sepia.SepiaPredict import SepiaXvalEmulatorPrediction
    res = {}
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res['gpu'] = torch.cuda.get_device_name(0)
    res['nvidia_smi'] = smi[0] if smi else None
    m, q, pu, ns = 512, 8, 10, 64
    pr = make_problem(m=m, q=q, pu=pu, n_x=64, n_t=16)
    data = SepiaData(t_sim=pr['t'], y_sim=pr['y'], y_ind_sim=np.arange(pr['y'].shape[1], dtype=float))
    data.transform_xt(t_notrans=np.arange(q)); data.standardize_y(y_mean=pr['mu'], y_sd=pr['sd']); data.create_K_basis(K=pr['K'])
    model = SepiaModel(data)
    samples = synthetic.posterior_samples(ns, model.num.p + q, pu, seed=3)

    # whole call: cold builds the 640 factors, warm finds them in the model's cache
    def cold():
        model._pred_cache = None
        SepiaXvalEmulatorPrediction(samples=samples, model=model)
    cold()
    res['class_cold_ms'] = wall(cold)
    res['class_warm_ms'] = wall(lambda: SepiaXvalEmulatorPrediction(samples=samples, model=model))
    xv = SepiaXvalEmulatorPrediction(samples=samples, model=model, storeRlz=False)
    P = model._pred_cache[1]
    B = P.B
    flop = B * m ** 3 / 3.0
    res['blocks'] = B
    res['model_flop'] = flop
    idx = torch.arange(m, dtype=torch.int32, device='cuda')
    perm = idx[torch.randperm(m, generator=torch.Generator().manual_seed(0)).cuda()]
    # alternate the two orders so that both see the same machine state
    asc, per = [], []
    for _ in range(3):
        asc.append(ev(lambda: P.xval_solve(idx), iters=20)[0])
        per.append(ev(lambda: P.xval_solve(perm), iters=20)[0])
    res['kernel_ascending_ms'] = min(asc)
    res['kernel_permuted_ms'] = min(per)
    res['kernel_ascending_tflops_vs_m3_3'] = flop / min(asc) / 1e9
    res['kernel_permuted_tflops_vs_m3_3'] = flop / min(per) / 1e9
    res['skip_speedup'] = min(per) / min(asc)

    # SEPIA's route: one sub-model per fold (factor the 511 x 511 S22 of every block, predict the held-out row)
    lamWOs = np.asarray(samples['lamWOs'], dtype=np.float64).reshape(-1, 1)
    _, beta, lamz, dadd, s11, W = xv._blocks()
    c = (1.0 / (model.num.LamSim[None, :] * lamWOs)).reshape(-1)
    mu_x, var_x, _ = P.xval([[i] for i in range(m)], c)
    mu_x, var_x = mu_x.cpu().numpy(), var_x.cpu().numpy()
    zt = model.num.zt
    folds = np.linspace(0, m - 1, 16).astype(int)
    dmu = dvar = 0.0
    refit_ms = []
    for i in folds:
        keep = np.setdiff1d(np.arange(m), [i])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sub = ops.Predictor(zt[keep], W[:, keep], beta, lamz, dadd, s11)
        mean, var = sub.predict(zt[i:i + 1])
        mean, var = mean.cpu().numpy()[:, 0], var.cpu().numpy()[:, 0]
        refit_ms.append((time.perf_counter() - t0) * 1e3)
        dmu = max(dmu, float(np.abs(mean - mu_x[:, i]).max() / np.abs(mu_x).max()))
        dvar = max(dvar, float(np.abs((var - var_x[:, i]) / var_x[:, i]).max()))
    res['refit_ms_per_fold'] = float(np.median(refit_ms[1:]))
    res['refit_ms_512_folds_extrapolated'] = res['refit_ms_per_fold'] * m
    res['refit_over_warm_class'] = res['refit_ms_512_folds_extrapolated'] / res['class_warm_ms']
    res['max_rel_diff_mean'] = dmu
    res['max_rel_diff_var'] = dvar
    print(json.dumps(res))


if __name__ == '__main__':
    main()
