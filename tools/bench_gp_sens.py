"""Developer benchmark: closed-form GP sensitivity at cfg3 (m = 512, q = 8, pu = 10) with 64 and 256 posterior samples.

For each sample count: the weights a = S22^-1 w / lamUz from the cached factors (emulator_expansion, warm), ops.gp_sens in
both modes ('samples': one function per (sample, PC) block; 'mean': the posterior-mean function per PC, every pair of
(sample, row) terms) and ops.main_effects, timed with CUDA events; pair-integrals per second count the q I2 integrals of
every evaluated pair (n <= n').  For comparison, the wall time of the Monte-Carlo route
PCA_saltelli_sensitivity_indices(emulator_mean_function(...), m=8, bootstrap=True) on the same model.  Prints one JSON
line (also written to DIR/bench_gp_sens.json with --out DIR)."""
import argparse
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
from gladsgp_b200 import ops, sensitivity, synthetic       # noqa: E402
from helpers import make_problem                             # noqa: E402


def ev(fn, iters, warm=1):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--samples', type=int, nargs='+', default=[64, 256])
    ap.add_argument('--out', default=None)
    ap.add_argument('--no-saltelli', action='store_true')
    args = ap.parse_args()
    from sepia.SepiaData import SepiaData
    from sepia.SepiaModel import SepiaModel
    res = {}
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res['gpu'] = torch.cuda.get_device_name(0)
    res['nvidia_smi'] = smi[0] if smi else None
    m, q, pu = 512, 8, 10
    pr = make_problem(m=m, q=q, pu=pu, n_x=64, n_t=16)
    data = SepiaData(t_sim=pr['t'], y_sim=pr['y'], y_ind_sim=np.arange(pr['y'].shape[1], dtype=float))
    data.transform_xt(t_notrans=np.arange(q)); data.standardize_y(y_mean=pr['mu'], y_sd=pr['sd']); data.create_K_basis(K=pr['K'])
    model = SepiaModel(data)
    pcvar = np.full(pu, 1.0 / pu)
    grid = np.linspace(0.0, 1.0, 21)
    for ns in args.samples:
        r = {}
        samples = synthetic.posterior_samples(ns, model.num.p + q, pu, seed=3)
        model._pred_cache = None
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        Z, beta, a, _ = sensitivity.emulator_expansion(model, samples)        # cold: builds and caches the factors
        torch.cuda.synchronize()
        r['expansion_cold_ms'] = (time.perf_counter() - t0) * 1e3
        r['weights_ms'] = ev(lambda: sensitivity.emulator_expansion(model, samples), iters=5)
        for option, mode in (('samples', 0), ('mean', 1)):
            aa = a if mode == 0 else a / ns
            N = m if mode == 0 else ns * m
            F = ns * pu if mode == 0 else pu
            pairs = F * N * (N + 1) / 2
            iters = 10 if pairs * q < 1e11 else 2
            t = ev(lambda: ops.gp_sens(Z, beta, aa, ns, pu, mode), iters=iters)
            r[option + '_ms'] = t
            r[option + '_pair_integrals'] = pairs * q
            r[option + '_pair_integrals_per_s'] = pairs * q / (t * 1e-3)
            r[option + '_main_effects_ms'] = ev(lambda: ops.main_effects(Z, beta, aa, ns, pu, grid, mode), iters=iters)
        t0 = time.perf_counter()
        sensitivity.gp_sensitivity_indices(model, samples, option='mean', pcvar=pcvar)
        r['gp_sensitivity_indices_mean_wall_ms'] = (time.perf_counter() - t0) * 1e3
        if not args.no_saltelli:
            func = sensitivity.emulator_mean_function(model, samples)
            np.random.seed(0)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            sensitivity.PCA_saltelli_sensitivity_indices(func, q, 8, pcvar, bootstrap=True)
            r['saltelli_m8_bootstrap_wall_ms'] = (time.perf_counter() - t0) * 1e3
        res['ns%d' % ns] = r
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'bench_gp_sens.json'), 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
