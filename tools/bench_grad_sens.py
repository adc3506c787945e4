"""Developer benchmark: closed-form gradient outer products (active subspaces, DGSM) at cfg3 (m = 512, q = 8, pu = 10) with
64 and 256 posterior samples.

For each sample count: ops.grad_sens in its four modes (0 per (sample, PC) block, 1 per PC over every sample, 2 per sample
over every PC with the field's Omega, 3 one function over everything), timed with CUDA events over several launches after
a warm-up launch; (pair, input) integrals per second count the q inputs of every evaluated pair n <= n', as
bench_gp_sens.py counts them.  In the same run: ops.gp_sens in its modes 0 and 1 (the Sobol' moments of the same
functions), and the finite-difference Monte-Carlo route, central differences of emulator_mean_function at 8192 Sobol'
points ((2q + 1) predictions per point).  A mode whose counted work exceeds --max-integrals is reported as not measured.
The card's name, power limit and maximum SM clock are read in the same run.  Prints one JSON line (also written to
DIR/bench_grad_sens.json with --out DIR)."""
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
    ap.add_argument('--max-integrals', type=float, default=1e12)
    ap.add_argument('--fd-points', type=int, default=8192)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    from sepia.SepiaData import SepiaData
    from sepia.SepiaModel import SepiaModel
    from scipy.stats import qmc
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
    omega = sensitivity._field_omega(model, None)
    for ns in args.samples:
        r = {}
        samples = synthetic.posterior_samples(ns, model.num.p + q, pu, seed=3)
        Z, beta, a, _ = sensitivity.emulator_expansion(model, samples)
        a_mean = a / ns
        for mode in range(4):
            N = m * (1, ns, pu, ns * pu)[mode]
            F = (ns * pu, pu, ns, 1)[mode]
            integrals = F * N * (N + 1) / 2 * q
            key = 'mode%d' % mode
            r[key + '_pair_integrals'] = integrals
            if integrals > args.max_integrals:
                r[key + '_ms'] = None
                continue
            aa = a_mean if mode in (1, 3) else a
            iters = 10 if integrals < 1e11 else 2
            t = ev(lambda: ops.grad_sens(Z, beta, aa, ns, pu, mode, omega), iters=iters)
            r[key + '_ms'] = t
            r[key + '_pair_integrals_per_s'] = integrals / (t * 1e-3)
        for mode in (0, 1):
            N = m * (1, ns)[mode]
            F = (ns * pu, pu)[mode]
            integrals = F * N * (N + 1) / 2 * q
            aa = a_mean if mode == 1 else a
            iters = 10 if integrals < 1e11 else 2
            t = ev(lambda: ops.gp_sens(Z, beta, aa, ns, pu, mode), iters=iters)
            r['gp_sens_mode%d_ms' % mode] = t
            r['gp_sens_mode%d_pair_integrals_per_s' % mode] = integrals / (t * 1e-3)
        # the Monte-Carlo route: central differences of the posterior-mean function at Sobol' points
        func = sensitivity.emulator_mean_function(model, samples)
        X = qmc.Sobol(q, seed=1).random(args.fd_points)
        h = 1e-5
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        G = np.empty((args.fd_points, pu, q))
        func(X)
        for k in range(q):
            e = np.zeros(q)
            e[k] = h
            G[:, :, k] = (func(X + e) - func(X - e)) / (2 * h)
        np.einsum('pjk,pjl->jkl', G, G) / args.fd_points
        r['fd_mc_wall_ms'] = (time.perf_counter() - t0) * 1e3
        r['fd_mc_predictions'] = args.fd_points * (2 * q + 1)
        t0 = time.perf_counter()
        sensitivity.gp_active_subspace(model, samples, option='samples', target='pc')
        r['gp_active_subspace_samples_pc_wall_ms'] = (time.perf_counter() - t0) * 1e3
        res['ns%d' % ns] = r
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'bench_grad_sens.json'), 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
