"""Developer benchmark: emulator Jacobians (ops.Predictor.jacobian, csrc/ggp_jacobian.cu) at cfg3 (m = 512, q = 8,
pu = 10) with 64 posterior samples and 8192 Sobol' points, against the central differences they replace.

Times, with CUDA events over several calls after a warm-up call, Predictor.jacobian in its full mode (the joint
(q+1) x (q+1) covariance per (block, design)) and its compact mode (2q + 1 values), and in the same run the 2q + 1
Predictor.predict calls of central differences (h = 1e-5 on the transformed scale).  The counted FP64 work per
(block, design) is
    (q+1) m^2 + (3d+2) m + q m + 2 (q+1)^2 Mp,
predict's flop model (tools/bench_predict.py) for each of the q + 1 rows, the derivative factors and the Gram.  Reports
the speed ratio to central differences and the largest difference between the two gradients (relative to the largest
gradient).  The card's name, power limit and maximum SM clock are read in the same run.  Prints one JSON line (also
written to DIR/bench_jacobian.json with --out DIR)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
from gladsgp_b200 import synthetic                          # noqa: E402
from gladsgp_b200.calibration import _designs, _predictor   # noqa: E402
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
    ap.add_argument('--samples', type=int, default=64)
    ap.add_argument('--points', type=int, default=8192)
    ap.add_argument('--iters', type=int, default=5)
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
    samples = synthetic.posterior_samples(args.samples, model.num.p + q, pu, seed=3)
    pred, ns = _predictor(model, samples)
    B, n, d, Mp = pred.B, args.points, pred.d, pred.Mp
    T = torch.as_tensor(qmc.Sobol(q, seed=1).random(n) * 0.98 + 0.01, device='cuda')
    X = _designs(T)
    res.update(m=m, q=q, pu=pu, samples=ns, points=n, blocks=B)
    flop = (q + 1) * m * m + (3 * d + 2) * m + q * m + 2 * (q + 1) ** 2 * Mp
    res['counted_flop_per_block_design'] = flop
    for full in (True, False):
        key = 'full' if full else 'compact'
        t = ev(lambda: pred.jacobian(X, 1, full=full), args.iters)
        res[key + '_ms'] = t
        res[key + '_pairs_per_s'] = B * n / (t * 1e-3)
        res[key + '_counted_tflops'] = B * n * flop / (t * 1e-3) * 1e-12
    h = 1e-5
    Xs = [X]
    for k in range(q):
        for sgn in (1.0, -1.0):
            Xk = X.clone()
            Xk[:, 1 + k] += sgn * h
            Xs.append(Xk)

    def central():
        return [pred.predict(x)[0] for x in Xs]
    t = ev(central, args.iters)
    res['central_differences_ms'] = t
    res['central_differences_predict_calls'] = len(Xs)
    res['speedup_full_vs_central'] = t / res['full_ms']
    res['speedup_compact_vs_central'] = t / res['compact_ms']
    mean, _ = pred.jacobian(X, 1, full=False)
    outs = central()
    fd = torch.stack([(outs[1 + 2 * k] - outs[2 + 2 * k]) / (2 * h) for k in range(q)], dim=-1)
    g = mean[..., 1:]
    res['max_abs_grad'] = float(g.abs().max())
    res['max_abs_diff_central_vs_jacobian'] = float((fd - g).abs().max())
    res['max_rel_diff_central_vs_jacobian'] = res['max_abs_diff_central_vs_jacobian'] / res['max_abs_grad']
    res['value_row_equals_predict'] = bool(torch.equal(mean[..., 0], outs[0]))
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'bench_jacobian.json'), 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
