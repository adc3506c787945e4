"""Developer benchmark: history matching (gladsgp_b200.history) at cfg3 (m = 512, q = 8, pu = 10) on the synthetic
GlaDS-shaped ensemble of 4000 sites x 365 days (1.46 M outputs), fitted as model.init_model does (the model of
tools/bench_design.py).

For S in {16, 64} posterior samples and two workloads -- N = 2^20 points against n_o = 2048 outputs spread over the field,
and N = 2^16 points against the full field -- the device time of the predictive moments (ggp_predict_f64) and of
ggp_hm_impl_f64 (mixture, DMMA pair and merge kernels), CUDA events around each, the moments computed for all N points at
once; and the whole history_match call behind a synchronise.  The counted flop of the pair products is
2 N n_o (Fe + Fv), given both with the padded feature widths the kernel multiplies (Fe = 16, Fv = 56 at pu = 10) and
unpadded (pu + 1 and pu (pu + 1) / 2 + 1), reported over bench.fp64_peak_tflops of the same run.  The observations are
the emulator's mean field at the centre of the input box.  The FP64 oracle is timed at a reduced size.  Prints one JSON
line (also written to DIR/bench_hm.json with --out DIR)."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench                                                                     # noqa: E402
from gladsgp_b200 import calibration as cal, history, model as gmodel, ops, synthetic   # noqa: E402
from oracle import calib_oracle as co, hm_oracle as ho, sepia_oracle as so     # noqa: E402

M, Q, PU = 512, 8, 10


def build_model(n_x, n_t):
    t = synthetic.design(M, Q, seed=synthetic.BASE_SEED)
    y = synthetic.ensemble(t, n_x=n_x, n_t=n_t, seed=synthetic.BASE_SEED + 3)
    with tempfile.TemporaryDirectory() as d:
        data, model = gmodel.init_model(t, y, 'hm', PU, data_dir=d)
    return model


def observations(model, samples, O):
    """Native y_obs at outputs O: the emulator's mixture mean at the centre of the box."""
    pred, S = cal._predictor(model, samples)
    mean, _ = pred.predict(cal._designs(torch.full((1, Q), 0.5, dtype=torch.float64, device='cuda')))
    m = mean.reshape(S, PU).mean(0)
    sd = model.data.sim_data
    Od = torch.as_tensor(O, device='cuda')
    K_O = sd.K_device()[:, Od].to(torch.float64)

    def at(v):
        v = np.asarray(v, dtype=np.float64).reshape(-1)
        return np.broadcast_to(v, (O.size,)) if v.size == 1 else v[O]
    ysd = at(sd.orig_y_sd)
    return (m @ K_O).cpu().numpy() * ysd + at(sd.orig_y_mean), K_O, ysd


def timed(model, samples, O, y, K_O, ysd, t, order, reps):
    """Device times (ms) of the moments of all points and of ggp_hm_impl_f64 on them."""
    pred, S = cal._predictor(model, samples)
    _, r, tau = cal._obs(model, y, O, 0.0)
    rho = float(np.mean(1.0 / np.asarray(samples['lamWOs'], dtype=np.float64).reshape(-1)))
    delta = 0.05 * np.ones(O.size)                                # disc_sd = 5 % of each output's sd
    rd = torch.as_tensor(r, device='cuda')
    cd = torch.as_tensor(rho + tau ** 2 + delta ** 2, device='cuda')
    X = cal._designs(torch.as_tensor(cal._to_trans(model, t), device='cuda'))
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    mean, var = pred.predict(X)
    ev[1].record()
    torch.cuda.synchronize()
    predict_ms = ev[0].elapsed_time(ev[1])
    ops.hm_impl(mean, var, K_O, rd, cd, order, 3.0)              # warm-up
    ms = []
    for _ in range(reps):
        ev[0].record()
        impl, _ = ops.hm_impl(mean, var, K_O, rd, cd, order, 3.0)
        ev[1].record()
        torch.cuda.synchronize()
        ms.append(ev[0].elapsed_time(ev[1]))
    del mean, var
    return dict(predict_ms=predict_ms, hm_ms=ms, hm_ms_median=float(np.median(ms)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--samples', type=int, nargs='+', default=[16, 64])
    ap.add_argument('--sites', type=int, default=4000)
    ap.add_argument('--log2-points', type=int, nargs=2, default=[20, 16], help='log2 N of the two workloads')
    ap.add_argument('--n-obs', type=int, default=2048, help='observed outputs of the first workload')
    ap.add_argument('--order', type=int, default=3)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    res = {}
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res['gpu'] = torch.cuda.get_device_name(0)
    res['nvidia_smi'] = smi[0] if smi else None
    model = build_model(args.sites, 365)
    n_y = model.num.n_y
    rng = np.random.default_rng(0)
    sd = model.data.sim_data
    lo, hi = np.asarray(sd.orig_t_min).reshape(-1), np.asarray(sd.orig_t_max).reshape(-1)
    peak = bench.fp64_peak_tflops(torch, sustained_s=2.0)        # cuBLAS FP64 GEMM: (burst, sustained) TFLOP/s
    res['fp64_peak_tflops'] = dict(burst=peak[0], sustained=peak[1])
    Fe, Fv = (PU + 1 + 7) // 8 * 8, (PU * (PU + 1) // 2 + 1 + 7) // 8 * 8
    Fe_u, Fv_u = PU + 1, PU * (PU + 1) // 2 + 1
    work = [('sparse', 1 << args.log2_points[0], np.sort(rng.choice(n_y, size=args.n_obs, replace=False))),
            ('field', 1 << args.log2_points[1], np.arange(n_y))]
    for S in args.samples:
        samples = synthetic.posterior_samples(S, 1 + Q, PU, seed=S)
        model._pred_cache = None
        cal._predictor(model, samples)
        for name, N, O in work:
            t = rng.uniform(lo, hi, (N, Q))
            y, K_O, ysd = observations(model, samples, O)
            r = timed(model, samples, O, y, K_O, ysd, t, args.order, args.reps if name == 'sparse' else max(2, args.reps // 2))
            del K_O
            flop = 2.0 * N * O.size * (Fe + Fv)
            r.update(N=N, n_o=int(O.size), order=args.order, flop_padded=flop,
                     flop_unpadded=2.0 * N * O.size * (Fe_u + Fv_u),
                     tflops_padded=flop / (r['hm_ms_median'] * 1e-3) / 1e12)
            r['fraction_of_peak_padded'] = dict(burst=r['tflops_padded'] / peak[0], sustained=r['tflops_padded'] / peak[1])
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = history.history_match(model, samples, y, t, obs_index=O, disc_sd=0.05 * ysd, order=args.order)
            torch.cuda.synchronize()
            r['history_match_wall_s'] = time.perf_counter() - t0
            r['nroy_fraction'] = out['nroy_fraction']
            res['S%d_%s' % (S, name)] = r
            print(json.dumps({('S%d_%s' % (S, name)): r}), file=sys.stderr)
            del out
    # FP64 oracle (feature route) at a reduced size: 2 samples, 64 points, 256 outputs
    samples = synthetic.posterior_samples(2, 1 + Q, PU, seed=2)
    K = np.asarray(sd.K, dtype=np.float64)
    num = so.OracleNum(model.num.zt[:, 1:], np.zeros((M, PU)), np.eye(PU))     # the model's weights set below
    num.w = model._w_pcs.T.copy()
    num.wv = num.w.reshape((-1, 1), order='F')
    num.LamSim = np.asarray(model.num.LamSim, dtype=np.float64)
    O = np.sort(rng.choice(n_y, size=256, replace=False))
    t0 = time.perf_counter()
    em = co.Emulator(num, samples)
    ho.history_match(em, rng.uniform(0, 1, (64, Q)), K[:, O], rng.standard_normal(256), np.full(256, 0.1), 3, 3.0)
    res['host_oracle'] = dict(samples=2, N=64, n_o=256, s=time.perf_counter() - t0)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'bench_hm.json'), 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
