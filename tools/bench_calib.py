"""Developer benchmark: emulator-based calibration (gladsgp_b200.calibration) at cfg3 (m = 512, q = 8, pu = 10) on the
synthetic GlaDS-shaped ensemble of 4000 sites x 365 days (n_y = 1 460 000 outputs), fitted as model.init_model does.

For S in {16, 64} posterior samples and C in {64, 256, 1024} chains: the device time of one step split into the predict
kernel (ggp_predict_f64 on the C candidates) and the step kernel (ggp_calib_step_f64), CUDA events around each over many
steps, and chain-steps/s from their sum and from a host clock around 200 whole steps (launch gaps included).  The predict
kernel's FP64 rate counts B n (m^2 + 4 m) flop per call (B = S pu blocks, n = C designs: the triangular solve and the mean
/ variance products; the cross covariance is not counted).  C = 64 shows what a call below the kernel's 256-design task
costs.  The one-off precompute (_obs_terms) is timed for n_o = 7300 (20 sites x 365 days) and for the full field, and the
FP64 host oracle's likelihood evaluations per second at S = 4 on 16 points.  Prints one JSON line (also written to
DIR/bench_calib.json with --out DIR)."""
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
from gladsgp_b200 import calibration as cal, model as gmodel, ops, synthetic     # noqa: E402
from oracle import calib_oracle as co, sepia_oracle as so                       # noqa: E402

M, Q, PU, N_SITES, N_DAYS = 512, 8, 10, 4000, 365


def build_model(n_x, n_t):
    t = synthetic.design(M, Q, seed=synthetic.BASE_SEED)
    y = synthetic.ensemble(t, n_x=n_x, n_t=n_t, seed=synthetic.BASE_SEED + 3)
    with tempfile.TemporaryDirectory() as d:
        data, model = gmodel.init_model(t, y, 'calib', PU, data_dir=d)
    return model, y


def timed_steps(pred, G, b, c0, C, n_steps, gen):
    """Per-step device times (ms) of the predict and step kernels over n_steps steps, and a host-clock total."""
    q = Q
    lo = torch.zeros(q, dtype=torch.float64, device='cuda')
    hi = torch.ones(q, dtype=torch.float64, device='cuda')
    L = torch.diag(torch.full((q,), 0.02, dtype=torch.float64, device='cuda'))
    theta = torch.rand((C, q), generator=gen, dtype=torch.float64, device='cuda')
    Xp = cal._designs(theta)
    mean, var = pred.predict(Xp)
    ll = ops.calib_loglik(mean, var, G, b, c0)
    z = torch.randn((n_steps, C, q), generator=gen, dtype=torch.float64, device='cuda')
    logu = torch.log(torch.rand((n_steps, C), generator=gen, dtype=torch.float64, device='cuda'))
    rt = torch.empty((C, q), dtype=torch.float64, device='cuda')
    rl = torch.empty(C, dtype=torch.float64, device='cuda')
    ra = torch.empty(C, dtype=torch.uint8, device='cuda')
    Xp[:, 1:] = theta + z[0] @ L.T

    def step(t, ev=None):
        if ev:
            ev[0].record()
        mean, var = pred.predict(Xp)
        if ev:
            ev[1].record()
        ops.calib_step(mean, var, G, b, c0, Xp, lo, hi, L, z[(t + 1) % n_steps], logu[t], theta, ll, rt, rl, ra)
        if ev:
            ev[2].record()
    for t in range(5):
        step(t)
    torch.cuda.synchronize()
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(n_steps)]
    for t in range(n_steps):
        step(t, evs[t])
    torch.cuda.synchronize()
    tp = float(np.median([e[0].elapsed_time(e[1]) for e in evs]))
    ts = float(np.median([e[1].elapsed_time(e[2]) for e in evs]))
    t0 = time.perf_counter()
    for t in range(n_steps):
        step(t)
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) * 1e3 / n_steps
    return tp, ts, wall


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--samples', type=int, nargs='+', default=[16, 64])
    ap.add_argument('--chains', type=int, nargs='+', default=[64, 256, 1024])
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--sites', type=int, default=N_SITES)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    res = {}
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res['gpu'] = torch.cuda.get_device_name(0)
    res['nvidia_smi'] = smi[0] if smi else None
    t0 = time.perf_counter()
    model, y = build_model(args.sites, N_DAYS)
    res['setup_s'] = time.perf_counter() - t0
    n_y = model.num.n_y
    res['n_y'] = n_y
    sites = np.linspace(0, args.sites - 1, 20).astype(np.int64)
    O7300 = (sites[:, None] * N_DAYS + np.arange(N_DAYS)[None, :]).reshape(-1)
    y_obs = np.asarray(y[17], dtype=np.float64)                        # one training run's field as the observation
    del y
    gen = torch.Generator(device='cuda')
    gen.manual_seed(0)
    m = M
    for S in args.samples:
        samples = synthetic.posterior_samples(S, 1 + Q, PU, seed=S)
        r = {}
        for name, O in (('n_o_7300', O7300), ('full_field', None)):
            yo = y_obs if O is None else y_obs[O]
            cal._obs_terms(model, samples, yo, O, 0.01)                 # warm-up (device copy of K)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            G, b, c0 = cal._obs_terms(model, samples, yo, O, 0.01)
            torch.cuda.synchronize()
            r['precompute_ms_' + name] = (time.perf_counter() - t0) * 1e3
        model._pred_cache = None
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        pred, _ = cal._predictor(model, samples)
        torch.cuda.synchronize()
        r['factor_build_ms'] = (time.perf_counter() - t0) * 1e3
        B = S * PU
        for C in args.chains:
            tp, ts, wall = timed_steps(pred, G, b, c0, C, args.steps, gen)
            flop = B * C * (m * m + 4.0 * m)
            r['C%d' % C] = dict(predict_ms=tp, step_kernel_ms=ts, step_fraction=ts / (tp + ts),
                                chain_steps_per_s_device=C / ((tp + ts) * 1e-3), wall_ms_per_step=wall,
                                chain_steps_per_s_wall=C / (wall * 1e-3), predict_flop=flop,
                                predict_tflops=flop / (tp * 1e-3) / 1e12)
        res['S%d' % S] = r
    # host oracle at a reduced size: 4 samples, 16 points, the same m and pu
    samples = synthetic.posterior_samples(4, 1 + Q, PU, seed=4)
    num = so.OracleNum(model.num.zt[:, 1:], np.zeros((M, 1)), None)
    num.pu, num.w = PU, model._w_pcs.T.copy()
    num.wv = num.w.reshape((-1, 1), order='F')
    num.LamSim = np.asarray(model.num.LamSim, dtype=np.float64)
    G, b, c0 = (x.cpu().numpy() for x in cal._obs_terms(model, samples, y_obs[O7300], O7300, 0.01))
    t0 = time.perf_counter()
    em = co.Emulator(num, samples)
    t1 = time.perf_counter()
    co.loglik(em, G, b, c0, np.random.default_rng(0).uniform(0, 1, (16, Q)))
    t2 = time.perf_counter()
    res['host_oracle'] = dict(samples=4, points=16, factor_s=t1 - t0, eval_s=t2 - t1, evals_per_s=16 / (t2 - t1))
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'bench_calib.json'), 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
