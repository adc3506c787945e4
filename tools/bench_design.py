"""Developer benchmark: greedy ALC sequential design (gladsgp_b200.design) at cfg3 (m = 512, q = 8, pu = 10) on the
synthetic GlaDS-shaped ensemble, fitted as model.init_model does (the model of tools/bench_calib.py).

For S in {16, 64} posterior samples, n_ref = 1024 reference and n_cand = 4096 candidate inputs and k = 16 picks: the
device time of the score call (ggp_design_score_f64: the DMMA score kernel, the row-variance and block-sum kernels) per
step and of the condition call, CUDA events around each over the k steps; the predict time of the V rows; the whole
next_runs call behind a synchronise.  The counted flop of one score step is 2 B n_ref n_cand (Mp + Kp) (B = S pu blocks,
Kp = 16 the pitch of A; the kernel reads only the columns of A in use, rounded up to 8), reported over
bench.fp64_peak_tflops.  The FP64 oracle's rank-one route is timed at a reduced size.  Prints one JSON line (also written
to DIR/bench_design.json with --out DIR)."""
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
from gladsgp_b200 import calibration as cal, design, model as gmodel, ops, synthetic   # noqa: E402
from oracle import design_oracle as do                                          # noqa: E402

M, Q, PU = 512, 8, 10


def build_model(n_x, n_t):
    t = synthetic.design(M, Q, seed=synthetic.BASE_SEED)
    y = synthetic.ensemble(t, n_x=n_x, n_t=n_t, seed=synthetic.BASE_SEED + 3)
    with tempfile.TemporaryDirectory() as d:
        data, model = gmodel.init_model(t, y, 'design', PU, data_dir=d)
    return model


def timed_design(model, samples, C, R, k):
    """Per-step device times (ms) of the score and condition calls with every block in one chunk, and of the predict
    calls that give V."""
    pred, S = cal._predictor(model, samples)
    B, Mp = pred.B, pred.Mp
    XC = cal._designs(torch.as_tensor(cal._to_trans(model, C), device='cuda'))
    XR = cal._designs(torch.as_tensor(cal._to_trans(model, R), device='cuda'))
    n_ref, n_cand = XR.shape[0], XC.shape[0]
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    ev[0].record()
    V_C = pred.predict(XC, want_V=True)[2]
    V_R = pred.predict(XR, want_V=True)[2]
    ev[1].record()
    torch.cuda.synchronize()
    predict_ms = ev[0].elapsed_time(ev[1])
    Kp = (k + 7) & ~7
    A_C = torch.zeros((B, n_cand, Kp), dtype=torch.float64, device='cuda')
    A_R = torch.zeros((B, n_ref, Kp), dtype=torch.float64, device='cuda')
    wgt = torch.full((B,), 1.0 / (S * n_ref), dtype=torch.float64, device='cuda')
    score = torch.empty(n_cand, dtype=torch.float64, device='cuda')
    imse = torch.empty(1, dtype=torch.float64, device='cuda')
    ws = ops.design_score(pred, 0, XR, XC, V_R, V_C, A_R, A_C, 0, wgt, score, imse, False)        # warm-up
    ts, tc = [], []
    for t in range(k):
        ev[0].record()
        ops.design_score(pred, 0, XR, XC, V_R, V_C, A_R, A_C, t, wgt, score, imse, False, ws)
        ev[1].record()
        ops.design_condition(pred, 0, XR, XC, V_R, V_C, A_R, A_C, t, t * 97 % n_cand)
        ev[2].record()
        torch.cuda.synchronize()
        ts.append(ev[0].elapsed_time(ev[1]))
        tc.append(ev[1].elapsed_time(ev[2]))
    del V_C, V_R, A_C, A_R
    return dict(B=B, Mp=Mp, Kp=Kp, predict_ms=predict_ms, score_ms=ts, condition_ms=tc)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--samples', type=int, nargs='+', default=[16, 64])
    ap.add_argument('--n-ref', type=int, default=1024)
    ap.add_argument('--n-cand', type=int, default=4096)
    ap.add_argument('--k', type=int, default=16)
    ap.add_argument('--sites', type=int, default=4000)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    res = {}
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res['gpu'] = torch.cuda.get_device_name(0)
    res['nvidia_smi'] = smi[0] if smi else None
    model = build_model(args.sites, 365)
    rng = np.random.default_rng(0)
    sd = model.data.sim_data
    lo, hi = np.asarray(sd.orig_t_min).reshape(-1), np.asarray(sd.orig_t_max).reshape(-1)
    C = rng.uniform(lo, hi, (args.n_cand, Q))
    R = rng.uniform(lo, hi, (args.n_ref, Q))
    peak = bench.fp64_peak_tflops(torch, sustained_s=2.0)        # cuBLAS FP64 GEMM: (burst, sustained) TFLOP/s
    res['fp64_peak_tflops'] = dict(burst=peak[0], sustained=peak[1])
    for S in args.samples:
        samples = synthetic.posterior_samples(S, 1 + Q, PU, seed=S)
        model._pred_cache = None
        cal._predictor(model, samples)
        r = timed_design(model, samples, C, R, args.k)
        flop = 2.0 * r['B'] * args.n_ref * args.n_cand * (r['Mp'] + r['Kp'])
        med = float(np.median(r['score_ms']))
        r.update(score_ms_median=med, condition_ms_median=float(np.median(r['condition_ms'])), score_flop=flop,
                 score_tflops=flop / (med * 1e-3) / 1e12)
        r['score_fraction_of_peak'] = dict(burst=r['score_tflops'] / peak[0], sustained=r['score_tflops'] / peak[1])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = design.next_runs(model, samples, C, args.k, reference=R)
        torch.cuda.synchronize()
        r['next_runs_wall_s'] = time.perf_counter() - t0
        r['imse'] = [float(out['imse'][0]), float(out['imse'][-1])]
        res['S%d' % S] = r
    # FP64 oracle (rank-one route) at a reduced size: 2 samples, 256 candidates, 128 reference points, 4 picks
    samples = synthetic.posterior_samples(2, 1 + Q, PU, seed=2)
    XC = do.designs(cal._to_trans(model, C[:256]))
    XR = do.designs(cal._to_trans(model, R[:128]))
    t0 = time.perf_counter()
    do.greedy_rank_one(model.num.zt, model.num.LamSim, samples, XR, XC, 4, design.field_weights(model))
    res['host_oracle'] = dict(samples=2, n_cand=256, n_ref=128, k=4, s=time.perf_counter() - t0)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'bench_design.json'), 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
