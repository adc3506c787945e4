"""Developer benchmark: cached-factor prediction + reconstruction + rSVD passes (cfg4 / cfg3 shapes, bounded)."""
import json, os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gladsgp_b200 import ops, synthetic, _lib
if os.environ.get('GGP_LIB'):                      # developer A/B runs against a variant library
    _lib.LIB_PATH = os.environ['GGP_LIB']


def ev(fn, iters=3, warm=1):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(iters):
        a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        best = min(best, a.elapsed_time(b))
    return best


def main():
    res = {}
    m, q, pu = 512, 8, 10
    d = q + 1
    nsamp = int(os.environ.get('NSAMP', 100)); n = int(os.environ.get('NPRED', 4096))
    t = synthetic.design(m, q)
    X = np.concatenate([0.5 * np.ones((m, 1)), t.astype(np.float64)], axis=1)
    s = synthetic.posterior_samples(nsamp, d, pu)
    rng = np.random.default_rng(1)
    W = rng.standard_normal((pu, m))
    beta = s['betaU'].astype(np.float64).reshape(nsamp, pu, d).reshape(nsamp * pu, d)
    lamz = s['lamUz'].astype(np.float64).reshape(-1)
    lamws = s['lamWs'].astype(np.float64).reshape(-1)
    lamwos = np.repeat(s['lamWOs'].astype(np.float64), pu, axis=1).reshape(-1)
    dadd = 1.0 / lamwos + 1.0 / lamws
    s11 = 1.0 / lamz + 1.0 / lamws
    Wb = np.broadcast_to(W[None], (nsamp, pu, m)).reshape(nsamp * pu, m).copy()
    B = nsamp * pu
    P = [None]
    tf = ev(lambda: P.__setitem__(0, ops.Predictor(X, Wb, beta, lamz, dadd, s11)), iters=2, warm=1)
    res['factor_ms'] = tf; res['factor_evals_per_s'] = B / tf * 1e3
    xp = np.concatenate([0.5 * np.ones((n, 1)), synthetic.test_design(n, q).astype(np.float64)], axis=1)
    xpd = torch.as_tensor(xp, device='cuda')
    tp = ev(lambda: P[0].predict(xpd), iters=3, warm=1)
    res['predict_ms'] = tp
    res['preds_per_s_pc_space'] = nsamp * n / tp * 1e3
    res['predict_tflops'] = B * n * (m * m + (3 * d + 2) * m) / tp / 1e9
    # reconstruction: R rows x n_y
    n_y = 1460000; R = 256
    w = torch.randn(R, pu, device='cuda'); K = torch.randn(pu, n_y, device='cuda')
    sd = torch.rand(n_y, device='cuda') + 0.5; mu = torch.randn(n_y, device='cuda')
    out = torch.empty((R, n_y), dtype=torch.float32, device='cuda')
    tr = ev(lambda: ops.reconstruct(w, K, sd, mu, out=out), iters=5, warm=2)
    res['reconstruct_ms'] = tr; res['reconstruct_gbs'] = 4.0 * R * n_y / tr / 1e6
    res['reconstruct_rows_per_s'] = R / tr * 1e3
    # fused statistics: 64 samples x 4 designs (assess_all_models.py batch), mean + 2.5/97.5 % quantiles
    ns_, np_ = 64, 4
    w3 = torch.randn(ns_, np_, pu, device='cuda'); nz = torch.randn(ns_, np_, device='cuda') * 0.1
    tst = ev(lambda: ops.reconstruct_stats(w3, K, sd, mu, q=0.025, noise=nz), iters=5, warm=2)
    res['stats_ms_64x4'] = tst
    res['stats_equiv_materialised_gbs'] = 4.0 * ns_ * np_ * n_y / tst / 1e6
    # the same pass with the test-error sums fused in and no field written (assess_all_models.py:523-538)
    yt = torch.randn(np_, n_y, device='cuda') + 2.0
    tes = ev(lambda: ops.reconstruct_errstats(w3, K, sd, mu, yt, 1.0, q=0.025, noise=nz), iters=5, warm=2)
    res['errstats_ms_64x4'] = tes
    del out, K
    # rSVD passes on a 512 x 1.46M float32 ensemble
    Xe = torch.randn(m, n_y, device='cuda')
    om = torch.randn(25, n_y, device='cuda')
    ws = torch.empty(_lib.load().ggp_rsvd_tc_workspace_bytes(m), dtype=torch.uint8, device='cuda')
    ts = ev(lambda: ops.rsvd_sketch_tc(Xe, om, ws), iters=3, warm=1)
    Y = ops.rsvd_sketch_tc(Xe, om, ws)
    tx = ev(lambda: ops.rsvd_xty_tc(Xe, Y), iters=3, warm=1)
    res['rsvd_sketch_ms'] = ts; res['rsvd_sketch_gbs'] = 4.0 * m * n_y / ts / 1e6
    res['rsvd_xty_ms'] = tx; res['rsvd_xty_gbs'] = 4.0 * m * n_y / tx / 1e6
    print(json.dumps(res, indent=1))
    os.makedirs('gpurun_out', exist_ok=True)
    json.dump(res, open('gpurun_out/bench_predict.json', 'w'), indent=1)


if __name__ == '__main__':
    main()
