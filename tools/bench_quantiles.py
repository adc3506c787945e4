"""Developer benchmark: posterior mean and quantile fields over the samples (ggp_reconstruct_quantiles_f32) at cfg4's
post-processing size (npred = 4 designs, n_y = 1 460 000 outputs, pu = 10, noise).

Cases, each timed with CUDA events after warm-up:
  (a) 1000 samples, quantiles (0.025, 0.975)
  (b) 1000 samples, quantiles (0.025, 0.25, 0.5, 0.75, 0.975)
  (c) 64 samples at pu = 20 (cfg5's PCs), (0.025, 0.975)
  (d) 64 samples at pu = 10: the fused kernel (ggp_reconstruct_stats_f32, 2.5 %) and the general one, alternated
  (e) for (a), the route without the kernel: ops.reconstruct into column chunks, torch.sort along the samples, the float32
      interpolation -- and the number of entries where it differs from (a)
Counted work: phase-1 flop nsamp npred n_y (2 pu + 3) and the key bytes phase 2 reads (the mean pass, plus 33 passes per
distinct order statistic).  K (58 MB) stays in L2 between passes; the work is bound by the arithmetic and the shared-memory
passes, not by HBM.  Prints one JSON line; with --out DIR it also writes it to DIR/bench_quantiles.json."""
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
from gladsgp_b200 import ops                                 # noqa: E402
from quantile_helpers import numpy_rank, quantile_sorted    # noqa: E402

NPRED, N_Y = 4, 1460000


def ev(fn, iters=5, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def inputs(ns, pu, seed):
    g = torch.Generator(device='cuda'); g.manual_seed(seed)
    w = torch.randn((ns, NPRED, pu), dtype=torch.float32, device='cuda', generator=g)
    K = torch.randn((pu, N_Y), dtype=torch.float32, device='cuda', generator=g)
    sd = torch.rand((N_Y,), dtype=torch.float32, device='cuda', generator=g) * 1.9 + 0.1
    mu = torch.randn((N_Y,), dtype=torch.float32, device='cuda', generator=g)
    nz = torch.randn((ns, NPRED), dtype=torch.float32, device='cuda', generator=g) * 0.1
    return w, K, sd, mu, nz


def work(ns, pu, qs, noise=True):
    n_rank = len({numpy_rank(ns, q)[0] for q in qs})
    flop = ns * NPRED * N_Y * (2 * pu + 3)
    key_bytes = NPRED * N_Y * ns * 4 * (1 + int(noise) + 33 * n_rank)
    return dict(phase1_flop=float(flop), phase2_key_bytes=float(key_bytes), distinct_ranks=n_rank)


def case(name, ns, pu, qs, seed, res):
    w, K, sd, mu, nz = inputs(ns, pu, seed)
    ms = ev(lambda: ops.reconstruct_quantiles(w, K, sd, mu, qs, noise=nz))
    wk = work(ns, pu, qs)
    res[name] = dict(nsamp=ns, pu=pu, quantiles=list(qs), ms=ms, **wk,
                     phase1_tflops=wk['phase1_flop'] / ms / 1e9, phase2_key_tb_per_s=wk['phase2_key_bytes'] / ms / 1e9)
    return w, K, sd, mu, nz


def sort_route(w, K, sd, mu, nz, qs, chunk=200000):
    ns, npred, pu = w.shape
    out = torch.empty((len(qs), npred, N_Y), dtype=torch.float32, device='cuda')
    for c0 in range(0, N_Y, chunk):
        c1 = min(N_Y, c0 + chunk)
        y = ops.reconstruct(w.reshape(ns * npred, pu), K[:, c0:c1], sd[c0:c1], mu[c0:c1]).reshape(ns, npred, -1)
        zs = torch.sort(y + sd[c0:c1] * nz[:, :, None], dim=0).values
        for k, q in enumerate(qs):
            out[k, :, c0:c1] = quantile_sorted(zs, q)
        del y, zs
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None, help='directory for bench_quantiles.json (default: print only)')
    args = ap.parse_args()
    res = {}
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res['gpu'] = torch.cuda.get_device_name(0)
    res['nvidia_smi'] = smi[0] if smi else None
    res['npred'], res['n_y'] = NPRED, N_Y
    q2 = (0.025, 0.975)
    w, K, sd, mu, nz = case('a_1000_samples_2q', 1000, 10, q2, 1, res)
    case('b_1000_samples_5q', 1000, 10, (0.025, 0.25, 0.5, 0.75, 0.975), 1, res)
    case('c_64_samples_pu20', 64, 20, q2, 2, res)

    # (e) the route without the kernel, on (a)'s inputs, and its agreement with (a)
    res['e_reconstruct_sort_ms'] = ev(lambda: sort_route(w, K, sd, mu, nz, q2), iters=3, warm=1)
    res['e_over_a'] = res['e_reconstruct_sort_ms'] / res['a_1000_samples_2q']['ms']
    _, yq = ops.reconstruct_quantiles(w, K, sd, mu, q2, noise=nz)
    res['e_entries_differing_from_a'] = int((sort_route(w, K, sd, mu, nz, q2) != yq).sum().item())
    del w, K, sd, mu, nz, yq

    # (d) fused versus general at 64 samples, pu = 10, alternated so that both see the same machine state
    w, K, sd, mu, nz = inputs(64, 10, 3)
    fused, general = [], []
    for _ in range(3):
        fused.append(ev(lambda: ops.reconstruct_stats(w, K, sd, mu, q=0.025, noise=nz)))
        general.append(ev(lambda: ops.reconstruct_quantiles(w, K, sd, mu, q2, noise=nz)))
    res['d_64_samples_fused_ms'] = min(fused)
    res['d_64_samples_general_ms'] = min(general)
    res['d_general_over_fused'] = min(general) / min(fused)
    res['d_work'] = work(64, 10, q2)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'bench_quantiles.json'), 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
