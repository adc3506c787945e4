"""Developer benchmark: MCMC convergence diagnostics on the device (ops.chain_diagnostics, csrc/ggp_chain_diag.cu).

Shapes:
  (a) the benchmark's sampler run: 944 chains x 1000 draws x 112 elements (111 parameters + logPost) of seeded sticky AR(1)
      draws (phi = 0.8; the previous value is repeated with probability 0.7, as Metropolis rejections do), 0.85 GB of FP64;
  (b) ModelBatch: 45 models x 12 elements x 512 draws, one chain each (the per-threshold scalar models at d = 9, pu = 1).
Each is timed with CUDA events, the median of 7 calls after 2 warm-up calls.  For (a) a separate torch.profiler run gives
the time of each phase (sort / rank, R-hat, ESS), and the bytes the sort passes move over the sort / rank kernel's time are
set against the device-to-device copy rate measured in the same run.  Counted sort bytes: per element and per sort, one key
generation pass (read x, write 12 B per key) plus, per digit pass that is not skipped, a histogram read (8 B per key) and a
scatter (12 B read + 12 B written per key).  The working set (0.85 GB of draws, 4.7 GB of workspace) is far larger than L2.
The FP64 oracle (oracle/chain_diag_oracle.py) runs once on the host at shape (a) for the ratio.
Prints one JSON line; with --out DIR it also writes it to DIR/bench_chain_diag.json."""
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
from gladsgp_b200 import ops                     # noqa: E402
from oracle import chain_diag_oracle as cdo      # noqa: E402


def ev(fn, iters=7, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def sticky_ar1(rng, n, C, E, phi=0.8, stick=0.7):
    x = np.empty((n, C, E))
    x[0] = rng.standard_normal((C, E))
    for i in range(1, n):
        move = rng.random((C, E)) >= stick
        x[i] = np.where(move, phi * x[i - 1] + rng.standard_normal((C, E)), x[i - 1])
    return x


def _keys(v):
    b = (np.asarray(v, dtype=np.float64) + 0.0).view(np.uint64)
    neg = (b >> np.uint64(63)).astype(bool)
    return np.where(neg, ~b, b | np.uint64(1 << 63))


def _passes(k):
    diff = np.bitwise_or.reduce(k ^ k[0])
    return sum(1 for d in range(8) if (int(diff) >> (8 * d)) & 0xff)


def sort_bytes(x):
    """Bytes the two sorts of every element move (see the module docstring)."""
    n, C, E = x.shape
    total = 0
    for e in range(E):
        a = x[:, :, e].T
        s = cdo.split_chains(a)
        for vals, nk in ((a.reshape(-1), a.size), (np.abs(s - np.median(s)).reshape(-1), s.size)):
            total += nk * (8 + 12) + _passes(_keys(vals)) * nk * (8 + 12 + 12)
    return float(total)


def phase_ms(x):
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ops.chain_diagnostics(x)
        torch.cuda.synchronize()
    ph = {'sort_rank': 0.0, 'rhat': 0.0, 'ess': 0.0}
    for evt in prof.key_averages():
        name = evt.key
        us = getattr(evt, 'device_time_total', None)
        if us is None:
            us = evt.cuda_time_total
        if 'chain_diag_rank_kernel' in name:
            ph['sort_rank'] += us / 1e3
        elif 'chain_diag_rhat_kernel' in name:
            ph['rhat'] += us / 1e3
        elif 'chain_diag_ess_kernel' in name or 'chain_diag_finish_kernel' in name:
            ph['ess'] += us / 1e3
    return ph


def copy_rate():
    a = torch.empty(1 << 28, dtype=torch.float64, device='cuda')      # 2 GiB
    b = torch.empty_like(a)
    ms = ev(lambda: b.copy_(a), iters=5, warm=1)
    return 2.0 * a.numel() * 8 / (ms * 1e-3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip().splitlines()
    rng = np.random.default_rng(2026)
    n, C, E = 1000, 944, 112
    x = sticky_ar1(rng, n, C, E)
    xd = torch.as_tensor(x, device='cuda')
    ms_big = ev(lambda: ops.chain_diagnostics(xd))
    ph = phase_ms(xd)
    xm = torch.as_tensor(sticky_ar1(rng, 512, 1, 45 * 12), device='cuda')
    ms_batch = ev(lambda: ops.chain_diagnostics(xm))
    sb = sort_bytes(x)
    peak = copy_rate()
    t0 = time.perf_counter()
    cdo.diagnose_all(x)
    host_s = time.perf_counter() - t0
    res = dict(
        gpu=smi[0] if smi else None,
        shape_sampler=dict(n_draws=n, n_chains=C, n_elem=E),
        sampler_ms=ms_big, sampler_phase_ms=ph,
        shape_modelbatch=dict(n_draws=512, n_chains=1, n_elem=45 * 12), modelbatch_ms=ms_batch,
        sort_bytes=sb, sort_rank_gbps=sb / (ph['sort_rank'] * 1e-3) / 1e9 if ph['sort_rank'] > 0 else None,
        hbm_copy_gbps=peak / 1e9,
        host_oracle_s=host_s, host_over_device=host_s / (ms_big * 1e-3),
    )
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'bench_chain_diag.json'), 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
