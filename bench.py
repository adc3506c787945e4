#!/usr/bin/env python
"""Benchmark of the GP-emulator hot path (contract: see the task brief / DESIGN.md section 6).

Metric (BASELINE.json): MCMC steps/s at m=512, q=8 (d=9), pu=10 -- one step = one SEPIA
mcmc_step = pu*(d+4) fused covariance+Cholesky block evaluations per chain.  A bench "step"
advances every chain of every rank by one mcmc_step; `value` = chain-steps per second over the
whole job.  Chains are independent (weak scaling: a fixed number of chains per GPU, no data-path
collective; one NCCL all_gather of the per-chain log-posteriors at the end).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--chains C] [--dump-outputs DIR]
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree untouched (it may be read-only)
DUMP_LIMIT_BYTES = 64 << 20

M, Q, PU = 512, 8, 10
D = Q + 1
P = D * PU + 2 * PU + 1
EVALS_PER_STEP = PU * (D + 4)
METRIC = 'mcmc_steps_per_s'
UNIT = 'chain-steps/s'
SWEEP_DRAM_BYTES_PER_EVAL = 196.85e9 / 25860.0     # ncu --set full of one step-kernel launch (profiles/r2a_sweep_kernel_summary.txt:
#                                                      164.09 GB read + 32.77 GB written, 25.86 k evaluations in the launch)
REF_RECORDED_MCMC_S = 1803.242                     # experiments/synthetic/analysis/data/models/timing.csv:11 (m=512, pu=10; hardware unknown)


def measured_peaks():
    """HBM GB/s from MEASURED_PEAKS.json (driver-written), else the profiling recipe's fallback."""
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md)'
WORKLOAD = 'cfg3 multivariate PCA emulator: m=512 sims, q=8 params (d=9), pu=10 PCs, SEPIA Metropolis-within-Gibbs'


def build_problem(n_x, n_t, seed=20240318 + 3, standardized=True):
    """Synthetic GlaDS-shaped ensemble (+ column mean / clamped sd as src/model.py:60-64)."""
    from gladsgp_b200 import synthetic
    t = synthetic.design(M, Q, seed=20240318)
    y = synthetic.ensemble(t, n_x=n_x, n_t=n_t, seed=seed)
    mu = np.mean(y, axis=0)
    sd = np.std(y, ddof=1, axis=0)
    sd[sd < 1e-6] = 1e-6
    if not standardized:
        return t, y, mu.astype(np.float32), sd.astype(np.float32)
    return t, y, ((y - mu) / sd).astype(np.float32), mu.astype(np.float32), sd.astype(np.float32)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for nme, v in zip(names, r[4:8]):
                    if v.lower().startswith('active'):
                        reasons.add(nme)
            except Exception:
                pass
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


def oracle_model(t, y_std, K, pc_prec, resid_ss=None):
    from oracle import sepia_oracle as so
    num = so.OracleNum(t, y_std, K, resid_ss=resid_ss)
    om = so.OracleModel(num)
    om.override_lamWOs(pc_prec)
    return om


def cpu_steps_per_s(om, n_steps, seed=1):
    rng = np.random.RandomState(seed)
    t0 = time.perf_counter()
    om.do_mcmc(n_steps, rng=rng)
    dt = time.perf_counter() - t0
    return n_steps / dt, dt


def blas_threads():
    try:
        from threadpoolctl import threadpool_info
        return max([p.get('num_threads', 1) for p in threadpool_info()] + [1])
    except Exception:
        return os.cpu_count() or 1


def small_setup(n_x, n_t):
    """Host-only set-up for the reference arm (no GPU): K from the oracle rSVD on a reduced field."""
    from oracle import svd_oracle
    t, y, y_std, mu, sd = build_problem(n_x, n_t)
    U, S, Vh = svd_oracle.randomized_svd(y_std, 25, k=0, q=1, rng=np.random.RandomState(0))
    K = svd_oracle.k_basis(S, Vh, PU, M).astype(np.float32)
    w = np.dot(np.linalg.pinv(K).T, y_std.T).T
    pc_prec = 1.0 / np.var(y_std - np.dot(w, K))
    return t, y_std, K, pc_prec


def _ref_worker_main(argv):
    """Child process of the reference arm: one single-thread chain (OMP/BLAS threads pinned to 1 by the parent's env)."""
    ref_nx, ref_nt, warm, steps, seed = [int(x) for x in argv]
    t, y_std, K, pc_prec = small_setup(ref_nx, ref_nt)
    om = oracle_model(t, y_std, K, pc_prec)
    rng = np.random.RandomState(seed)
    om.do_mcmc(warm, rng=rng)
    t0 = time.perf_counter()
    om.do_mcmc(steps, rng=rng)
    print(json.dumps({'dt': time.perf_counter() - t0}))


def host_cpu_modes(ref_nx, ref_nt, warm, steps, om=None):
    """The CPU port on this box's host cores, both ways (BASELINE.md 3.2): (a) ONE chain with every BLAS thread the
    box has -- the reference's own usage, src/model.py:234-235; (b) one single-thread chain per core in parallel
    processes -- the fair aggregate for a throughput comparison (a 512 x 512 problem does not scale over BLAS threads).
    Returns dict(one_chain=..., per_core_chains=...), each with value (chain-steps/s), threads / processes, seconds."""
    cores = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    out = {}
    try:
        from threadpoolctl import threadpool_limits
        ctx = threadpool_limits(limits=cores)
    except Exception:
        ctx = None
    if om is None:
        t, y_std, K, pc_prec = small_setup(ref_nx, ref_nt)
        om = oracle_model(t, y_std, K, pc_prec)
    rng = np.random.RandomState(1)
    om.do_mcmc(warm, rng=rng)
    t0 = time.perf_counter()
    om.do_mcmc(steps, rng=rng)
    dt = time.perf_counter() - t0
    out['one_chain'] = {'value': steps / dt, 'chains': 1, 'blas_threads': blas_threads(), 'seconds': dt, 'steps': steps}
    if ctx is not None:
        ctx.unregister() if hasattr(ctx, 'unregister') else None
    nproc = max(1, min(cores, int(os.environ.get('BENCH_REF_PROCS', cores))))
    env = dict(os.environ)
    for k in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS', 'NUMEXPR_NUM_THREADS'):
        env[k] = '1'
    env['CUDA_VISIBLE_DEVICES'] = ''
    t0 = time.perf_counter()
    procs = [subprocess.Popen([sys.executable, os.path.abspath(__file__), '--ref-worker', str(ref_nx), str(ref_nt), str(warm),
                               str(steps), str(100 + i)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, env=env)
             for i in range(nproc)]
    dts = []
    for pr in procs:
        o, _ = pr.communicate()
        try:
            dts.append(json.loads(o.strip().splitlines()[-1])['dt'])
        except Exception:
            pass
    wall = time.perf_counter() - t0
    if dts:
        out['per_core_chains'] = {'value': len(dts) * steps / max(dts), 'chains': len(dts), 'blas_threads': 1,
                                  'seconds': max(dts), 'wall_incl_startup_s': wall, 'steps': steps,
                                  'per_chain_steps_per_s': steps / float(np.mean(dts))}
    return out, cores


def run_reference(args):
    """Reference arm: the reference's CPU implementation of the path (NumPy/SciPy SEPIA restatement in oracle/,
    `kind: port` -- the sepia package itself is not installable here) on this box's host cores, run both as one chain
    with all BLAS threads and as one single-thread chain per core; `value` is the better of the two."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    modes, cores = host_cpu_modes(args.ref_nx, args.ref_nt, args.warmup, args.steps)
    best_name = max(modes, key=lambda k: modes[k]['value'])
    best = modes[best_name]
    val = best['value']
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': 1e3 * best['seconds'] / args.steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': WORKLOAD, 'chains': best['chains'], 'field_n_y_for_setup': args.ref_nx * args.ref_nt,
                   'evals_per_step': EVALS_PER_STEP, 'mode': best_name},
        'cpu_baseline': {'value': val, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                         'sample': '%d mcmc_steps per chain (oracle/sepia_oracle.py, NumPy/SciPy FP64): best of one chain x '
                                   'all BLAS threads and one single-thread chain per core' % args.steps,
                         'modes': modes},
        'e2e': {'value': val, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))


def fp64_peak_tflops(torch, sustained_s=0.0):
    """cuBLAS FP64 GEMM 8192^3 (MEASURED_PEAKS.json has no FP64 figure): best single call (burst) and, with sustained_s > 0,
    the average of back-to-back calls over that many seconds (the part runs into its 1 kW power cap within a second or two of
    FP64 tensor work: the sustained figure is the one a seconds-long step can be held against, B200_PROFILING.md)."""
    n = 8192
    a = torch.randn(n, n, dtype=torch.float64, device='cuda'); b = torch.randn(n, n, dtype=torch.float64, device='cuda')
    c = torch.empty_like(a)
    torch.matmul(a, b, out=c); torch.cuda.synchronize()
    best = 1e9
    for _ in range(3):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); torch.matmul(a, b, out=c); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    burst = 2.0 * n ** 3 / best / 1e9
    if sustained_s <= 0:
        del a, b, c
        return burst
    reps = max(4, int(sustained_s * 1e3 / best))
    for _ in range(reps // 2):                       # bring the part to its sustained state first
        torch.matmul(a, b, out=c)
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        torch.matmul(a, b, out=c)
    e1.record(); torch.cuda.synchronize()
    sustained = 2.0 * n ** 3 * reps / e0.elapsed_time(e1) / 1e9
    del a, b, c
    return burst, sustained


def prediction_bench(torch, model, args, rank, world):
    """Emulator predictions/s: one prediction = one (posterior sample, test design) pair -> pu PC means and
    variances.  nsamp x pu covariance factors are cached once; test designs are sharded across ranks."""
    import torch.distributed as dist
    from gladsgp_b200 import ops, synthetic
    from sepia.SepiaPredict import SepiaEmulatorPrediction
    nsamp, npred = args.pred_samples, args.pred_designs
    samples = synthetic.posterior_samples(nsamp, D, PU, seed=77)
    tp = synthetic.test_design(npred * world, Q)[rank * npred:(rank + 1) * npred]
    pr = SepiaEmulatorPrediction(t_pred=tp[:4], samples=samples, model=model, do_call=False)
    ns, beta, lamz, dadd, s11, W = pr._blocks()
    torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True); e2 = torch.cuda.Event(enable_timing=True)
    P0 = ops.Predictor(model.num.zt, W, beta, lamz, dadd, s11)            # warm-up (also keeps the factors)
    xp = torch.as_tensor(np.concatenate([0.5 * np.ones((npred, 1)), tp.astype(np.float64)], axis=1), device='cuda')
    P0.predict(xp[:512])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0.record()
    P1 = ops.Predictor(model.num.zt, W, beta, lamz, dadd, s11)
    e1.record()
    mean, var = P1.predict(xp)
    e2.record()
    torch.cuda.synchronize()
    fac_ms, prd_ms = e0.elapsed_time(e1), e1.elapsed_time(e2)
    for _ in range(2):                       # the pass is ~50 ms: best of three against clock ramps after the host-side sections
        a0 = torch.cuda.Event(enable_timing=True); a1 = torch.cuda.Event(enable_timing=True)
        a0.record(); mean, var = P1.predict(xp); a1.record(); torch.cuda.synchronize()
        prd_ms = min(prd_ms, a0.elapsed_time(a1))
    # end to end through the reference-facing class with host buffers and its default behaviour (joint predictive
    # covariance + one multivariate-normal realisation per sample, as SEPIA's wPred): calls of 256 designs, the
    # largest size a reference caller uses (sensitivity_indices.py:96), over E2E_CALLS different design blocks
    n_call, E2E_CALLS = 256, 4
    SepiaEmulatorPrediction(t_pred=tp[:n_call], samples=samples, model=model)          # warm the path
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(E2E_CALLS):
        pe = SepiaEmulatorPrediction(t_pred=tp[i * n_call:(i + 1) * n_call], samples=samples, model=model)
    e2e_s = time.perf_counter() - t0
    # the same joint work, device-timed with resident inputs (the e2e number's own ceiling): predict with V, joint covariance,
    # Cholesky draw
    xj = xp[:n_call].contiguous()
    zj = torch.randn(ns * PU, n_call, dtype=torch.float64, device='cuda')

    def joint_pass():
        mj, vj, Vj = P1.predict(xj, want_V=True)
        Sj = P1.pred_cov(xj, Vj)
        return ops.chol_draw(Sj, zj)
    joint_ms = _ev_ms(torch, joint_pass)
    # reconstruction of a batch of fields (get_y), float32
    w32 = pe.w[:, :4, :].astype(np.float32).reshape(-1, PU)
    sd_ = model.data.sim_data
    Kd = torch.as_tensor(np.asarray(sd_.K), device='cuda'); sdd = torch.as_tensor(np.asarray(sd_.orig_y_sd), device='cuda')
    mud = torch.as_tensor(np.asarray(sd_.orig_y_mean), device='cuda'); wd = torch.as_tensor(w32, device='cuda')
    out = ops.reconstruct(wd, Kd, sdd, mud)
    torch.cuda.synchronize()
    r0 = torch.cuda.Event(enable_timing=True); r1 = torch.cuda.Event(enable_timing=True)
    r0.record(); ops.reconstruct(wd, Kd, sdd, mud, out=out); r1.record(); torch.cuda.synchronize()
    rec_ms = r0.elapsed_time(r1)
    t = torch.tensor([fac_ms, prd_ms, e2e_s * 1e3, rec_ms, joint_ms], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    fac_ms, prd_ms, e2e_ms, rec_ms, joint_ms = [float(x) for x in t.cpu()]
    n_y = int(Kd.shape[1])
    res = {
        'metric': 'emulator_preds_per_s', 'unit': '(sample,design) pairs/s, all pu PCs',
        'config': {'posterior_samples': nsamp, 'designs_per_gpu': npred, 'pu': PU, 'm': M, 'blocks_factored': nsamp * PU},
        'value_pc_space': nsamp * npred * world / (prd_ms * 1e-3),
        'value_pc_space_incl_factorisation': nsamp * npred * world / ((prd_ms + fac_ms) * 1e-3),
        'factor_ms': fac_ms, 'predict_ms': prd_ms,
        'predict_tflops_fp64': nsamp * PU * npred * (M * M + (3 * D + 2) * M) / (prd_ms * 1e-3) / 1e12,
        'value_joint_256': nsamp * n_call * world / (joint_ms * 1e-3),
        'joint_256_note': 'device-timed, resident inputs: one call of 256 designs with the joint covariance and the Cholesky draw '
                          '(predict_kernel + pred_cov_kernel + chol_draw_kernel), the work the e2e figure below includes',
        'e2e': {'value': nsamp * n_call * E2E_CALLS * world / (e2e_ms * 1e-3),
                'api': 'SepiaEmulatorPrediction(t_pred=256 designs, samples, model), %d calls, default (joint) behaviour' % E2E_CALLS,
                'note': 'host numpy in; joint covariance per (sample, PC), one realisation per sample from the global np.random '
                        'stream, pred.w (nsamp,npred,pu) back on the host'},
        'roofline': {'bound': 'tensor', 'kernel': 'ggp::predict_kernel (V = S21^T L^-T through the cached factor, mean, variance)',
                     'achieved': nsamp * PU * npred * (M * M + (3 * D + 2) * M) / (prd_ms * 1e-3) / 1e12, 'unit': 'TFLOP/s',
                     'peak': None, 'frac': None, 'traffic': None},
        'reconstruct': {'rows': int(w32.shape[0]), 'n_y': n_y, 'ms': rec_ms, 'gbs': 4.0 * w32.shape[0] * n_y / rec_ms / 1e6,
                        'frac_of_hbm_peak': 4.0 * w32.shape[0] * n_y / rec_ms / 1e6 / 6533.8},
    }
    if rank == 0:
        # CPU baseline: SEPIA-style w_pred (fresh S22 solve per sample, PC and call), tiny sample
        from oracle import sepia_oracle as so
        num = so.OracleNum(model.data.sim_data.t_trans, model.data.sim_data.y_std[:, :64], np.asarray(sd_.K)[:, :64], resid_ss=0.0)
        num.w = model._w_pcs.T.copy(); num.wv = num.w.reshape((-1, 1), order='F'); num.LamSim = model.num.LamSim
        s2 = {k: v[:2] for k, v in samples.items()}
        t0 = time.perf_counter()
        so.w_pred(num, tp[:4], s2, rng=np.random.RandomState(0))
        dt = time.perf_counter() - t0
        res['cpu_baseline'] = {'value': 2 * 4 / dt, 'unit': res['unit'], 'kind': 'port', 'cores': blas_threads(),
                               'sample': '2 samples x 4 designs in one SEPIA-style call (%.2f s)' % dt}
    return res


def _ev_ms(torch, fn, reps=3):
    """Best-of-reps device time (ms) of fn() with CUDA events on the current stream."""
    fn(); torch.cuda.synchronize()
    best = 1e30
    for _ in range(reps):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return best


def single_chain_bench(torch, model):
    """The reference's own workload (src/model.py:234-235): ONE chain, tune_step_sizes(100, 5) then do_mcmc(512), wall clock
    through the public API, next to the 1803.242 s the reference recorded for m=512, pu=10 (timing.csv:11, hardware unknown)."""
    import contextlib
    import io
    np.random.seed(2024)
    model.do_mcmc(8, prog=False)                      # warm the single-chain (cluster) kernels
    model.clear_samples()
    torch.cuda.synchronize()
    buf = io.StringIO()
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(buf):             # tune_step_sizes prints the step sizes, as SEPIA does
        model.tune_step_sizes(100, 5, prog=False)
    t1 = time.perf_counter()
    model.do_mcmc(512, prog=False)
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    return {'api': 'model.tune_step_sizes(100, 5); model.do_mcmc(512)   (src/model.py:234-235)', 'chains': 1,
            'mcmc_steps': 10 + 100 * 5 + 512, 'wall_s': t2 - t0, 'tune_s': t1 - t0, 'do_mcmc_512_s': t2 - t1,
            'do_mcmc_steps_per_s': 512 / (t2 - t1), 'reference_recorded_s': REF_RECORDED_MCMC_S,
            'reference_recorded_source': 'experiments/synthetic/analysis/data/models/timing.csv:11 (hardware not recorded)',
            'speedup_vs_recorded': REF_RECORDED_MCMC_S / (t2 - t0)}


def rsvd_bench(torch, data, svd_s):
    """The two streaming products of src/svd.py on the device-resident ensemble: GB/s of each pass against the HBM peak."""
    from gladsgp_b200 import ops, _lib
    X = data.sim_data.y_std_device()
    m, n = X.shape
    r = 25
    g = torch.Generator(device='cuda'); g.manual_seed(1)
    omT = torch.randn((r, n), dtype=torch.float32, device='cuda', generator=g)
    Y = torch.randn((m, r), dtype=torch.float32, device='cuda', generator=g)
    ws = torch.empty(_lib.load().ggp_rsvd_tc_workspace_bytes(m), dtype=torch.uint8, device='cuda')
    sk = _ev_ms(torch, lambda: ops.rsvd_sketch_tc(X, omT, ws))
    xt = _ev_ms(torch, lambda: ops.rsvd_xty_tc(X, Y))
    peak, src = measured_peaks()
    byt = 4.0 * m * n
    return {'m': int(m), 'n_y': int(n), 'rank': r, 'randomized_svd_s': svd_s,
            'sketch_pass': {'kernel': 'ggp::sketch_tma_kernel (Y = X Omega, tcgen05 3xTF32, X tiles by TMA; GGP_TMA=0: ggp::sketch_tc_kernel)' if os.environ.get('GGP_TMA', '3') != '0' else 'ggp::sketch_tc_kernel (Y = X Omega, tcgen05 3xTF32)', 'ms': sk, 'gbs': byt / sk / 1e6,
                            'frac_of_hbm_peak': byt / sk / 1e6 / peak},
            'xty_pass': {'kernel': 'ggp::xty_ts_kernel (B = Y^T X, tcgen05 3xTF32)', 'ms': xt, 'gbs': byt / xt / 1e6,
                         'frac_of_hbm_peak': byt / xt / 1e6 / peak},
            'algorithmic_bytes_per_pass': byt, 'hbm_peak_gbs': peak, 'hbm_peak_source': src}


def cfg5_bench(torch, rank, world, steps=2):
    """BASELINE.json configs[4]: m=4096 sims, 16 parameters (d=17), 20 PCs -- one chain per GPU (8 chains on 8 GPUs), and,
    with more than one GPU, ONE chain with its PCs spread over the GPUs (one NCCL all_gather of per-PC rows per step)."""
    import torch.distributed as dist
    from gladsgp_b200 import synthetic, dist as gdist
    from sepia.SepiaData import SepiaData
    from sepia.SepiaModel import SepiaModel
    m, q, pu = 4096, 16, 20
    d = q + 1
    t = synthetic.design(m, q, seed=20240318)
    rng = np.random.default_rng(5)
    n_y = 4000                                        # the field size is free in cfg5
    modes = rng.standard_normal((24, n_y))
    coef = np.stack([np.sin((k + 1) * t @ rng.uniform(0.2, 1.5, size=q)) for k in range(24)], axis=1) / (1 + np.arange(24))
    y = (coef @ modes + 0.02 * rng.standard_normal((m, n_y))).astype(np.float32)
    dd = SepiaData(t_sim=t, y_sim=y, y_ind_sim=np.linspace(0, 1, n_y))
    dd.transform_xt(t_notrans=np.arange(q)); dd.standardize_y()
    dd.create_K_basis(n_pc=pu)
    mod = SepiaModel(dd)
    eng, tb = mod._get_engine(1)
    P = tb['theta'].size
    evals = pu * (d + 4)
    flop_eval = m ** 3 / 3.0 + m * m + 2 * m + (3 * d + 2) * m * (m - 1) / 2.0
    us = np.random.RandomState(900 + rank).random_sample((1, 2 * P * (steps + 1)))
    eng.run(1, tb['step'], uniforms=us[:, :2 * P], record=False)                  # warm-up step (also the per-PC terms)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record(); out = eng.run(steps, tb['step'], uniforms=us[:, 2 * P:], init_sigwl=False); e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    res = {'workload': 'cfg5: m=4096, d=17, pu=20, %d block evaluations per step' % evals, 'steps': steps,
           'one_chain_per_gpu': {'chains': world, 's_per_step': ms / steps / 1e3, 'chain_steps_per_s': world * steps / (ms * 1e-3),
                                 'tflops_fp64_per_gpu': steps * evals * flop_eval / (ms * 1e-3) / 1e12,
                                 'lp_finite': bool(torch.isfinite(out['lp']).all().item())}}
    if world > 1:
        # strong scaling: the same single chain (rank 0's stream on every rank), PCs spread over the ranks
        us0 = np.random.RandomState(900).random_sample((1, 2 * P * (steps + 1)))
        eng.set_state(tb['theta'])
        gdist.mcmc_by_pc(eng, 1, tb['step'], uniforms=us0[:, :2 * P], record=False)
        torch.cuda.synchronize(); dist.barrier()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); o2 = gdist.mcmc_by_pc(eng, steps, tb['step'], uniforms=us0[:, 2 * P:], init_sigwl=False); e1.record()
        torch.cuda.synchronize()
        ms2 = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device='cuda')
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
        ms2 = float(ms2.item())
        cp = -(-pu // world)
        res['one_chain_by_pc'] = {'gpus': world, 'pcs_per_gpu_max': cp, 's_per_step': ms2 / steps / 1e3,
                                  'speedup_vs_one_gpu': ms / ms2, 'strong_scaling_efficiency': ms / ms2 / world,
                                  'ideal_speedup_for_this_split': pu / float(cp),
                                  'collective': 'NCCL all_gather_into_tensor of %d B per rank per step (%d calls)'
                                                % (cp * (2 * d + 6) * 8, o2['collective_calls']),
                                  'tflops_fp64_total': steps * evals * flop_eval / (ms2 * 1e-3) / 1e12}
    del eng, mod
    torch.cuda.empty_cache()
    return res


def sharded_collectives_bench(torch, model, data, rank, world, nsamp=64, npred_total=16384):
    """The two data-path collectives that move real data, timed on the device with the collective inside the timed region:
    prediction sharded by test-design block (all_gather of the moments) and the rSVD sharded by output-column slab (all_reduce of
    the m x r sketches).  Shares of the collectives are measured by timing the same region with the collective replaced by a
    local no-op."""
    import torch.distributed as dist
    from gladsgp_b200 import ops, synthetic, dist as gdist
    from sepia.SepiaPredict import SepiaEmulatorPrediction
    res = {}
    samples = synthetic.posterior_samples(nsamp, D, PU, seed=77)
    tp = synthetic.test_design(npred_total, Q)
    pr = SepiaEmulatorPrediction(t_pred=tp[:4], samples=samples, model=model, do_call=False)
    ns, beta, lamz, dadd, s11, W = pr._blocks()
    Pd = ops.Predictor(model.num.zt, W, beta, lamz, dadd, s11)
    xp = np.concatenate([0.5 * np.ones((npred_total, 1)), tp.astype(np.float64)], axis=1)
    lo, hi = gdist.shard_bounds(npred_total, rank, world)
    xloc = torch.as_tensor(np.ascontiguousarray(xp[lo:hi]), device='cuda')

    def timed(fn):
        fn(); torch.cuda.synchronize(); dist.barrier()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device='cuda')
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    full = timed(lambda: gdist.predict_sharded(Pd, xp))
    local = timed(lambda: Pd.predict(xloc))
    res['predict_sharded'] = {'pairs': nsamp * npred_total, 'ms': full, 'ms_without_gather': local,
                              'pairs_per_s': nsamp * npred_total / (full * 1e-3),
                              'collective': 'NCCL all_gather of (B=%d, n/world) float64 means and variances: %d B per rank'
                                            % (nsamp * PU, 2 * 8 * nsamp * PU * (hi - lo)),
                              'collective_share': max(0.0, 1.0 - local / full)}
    # rSVD by output-column slab
    X = data.sim_data.y_std_device()
    m, n = X.shape
    clo, chi = gdist.shard_bounds(n, rank, world)
    clo -= clo % 4                                      # keep slabs 16-byte aligned
    Xs = X[:, clo:chi].contiguous()
    om = torch.as_tensor(np.random.RandomState(3).normal(size=(chi - clo, 25)).astype(np.float32), device='cuda')   # test matrix resident
    full = timed(lambda: gdist.randomized_svd_sharded(Xs, 25, k=0, q=1, omega_slab=om))
    res['rsvd_sharded'] = {'m': int(m), 'n_y_per_rank': int(chi - clo), 'ms': full,
                           'note': 'whole decomposition with the slab and the test matrix resident: 4 streaming passes + m x 25 QR, '
                                   '25 x n Gram, 25 x 25 eigh (torch) + the all_reduces',
                           'passes_min_ms_at_hbm_peak': 4 * 4.0 * m * (chi - clo) / 6533.8e6,
                           'collective': 'NCCL all_reduce of the (m, 25) float32 sketch per pass (2 passes) + (25, 25) float64 Gram',
                           'gbs_aggregate_4_passes': 4 * 4.0 * m * (chi - clo) * world / full / 1e6}
    return res


def cfg4_full_bench(torch, model, rank, world):
    """BASELINE.json configs[3] at full size: 1000 posterior samples x 100 000 test designs, designs sharded across the GPUs."""
    import torch.distributed as dist
    from gladsgp_b200 import ops, synthetic, dist as gdist
    from sepia.SepiaPredict import SepiaEmulatorPrediction
    nsamp, npred = 1000, 100000
    samples = synthetic.posterior_samples(nsamp, D, PU, seed=78)
    tp = synthetic.test_design(npred, Q)
    pr = SepiaEmulatorPrediction(t_pred=tp[:4], samples=samples, model=model, do_call=False)
    ns, beta, lamz, dadd, s11, W = pr._blocks()
    torch.cuda.synchronize(); dist.barrier() if world > 1 else None
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True); e2 = torch.cuda.Event(enable_timing=True)
    e0.record()
    Pd = ops.Predictor(model.num.zt, W, beta, lamz, dadd, s11)
    e1.record()
    lo, hi = gdist.shard_bounds(npred, rank, world)
    xp = torch.as_tensor(np.concatenate([0.5 * np.ones((hi - lo, 1)), tp[lo:hi].astype(np.float64)], axis=1), device='cuda')
    chunk = 4096
    msum = torch.zeros(ns * PU, dtype=torch.float64, device='cuda')
    for c0 in range(0, hi - lo, chunk):
        mean, var = Pd.predict(xp[c0:c0 + chunk])
        msum += mean.sum(dim=1)
    e2.record(); torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1), e1.elapsed_time(e2)], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    fac_ms, prd_ms = [float(x) for x in t.cpu()]
    del Pd
    torch.cuda.empty_cache()
    return {'workload': 'cfg4: 1000 samples x 100 000 designs, all 10 PC means and variances', 'gpus': world,
            'factor_s': fac_ms / 1e3, 'predict_s': prd_ms / 1e3, 'pairs_per_s': nsamp * npred / ((fac_ms + prd_ms) * 1e-3),
            'tflops_fp64_aggregate': nsamp * PU * npred * (M * M + (3 * D + 2) * M) / (prd_ms * 1e-3) / 1e12,
            'checksum_finite': bool(torch.isfinite(msum).all().item())}


def dump_outputs(dirname, arrays):
    """arrays: name -> array with one row per chain.  Writes dirname/<name>.npy; when all rows together exceed
    DUMP_LIMIT_BYTES, the same seeded sample of chains is kept in every array."""
    os.makedirs(dirname, exist_ok=True)
    n = len(next(iter(arrays.values())))
    row_bytes = sum(a[0].nbytes for a in arrays.values())
    keep = np.arange(n)
    if n * row_bytes > DUMP_LIMIT_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(n, DUMP_LIMIT_BYTES // row_bytes, replace=False))
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + '.npy'), np.ascontiguousarray(a[keep]))


def run_ours(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm')
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    from gladsgp_b200 import svd, model as gmodel, ops
    from sepia.SepiaData import SepiaData
    from sepia.SepiaModel import SepiaModel

    # ---------------- set-up through the public API (untimed): standardise, rSVD, K, SepiaModel
    t_set = time.perf_counter()
    nx = args.nx if (world == 1 or rank == 0) else max(args.nx // 10, 64)   # host RAM: one full field per box
    t, y, mu, sd = build_problem(nx, args.nt, standardized=False)
    data = SepiaData(t_sim=t, y_sim=y, y_ind_sim=np.linspace(0, 1, y.shape[1]))
    data.transform_xt(t_notrans=np.arange(Q))
    data.standardize_y(y_mean=mu, y_sd=sd)
    np.random.seed(1234)
    torch.cuda.synchronize(); t_svd = time.perf_counter()
    U, S, Vh = svd.randomized_svd(data.sim_data.y_std_device(), 25, k=0, q=1)   # device-resident since standardize_y
    torch.cuda.synchronize(); svd_s = time.perf_counter() - t_svd
    K = ((S[:PU, None] * Vh[:PU]) / np.sqrt(M)).astype(np.float32)
    data.create_K_basis(K=K)
    model = SepiaModel(data)
    pc_prec = gmodel.pc_precision(data.sim_data)
    gmodel.override_lamWOs(model, pc_prec)
    setup_s = time.perf_counter() - t_set
    chains = args.chains

    # ---------------- device-resident timing (`value`): inputs already in HBM
    eng, tb = model._get_engine(chains)
    rs = np.random.RandomState(100 + rank)
    nsteps_tot = args.warmup + args.steps
    us = torch.as_tensor(rs.random_sample((chains, 2 * P * nsteps_tot))).to('cuda')
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # clocks / throttle reasons are sampled from here (spin-up + warm-up + timed region, all under load)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    # clock spin-up after the long host-side set-up (the GPU has been idle), then the W contract warm-up steps
    spin = torch.as_tensor(rs.random_sample((chains, 2 * P * 12))).to('cuda')
    eng.run(12, tb['step'], uniforms=spin, record=False)
    out = eng.run(args.warmup, tb['step'], uniforms=us[:, :2 * P * args.warmup].contiguous(), record=False, init_sigwl=False)
    us_t = us[:, 2 * P * args.warmup:].contiguous()
    theta0, sig0 = eng.theta.clone(), eng.sigwl.clone()
    barrier()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    out = eng.run(args.steps, tb['step'], uniforms=us_t, init_sigwl=False, record=True)
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    dev_ms = e0.elapsed_time(e1)
    lp_last = out['lp'][-1].clone()
    if args.dump_outputs and rank == 0:
        # what the timed run returns for its last step: every chain's parameter vector and log-posterior (float64)
        dump_outputs(args.dump_outputs, {'draws': out['draws'][-1].cpu().numpy(), 'lp': lp_last.cpu().numpy()})
    # same K steps again from the same state with per-kernel CUDA-event timers and evaluation counters
    # (instrumented pass: feeds `roofline` only)
    eng.theta.copy_(theta0); eng.sigwl.copy_(sig0)
    out2 = eng.run(args.steps, tb['step'], uniforms=us_t, init_sigwl=False, record=True, time_kernels=True)
    sweep_ms, wos_ms = out2['kernel_ms']
    n_valid = int(out2['eval_count'][0]) + int(out2['eval_count'][1])   # block evaluations inside the step kernels (sites + lamWOs terms)
    assert torch.equal(out2['lp'][-1], lp_last), 'instrumented pass must reproduce the timed pass bit for bit'

    # ---------------- end-to-end through the public API with host buffers (`e2e`)
    np.random.seed(4321 + rank)
    model.do_mcmc_chains(max(args.warmup, args.steps), chains)        # warm the path (staging buffers at full size)
    barrier()
    t0 = time.perf_counter()
    draws, lps = model.do_mcmc_chains(args.steps, chains)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()
    if os.environ.get('BENCH_E2E_DEBUG'):
        for _ in range(5):
            t0 = time.perf_counter(); model.do_mcmc_chains(args.steps, chains); torch.cuda.synchronize()
            sys.stderr.write('e2e repeat %.1f ms (first %.1f ms, device pass %.1f ms)\n' % ((time.perf_counter() - t0) * 1e3, e2e_s * 1e3, dev_ms))
    h2d = 2 * P * chains * 8
    d2h = (P + 1) * chains * 8 + 8 * chains / max(args.steps, 1)

    # ---------------- second half of the metric: emulator predictions/s (cfg4 shape, bounded sample)
    pred = prediction_bench(torch, model, args, rank, world)
    extra = {}
    if not args.no_extras:
        extra['rsvd'] = rsvd_bench(torch, data, svd_s) if rank == 0 else None
        if world > 1:
            extra['sharded_collectives'] = sharded_collectives_bench(torch, model, data, rank, world)
        if world >= 8 or args.cfg4_full:
            extra['cfg4_full'] = cfg4_full_bench(torch, model, rank, world)
        extra['cfg5'] = cfg5_bench(torch, rank, world, steps=args.cfg5_steps)
        if world == 1:
            extra['single_chain'] = single_chain_bench(torch, model)

    tm = torch.tensor([dev_ms, e2e_s * 1e3, sweep_ms, wos_ms], dtype=torch.float64, device='cuda')
    cnt = torch.tensor([float(n_valid)], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
        gathered = [torch.empty_like(lp_last) for _ in range(world)]
        dist.all_gather(gathered, lp_last)                            # the path's one collective: log-posteriors
    dev_ms, e2e_ms, sweep_ms, wos_ms = [float(x) for x in tm.cpu()]
    n_valid_all = float(cnt.cpu()[0])

    if rank == 0:
        total_chains = chains * world
        value = total_chains * args.steps / (dev_ms * 1e-3)
        e2e_val = total_chains * args.steps / (e2e_ms * 1e-3)
        # roofline of the dominant kernel (sweep_kernel): algorithmic FP64 flops per evaluated site
        # = m^3/3 + m^2 + 2m (Cholesky + solve, SURVEY 8d) + (3d+2) m(m-1)/2 (covariance build)
        flop_eval = M ** 3 / 3.0 + M * M + 2 * M + (3 * D + 2) * M * (M - 1) / 2.0
        sweep_evals = n_valid_all / world          # counted on the device (per-rank average)
        achieved = sweep_evals * flop_eval / (sweep_ms * 1e-3) / 1e12
        peak_burst, peak_sust = fp64_peak_tflops(torch, sustained_s=max(1.0, min(3.0, dev_ms * 1e-3)))
        peak = peak_sust
        # CPU baseline: the oracle port on this box's host cores, bounded sample
        om = oracle_model(t, data.sim_data.y_std, K, pc_prec, resid_ss=0.0)
        modes, cores = host_cpu_modes(args.ref_nx, args.ref_nt, 1, args.cpu_steps, om=om)
        best_mode = max(modes, key=lambda k: modes[k]['value'])
        cpu_val, cpu_dt = modes[best_mode]['value'], modes[best_mode]['seconds']
        pk = fp64_peak_tflops(torch) if pred.get('roofline') else None
        if pk:
            pred['roofline']['peak'] = pk
            pred['roofline']['frac'] = pred['roofline']['achieved'] / pk
            pred['roofline']['peak_source'] = 'cuBLAS FP64 GEMM 8192^3 measured in this run'
            pred['roofline']['traffic_note'] = 'no ncu capture of this kernel in this round (profiles/r1_predict_kernel_summary.txt: DMMA pipe 65.6 %)' 
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': dev_ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f64', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'chains_per_gpu': chains, 'chains_total': total_chains,
                       'evals_per_step_per_chain': EVALS_PER_STEP, 'field_n_y': int(y.shape[1]),
                       'l2': 'working set (factor workspaces %d MB/GPU) exceeds L2; no flush needed'
                             % (chains * PU * ops._lib.load().ggp_factor_doubles(M) * 8 >> 20),
                       'rsvd_setup_s': svd_s, 'setup_s': setup_s},
            'single_chain_equiv_steps_per_s': value / total_chains,
            'e2e': {'value': e2e_val, 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': int(d2h),
                    'api': 'SepiaModel.do_mcmc_chains (host np.random stream -> device, draws -> host)',
                    'note': 'a separate pass of the same K steps (own np.random stream, chains continue from where the device pass '
                            'left them): the two passes evaluate slightly different numbers of sites (proposals outside the bounds '
                            'are rejected without an evaluation), hence a few per cent either way'},
            'gpu_launches': args.steps,            # one ggp::sweep_kernel (step kernel) launch per mcmc_step in the timed region
            'roofline': {'bound': 'tensor', 'kernel': 'ggp::sweep_kernel (step kernel: fused cov build + DMMA Cholesky + solve per site, lamWOs terms, close)',
                         'achieved': achieved, 'peak': peak, 'unit': 'TFLOP/s', 'frac': achieved / peak,
                         'peak_source': 'cuBLAS FP64 GEMM 8192^3 measured in this run, back to back for as long as the timed region (sustained, '
                                        'under the power cap like the step kernels); MEASURED_PEAKS.json has no FP64 figure',
                         'peak_burst': peak_burst, 'frac_of_burst_peak': achieved / peak_burst,
                         'traffic': SWEEP_DRAM_BYTES_PER_EVAL * sweep_evals / args.steps,
                         'traffic_source': 'dram__bytes_read+write of one ncu --set full capture of ggp::sweep_kernel '
                                           '(profiles/r2a_sweep_kernel_summary.txt: 196.85 GB / 25.86 k evaluations), scaled to '
                                           'the evaluations of one launch of this run; algorithmic bytes: 37 KB of design read, one scalar back',
                         'evals_in_timed_launches': sweep_evals, 'kernel_ms_total': sweep_ms,
                         'kernel_share_of_step': sweep_ms / dev_ms, 'lamWOs_wave_ms_total': wos_ms, 'flop_per_eval': flop_eval},
            'cpu_baseline': {'value': cpu_val, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                             'sample': '%d mcmc_steps per chain (oracle/sepia_oracle.py, NumPy/SciPy FP64; SEPIA parity unpinned): best of '
                                       'one chain x all BLAS threads and one single-thread chain per core (%s, %.1f s)'
                                       % (args.cpu_steps, best_mode, cpu_dt),
                             'modes': modes},
            'clocks': clocks,
            'prediction': pred,
        }
        line.update({k: v for k, v in extra.items() if v is not None})
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--chains', type=int, default=944,
                    help='independent chains per GPU: 59 chains x 10 PCs = 590 CTAs fill the 148 SMs x 4 resident CTAs once; '
                         'several such waves let finished CTAs be replaced while the slowest of a wave still run '
                         '(round 1: 59: 3265, 118: 3400, 236: 3540, 944: 3630 chain-steps/s; round 2: 236: 3649, 944: 3729)')
    ap.add_argument('--nx', type=int, default=4000, help='field nodes (cfg3: 4k)')
    ap.add_argument('--nt', type=int, default=365, help='field time steps (cfg3: 365)')
    ap.add_argument('--ref-nx', type=int, default=400)
    ap.add_argument('--ref-nt', type=int, default=36)
    ap.add_argument('--cpu-steps', type=int, default=4)
    ap.add_argument('--pred-samples', type=int, default=64)
    ap.add_argument('--pred-designs', type=int, default=8192)
    ap.add_argument('--cfg5-steps', type=int, default=2)
    ap.add_argument('--cfg4-full', action='store_true', help='run cfg4 at full size (1000 x 100 000) also with fewer than 8 GPUs')
    ap.add_argument('--no-extras', action='store_true', help='skip the rsvd / cfg5 / cfg4 / single-chain blocks')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write the last step of the timed run as DIR/draws.npy (chains, P) and '
                         'DIR/lp.npy (chains,), float64 (rank 0\'s chains; a seeded sample of chains above 64 MB in all)')
    if len(sys.argv) > 1 and sys.argv[1] == '--ref-worker':
        return _ref_worker_main(sys.argv[2:])
    args = ap.parse_args()
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
