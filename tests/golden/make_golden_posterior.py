"""Golden posterior draws: burned-in chains of the oracle sampler (oracle/sepia_oracle.py) at default SEPIA priors.

    python tests/golden/make_golden_posterior.py [cfg1 cfg2 cfg3] [--out DIR]

For each configuration the oracle runs `n_steps` steps from the prior defaults (betaU 0.1, lamUz 1, lamWs 1000) with
the default step sizes, then `n_replay` further steps with its per-site trace recorded.  Stored:

  problem       builder arguments (tests/helpers.py make_problem / make_scalar_problem) and chain seed
  w, LamSim     the model data the sampler reads (zt is rebuilt from the design, which involves no BLAS)
  tb_*          the sampler tables, as in chain_cfg*.npz (tb_theta is the prior-default start of the run)
  draws         S = 64 draws thinned evenly from the second half of the run, float64, in sampling order
                [betaU (d x pu, column-major), lamUz (pu), lamWs (pu), lamWOs (1)]; draw_steps, draw_lp beside them
  state, lp     the final state of the run and its log-posterior
  rp_*, chain_* the replay record of the n_replay steps from `state`, in the layout of chain_cfg*.npz

These are the draws a real chain returns: betaU spanning four decades within one PC, lamWOs at the lower prior
bound, lamWs well below the prior default -- the inputs every posterior consumer meets in use.

  cfg1  m=100, q=8 (d=9), pu=5, n_y=200           600 steps + 60 replay steps   (~10 s)
  cfg2  1-D GP regression, m=1000, d=2, pu=1      400 steps + 50 replay steps   (~1 min)
  cfg3  m=512, q=8 (d=9), pu=10, n_y=200          300 steps + 20 replay steps   (~15 min)

BLAS runs on one thread so that a rerun reproduces the files bit for bit (tests/test_posterior_fixture_cpu.py).
"""
import os
import sys
import time

os.environ['OPENBLAS_NUM_THREADS'] = '1'
os.environ['OMP_NUM_THREADS'] = '1'
os.environ['MKL_NUM_THREADS'] = '1'

import numpy as np  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from helpers import so, tables_from_oracle, replay_from_trace, make_problem, make_scalar_problem  # noqa: E402

S = 64
CONFIGS = {
    'cfg1': dict(kind='pca', args=dict(m=100, q=8, pu=5, n_x=20, n_t=10, seed=5), seed=3, n_steps=600, n_replay=60),
    'cfg2': dict(kind='scalar', args=dict(m=1000, seed=20240320), seed=4, n_steps=400, n_replay=50),
    'cfg3': dict(kind='pca', args=dict(m=512, q=8, pu=10, n_x=20, n_t=10, seed=7), seed=5, n_steps=300, n_replay=20),
}


def build(cfg):
    c = CONFIGS[cfg]
    return make_problem(**c['args']) if c['kind'] == 'pca' else make_scalar_problem(**c['args'])


def _draws(mod, lo, hi):
    s = mod.get_samples()
    d = np.concatenate([s['betaU'], s['lamUz'], s['lamWs'], s['lamWOs']], axis=1)
    return d[lo:hi], s['logPost'][lo:hi, 0]


def run(cfg):
    c = CONFIGS[cfg]
    num = build(cfg)['num']
    mod = so.OracleModel(num)
    tb = tables_from_oracle(mod)
    P = tb['theta'].size
    rng = np.random.RandomState(c['seed'])
    n, nr = c['n_steps'], c['n_replay']
    t0 = time.time()
    mod.do_mcmc(n, rng=rng)
    chain, chain_lp = _draws(mod, 0, n)
    steps = n // 2 + np.round(np.linspace(0, n - n // 2 - 1, S)).astype(np.int64)
    mod.trace = []
    mod.do_mcmc(nr, rng=rng)                          # the same stream, continued from the final state
    dt = time.time() - t0
    replay, acc = replay_from_trace(mod.trace, nr, P)
    rd, rlp = _draws(mod, n, n + nr)
    out = dict(kind=np.array(c['kind']), seed=np.array(c['seed']), n_steps=np.array(nr), n_burn=np.array(n),
               w=num.w, LamSim=np.asarray(num.LamSim, dtype=np.float64),
               draws=chain[steps], draw_steps=steps, draw_lp=chain_lp[steps], state=chain[-1], lp=chain_lp[-1],
               chain_acc=acc, chain_draws=rd, chain_lp=rlp)
    out.update({'arg_' + k: np.array(v) for k, v in c['args'].items()})
    out.update({'tb_' + k: v for k, v in tb.items()})
    out.update({'rp_' + k: v for k, v in replay.items()})
    return out, dt


def main():
    argv = sys.argv[1:]
    out_dir = HERE
    if '--out' in argv:
        i = argv.index('--out')
        out_dir = argv[i + 1]
        argv = argv[:i] + argv[i + 2:]
    for cfg in argv or list(CONFIGS):
        if cfg not in CONFIGS:
            raise SystemExit('unknown configuration ' + cfg)
        out, dt = run(cfg)
        path = os.path.join(out_dir, 'posterior_%s.npz' % cfg)
        np.savez_compressed(path, **out)
        d = out['draws']
        nb = int(out['tb_prior_kind'].size - 2 * out['LamSim'].size - 1)
        print(cfg, 'betaU %.3g .. %.3g' % (d[:, :nb].min(), d[:, :nb].max()),
              'lamWOs %.4g .. %.4g' % (d[:, -1].min(), d[:, -1].max()),
              'replay accept rate %.3f' % out['chain_acc'].mean(), '%.1f s' % dt, os.path.getsize(path), 'bytes')


if __name__ == '__main__':
    main()
