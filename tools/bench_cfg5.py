"""cfg5 (BASELINE.json configs[4]): m = 4096 sims, 16 parameters (d = 17), 20 PCs, 8 chains -- MCMC steps/s on this GPU.
Usage: python tools/bench_cfg5.py [n_chains] [steps]   (8 chains on one GPU, or 1 chain per GPU on an 8-GPU box)."""
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gladsgp_b200 import synthetic, _lib  # noqa: E402
if os.environ.get('GGP_LIB'):                      # developer A/B runs against a variant library
    _lib.LIB_PATH = os.environ['GGP_LIB']
from sepia.SepiaData import SepiaData  # noqa: E402
from sepia.SepiaModel import SepiaModel  # noqa: E402


def main():
    chains = int(sys.argv[1]) if len(sys.argv) > 1 else 8
    steps = int(sys.argv[2]) if len(sys.argv) > 2 else 2
    m, q, pu = 4096, 16, 20
    t = synthetic.design(m, q, seed=20240318)
    rng = np.random.default_rng(5)
    # small synthetic field (the field size is free in cfg5): n_y = 4000 outputs, 24 smooth modes + noise
    n_y = 4000
    modes = rng.standard_normal((24, n_y))
    coef = np.stack([np.sin((k + 1) * t @ rng.uniform(0.2, 1.5, size=q)) for k in range(24)], axis=1) / (1 + np.arange(24))
    y = (coef @ modes + 0.02 * rng.standard_normal((m, n_y))).astype(np.float32)
    d = SepiaData(t_sim=t, y_sim=y, y_ind_sim=np.linspace(0, 1, n_y))
    d.transform_xt(t_notrans=np.arange(q)); d.standardize_y()
    d.create_K_basis(n_pc=pu)
    model = SepiaModel(d)
    np.random.seed(0)
    t0 = time.perf_counter(); model.do_mcmc_chains(1, chains); torch.cuda.synchronize(); warm = time.perf_counter() - t0
    t0 = time.perf_counter(); draws, lp = model.do_mcmc_chains(steps, chains); torch.cuda.synchronize(); dt = time.perf_counter() - t0
    evals = pu * (m * 0 + 17 + 4)
    flop_eval = m ** 3 / 3.0 + m * m + 2 * m + (3 * 17 + 2) * m * (m - 1) / 2.0
    res = dict(m=m, d=17, pu=pu, chains=chains, steps=steps, s_per_step=dt / steps, chain_steps_per_s=chains * steps / dt,
               evals_per_step_per_chain=evals, tflops_fp64=chains * steps * evals * flop_eval / dt / 1e12,
               first_step_s=warm, lp_finite=bool(np.all(np.isfinite(lp))))
    print(json.dumps(res))


if __name__ == '__main__':
    main()
