"""MCMC convergence diagnostics on the device: rank-normalized split R-hat, bulk ESS and tail ESS (DESIGN.md section 2).

The reference checks convergence by eye, repeating a chain and comparing QQ plots and histograms
(mcmc_diagnostics_advanced.py:50-54,86-110).  With many chains per run the quantitative multi-chain check of Vehtari et al.
(2021) is available instead; csrc/ggp_chain_diag.cu computes it where the draws live, without downloading them.
"""
import numpy as np

from . import _lib, ops


def _device(a):
    torch = _lib.require_cuda()
    if torch.is_tensor(a):
        return a.to(device='cuda', dtype=torch.float64)
    return torch.as_tensor(np.ascontiguousarray(np.asarray(a, dtype=np.float64)), device='cuda')


def chain_diagnostics(draws, lp=None, nburn=0):
    """draws (n, C, P) as a NumPy array or a CUDA tensor; lp (n, C) or None, appended as the last element.  The first nburn
    draws of every chain are left out.  Returns dict(rhat, ess_bulk, ess_tail) of NumPy (P,) arrays, (P + 1,) with lp."""
    nburn = int(nburn)
    x = _device(draws)
    if x.dim() != 3:
        raise ValueError('draws must be (n_draws, n_chains, n_params)')
    parts = [ops.chain_diagnostics(x[nburn:])]
    if lp is not None:
        l = _device(lp)
        if l.dim() != 2 or tuple(l.shape) != tuple(x.shape[:2]):
            raise ValueError('lp must be (n_draws, n_chains), matching draws')
        parts.append(ops.chain_diagnostics(l[nburn:, :, None]))
    keys = ('rhat', 'ess_bulk', 'ess_tail')
    return {k: np.concatenate([p[i].cpu().numpy() for p in parts]) for i, k in enumerate(keys)}


def by_block(blocks, res):
    """Flat per-element results in the sampler's element order (res: dict of (P + 1,) arrays, logPost last) ->
    {name: dict(rhat, ess_bulk, ess_tail)} with every block's arrays in its val_shape (Fortran order) and logPost scalars."""
    out = {}
    o = 0
    for b in blocks:
        n = int(np.prod(b.val_shape))
        out[b.name] = {k: v[o:o + n].reshape(b.val_shape, order='F').copy() for k, v in res.items()}
        o += n
    out['logPost'] = {k: np.float64(v[o]) for k, v in res.items()}
    return out
