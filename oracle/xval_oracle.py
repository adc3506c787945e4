"""CPU oracle for SepiaXvalEmulatorPrediction.  TEST INFRASTRUCTURE ONLY.

Restates SEPIA's literal cross-validation route on top of the wPred restatement in oracle/sepia_oracle.py: per fold, a
sub-problem with the fold's zt / w rows removed (same K basis, LamSim and posterior samples -- SEPIA does not refit the
hyper-parameters), then w_pred at the held-out rows.  Like the rest of the SEPIA restatement this is from the published
algorithm, not from the package source: parity unpinned.  The conventions it freezes are listed in DESIGN.md section 2.
"""
from __future__ import annotations

import copy

import numpy as np

from oracle.sepia_oracle import OracleNum, w_pred


def xval_pred(num: OracleNum, samples, leave_out_inds=None, rng=np.random, draw=True):
    """leave_out_inds: list of folds (arrays of training rows); default leave-one-out [[0], ..., [m-1]].
    Returns (w_draws (nsamp, sum |F|, pu) fold-major or None, mu list, Sigma list): one (nsamp, pu |F|) /
    (nsamp, pu |F|, pu |F|) entry per fold, PC-major.  The draws consume rng.normal fold by fold, then sample by sample
    (pu |F| values each)."""
    m = num.m
    folds = [[i] for i in range(m)] if leave_out_inds is None else leave_out_inds
    ws, mus, Sigs = [], [], []
    for f in folds:
        f = np.asarray(f, dtype=np.int64).reshape(-1)
        keep = np.setdiff1d(np.arange(m), f)
        sub = copy.copy(num)
        sub.m = keep.size
        sub.zt = num.zt[keep]
        sub.iu = np.triu_indices(sub.m, 1)
        sub.sqdist = np.square(sub.zt[sub.iu[0]] - sub.zt[sub.iu[1]])
        sub.w = num.w[keep]
        sub.wv = sub.w.reshape((-1, 1), order='F')
        w, mu, Sig = w_pred(sub, num.zt[f, 1:], samples, rng=rng, draw=draw)
        ws.append(w)
        mus.append(mu)
        Sigs.append(Sig)
    return (np.concatenate(ws, axis=1) if draw else None), mus, Sigs
