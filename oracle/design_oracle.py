"""CPU oracle of greedy ALC sequential design (gladsgp_b200.design; DESIGN.md section 2 item 10).  TEST INFRASTRUCTURE
ONLY: NumPy / SciPy FP64.

Blocks b = (s, j) of SepiaEmulatorPrediction._blocks() with addResidVar=False: k_b(x, x') = exp(-sum_k beta_k (x_k -
x'_k)^2) / lamUz (nugget-free, for every pair of distinct index entries), s11 = 1/lamUz + 1/lamWs, the S22 nugget
dadd = 1/lamWs + 1/(LamSim_j lamWOs).  Designs are rows [0.5 (dummy x), t_trans].

* greedy_rank_one: the rank-one form the device computes (V = L^-1 k(X, x), one appended column A per pick), with the
  top-two score margin at every step;
* greedy_direct: S22 re-factored with the chosen points appended as training rows (nugget dadd), v_t and every score by
  brute-force augmentation with the candidate.
Both return dict(index, score, imse, scores (k, n_cand), margin (k,)).
"""
from __future__ import annotations

import numpy as np
import scipy.linalg

from oracle import sepia_oracle as so


def designs(t_trans):
    t_trans = np.asarray(t_trans, dtype=np.float64)
    return np.concatenate([np.full((t_trans.shape[0], 1), 0.5), t_trans], axis=1)


def blocks(zt, LamSim, samples):
    """[(beta (d,), lamUz, s11, dadd)] in block order b = s * pu + j."""
    zt = np.asarray(zt, dtype=np.float64)
    d = zt.shape[1]
    LamSim = np.asarray(LamSim, dtype=np.float64).reshape(-1)
    pu = LamSim.size
    lamUz = np.asarray(samples['lamUz'], dtype=np.float64).reshape(-1, pu)
    lamWs = np.asarray(samples['lamWs'], dtype=np.float64).reshape(-1, pu)
    lamWOs = np.asarray(samples['lamWOs'], dtype=np.float64).reshape(-1)
    S = lamUz.shape[0]
    bU = np.asarray(samples['betaU'], dtype=np.float64).reshape(S, pu, d)
    out = []
    for s in range(S):
        for j in range(pu):
            out.append((bU[s, j], lamUz[s, j], 1.0 / lamUz[s, j] + 1.0 / lamWs[s, j],
                        1.0 / lamWs[s, j] + 1.0 / (LamSim[j] * lamWOs[s])))
    return out, S, pu


def _kern(A, B, beta, lamz):
    return so.cov_cross(A, B, beta, lamz)


def _select(score, taken):
    sc = np.where(taken, -np.inf, score)
    c = int(np.argmax(sc))                                   # first maximum: ties to the lowest index
    rest = np.delete(sc, c)
    margin = sc[c] - (rest.max() if rest.size else -np.inf)
    return c, margin


def greedy_rank_one(zt, LamSim, samples, XR, XC, k, weights):
    """XR (n_ref, d), XC (n_cand, d) designs; weights (pu,).  Scores and integrated variances of the rank-one form."""
    bl, S, pu = blocks(zt, LamSim, samples)
    n_ref, n_cand = XR.shape[0], XC.shape[0]
    st = []
    for b, (beta, lamz, s11, dadd) in enumerate(bl):
        L = np.linalg.cholesky(so.cov_cross(zt, zt, beta, lamz) + dadd * np.eye(zt.shape[0]))
        VR = scipy.linalg.solve_triangular(L, _kern(zt, XR, beta, lamz), lower=True).T      # (n_ref, m)
        VC = scipy.linalg.solve_triangular(L, _kern(zt, XC, beta, lamz), lower=True).T
        st.append(dict(w=weights[b % pu] / (S * n_ref), Sig=_kern(XR, XC, beta, lamz) - VR @ VC.T,
                       SigCC=_kern(XC, XC, beta, lamz) - VC @ VC.T,
                       vR=s11 - np.sum(VR * VR, axis=1), den=1.0 / lamz + dadd - np.sum(VC * VC, axis=1)))
    taken = np.zeros(n_cand, dtype=bool)
    out = dict(index=[], score=[], imse=[], scores=[], margin=[])
    for t in range(k + 1):
        score = np.zeros(n_cand)
        imse = 0.0
        for x in st:
            score = score + x['w'] * np.sum(x['Sig'] ** 2, axis=0) / x['den']
            imse = imse + x['w'] * np.sum(np.maximum(x['vR'], 0.0))
        out['imse'].append(imse)
        if t == k:
            break
        c, margin = _select(score, taken)
        taken[c] = True
        out['index'].append(c); out['score'].append(score[c]); out['scores'].append(score); out['margin'].append(margin)
        for x in st:                                         # append column t: a(x) = Sigma_t(x, c) / sqrt(den_t(c))
            sd = np.sqrt(x['den'][c])
            aR = x['Sig'][:, c] / sd
            aC = x['SigCC'][:, c] / sd
            x['Sig'] = x['Sig'] - np.outer(aR, aC)
            x['SigCC'] = x['SigCC'] - np.outer(aC, aC)
            x['vR'] = x['vR'] - aR * aR
            x['den'] = x['den'] - aC * aC
    return {key: np.asarray(v) for key, v in out.items()}


def greedy_direct(zt, LamSim, samples, XR, XC, k, weights):
    """The same greedy design with every quantity from a fresh factorisation of the enlarged S22."""
    bl, S, pu = blocks(zt, LamSim, samples)
    n_ref, n_cand = XR.shape[0], XC.shape[0]

    def variance(beta, lamz, s11, dadd, train):
        """v(r) at the reference points with the training rows `train` (S22 = k + dadd I)."""
        K = _kern(train, train, beta, lamz) + dadd * np.eye(train.shape[0])
        cf = scipy.linalg.cho_factor(K, lower=True)
        kr = _kern(train, XR, beta, lamz)
        return s11 - np.sum(kr * scipy.linalg.cho_solve(cf, kr), axis=0)

    chosen = []
    taken = np.zeros(n_cand, dtype=bool)
    out = dict(index=[], score=[], imse=[], scores=[], margin=[])
    for t in range(k + 1):
        train = np.concatenate([zt, XC[chosen]], axis=0)
        score = np.zeros(n_cand)
        imse = 0.0
        for b, (beta, lamz, s11, dadd) in enumerate(bl):
            w = weights[b % pu] / (S * n_ref)
            v = variance(beta, lamz, s11, dadd, train)
            imse = imse + w * np.sum(np.maximum(v, 0.0))
            if t < k:
                for c in range(n_cand):
                    if not taken[c]:
                        vc = variance(beta, lamz, s11, dadd, np.concatenate([train, XC[c:c + 1]], axis=0))
                        score[c] += w * np.sum(v - vc)
        out['imse'].append(imse)
        if t == k:
            break
        c, margin = _select(score, taken)
        taken[c] = True
        chosen.append(c)
        out['index'].append(c); out['score'].append(score[c]); out['scores'].append(score); out['margin'].append(margin)
    return {key: np.asarray(v) for key, v in out.items()}
