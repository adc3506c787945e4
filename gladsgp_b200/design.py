"""Sequential design: the next simulator runs that most reduce the emulator's integrated predictive variance, chosen by
greedy ALC ("active learning Cohn"; DESIGN.md section 2 item 10).

A GP's predictive variance does not depend on the simulator's output, so the whole batch of n_new runs is chosen before
any of them is made, from the prediction factors cached with the model (model._pred_cache, shared with
SepiaEmulatorPrediction, cross-validation, sensitivity and calibration).  For every (sample, PC) block the rows
V = S21^T L^-T of the reference and candidate designs come from ggp_predict_f64; each pick appends one column A (a
rank-one update of the enlarged Cholesky factor), and nothing is factored again.  The score of candidate c is the drop of
the integrated variance that adding c as a training run would give,
    score_t(c) = (1/S) sum_s sum_j w_j (1/n_ref) sum_r Sigma_t(r, c)^2 / den_t(c),
with w_j the native-unit field variance carried by PC j; the greedy step takes the unselected candidate with the largest
score (ties: the lowest index).  The scores are dense FP64 products on the tensor cores (csrc/ggp_design.cu).
"""
import numpy as np

from . import _lib, ops
from .calibration import _check_t_model, _designs, _predictor, _to_trans

DESIGN_V_BYTES = 1 << 34      # V of the reference and candidate designs: at most 16 GiB, more blocks in several chunks
MAX_NEW = 128                 # runs per call: the pitch of the appended columns A


def _points(t, name, q):
    t = np.asarray(t, dtype=np.float64)
    if t.ndim != 2 or t.shape[1] != q or t.shape[0] < 1:
        raise ValueError('%s must be (n, %d) with n >= 1' % (name, q))
    if not np.all(np.isfinite(t)):
        raise ValueError('%s holds a non-finite value' % name)
    return t


def field_weights(model):
    """w_j = sum_k (K_jk orig_y_sd_k)^2 (pu,): the native-unit field variance per unit of PC j's weight (K = [[1]] for a
    scalar-output model)."""
    sd = model.data.sim_data
    ysd = np.asarray(sd.orig_y_sd, dtype=np.float64).reshape(-1)
    if model.data.scalar_out:
        return np.array([float(ysd[0]) ** 2])
    K = np.asarray(sd.K, dtype=np.float64)
    ysd = np.broadcast_to(ysd, (K.shape[1],))
    return np.einsum('jk,k->j', K * K, ysd * ysd)


def next_runs(model, samples, candidates, n_new, reference=None, pc_weights=None):
    """Choose n_new simulator runs among `candidates` (n_cand, q) by greedy ALC over the posterior samples: each step takes
    the candidate whose addition as a training run most reduces the predictive variance integrated over `reference`
    (n_ref, q; default: the candidates), then conditions on it.  Both are native `t` values.  pc_weights (pu,): the
    weight of each PC's variance (default: field_weights(model), the native-unit field variance it carries).

    Returns dict(index (n_new,) int64 in selection order, t (n_new, q) native, score (n_new,): the chosen candidate's score
    at its step, imse (n_new + 1,): the weighted integrated variance before each step and after the last, pc_weights)."""
    _check_t_model(model, 'sequential design', 'design over')
    q, pu = model.num.q, model.num.pu
    C = _points(candidates, 'candidates', q)
    R = None if reference is None else _points(reference, 'reference', q)
    n_cand = C.shape[0]
    if isinstance(n_new, bool) or int(n_new) != n_new or not 1 <= int(n_new) <= min(n_cand, MAX_NEW):
        raise ValueError('n_new must be an integer in [1, min(n_cand, %d)] = [1, %d]' % (MAX_NEW, min(n_cand, MAX_NEW)))
    n_new = int(n_new)
    if pc_weights is None:
        w = field_weights(model)
    else:
        w = np.asarray(pc_weights, dtype=np.float64)
        if w.shape != (pu,):
            raise ValueError('pc_weights must be (%d,)' % pu)
        if not np.all(np.isfinite(w)) or np.any(w < 0):
            raise ValueError('pc_weights must be finite and >= 0')
    torch = _lib.require_cuda()
    pred, S = _predictor(model, samples)
    B, Mp = pred.B, pred.Mp
    XC = _designs(torch.as_tensor(_to_trans(model, C), device='cuda'))
    XR = XC if R is None else _designs(torch.as_tensor(_to_trans(model, R), device='cuda'))
    n_ref = XR.shape[0]
    wgt = torch.as_tensor(np.tile(w / (S * n_ref), S), device='cuda')          # block b = s * pu + j
    Kp = (n_new + 7) & ~7
    A_C = torch.zeros((B, n_cand, Kp), dtype=torch.float64, device='cuda')
    A_R = A_C if R is None else torch.zeros((B, n_ref, Kp), dtype=torch.float64, device='cuda')
    per = ((0 if R is None else n_ref) + n_cand) * Mp * 8
    chunk = max(1, min(B, DESIGN_V_BYTES // per))
    chunks = [(b0, min(chunk, B - b0)) for b0 in range(0, B, chunk)]
    cached = {}

    def rows(b0, nb):
        """V_R, V_C of blocks [b0, b0+nb): computed once with one chunk, again at every step with several."""
        if b0 in cached:
            return cached[b0]
        V_C = pred.predict(XC, want_V=True, b0=b0, nb=nb)[2]
        V_R = V_C if R is None else pred.predict(XR, want_V=True, b0=b0, nb=nb)[2]
        if len(chunks) == 1:
            cached[b0] = (V_R, V_C)
        return V_R, V_C

    score = torch.empty(n_cand, dtype=torch.float64, device='cuda')
    imse = torch.empty(n_new + 1, dtype=torch.float64, device='cuda')
    taken = torch.zeros(n_cand, dtype=torch.bool, device='cuda')
    index = np.empty(n_new, dtype=np.int64)
    best = torch.empty(n_new, dtype=torch.float64, device='cuda')
    ws = None
    for t in range(n_new + 1):
        for b0, nb in chunks:
            V_R, V_C = rows(b0, nb)
            sl = slice(b0, b0 + nb)
            if t > 0:
                ops.design_condition(pred, b0, XR, XC, V_R, V_C, A_R[sl], A_C[sl], t - 1, index[t - 1])
            ws = ops.design_score(pred, b0, XR, XC, V_R, V_C, A_R[sl], A_C[sl], t, wgt[sl],
                                  score if t < n_new else None, imse[t:t + 1], b0 > 0, ws)
        del V_R, V_C
        if t < n_new:
            sc = torch.where(taken, torch.full_like(score, -np.inf), score)
            c = int(torch.argmax(sc))                       # the first maximum: ties go to the lowest index
            index[t] = c
            best[t] = score[c]
            taken[c] = True
    return dict(index=index, t=C[index], score=best.cpu().numpy(), imse=imse.cpu().numpy(), pc_weights=w)
