"""Developer timing of the materialised covariance build (592 matrices of 512 x 512, d = 9): tile kernel vs row-block kernel.

m = 512 is a multiple of the 64-row block, so a 16-byte aligned output takes the row-block kernel; the same call on an output
offset by 8 bytes takes the tile kernel.  Both results are compared bit for bit."""
import json, os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gladsgp_b200 import ops, synthetic, _lib
m, q = 512, 8
B = int(sys.argv[1]) if len(sys.argv) > 1 else 592
d = q + 1
t = synthetic.design(m, q)
X = np.concatenate([0.5 * np.ones((m, 1)), t.astype(np.float64)], axis=1)
rng = np.random.default_rng(0)
beta = np.exp(rng.uniform(np.log(0.05), np.log(3.0), size=(B, d)))
lamz = rng.uniform(0.5, 2.0, B); dadd = rng.uniform(1e-3, 1e-2, B)
Xd, bd, ld, dd = [torch.as_tensor(a, device='cuda') for a in (X, beta, lamz, dadd)]
lib = _lib.load()
def cov_build_into(out):
    _lib.check(lib.ggp_cov_build_f64(_lib.ptr(Xd), m, d, _lib.ptr(bd), _lib.ptr(ld), _lib.ptr(dd), B, _lib.ptr(out),
                                     _lib.stream_ptr()), 'ggp_cov_build_f64')
def ev(fn, reps=7):
    fn(); torch.cuda.synchronize(); best = 1e9
    for _ in range(reps):
        a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize(); best = min(best, a.elapsed_time(b))
    return best
res = {}
outs = {}
buf = torch.empty(B * m * m + 2, dtype=torch.float64, device='cuda')
for mode, off in (('0', 1), ('1', 0)):          # covrows0: tile kernel (8-byte offset output), covrows1: row-block kernel
    out = buf[off:off + B * m * m]
    assert (out.data_ptr() % 16 == 0) == (mode == '1')
    ms = ev(lambda: cov_build_into(out))
    outs[mode] = out.view(B, m, m).clone()
    res['covrows' + mode] = dict(ms=ms, gbs=B * m * m * 8 / ms / 1e6, frac=B * m * m * 8 / ms / 1e6 / 6533.8)
res['identical'] = bool(torch.equal(outs['0'], outs['1']))
res['symmetric'] = bool(torch.equal(outs['1'], outs['1'].transpose(1, 2)))
n = 4096
tp = synthetic.test_design(n, q)
Xp = torch.as_tensor(np.concatenate([0.5 * np.ones((n, 1)), tp.astype(np.float64)], axis=1), device='cuda')
Bc = 64
ms = ev(lambda: ops.cross_cov(Xd, Xp, bd[:Bc], ld[:Bc]))
res['cross_cov'] = dict(ms=ms, gbs=Bc * m * n * 8 / ms / 1e6, frac=Bc * m * n * 8 / ms / 1e6 / 6533.8)
print(json.dumps(res))
