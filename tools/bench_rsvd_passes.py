"""Developer timing of the two rSVD passes at cfg3 size (512 x 1.46 M float32, r = 25), with a SHA-1 of every output.

sketch_tma: X and Omega^T 16-byte aligned (row pitch 4 n a multiple of 16 B) -> sketch_tma_kernel.
sketch_reg: the same values with X at a 4-byte misaligned base -> sketch_tc_kernel (scalar loads), the path of any ensemble
whose row pitch is not a multiple of 16 B.
xty: Y^T X -> xty_ts_kernel.  torch_sum_read_only: one read of X by torch.sum, the floor a streaming pass can reach.
GGP_LIB=<path> times another build of the library (e.g. one from an earlier commit) on the same seeded inputs."""
import hashlib, json, os, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gladsgp_b200 import _lib
if os.environ.get('GGP_LIB'):                      # developer A/B runs against a variant library
    _lib.LIB_PATH = os.environ['GGP_LIB']
from gladsgp_b200 import ops
m, n, r = 512, 1460000, 25
HBM_GBS = 6533.8                                   # measured HBM read peak of one B200 (DESIGN.md)
g = torch.Generator(device='cuda'); g.manual_seed(0)
X = torch.randn((m, n), dtype=torch.float32, device='cuda', generator=g)
omT = torch.randn((r, n), dtype=torch.float32, device='cuda', generator=g)
Y = torch.randn((m, r), dtype=torch.float32, device='cuda', generator=g)
buf = torch.empty(m * n + 1, dtype=torch.float32, device='cuda')
buf[1:] = X.view(-1)
X_mis = buf[1:].view(m, n)                         # base 4 bytes past a 16-byte boundary
ws = torch.empty(_lib.load().ggp_rsvd_tc_workspace_bytes(m), dtype=torch.uint8, device='cuda')


def ev(fn, reps=7):
    fn(); torch.cuda.synchronize(); best = 1e9
    for _ in range(reps):
        a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize(); best = min(best, a.elapsed_time(b))
    return best


def sha1(t):
    return hashlib.sha1(t.contiguous().cpu().numpy().tobytes()).hexdigest()


res = {'lib': _lib.LIB_PATH, 'device': torch.cuda.get_device_name()}
passes = {'sketch_tma': lambda: ops.rsvd_sketch_tc(X, omT, ws),
          'sketch_reg': lambda: ops.rsvd_sketch_tc(X_mis, omT, ws),
          'xty': lambda: ops.rsvd_xty_tc(X, Y)}
for name, fn in passes.items():
    ms = ev(fn)
    res[name] = dict(ms=ms, gbs=4.0 * m * n / ms / 1e6, frac=4.0 * m * n / ms / 1e6 / HBM_GBS, sha1=sha1(fn()))
x1 = X.view(-1)
ms = ev(lambda: x1.sum())
res['torch_sum_read_only'] = dict(ms=ms, gbs=4.0 * m * n / ms / 1e6)
print(json.dumps(res))
