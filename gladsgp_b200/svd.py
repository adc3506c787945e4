"""B200 randomized SVD: drop-in for /root/reference/src/svd.py:12-82 (`randomized_svd`).

Same signature and return shapes; the three products over the (m, n) float32 ensemble
(src/svd.py:52,56,60) run as streaming passes on the tcgen05 tensor cores (3xTF32 split products with
FP32-level accuracy, csrc/ggp_rsvd_tc.cu), the m x r QR and the r x r eigen-problem run in FP64 in
torch/cuSOLVER on the device.  The Gaussian test matrix is drawn from the global np.random stream exactly as the reference does
(src/svd.py:51) unless `omega` is injected.
"""
import numpy as np

from . import ops, _lib


def randomized_svd(X, p, k=None, q=1, return_error=False, omega=None, return_device=False):
    torch = _lib.require_cuda()
    if k is None:
        k = p
    r = p + k
    if torch.is_tensor(X):
        Xd = X.to(device='cuda', dtype=torch.float32).contiguous()
    else:
        Xh = np.ascontiguousarray(X, dtype=np.float32)
        Xd = torch.as_tensor(Xh).pin_memory().to('cuda', non_blocking=True) if Xh.nbytes < (8 << 30) else torch.as_tensor(Xh).to('cuda')
    m, n = Xd.shape
    if omega is None:
        omega = np.random.normal(size=(n, r)).astype(np.float32)              # svd.py:51
    omT = torch.as_tensor(np.ascontiguousarray(np.asarray(omega, dtype=np.float32).T), device='cuda')
    ws = torch.empty(_lib.load().ggp_rsvd_tc_workspace_bytes(m), dtype=torch.uint8, device='cuda')
    Y = ops.rsvd_sketch_tc(Xd, omT, ws)                                       # svd.py:52  Y = X @ omega
    for _ in range(q):                                                        # svd.py:55-56  Y = X @ X.T @ Y
        Zt = ops.rsvd_xty_tc(Xd, Y)                                           #   (X^T Y)^T, (r, n)
        Y = ops.rsvd_sketch_tc(Xd, Zt, ws)                                    #   X (X^T Y)
    # svd.py:59 -- the m x r orthonormalisation runs in FP64 (it costs nothing at this size, and a float32 QR leaves Q
    # orthonormal to ~1e-6 only, which is what then limits the singular values); Q is rounded to float32 for the product pass
    Qd, _ = torch.linalg.qr(Y.double(), mode='reduced')
    Q = Qd.float()
    B = ops.rsvd_xty_tc(Xd, Q.contiguous())                                   # svd.py:60  B = Q.T @ X, (r, n)
    # small SVD of B via the r x r Gram matrix in FP64 (svd.py:63)
    Bd = B.double()
    lam, E = torch.linalg.eigh(Bd @ Bd.T)
    lam = torch.flip(lam, dims=[0]).clamp_min(0.0)
    E = torch.flip(E, dims=[1])
    S = torch.sqrt(lam)
    U = (Qd @ E).float()                                                      # svd.py:64
    Vh = ((E.T @ Bd) / S.clamp_min(1e-300)[:, None]).float()
    U, S, Vh = U[:, :p], S[:p].float(), Vh[:p, :]                             # svd.py:66-68
    if not return_device:
        U, S, Vh = U.cpu().numpy(), S.cpu().numpy(), Vh.cpu().numpy()
    svd = (U, S, Vh)
    if return_error:
        # the reference reads S[p] after truncating S to p entries (svd.py:67,73-76): always 0
        return svd, 0.0
    return svd
